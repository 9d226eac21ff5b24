/* nnsp_model_text.c -- the reference's ON-DISK model format, read and written without a C compiler.
 *
 * A trained ns-nnsp model ships as generated C source, `evb/src/def_nn{id}_{name}.c`, written by
 * python/c_code_table_converter.py:143-347: the normalisation statistics, one hex array per weight / bias
 * table (ARM 4-row interleave, python/nnsp_pack/c_weight_man.py:5-124) and a `NeuralNetClass net_{name}`
 * struct literal (layer sizes, layer types, Q-formats, activations, function-pointer tables with an
 * `#ifdef DEF_ACC32BIT_OPT` alternative). "Loading a model" in the reference means compiling that file.
 * This translation unit parses the text directly (a small C-subset reader: comments, one level of
 * #ifdef/#else/#endif, array definitions, one brace initialiser) and emits the same text back from a model,
 * byte for byte in the layout the shipped files use, so tables round-trip. Host code only. */
#include <ctype.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "nnsp_compat/nnsp_legacy_api.h"
#include "nnsp_model.h"

void nnsp_model_layer_to_table(const nnsp_layer *L, int8_t *kernel, int8_t *kernel_rec, int16_t *bias);

/* ---------------------------------------------------------------------------------------------------- */
/* reader                                                                                                */
/* ---------------------------------------------------------------------------------------------------- */
typedef struct {
    char      name[96];
    int       elem_bits;        /* 8, 16 or 32 */
    long long *v;
    size_t    n;
} text_array;

typedef struct {
    text_array *arr;
    size_t      narr, cap;
    char       *net;            /* text of the NeuralNetClass initialiser, between its outer braces */
    char        net_name[96];
} text_unit;

static void unit_free(text_unit *u)
{
    for (size_t i = 0; i < u->narr; i++) free(u->arr[i].v);
    free(u->arr);
    free(u->net);
}

/* strip comments, resolve `#ifdef DEF_ACC32BIT_OPT` (defined iff acc32) and drop other directives */
static char *preprocess(const char *text, size_t len, int acc32)
{
    char *out = (char *)malloc(len + 2);
    if (!out) return NULL;
    size_t o = 0, i = 0;
    int skipping = 0, depth = 0, skip_depth = 0;
    int line_start = 1;
    while (i < len) {
        if (text[i] == '/' && i + 1 < len && text[i + 1] == '/') { while (i < len && text[i] != '\n') i++; continue; }
        if (text[i] == '/' && i + 1 < len && text[i + 1] == '*') {
            i += 2;
            while (i + 1 < len && !(text[i] == '*' && text[i + 1] == '/')) i++;
            i = (i + 2 <= len) ? i + 2 : len;
            continue;
        }
        if (line_start) {
            size_t j = i;
            while (j < len && (text[j] == ' ' || text[j] == '\t')) j++;
            if (j < len && text[j] == '#') {
                size_t e = j;
                while (e < len && text[e] != '\n') e++;
                char dir[64] = { 0 }, arg[64] = { 0 };
                sscanf(text + j, "#%63s %63s", dir, arg);      /* bounded by the NUL the caller guarantees */
                if (!strcmp(dir, "ifdef") || !strcmp(dir, "ifndef")) {
                    depth++;
                    if (!skipping) {
                        const int defined = !strcmp(arg, "DEF_ACC32BIT_OPT") && acc32;
                        if ((dir[2] == 'd') ? !defined : defined) { skipping = 1; skip_depth = depth; }
                    }
                } else if (!strcmp(dir, "else")) {
                    if (skipping && skip_depth == depth) skipping = 0;
                    else if (!skipping) { skipping = 1; skip_depth = depth; }
                } else if (!strcmp(dir, "endif")) {
                    if (skipping && skip_depth == depth) skipping = 0;
                    if (depth > 0) depth--;
                }
                i = e;
                continue;
            }
        }
        line_start = (text[i] == '\n');
        if (!skipping) out[o++] = text[i];
        i++;
    }
    out[o] = 0;
    return out;
}

static const char *skip_ws(const char *p) { while (*p && isspace((unsigned char)*p)) p++; return p; }
static int is_ident(int c) { return isalnum(c) || c == '_'; }

/* one `type name[...] = { numbers };` definition starting at p (after qualifiers were skipped by the caller) */
static int parse_numbers(const char *p, const char **end, long long **vals, size_t *n)
{
    size_t cap = 256, cnt = 0;
    long long *v = (long long *)malloc(cap * sizeof *v);
    if (!v) return NNSP_B200_ERR_NOMEM;
    for (;;) {
        p = skip_ws(p);
        if (*p == '}') { p++; break; }
        if (*p == ',') { p++; continue; }
        if (!*p) { free(v); return NNSP_B200_ERR_ARG; }
        char *e;
        const long long x = strtoll(p, &e, 0);
        if (e == p) { free(v); return NNSP_B200_ERR_ARG; }
        if (cnt == cap) {
            cap *= 2;
            long long *t = (long long *)realloc(v, cap * sizeof *v);
            if (!t) { free(v); return NNSP_B200_ERR_NOMEM; }
            v = t;
        }
        v[cnt++] = x;
        p = e;
    }
    *end = p; *vals = v; *n = cnt;
    return NNSP_B200_OK;
}

static int read_unit(const char *src, text_unit *u)
{
    const char *p = src;
    memset(u, 0, sizeof *u);
    for (;;) {
        p = skip_ws(p);
        if (!*p) break;
        /* collect the tokens of one declaration up to '=' , ';' or '[' */
        char words[6][96];
        int nw = 0;
        while (*p && *p != '=' && *p != ';' && *p != '[' && *p != '{') {
            if (is_ident((unsigned char)*p)) {
                int k = 0;
                while (is_ident((unsigned char)*p)) { if (k < 95) words[nw < 6 ? nw : 5][k++] = *p; p++; }
                words[nw < 6 ? nw : 5][k] = 0;
                if (nw < 6) nw++;
            } else p++;
        }
        if (!*p) break;
        if (nw == 0) { p++; continue; }
        const char *name = words[nw - 1];
        int is_net = 0, bits = 0;
        for (int i = 0; i < nw - 1; i++) {
            if (!strcmp(words[i], "NeuralNetClass")) is_net = 1;
            if (!strcmp(words[i], "uint8_t") || !strcmp(words[i], "int8_t")) bits = 8;
            if (!strcmp(words[i], "uint16_t") || !strcmp(words[i], "int16_t")) bits = 16;
            if (!strcmp(words[i], "uint32_t") || !strcmp(words[i], "int32_t")) bits = 32;
        }
        if (*p == '[') { while (*p && *p != ']') p++; if (*p) p++; p = skip_ws(p); }
        if (*p == ';') { p++; continue; }                      /* state arrays: `int32_t cstate_layer1_vad[28];` */
        if (*p != '=') { nnsp_set_error("model text: unexpected '%c' after '%s'", *p, name); return NNSP_B200_ERR_ARG; }
        p = skip_ws(p + 1);
        if (*p != '{') { nnsp_set_error("model text: '%s' is not a brace initialiser", name); return NNSP_B200_ERR_ARG; }
        if (is_net) {
            const char *b = p + 1;
            int d = 1;
            const char *q = b;
            while (*q && d) { if (*q == '{') d++; else if (*q == '}') d--; q++; }
            if (d) { nnsp_set_error("model text: unterminated NeuralNetClass initialiser"); return NNSP_B200_ERR_ARG; }
            free(u->net);
            u->net = (char *)malloc((size_t)(q - b));
            if (!u->net) return NNSP_B200_ERR_NOMEM;
            memcpy(u->net, b, (size_t)(q - 1 - b));
            u->net[q - 1 - b] = 0;
            snprintf(u->net_name, sizeof u->net_name, "%s", name);
            p = q;
        } else {
            if (!bits) { nnsp_set_error("model text: array '%s' has no integer element type", name); return NNSP_B200_ERR_ARG; }
            if (u->narr == u->cap) {
                u->cap = u->cap ? 2 * u->cap : 32;
                text_array *t = (text_array *)realloc(u->arr, u->cap * sizeof *t);
                if (!t) return NNSP_B200_ERR_NOMEM;
                u->arr = t;
            }
            text_array *a = &u->arr[u->narr];
            memset(a, 0, sizeof *a);
            snprintf(a->name, sizeof a->name, "%s", name);
            a->elem_bits = bits;
            const int rc = parse_numbers(p + 1, &p, &a->v, &a->n);
            if (rc) { nnsp_set_error("model text: bad number list in '%s'", name); return rc; }
            u->narr++;
        }
        p = skip_ws(p);
        if (*p == ';') p++;
    }
    if (!u->net) { nnsp_set_error("model text: no `NeuralNetClass net_<name> = {...}` definition"); return NNSP_B200_ERR_ARG; }
    return NNSP_B200_OK;
}

static const text_array *find_array(const text_unit *u, const char *name)
{
    for (size_t i = 0; i < u->narr; i++)
        if (!strcmp(u->arr[i].name, name)) return &u->arr[i];
    return NULL;
}

/* the k-th top-level item of a brace list: either a nested `{...}` (returned without braces) or an expression */
static int list_item(const char *list, int k, char *out, size_t cap)
{
    const char *p = list;
    for (int idx = 0;; idx++) {
        p = skip_ws(p);
        if (!*p) return 0;
        const char *b = p;
        int d = 0;
        while (*p && !(d == 0 && *p == ',')) {
            if (*p == '{' || *p == '(') d++;
            else if (*p == '}' || *p == ')') d--;
            p++;
        }
        if (idx == k) {
            const char *e = p;
            while (e > b && isspace((unsigned char)e[-1])) e--;
            if (*b == '{' && e > b && e[-1] == '}') { b++; e--; }
            size_t n = (size_t)(e - b);
            if (n >= cap) n = cap - 1;
            memcpy(out, b, n);
            out[n] = 0;
            return 1;
        }
        if (*p == ',') p++;
    }
}
/* last identifier or number of an expression such as `(int8_t*) vad_kernel0` or `(...) &tanh_fix` */
static void last_word(const char *expr, char *out, size_t cap)
{
    const char *e = expr + strlen(expr);
    while (e > expr && !is_ident((unsigned char)e[-1])) e--;
    const char *b = e;
    while (b > expr && is_ident((unsigned char)b[-1])) b--;
    size_t n = (size_t)(e - b);
    if (n >= cap) n = cap - 1;
    memcpy(out, b, n);
    out[n] = 0;
}

int nnsp_b200_model_from_table_text(const char *text, size_t nbytes, int nn_id, int acc32, nnsp_b200_model **out)
{
    if (!text || !out) return NNSP_B200_ERR_ARG;
    char *z = (char *)malloc(nbytes + 1);                      /* NUL-terminated private copy */
    if (!z) return NNSP_B200_ERR_NOMEM;
    memcpy(z, text, nbytes);
    z[nbytes] = 0;
    char *src = preprocess(z, nbytes, acc32 > 0);
    free(z);
    if (!src) return NNSP_B200_ERR_NOMEM;
    text_unit u;
    int rc = read_unit(src, &u);
    free(src);
    if (rc) { unit_free(&u); return rc; }

    const char *nn_name = !strncmp(u.net_name, "net_", 4) ? u.net_name + 4 : u.net_name;
    if (nn_id < 0) {                                           /* nnsp_identification.h:3-9 */
        if (!strcmp(nn_name, "s2i")) nn_id = NNSP_B200_ID_S2I;
        else if (!strcmp(nn_name, "vad")) nn_id = NNSP_B200_ID_VAD;
        else if (!strncmp(nn_name, "kws", 3)) nn_id = NNSP_B200_ID_KWS;
        else { nnsp_set_error("model text: cannot infer the NNSP id of '%s'; pass nn_id", nn_name); unit_free(&u); return NNSP_B200_ERR_ARG; }
    }
    char nm[128], item[1 << 12], sub[256], word[96];
    NeuralNetClass net;
    memset(&net, 0, sizeof net);
    int8_t *kern[NNSP_B200_MAX_LAYERS] = { 0 }, *krec[NNSP_B200_MAX_LAYERS] = { 0 };
    int16_t *bias[NNSP_B200_MAX_LAYERS] = { 0 };
    int32_t mean[NNSP_B200_NMEL], stdr[NNSP_B200_NMEL];
#define FAIL(...) do { nnsp_set_error(__VA_ARGS__); rc = NNSP_B200_ERR_ARG; goto done; } while (0)
    /* field order of NeuralNetClass, neural_nets.h:15-32 */
    if (!list_item(u.net, 0, item, sizeof item)) FAIL("model text: empty initialiser");
    net.numlayers = (int8_t)strtol(item, NULL, 0);
    const int nl = net.numlayers;
    if (nl < 1 || nl > NNSP_B200_MAX_LAYERS) FAIL("model text: numlayers %d outside 1..%d", nl, NNSP_B200_MAX_LAYERS);
    if (!list_item(u.net, 1, item, sizeof item)) FAIL("model text: missing size_layer");
    for (int i = 0; i <= nl; i++) {
        if (!list_item(item, i, sub, sizeof sub) || !*sub) FAIL("model text: size_layer has fewer than %d entries", nl + 1);
        net.size_layer[i] = (int16_t)strtol(sub, NULL, 0);
        if (net.size_layer[i] < 1 || net.size_layer[i] > 4096) FAIL("model text: layer width %d out of range", net.size_layer[i]);
    }
    for (int f = 2; f <= 6; f++) {
        if (!list_item(u.net, f, item, sizeof item)) FAIL("model text: initialiser field %d missing", f);
        for (int i = 0; i < nl; i++) {
            if (!list_item(item, i, sub, sizeof sub) || !*sub) FAIL("model text: field %d has fewer than %d entries", f, nl);
            last_word(sub, word, sizeof word);
            if (f == 2) {
                if (!strcmp(word, "fc")) net.net_layer_type[i] = fc;
                else if (!strcmp(word, "lstm")) net.net_layer_type[i] = lstm;
                else FAIL("model text: unknown layer type '%s'", word);
            } else if (f == 6) {
                if (!strcmp(word, "relu6")) net.activation_type[i] = relu6;
                else if (!strcmp(word, "ftanh")) net.activation_type[i] = ftanh;
                else if (!strcmp(word, "sigmoid") || !strcmp(word, "fsigmoid")) net.activation_type[i] = sigmoid;
                else if (!strcmp(word, "linear")) net.activation_type[i] = linear;
                else FAIL("model text: unknown activation '%s'", word);
            } else {
                const int8_t q = (int8_t)strtol(word, NULL, 0);
                if (f == 3) net.qbit_kernel[i] = q; else if (f == 4) net.qbit_input[i] = q; else net.qbit_bias[i] = q;
            }
        }
        /* qbit_input[nl]: the qbit_input_rec of a last LSTM layer (neural_nets.c:108); 0 when the initialiser stops at nl */
        if (f == 4 && nl < NNSP_B200_MAX_LAYERS && list_item(item, nl, sub, sizeof sub) && *sub) {
            last_word(sub, word, sizeof word);
            net.qbit_input[nl] = (int8_t)strtol(word, NULL, 0);
        }
    }
    /* fields 7, 8: state pointers (owned by the engine here). 9: act_func, 10: layer_func, 11..13: tables */
    for (int i = 0; i < nl; i++) {
        if (list_item(u.net, 9, item, sizeof item) && list_item(item, i, sub, sizeof sub)) {
            last_word(sub, word, sizeof word);
            if (!strcmp(word, "tanh_fix")) net.act_func[i] = (void *(*)(void *, int32_t *, int))&tanh_fix;
            else if (!strcmp(word, "sigmoid_fix")) net.act_func[i] = (void *(*)(void *, int32_t *, int))&sigmoid_fix;
            else if (!strcmp(word, "relu6_fix")) net.act_func[i] = (void *(*)(void *, int32_t *, int))&relu6_fix;
            else if (!strcmp(word, "linear_fix")) net.act_func[i] = (void *(*)(void *, int32_t *, int))&linear_fix;
            else FAIL("model text: unknown activation function '%s'", word);
        } else FAIL("model text: activation function table missing");
        if (list_item(u.net, 10, item, sizeof item) && list_item(item, i, sub, sizeof sub)) {
            last_word(sub, word, sizeof word);
            int want_lstm = net.net_layer_type[i] == lstm;
            if (!strcmp(word, "fc_8x16") && !want_lstm) net.layer_func[i] = (int *(*)())&fc_8x16;
            else if (!strcmp(word, "fc_8x16_acc32b") && !want_lstm) net.layer_func[i] = (int *(*)())&fc_8x16_acc32b;
            else if (!strcmp(word, "lstm_8x16") && want_lstm) net.layer_func[i] = (int *(*)())&lstm_8x16;
            else if (!strcmp(word, "lstm_8x16_acc32b") && want_lstm) net.layer_func[i] = (int *(*)())&lstm_8x16_acc32b;
            else FAIL("model text: layer function '%s' does not match layer %d", word, i);
        } else FAIL("model text: layer function table missing");
        const int rows = net.size_layer[i + 1], cols = net.size_layer[i];
        const size_t nr = (net.net_layer_type[i] == lstm) ? 4u * (size_t)rows : (size_t)rows;
        for (int f = 11; f <= 13; f++) {
            if (!list_item(u.net, f, item, sizeof item) || !list_item(item, i, sub, sizeof sub)) FAIL("model text: table pointer field %d missing", f);
            last_word(sub, word, sizeof word);
            const int is_null = !strcmp(word, "0") || !strcmp(word, "NULL") || !*word;
            if (f == 13 && net.net_layer_type[i] != lstm) continue;
            if (is_null) FAIL("model text: layer %d lacks table %d", i, f);
            const text_array *a = find_array(&u, word);
            if (!a) FAIL("model text: array '%s' is not defined", word);
            const size_t need = (f == 11) ? nr * (size_t)cols : (f == 12 ? nr : nr * (size_t)rows);
            if (a->n != need || a->elem_bits != (f == 12 ? 16 : 8))
                FAIL("model text: '%s' has %zu x %d-bit elements, layer %d needs %zu", word, a->n, a->elem_bits, i, need);
            if (f == 12) {
                bias[i] = (int16_t *)malloc(need * 2 + 2);
                if (!bias[i]) { rc = NNSP_B200_ERR_NOMEM; goto done; }
                for (size_t k = 0; k < need; k++) bias[i][k] = (int16_t)(uint16_t)a->v[k];
                net.pt_bias[i] = bias[i];
            } else {
                int8_t *w = (int8_t *)malloc(need + 1);
                if (!w) { rc = NNSP_B200_ERR_NOMEM; goto done; }
                for (size_t k = 0; k < need; k++) w[k] = (int8_t)(uint8_t)a->v[k];
                if (f == 11) { kern[i] = w; net.pt_kernel[i] = w; } else { krec[i] = w; net.pt_kernel_rec[i] = w; }
            }
        }
    }
    {
        snprintf(nm, sizeof nm, "feature_mean_%s", nn_name);
        const text_array *am = find_array(&u, nm);
        snprintf(nm, sizeof nm, "feature_stdR_%s", nn_name);
        const text_array *as = find_array(&u, nm);
        if (!am || !as || am->n < NNSP_B200_NMEL || as->n < NNSP_B200_NMEL) FAIL("model text: feature_mean_%s / feature_stdR_%s missing or short", nn_name, nn_name);
        for (int i = 0; i < NNSP_B200_NMEL; i++) { mean[i] = (int32_t)(uint32_t)am->v[i]; stdr[i] = (int32_t)(uint32_t)as->v[i]; }
    }
    rc = nnsp_b200_model_from_net(&net, mean, stdr, nn_id, out);
    if (rc == NNSP_B200_OK && acc32 >= 0) nnsp_b200_model_set_acc32(*out, acc32);
done:
#undef FAIL
    for (int i = 0; i < NNSP_B200_MAX_LAYERS; i++) { free(kern[i]); free(krec[i]); free(bias[i]); }
    unit_free(&u);
    return rc;
}

/* ---------------------------------------------------------------------------------------------------- */
/* writer: the text python/c_code_table_converter.py:143-347 produces (as shipped in evb/src/def_nn*.c)  */
/* ---------------------------------------------------------------------------------------------------- */
typedef struct { char *buf; size_t cap, len; } sink;
static void put(sink *s, const char *fmt, ...)
{
    char tmp[256];
    va_list ap;
    va_start(ap, fmt);
    const int n = vsnprintf(tmp, sizeof tmp, fmt, ap);
    va_end(ap);
    if (n <= 0) return;
    if (s->buf && s->len + (size_t)n <= s->cap) memcpy(s->buf + s->len, tmp, (size_t)n);
    s->len += (size_t)n;
}

int nnsp_b200_model_to_table_text(const nnsp_b200_model *m, const char *nn_name, char *buf, size_t cap, size_t *nbytes)
{
    if (!m || !nn_name || !*nn_name || strlen(nn_name) > 40) return NNSP_B200_ERR_ARG;
    sink s = { buf, cap, 0 };
    static const char *act_enum[] = { "relu6", "ftanh", "sigmoid", "linear" };   /* ACTIVATION_TYPE, activation.h:16-22 */
    static const char *act_fn[] = { "relu6_fix", "tanh_fix", "sigmoid_fix", "linear_fix" };
    const int nl = m->numlayers;
    const nnsp_layer *Ll = &m->layer[nl - 1];
    /* A last LSTM layer reads its qbit_input_rec from qbit_input[nl] (neural_nets.c:108). With 10 layers that entry lies
     * past the array, on qbit_bias[0] (what nnsp_b200_model_from_net reads too): a table cannot hold any other value. */
    const int emit_qi_next = Ll->type == NNSP_LAYER_LSTM && nl < NNSP_B200_MAX_LAYERS;
    if (Ll->type == NNSP_LAYER_LSTM && nl == NNSP_B200_MAX_LAYERS && Ll->qi_next != m->layer[0].qb) {
        nnsp_set_error("model to table text: the last of %d layers is an LSTM whose qbit_input_rec %d differs from "
                       "qbit_bias[0] %d; a %d-layer table reads qbit_bias[0] there", nl, Ll->qi_next, m->layer[0].qb, nl);
        return NNSP_B200_ERR_UNSUPPORTED;
    }
    put(&s, "#include <stdint.h>\n#include \"neural_nets.h\"\n#include \"activation.h\"\n#include \"affine.h\"\n"
            "#include \"affine_acc32b.h\"\n#include \"lstm.h\"\n/*************stats***********/\n");
    put(&s, "const int32_t feature_mean_%s[] = {", nn_name);
    for (int i = 0; i < NNSP_B200_NMEL; i++) put(&s, "0x%08x, ", (unsigned)m->mean[i]);
    put(&s, "};\nconst int32_t feature_stdR_%s[] = {", nn_name);
    for (int i = 0; i < NNSP_B200_NMEL; i++) put(&s, "0x%08x, ", (unsigned)m->stdR[i]);
    put(&s, "};\n");
    for (int i = 0; i < nl; i++) {
        const nnsp_layer *L = &m->layer[i];
        const int is_lstm = L->type == NNSP_LAYER_LSTM;
        const size_t nr = is_lstm ? 4u * (size_t)L->rows : (size_t)L->rows;
        int8_t *k = (int8_t *)malloc(nr * L->cols + 1), *kr = (int8_t *)malloc(nr * L->rows + 1);
        int16_t *b = (int16_t *)malloc(nr * 2 + 2);
        if (!k || !kr || !b) { free(k); free(kr); free(b); return NNSP_B200_ERR_NOMEM; }
        nnsp_model_layer_to_table(L, k, kr, b);
        put(&s, "// layer %d\nconst uint8_t %s_kernel%d[]={", i, nn_name, i);
        for (size_t j = 0; j < nr * L->cols; j++) put(&s, "0x%02x,", (unsigned)(uint8_t)k[j]);
        put(&s, "};\n");
        if (is_lstm) {
            put(&s, "const uint8_t %s_kernel_rec%d[]={", nn_name, i);
            for (size_t j = 0; j < nr * L->rows; j++) put(&s, "0x%02x,", (unsigned)(uint8_t)kr[j]);
            put(&s, "};\n");
        }
        put(&s, "const uint16_t %s_bias%d[]={", nn_name, i);
        for (size_t j = 0; j < nr; j++) put(&s, "0x%04x,", (unsigned)(uint16_t)b[j]);
        put(&s, "};\n");
        free(k); free(kr); free(b);
    }
    put(&s, "// lstm states\n");
    for (int i = 0; i < nl; i++)
        if (m->layer[i].type == NNSP_LAYER_LSTM)
            put(&s, "int32_t cstate_layer%d_%s[%d];\nint16_t hstate_layer%d_%s[%d];\n", i, nn_name, m->layer[i].rows, i, nn_name, m->layer[i].rows);
    put(&s, "NeuralNetClass net_%s = {\n\n\t%d, // layers\n\n\t{", nn_name, nl);
    for (int i = 0; i <= nl; i++) put(&s, "%d,", m->size_layer[i]);
    put(&s, "}, // nn size for each layer, including the input layer\n\n\t{");
    for (int i = 0; i < nl; i++) put(&s, "%s,", m->layer[i].type == NNSP_LAYER_LSTM ? "lstm" : "fc");
    put(&s, "}, // layer type\n\n\t{");
    for (int i = 0; i < nl; i++) put(&s, "%d,", m->layer[i].qk);
    put(&s, "}, // fractional bits (kernel)\n\n\t{");
    for (int i = 0; i < nl; i++) put(&s, "%d,", m->layer[i].qi);
    if (emit_qi_next) put(&s, "%d,", Ll->qi_next);
    put(&s, "}, // qbit_i\n\n\t{");
    for (int i = 0; i < nl; i++) put(&s, "%d,", m->layer[i].qb);
    put(&s, "}, // fractional bits (bias)\n\n\t{");
    for (int i = 0; i < nl; i++) put(&s, "%s,", act_enum[m->layer[i].act]);
    put(&s, "}, // activations\n\n\t{\n");
    for (int i = 0; i < nl; i++) {
        if (m->layer[i].type == NNSP_LAYER_LSTM) put(&s, "\t\t(int32_t*) cstate_layer%d_%s,\n", i, nn_name);
        else put(&s, "\t\t(int32_t*) 0,\n");
    }
    put(&s, "\t}, // cstates lstm\n\n\t{\n");
    for (int i = 0; i < nl; i++) {
        if (m->layer[i].type == NNSP_LAYER_LSTM) put(&s, "\t\t(int16_t*) hstate_layer%d_%s,\n", i, nn_name);
        else put(&s, "\t\t(int16_t*) 0,\n");
    }
    put(&s, "\t}, // hstates lstm\n\n\t{\n");
    for (int i = 0; i < nl; i++) put(&s, "\t\t(void* (*)(void*, int32_t*, int)) &%s,\n", act_fn[m->layer[i].act]);
    put(&s, "\t}, // activation function\n#ifdef DEF_ACC32BIT_OPT\n\t{\n");
    for (int i = 0; i < nl; i++) put(&s, "\t\t(int* (*)()) &%s_8x16_acc32b,\n", m->layer[i].type == NNSP_LAYER_LSTM ? "lstm" : "fc");
    put(&s, "\t}, // net layer type\n#else\n\t{\n");
    for (int i = 0; i < nl; i++) put(&s, "\t\t(int* (*)()) &%s_8x16,\n", m->layer[i].type == NNSP_LAYER_LSTM ? "lstm" : "fc");
    put(&s, "\t}, // net layer type\n#endif\n\n\t{\n");
    for (int i = 0; i < nl; i++) put(&s, "\t\t(int8_t*) %s_kernel%d,\n", nn_name, i);
    put(&s, "\t}, // kernel\n\n\t{\n");
    for (int i = 0; i < nl; i++) put(&s, "\t\t(int16_t*) %s_bias%d,\n", nn_name, i);
    put(&s, "\t}, // bias\n\n\t{\n");
    for (int i = 0; i < nl; i++) {
        if (m->layer[i].type == NNSP_LAYER_LSTM) put(&s, "\t\t(int8_t*) %s_kernel_rec%d,\n", nn_name, i);
        else put(&s, "\t\t(int8_t*) 0,\n");
    }
    put(&s, "\t}, // kernel_rec\n\n};\n");
    if (nbytes) *nbytes = s.len;
    if (buf && s.len > cap) { nnsp_set_error("table text needs %zu bytes, buffer has %zu", s.len, cap); return NNSP_B200_ERR_ARG; }
    return NNSP_B200_OK;
}
