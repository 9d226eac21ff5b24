/* nnsp_model.c -- model container ("NNSPM1" blob) and the ARM weight interleave.
 * Layout rules follow python/nnsp_pack/c_weight_man.py:5-124 and the readers in
 * ns-nnsp/src/affine.c:74-184 (4/3/2/1-row groups, odd-column tail) and lstm.c:48-124. */
#include "nnsp_model.h"
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static __thread char g_err[256];

void nnsp_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
const char *nnsp_b200_last_error(void) { return g_err; }

const char *nnsp_b200_strerror(int code)
{
    switch (code) {
    case NNSP_B200_OK: return "ok";
    case NNSP_B200_ERR_ARG: return "invalid argument or malformed model";
    case NNSP_B200_ERR_CUDA: return "CUDA failure or no usable sm_100 device (there is no CPU fallback)";
    case NNSP_B200_ERR_NOMEM: return "out of memory";
    case NNSP_B200_ERR_UNSUPPORTED: return "model outside the limits of the engine";
    }
    return "unknown error";
}

/* ---- one K-row block (K = 1..4), c_weight_man.py:23-47 -------------------------------- */
static size_t block_xfer(int8_t *table, int8_t *rowmajor, int K, int cols, int ld, int to_table)
{
    size_t p = 0;
    const int pairs = cols >> 1;
    for (int cp = 0; cp < pairs; cp++) {
        const int c = 2 * cp;
        for (int rp = 0; rp < (K >> 1); rp++) {          /* 2x2 tile stored transposed */
            const int r = 2 * rp;
            int8_t *q[4] = { &rowmajor[r * ld + c], &rowmajor[(r + 1) * ld + c],
                             &rowmajor[r * ld + c + 1], &rowmajor[(r + 1) * ld + c + 1] };
            for (int k = 0; k < 4; k++, p++) {
                if (to_table) table[p] = *q[k]; else *q[k] = table[p];
            }
        }
        if (K & 1) {                                     /* odd last row: two columns in order */
            const int r = K - 1;
            for (int k = 0; k < 2; k++, p++) {
                if (to_table) table[p] = rowmajor[r * ld + c + k]; else rowmajor[r * ld + c + k] = table[p];
            }
        }
    }
    if (cols & 1) {                                      /* odd last column, stored column-wise */
        for (int r = 0; r < K; r++, p++) {
            if (to_table) table[p] = rowmajor[r * ld + cols - 1]; else rowmajor[r * ld + cols - 1] = table[p];
        }
    }
    return p;
}

static size_t matrix_xfer(int8_t *table, int8_t *rowmajor, int rows, int cols, int to_table)
{
    size_t p = 0;
    int r = 0;
    for (; r + 4 <= rows; r += 4) p += block_xfer(table + p, rowmajor + (size_t)r * cols, 4, cols, cols, to_table);
    if (rows - r) p += block_xfer(table + p, rowmajor + (size_t)r * cols, rows - r, cols, cols, to_table);
    return p;
}

size_t nnsp_deinterleave_arm(const int8_t *src, int rows, int cols, int8_t *dst)
{
    return matrix_xfer((int8_t *)src, dst, rows, cols, 0);
}
size_t nnsp_interleave_arm(const int8_t *src, int rows, int cols, int8_t *dst)
{
    return matrix_xfer(dst, (int8_t *)src, rows, cols, 1);
}

/* lstm kernels: per 4-unit group the table holds the i, j, f, o blocks back to back
 * (c_weight_man.py:61-92); canonical row = gate*H + unit */
static size_t lstm_xfer(int8_t *table, int8_t *canon, int H, int cols, int to_table)
{
    size_t p = 0;
    for (int u = 0; u < H; u += 4) {
        const int K = (H - u) < 4 ? (H - u) : 4;
        for (int g = 0; g < 4; g++)
            p += block_xfer(table + p, canon + ((size_t)g * H + u) * cols, K, cols, cols, to_table);
    }
    return p;
}
static void lstm_bias_xfer(int16_t *table, int16_t *canon, int H, int to_table)
{
    size_t p = 0;
    for (int u = 0; u < H; u += 4) {
        const int K = (H - u) < 4 ? (H - u) : 4;
        for (int g = 0; g < 4; g++)
            for (int k = 0; k < K; k++, p++) {
                if (to_table) table[p] = canon[g * H + u + k]; else canon[g * H + u + k] = table[p];
            }
    }
}

/* ---- internal constructors shared with nnsp_model_net.c ------------------------------- */
int nnsp_model_alloc_layer(nnsp_layer *L)
{
    const size_t nr = (L->type == NNSP_LAYER_LSTM) ? 4u * L->rows : (size_t)L->rows;
    L->w = (int8_t *)calloc(nr * L->cols + 1, 1);
    L->bias = (int16_t *)calloc(nr + 1, sizeof(int16_t));
    L->wrec = (L->type == NNSP_LAYER_LSTM) ? (int8_t *)calloc(nr * L->rows + 1, 1) : NULL;
    if (!L->w || !L->bias || (L->type == NNSP_LAYER_LSTM && !L->wrec)) return NNSP_B200_ERR_NOMEM;
    return NNSP_B200_OK;
}

/* fill canonical arrays of layer L from table-layout arrays (what def_nn*.c holds) */
void nnsp_model_layer_from_table(nnsp_layer *L, const int8_t *kernel, const int8_t *kernel_rec,
                                 const int16_t *bias)
{
    if (L->type == NNSP_LAYER_LSTM) {
        lstm_xfer((int8_t *)kernel, L->w, L->rows, L->cols, 0);
        lstm_xfer((int8_t *)kernel_rec, L->wrec, L->rows, L->rows, 0);
        lstm_bias_xfer((int16_t *)bias, L->bias, L->rows, 0);
    } else {
        matrix_xfer((int8_t *)kernel, L->w, L->rows, L->cols, 0);
        memcpy(L->bias, bias, (size_t)L->rows * sizeof(int16_t));
    }
}

/* the inverse: table-layout arrays of layer L from its canonical arrays */
void nnsp_model_layer_to_table(const nnsp_layer *L, int8_t *kernel, int8_t *kernel_rec, int16_t *bias)
{
    if (L->type == NNSP_LAYER_LSTM) {
        lstm_xfer(kernel, L->w, L->rows, L->cols, 1);
        lstm_xfer(kernel_rec, L->wrec, L->rows, L->rows, 1);
        lstm_bias_xfer(bias, L->bias, L->rows, 1);
    } else {
        matrix_xfer(kernel, L->w, L->rows, L->cols, 1);
        memcpy(bias, L->bias, (size_t)L->rows * sizeof(int16_t));
    }
}

int nnsp_model_validate(const struct nnsp_b200_model *m)
{
    if (m->numlayers < 1 || m->numlayers > NNSP_B200_MAX_LAYERS) {
        nnsp_set_error("numlayers %d outside 1..%d", m->numlayers, NNSP_B200_MAX_LAYERS);
        return NNSP_B200_ERR_ARG;
    }
    if (m->size_layer[0] != NNSP_B200_NMEL * NNSP_B200_NCTX) {
        nnsp_set_error("input width %d: the front end feeds %d (6 x 40 context)", m->size_layer[0],
                       NNSP_B200_NMEL * NNSP_B200_NCTX);
        return NNSP_B200_ERR_UNSUPPORTED;
    }
    for (int i = 0; i < m->numlayers; i++) {
        const nnsp_layer *L = &m->layer[i];
        if (L->rows < 1 || L->cols < 1 || L->rows != m->size_layer[i + 1] || L->cols != m->size_layer[i]) {
            nnsp_set_error("layer %d: inconsistent shape %dx%d", i, L->rows, L->cols);
            return NNSP_B200_ERR_ARG;
        }
        if (L->type != NNSP_LAYER_FC && L->type != NNSP_LAYER_LSTM) {
            nnsp_set_error("layer %d: unknown layer type %d", i, L->type);
            return NNSP_B200_ERR_ARG;
        }
        if (L->act < NNSP_ACT_RELU6 || L->act > NNSP_ACT_LINEAR) {
            nnsp_set_error("layer %d: unknown activation %d", i, L->act);
            return NNSP_B200_ERR_ARG;
        }
        if (L->act == NNSP_ACT_LINEAR && i != m->numlayers - 1 && L->type == NNSP_LAYER_FC) {
            /* a linear layer writes int32 into the int16 ping-pong buffer (neural_nets.c:152-158,
             * activation.c:19-29); only meaningful as the last layer */
            nnsp_set_error("layer %d: linear activation is only supported on the last layer", i);
            return NNSP_B200_ERR_UNSUPPORTED;
        }
        const int last = (i == m->numlayers - 1);
        const int limit = (last && L->act == NNSP_ACT_LINEAR && NNSP_B200_MAX_OUT < NNSP_B200_MAX_WIDTH) ? NNSP_B200_MAX_OUT : NNSP_B200_MAX_WIDTH;
        if (L->rows > limit) {
            nnsp_set_error("layer %d: width %d exceeds the engine limit of %d units", i, L->rows, limit);
            return NNSP_B200_ERR_UNSUPPORTED;
        }
        if (L->qk < 0 || L->qk > 15 || L->qi < 0 || L->qi > 15 || L->qb < 0 || L->qb > 15 ||
            L->qi_next < 0 || L->qi_next > 15) {
            nnsp_set_error("layer %d: q-format outside 0..15", i);
            return NNSP_B200_ERR_UNSUPPORTED;
        }
    }
    return NNSP_B200_OK;
}

void nnsp_b200_model_free(nnsp_b200_model *m)
{
    if (!m) return;
    for (int i = 0; i < NNSP_B200_MAX_LAYERS; i++) {
        free(m->layer[i].w);
        free(m->layer[i].wrec);
        free(m->layer[i].bias);
    }
    free(m);
}

int nnsp_b200_model_set_acc32(nnsp_b200_model *m, int acc32)
{
    if (!m) return NNSP_B200_ERR_ARG;
    for (int i = 0; i < m->numlayers; i++) m->layer[i].acc32 = acc32 ? 1 : 0;
    return NNSP_B200_OK;
}

int nnsp_b200_model_info(const nnsp_b200_model *m, int *nn_id, int *numlayers,
                         int16_t size_layer[NNSP_B200_MAX_LAYERS + 1], int *acc32)
{
    if (!m) return NNSP_B200_ERR_ARG;
    if (nn_id) *nn_id = m->nn_id;
    if (numlayers) *numlayers = m->numlayers;
    if (size_layer) memcpy(size_layer, m->size_layer, sizeof m->size_layer);
    if (acc32) *acc32 = m->layer[0].acc32;
    return NNSP_B200_OK;
}

/* ---- blob ------------------------------------------------------------------------------
 * little-endian:
 *   char   magic[8] = "NNSPM1\0\0"
 *   int32  nn_id, numlayers
 *   int16  size_layer[11], pad
 *   int32  mean[40], stdR[40]
 *   int32  layer[10][10] = {type, act, qk, qi, qb, acc32, kernel_bytes, rec_bytes, bias_count, qi_next}
 *   then per layer: kernel | kernel_rec | bias(int16), each padded to 4 bytes, all in the
 *   table layout of def_nn*.c (ARM interleave, lstm gate grouping)                        */
#define BLOB_HDR (8 + 8 + 24 + 320 + 400)
static size_t pad4(size_t n) { return (n + 3u) & ~(size_t)3u; }

static void layer_sizes(const nnsp_layer *L, size_t *kb, size_t *rb, size_t *bc)
{
    const size_t nr = (L->type == NNSP_LAYER_LSTM) ? 4u * L->rows : (size_t)L->rows;
    *kb = nr * L->cols;
    *rb = (L->type == NNSP_LAYER_LSTM) ? nr * L->rows : 0;
    *bc = nr;
}

int nnsp_b200_model_to_blob(const nnsp_b200_model *m, void *buf, size_t cap, size_t *nbytes)
{
    if (!m) return NNSP_B200_ERR_ARG;
    size_t need = BLOB_HDR;
    for (int i = 0; i < m->numlayers; i++) {
        size_t kb, rb, bc;
        layer_sizes(&m->layer[i], &kb, &rb, &bc);
        need += pad4(kb) + pad4(rb) + pad4(bc * 2);
    }
    if (nbytes) *nbytes = need;
    if (!buf) return NNSP_B200_OK;
    if (cap < need) { nnsp_set_error("blob buffer too small: %zu < %zu", cap, need); return NNSP_B200_ERR_ARG; }
    unsigned char *p = (unsigned char *)buf;
    memset(p, 0, need);
    memcpy(p, "NNSPM1\0\0", 8);
    int32_t v = m->nn_id; memcpy(p + 8, &v, 4);
    v = m->numlayers; memcpy(p + 12, &v, 4);
    memcpy(p + 16, m->size_layer, 22);
    memcpy(p + 40, m->mean, 160);
    memcpy(p + 200, m->stdR, 160);
    size_t off = BLOB_HDR;
    for (int i = 0; i < m->numlayers; i++) {
        const nnsp_layer *L = &m->layer[i];
        size_t kb, rb, bc;
        layer_sizes(L, &kb, &rb, &bc);
        int32_t rec[10] = { L->type, L->act, L->qk, L->qi, L->qb, L->acc32, (int32_t)kb, (int32_t)rb, (int32_t)bc, L->qi_next };
        memcpy(p + 360 + 40 * i, rec, 40);
        if (L->type == NNSP_LAYER_LSTM) {
            lstm_xfer((int8_t *)p + off, L->w, L->rows, L->cols, 1); off += pad4(kb);
            lstm_xfer((int8_t *)p + off, L->wrec, L->rows, L->rows, 1); off += pad4(rb);
            lstm_bias_xfer((int16_t *)(p + off), L->bias, L->rows, 1); off += pad4(bc * 2);
        } else {
            matrix_xfer((int8_t *)p + off, L->w, L->rows, L->cols, 1); off += pad4(kb);
            memcpy(p + off, L->bias, bc * 2); off += pad4(bc * 2);
        }
    }
    return NNSP_B200_OK;
}

int nnsp_b200_model_from_blob(const void *blob, size_t n, nnsp_b200_model **out)
{
    if (!blob || !out) return NNSP_B200_ERR_ARG;
    const unsigned char *p = (const unsigned char *)blob;
    if (n < BLOB_HDR || memcmp(p, "NNSPM1\0\0", 8) != 0) { nnsp_set_error("not an NNSPM1 blob"); return NNSP_B200_ERR_ARG; }
    nnsp_b200_model *m = (nnsp_b200_model *)calloc(1, sizeof *m);
    if (!m) return NNSP_B200_ERR_NOMEM;
    int32_t v;
    memcpy(&v, p + 8, 4); m->nn_id = v;
    memcpy(&v, p + 12, 4); m->numlayers = v;
    memcpy(m->size_layer, p + 16, 22);
    memcpy(m->mean, p + 40, 160);
    memcpy(m->stdR, p + 200, 160);
    if (m->numlayers < 1 || m->numlayers > NNSP_B200_MAX_LAYERS) { nnsp_b200_model_free(m); nnsp_set_error("bad layer count"); return NNSP_B200_ERR_ARG; }
    size_t off = BLOB_HDR;
    int rc = NNSP_B200_OK;
    for (int i = 0; i < m->numlayers && rc == NNSP_B200_OK; i++) {
        nnsp_layer *L = &m->layer[i];
        int32_t rec[10];
        memcpy(rec, p + 360 + 40 * i, 40);
        L->type = rec[0]; L->act = rec[1]; L->qk = rec[2]; L->qi = rec[3]; L->qb = rec[4]; L->acc32 = rec[5]; L->qi_next = rec[9];
        L->rows = m->size_layer[i + 1]; L->cols = m->size_layer[i];
        if (L->rows < 1 || L->cols < 1 || L->rows > 4096 || L->cols > 4096) { rc = NNSP_B200_ERR_ARG; break; }
        size_t kb, rb, bc;
        layer_sizes(L, &kb, &rb, &bc);
        if ((size_t)rec[6] != kb || (size_t)rec[7] != rb || (size_t)rec[8] != bc ||
            off + pad4(kb) + pad4(rb) + pad4(bc * 2) > n) { nnsp_set_error("layer %d: size fields disagree with shapes", i); rc = NNSP_B200_ERR_ARG; break; }
        rc = nnsp_model_alloc_layer(L);
        if (rc) break;
        const int8_t *k = (const int8_t *)p + off; off += pad4(kb);
        const int8_t *kr = (const int8_t *)p + off; off += pad4(rb);
        const int16_t *b = (const int16_t *)(p + off); off += pad4(bc * 2);
        nnsp_model_layer_from_table(L, k, kr, b);
    }
    if (rc == NNSP_B200_OK) rc = nnsp_model_validate(m);
    if (rc != NNSP_B200_OK) { nnsp_b200_model_free(m); return rc; }
    *out = m;
    return NNSP_B200_OK;
}
