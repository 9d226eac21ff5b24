/* tests/dropin_driver.c -- TEST INFRASTRUCTURE: an application of the nine legacy entry points.
 *
 * It includes only include/nnsp_compat and calls NNSPClass_*, FeatureClass_* and NeuralNetClass_* the way code
 * written for ns-nnsp does. tests/test_gpu_dropin.py compiles it, links it to libnnsp_b200.so and drives it with
 * model tables emitted by nnsp_b200_model_to_table_text. The tap layout and the shadow evaluation of every layer
 * are those of oracle/ref_glue.c (ref_nnsp_run, ref_net_eval), so the taps compare with the oracle's and with the
 * hashes recorded from the reference.
 *
 * Unlike the reference glue it keeps no global state: every instance lives on the heap with its own NNSPClass,
 * FeatureClass and thresholds, so several instances run side by side and from several threads. */
#include <stdlib.h>
#include <string.h>

#include "feature_module.h"
#include "neural_nets.h"
#include "nn_speech.h"

typedef struct { int16_t trigger; int16_t outputs[3]; } drv_result;       /* == nnsp_b200_result */

typedef struct {
    NNSPClass inst;
    FeatureClass feat;
    int16_t thresh_prob, th_count;              /* read by NNSPClass_exec through the pointers NNSPClass_init took */
    NeuralNetClass *net;
    const int32_t *mean, *stdR;
    int nn_id;
} drv_inst;

#define DRV_MAXW 1024

static int act_stride(const NeuralNetClass *n)
{
    int i, s = 0;
    for (i = 1; i < n->numlayers; i++) s += n->size_layer[i];
    return s;
}
static int h_stride(const NeuralNetClass *n)
{
    int i, s = 0;
    for (i = 0; i < n->numlayers; i++) if (n->net_layer_type[i] == lstm) s += n->size_layer[i + 1];
    return s;
}
void drv_strides(const NeuralNetClass *n, int *act, int *h, int *n_out)
{
    *act = act_stride(n); *h = h_stride(n); *n_out = n->size_layer[n->numlayers];
}

static void save_hc(const NeuralNetClass *n, int16_t *h, int32_t *c)
{
    int i, j, o = 0;
    for (i = 0; i < n->numlayers; i++)
        if (n->net_layer_type[i] == lstm)
            for (j = 0; j < n->size_layer[i + 1]; j++, o++) { h[o] = n->pt_hstate[i][j]; c[o] = n->pt_cstate[i][j]; }
}
static void load_hc(NeuralNetClass *n, const int16_t *h, const int32_t *c)
{
    int i, j, o = 0;
    for (i = 0; i < n->numlayers; i++)
        if (n->net_layer_type[i] == lstm)
            for (j = 0; j < n->size_layer[i + 1]; j++, o++) { n->pt_hstate[i][j] = h[o]; n->pt_cstate[i][j] = c[o]; }
}

/* with the LSTM state set to (h0, c0), run the first k layers for k = 1..L through debug_layer and record every
 * layer's output; the live state is put back afterwards (ref_glue.c shadow_layers) */
static void shadow_layers(NeuralNetClass *n, int16_t *ctx, const int16_t *h0, const int32_t *c0, int16_t *act,
                          int32_t *logits)
{
    int16_t hl[DRV_MAXW];
    int32_t cl[DRV_MAXW], out[DRV_MAXW];
    int k, o = 0, j;
    save_hc(n, hl, cl);
    for (k = 1; k <= n->numlayers; k++) {
        load_hc(n, h0, c0);
        NeuralNetClass_exe(n, ctx, out, (int8_t)k);
        if (k < n->numlayers) {
            if (act) memcpy(act + o, out, n->size_layer[k] * sizeof(int16_t));
            o += n->size_layer[k];
        } else if (logits) {
            if (n->activation_type[k - 1] == linear) memcpy(logits, out, n->size_layer[k] * sizeof(int32_t));
            else for (j = 0; j < n->size_layer[k]; j++) logits[j] = ((int16_t *)out)[j];
        }
    }
    load_hc(n, hl, cl);
}

static void fill_post(int16_t *post, const NNSPClass *p, int ran_nn, int stage)
{
    int i;
    post[0] = p->trigger;
    for (i = 0; i < 3; i++) post[1 + i] = p->outputs[i];
    for (i = 0; i < 8; i++) post[4 + i] = p->counts_category[i];
    post[12] = p->argmax_last;
    post[13] = p->slides;
    post[14] = (int16_t)ran_nn;
    post[15] = (int16_t)stage;
}

/* ---- instances --------------------------------------------------------------------------------------------- */
drv_inst *drv_new(NeuralNetClass *net, const int32_t *mean, const int32_t *stdR, int nn_id)
{
    drv_inst *d = (drv_inst *)calloc(1, sizeof *d);
    if (!d) return NULL;
    d->net = net; d->mean = mean; d->stdR = stdR; d->nn_id = nn_id;
    d->thresh_prob = 16383; d->th_count = 4;
    return d;
}

void drv_free(drv_inst *d) { free(d); }

/* the application changes the values behind the pointers NNSPClass_init took: the next frame uses them */
void drv_set_thresholds(drv_inst *d, int16_t thresh_prob, int16_t th_count)
{
    d->thresh_prob = thresh_prob;
    d->th_count = th_count;
}

/* T frames through NNSPClass_exec. reset: 0 continue, 1 a brand-new instance (zeroed structs, init, reset),
 * 2 NNSPClass_reset of the live instance. Any tap may be null; taps of frames without an inference hold zeros
 * in act and logits (ref_glue.c ref_nnsp_run). */
int drv_run(drv_inst *d, int reset, const int16_t *pcm, int n_frames, drv_result *results, int32_t *tap_logmel,
            int16_t *tap_feat, int16_t *tap_act, int32_t *tap_logits, int16_t *tap_h, int32_t *tap_c, int16_t *tap_post)
{
    NeuralNetClass *net = d->net;
    const int as = act_stride(net), hs = h_stride(net), no = net->size_layer[net->numlayers];
    int16_t frame[160], h0[DRV_MAXW];
    int32_t c0[DRV_MAXW];
    FeatureClass shadow;
    int t, i;
    if (hs > DRV_MAXW || no > DRV_MAXW) return -1;
    if (reset == 1) {
        memset(&d->inst, 0, sizeof d->inst);
        memset(&d->feat, 0, sizeof d->feat);
        NNSPClass_init(&d->inst, net, &d->feat, (char)d->nn_id, d->mean, d->stdR, &d->thresh_prob, &d->th_count);
        NNSPClass_reset(&d->inst);
    } else if (reset == 2) {
        NNSPClass_reset(&d->inst);
    }
    for (t = 0; t < n_frames; t++) {
        memcpy(frame, pcm + (size_t)t * 160, sizeof frame);
        const int ran = (d->inst.slides == 1);
        if (ran && (tap_act || tap_logits)) {
            shadow = d->feat;
            FeatureClass_execute(&shadow, frame);
            save_hc(net, h0, c0);
            shadow_layers(net, shadow.normFeatContext, h0, c0, tap_act ? tap_act + (size_t)t * as : 0,
                          tap_logits ? tap_logits + (size_t)t * no : 0);
        } else {
            if (tap_act) memset(tap_act + (size_t)t * as, 0, as * sizeof(int16_t));
            if (tap_logits) memset(tap_logits + (size_t)t * no, 0, no * sizeof(int32_t));
        }
        int16_t trig = NNSPClass_exec(&d->inst, frame);
        if (results) { results[t].trigger = trig; for (i = 0; i < 3; i++) results[t].outputs[i] = d->inst.outputs[i]; }
        if (tap_logmel) memcpy(tap_logmel + (size_t)t * 40, d->feat.feature, 40 * sizeof(int32_t));
        if (tap_feat) memcpy(tap_feat + (size_t)t * 40, d->feat.normFeatContext + 5 * 40, 40 * sizeof(int16_t));
        if (tap_h || tap_c) {
            save_hc(net, h0, c0);
            if (tap_h) memcpy(tap_h + (size_t)t * hs, h0, hs * sizeof(int16_t));
            if (tap_c) memcpy(tap_c + (size_t)t * hs, c0, hs * sizeof(int32_t));
        }
        if (tap_post) fill_post(tap_post + (size_t)t * 16, &d->inst, ran, d->nn_id);
    }
    return 0;
}

/* ---- one network evaluation on an explicit input and LSTM state (ref_glue.c ref_net_eval) ------------------- */
/* h / c: the state of every LSTM layer back to back (in / out); act = layers 0..L-2, logits = layer L-1. The
 * table's own state arrays are left holding the new state, as NeuralNetClass_exe leaves them. final (may be null)
 * receives the output buffer of the full evaluation as NeuralNetClass_exe wrote it: int32 values after a linear
 * last layer, int16 values otherwise (neural_nets.c:152-167). */
int drv_net_eval(NeuralNetClass *net, const int16_t *input, int16_t *h, int32_t *c, int16_t *act, int32_t *logits,
                 int32_t *final)
{
    int16_t in[512];
    int32_t out[DRV_MAXW];
    if (net->size_layer[0] > 512 || h_stride(net) > DRV_MAXW || net->size_layer[net->numlayers] > DRV_MAXW) return -1;
    memcpy(in, input, net->size_layer[0] * sizeof(int16_t));
    shadow_layers(net, in, h, c, act, logits);
    load_hc(net, h, c);
    NeuralNetClass_exe(net, in, out, -1);
    save_hc(net, h, c);
    if (final) memcpy(final, out, net->size_layer[net->numlayers] * sizeof(int32_t));
    return 0;
}

/* NeuralNetClass_exe as the application calls it */
void drv_net_exe(NeuralNetClass *net, int16_t *input, int32_t *output, int debug_layer)
{
    NeuralNetClass_exe(net, input, output, (int8_t)debug_layer);
}

/* the LSTM state the table's own arrays hold, back to back */
void drv_table_state(const NeuralNetClass *net, int16_t *h, int32_t *c) { save_hc(net, h, c); }

/* ---- the front end on one 480-sample window (ref_glue.c ref_feature_stages) ----------------------------------- */
/* FeatureClass_execute slides dataBuffer by one hop and appends the frame: preload it so that the analysis buffer
 * equals win480. ctx receives normFeatContext (6 rows of 40) after the call; rows 0..4 hold the standardised silence
 * row of FeatureClass_setDefault, slid up by one. */
void drv_feature(const NeuralNetClass *net, const int32_t *mean, const int32_t *stdR, const int16_t *win480,
                 int32_t *logmel, int16_t *ctx)
{
    FeatureClass f;
    int16_t frame[160];
    int i;
    memset(&f, 0, sizeof f);
    FeatureClass_construct(&f, mean, stdR, net->qbit_input[0]);          /* as NNSPClass_init does */
    FeatureClass_setDefault(&f);
    for (i = 0; i < 320; i++) f.state_stftModule.dataBuffer[160 + i] = win480[i];
    memcpy(frame, win480 + 320, sizeof frame);
    FeatureClass_execute(&f, frame);
    memcpy(logmel, f.feature, 40 * sizeof(int32_t));
    memcpy(ctx, f.normFeatContext, 240 * sizeof(int16_t));
}

long long drv_net_bytes(void) { return (long long)sizeof(NeuralNetClass); }
