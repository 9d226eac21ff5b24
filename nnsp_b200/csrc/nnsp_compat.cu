/* nnsp_compat.cu -- the nine legacy ns-nnsp entry points, same signatures, same caller-owned state,
 * computed on the GPU (batch of one). This is the literal drop-in boundary: code written against
 * nn_speech.h / feature_module.h / neural_nets.h -- including the reference's own controllers
 * evb/src/nnCntrlClass.c and s2iCntrlClass.c -- links against libnnsp_b200.so unchanged.
 *
 *   NNSPClass_init / _reset / _exec ............ ns-nnsp/src/nn_speech.c:23-127
 *   FeatureClass_construct / _setDefault / _execute ... ns-nnsp/src/feature_module.c:12-75
 *   NeuralNetClass_init / _setDefault / _exe ... ns-nnsp/src/neural_nets.c:22-168
 *
 * State stays where the reference keeps it (the caller's structs and the model table's h/c arrays);
 * each call ships the needed state to the device, runs ONE kernel built from the same device functions
 * as the batched engine (frame_logmel, net_forward, post_*), and writes the new state back. One launch
 * and two small copies per call: this path is for compatibility and parity, the batched API is for speed.
 * The legacy functions have no error channel; on a CUDA failure they print the error and abort()
 * (there is no CPU fallback to fall back to). */
#include <cuda_runtime.h>
#include <map>
#include <mutex>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "nnsp_compat/nnsp_legacy_api.h"
#include "nnsp_feat.cuh"
#include "nnsp_host.h"
#include "nnsp_net.cuh"

namespace nnsp {

enum { LG_FEATURE = 1, LG_NET = 2, LG_POST = 4 };

struct LegacyIO {
    /* in */
    int      mode, nn_id, numlayers_run, rshift;
    int16_t  thresh_prob, th_count, pad0, pad1;
    int32_t  mean[40], stdR[40];
    alignas(16) int16_t win[480];          /* stftModule.dataBuffer after the slide (spectrogram_module.c:55-60) */
    /* in/out */
    alignas(16) int16_t ctx[240];          /* FeatureClass.normFeatContext, already slid by one row          */
    int16_t  h[NNSP_B200_MAX_WIDTH];
    int32_t  c[NNSP_B200_MAX_WIDTH];
    int16_t  scal[SC_N];
    /* out */
    int32_t  logmel[40];
    int16_t  act[4 * NNSP_B200_MAX_WIDTH * 3];
    int32_t  logits[NNSP_B200_MAX_WIDTH];
};

struct LegacySmem {
    FeatSmemTables ft;
    FrameScratch fs;
    WarpScratch ws;
    int16_t tanh_lut[384];
    DevModel model;
};

/* one warp: optional front end, optional network (weights read straight from global memory), optional
 * post-processing */
__global__ void __launch_bounds__(32) legacy_kernel(LegacyIO *io, const DevTables *__restrict__ tables,
                                                    const DevModel *__restrict__ model, const uint32_t *__restrict__ wimg,
                                                    const int16_t *__restrict__ bimg)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    LegacySmem &sm = *reinterpret_cast<LegacySmem *>(smem_raw);
    const int lane = threadIdx.x;
    const int mode = io->mode;
    load_feat_tables(&sm.ft, tables, lane, 32);
    for (int i = lane; i < 384; i += 32) sm.tanh_lut[i] = tables->tanh_lut[i];
    if (model) {
        const int *src = reinterpret_cast<const int *>(model);
        int *dst = reinterpret_cast<int *>(&sm.model);
        for (int i = lane; i < (int)(sizeof(DevModel) / 4); i += 32) dst[i] = src[i];
    }
    WarpScratch *ws = &sm.ws;
    for (int i = lane; i < 240; i += 32) ws->ctx[i] = io->ctx[i];
    for (int i = lane; i < NNSP_B200_MAX_WIDTH; i += 32) { ws->h[i] = io->h[i]; ws->c[i] = io->c[i]; }
    if (lane < SC_N) ws->scal[lane] = io->scal[lane];
    __syncwarp();
    if (mode & LG_FEATURE) {
        const int16_t *w = io->win;
        auto load_pair = [&](int, int p) -> uint32_t { return *reinterpret_cast<const unsigned int *>(w + 2 * p); };
        frame_logmel<false>(sm.ft, sm.fs, lane & 15, load_pair, io->logmel, lane < 16, FeatDump{});
        __syncwarp();
        __threadfence_block();
        const int32_t lm0 = io->logmel[lane], lm1 = (lane < 8) ? io->logmel[32 + lane] : 0;
        ws->ctx[200 + lane] = standardise(lm0, io->mean[lane], io->stdR[lane], io->rshift);            /* feature_module.c:67-73 */
        if (lane < 8) ws->ctx[232 + lane] = standardise(lm1, io->mean[32 + lane], io->stdR[32 + lane], io->rshift);
        __syncwarp();
    }
    if ((mode & LG_NET) && model) {
        DevModel &M = sm.model;
        M.numlayers = io->numlayers_run;                      /* debug_layer tap: run only the first k layers (neural_nets.c:65) */
        __syncwarp();
        net_forward(M, wimg, bimg, sm.tanh_lut, ws, lane, io->act, io->logits);
        if ((mode & LG_POST) && lane == 0) {
            if (io->nn_id == NNSP_B200_ID_S2I) post_s2i(ws->scal, ws->logits, io->th_count);            /* nn_speech.c:97-119 */
            else if (io->nn_id == NNSP_B200_ID_VAD || io->nn_id == NNSP_B200_ID_KWS) post_binary(ws->scal, ws->logits, io->thresh_prob, io->th_count);
        }
        __syncwarp();
    }
    for (int i = lane; i < 240; i += 32) io->ctx[i] = ws->ctx[i];
    for (int i = lane; i < NNSP_B200_MAX_WIDTH; i += 32) { io->h[i] = ws->h[i]; io->c[i] = ws->c[i]; }
    if (lane < SC_N) io->scal[lane] = ws->scal[lane];
}

/* an uploaded model and the bytes of the NeuralNetClass it was built from */
struct LegacyModel {
    NeuralNetClass net;
    DeviceModel *dm;
};

struct LegacyCtx {
    int device = 0;
    bool ready = false;
    const DevTables *tables = nullptr;
    LegacyIO *h_io = nullptr, *d_io = nullptr;
    cudaStream_t stream = nullptr;
    std::map<const void *, LegacyModel> models;            /* keyed by NeuralNetClass* */
};
static LegacyCtx g_lg;
static std::mutex g_lg_mu;

static void legacy_die(const char *what)
{
    fprintf(stderr, "nnsp-b200: %s failed: %s\nnnsp-b200 has no CPU fallback; aborting.\n", what, nnsp_b200_last_error());
    abort();
}

static void legacy_init()
{
    if (g_lg.ready) return;
    const char *dev = getenv("NNSP_B200_DEVICE");
    g_lg.device = dev ? atoi(dev) : 0;
    if (select_device(g_lg.device)) legacy_die("select_device");
    if (get_device_tables(g_lg.device, &g_lg.tables)) legacy_die("constant tables");
    if (cudaMallocHost(&g_lg.h_io, sizeof(LegacyIO)) != cudaSuccess || cudaMalloc(&g_lg.d_io, sizeof(LegacyIO)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&g_lg.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaFuncSetAttribute(legacy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LegacySmem)) != cudaSuccess) {
        nnsp_set_error("%s", cudaGetErrorString(cudaGetLastError()));
        legacy_die("legacy context allocation");
    }
    memset(g_lg.h_io, 0, sizeof(LegacyIO));
    g_lg.ready = true;
}

/* The reference reads the NeuralNetClass on every call, so an application may fill one struct with another table
 * between calls. The cached upload is reused only while the struct's bytes are the ones it was built from; tables
 * rewritten in place behind unchanged pointers are not detected. The first call on a struct builds the entry: from
 * NeuralNetClass_exe with nn_id -1 and zero statistics, which legacy_kernel never reads (LegacyIO carries them). */
static DeviceModel *legacy_model(const NeuralNetClass *net, const int32_t *mean, const int32_t *stdR, int nn_id)
{
    auto it = g_lg.models.find(net);
    if (it != g_lg.models.end()) {
        if (!memcmp(&it->second.net, net, sizeof *net)) return it->second.dm;
        cudaSetDevice(g_lg.device);
        free_model(it->second.dm);
        delete it->second.dm;
        g_lg.models.erase(it);
    }
    static const int32_t zeros[40] = { 0 };
    nnsp_b200_model *m = nullptr;
    if (nnsp_b200_model_from_net(net, mean ? mean : zeros, stdR ? stdR : zeros, nn_id, &m)) legacy_die("nnsp_b200_model_from_net");
    DeviceModel *dm = new DeviceModel();
    cudaSetDevice(g_lg.device);
    if (upload_model(m, dm) || cudaDeviceSynchronize() != cudaSuccess) legacy_die("model upload");
    nnsp_b200_model_free(m);
    LegacyModel &e = g_lg.models[net];
    memcpy(&e.net, net, sizeof e.net);
    e.dm = dm;
    return dm;
}

static void legacy_run(const DeviceModel *dm)
{
    cudaSetDevice(g_lg.device);
    cudaError_t e = cudaMemcpyAsync(g_lg.d_io, g_lg.h_io, sizeof(LegacyIO), cudaMemcpyHostToDevice, g_lg.stream);
    if (e == cudaSuccess) {
        legacy_kernel<<<1, 32, sizeof(LegacySmem), g_lg.stream>>>(g_lg.d_io, g_lg.tables, dm ? dm->d : nullptr,
                                                                 dm ? dm->wimg : nullptr, dm ? dm->bimg : nullptr);
        g_launches.fetch_add(1);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(g_lg.h_io, g_lg.d_io, sizeof(LegacyIO), cudaMemcpyDeviceToHost, g_lg.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g_lg.stream);
    if (e != cudaSuccess) { nnsp_set_error("%s", cudaGetErrorString(e)); legacy_die("legacy kernel"); }
}

/* h/c of every lstm layer, back to back, between the table's arrays and the IO block */
static void gather_hc(const NeuralNetClass *n, LegacyIO *io)
{
    int o = 0;
    for (int i = 0; i < n->numlayers; i++)
        if (n->net_layer_type[i] == lstm)
            for (int j = 0; j < n->size_layer[i + 1] && o < NNSP_B200_MAX_WIDTH; j++, o++) { io->h[o] = n->pt_hstate[i][j]; io->c[o] = n->pt_cstate[i][j]; }
}
static void scatter_hc(NeuralNetClass *n, const LegacyIO *io, int layers_run)
{
    int o = 0;
    for (int i = 0; i < n->numlayers; i++)
        if (n->net_layer_type[i] == lstm)
            for (int j = 0; j < n->size_layer[i + 1] && o < NNSP_B200_MAX_WIDTH; j++, o++)
                if (i < layers_run) { n->pt_hstate[i][j] = io->h[o]; n->pt_cstate[i][j] = io->c[o]; }
}

}  // namespace nnsp

using namespace nnsp;

extern "C" {

/* ---- FeatureClass -------------------------------------------------------------------------------- */
void FeatureClass_construct(FeatureClass *ps, const int32_t *norm_mean, const int32_t *norm_stdR, int8_t qbit_output)
{
    const nnsp_tables *t = nnsp_tables_get();
    if (!t) { nnsp_set_error("constant-table self check failed"); legacy_die("FeatureClass_construct"); }
    ps->state_stftModule.len_win = LEN_STFT_WIN_COEFF;     /* stftModule_construct, spectrogram_module.c:14-24 */
    ps->state_stftModule.hop = LEN_STFT_HOP;
    ps->state_stftModule.len_fft = LEN_FFT_NNSP;
    ps->state_stftModule.window = t->stft_win;
    ps->pt_norm_mean = norm_mean;
    ps->pt_norm_stdR = norm_stdR;
    ps->num_context = NUM_FEATURE_CONTEXT;
    ps->dim_feat = DIMEMSION_FEATURE;
    ps->qbit_output = qbit_output;
}

/* State initialisation only (no signal processing): zero the analysis buffer, pre-fill context rows 0..4
 * with the standardised log10(2^-15) row; row 5 is left as it is, exactly like feature_module.c:26-45. */
void FeatureClass_setDefault(FeatureClass *ps)
{
    for (int i = 0; i < ps->state_stftModule.len_win; i++) ps->state_stftModule.dataBuffer[i] = 0;
    for (int i = 0; i < ps->dim_feat; i++) {
        int64_t t = ((int64_t)-147963 - (int64_t)ps->pt_norm_mean[i]) * (int64_t)ps->pt_norm_stdR[i];
        t >>= (30 - ps->qbit_output);
        t = t > 32767 ? 32767 : (t < -32768 ? -32768 : t);
        for (int j = 0; j < ps->num_context - 1; j++) ps->normFeatContext[i + j * ps->dim_feat] = (int16_t)t;
    }
}

static void legacy_stage_feature(FeatureClass *ps, const int16_t *input, LegacyIO *io)
{
    /* slide the caller's buffers (data movement), then hand the window and context to the device */
    int16_t *db = ps->state_stftModule.dataBuffer;
    memmove(db, db + LEN_STFT_HOP, (LEN_STFT_WIN_COEFF - LEN_STFT_HOP) * sizeof(int16_t));
    memcpy(db + LEN_STFT_WIN_COEFF - LEN_STFT_HOP, input, LEN_STFT_HOP * sizeof(int16_t));
    for (int r = 0; r < 5; r++) memmove(ps->normFeatContext + r * 40, ps->normFeatContext + (r + 1) * 40, 40 * sizeof(int16_t));
    memcpy(io->win, db, sizeof io->win);
    memcpy(io->ctx, ps->normFeatContext, sizeof io->ctx);
    memcpy(io->mean, ps->pt_norm_mean, sizeof io->mean);
    memcpy(io->stdR, ps->pt_norm_stdR, sizeof io->stdR);
    io->rshift = 30 - ps->qbit_output;
}

void FeatureClass_execute(FeatureClass *ps, int16_t *input)
{
    std::lock_guard<std::mutex> lk(g_lg_mu);
    legacy_init();
    LegacyIO *io = g_lg.h_io;
    io->mode = LG_FEATURE;
    legacy_stage_feature(ps, input, io);
    legacy_run(nullptr);
    memcpy(ps->normFeatContext, io->ctx, sizeof io->ctx);
    memcpy(ps->feature, io->logmel, sizeof io->logmel);
}

/* ---- NeuralNetClass ------------------------------------------------------------------------------- */
void NeuralNetClass_init(NeuralNetClass *pt_inst) { (void)pt_inst; }       /* neural_nets.c:22-25 is empty too */

void NeuralNetClass_setDefault(NeuralNetClass *pt_inst)                    /* neural_nets.c:27-42: state initialisation */
{
    for (int i = 0; i < pt_inst->numlayers; i++)
        if (pt_inst->net_layer_type[i] == lstm)
            for (int j = 0; j < pt_inst->size_layer[i + 1]; j++) { pt_inst->pt_cstate[i][j] = 0; pt_inst->pt_hstate[i][j] = 0; }
}

static void legacy_net_outputs(const NeuralNetClass *n, const LegacyIO *io, int layers, int32_t *output)
{
    const int rows = n->size_layer[layers];
    /* activation_type decides int32 vs int16 copy-out, like neural_nets.c:152-167 */
    if (n->activation_type[layers - 1] == linear) memcpy(output, io->logits, (size_t)rows * sizeof(int32_t));
    else { int16_t *o16 = (int16_t *)output; for (int j = 0; j < rows; j++) o16[j] = (int16_t)io->logits[j]; }
}

void NeuralNetClass_exe(NeuralNetClass *pt_inst, int16_t *input, int32_t *output, int8_t debug_layer)
{
    const int layers = (debug_layer < 0) ? pt_inst->numlayers : debug_layer;
    if (layers == 0) {                                                    /* neural_nets.c:85-91 */
        memcpy(output, input, (size_t)pt_inst->size_layer[0] * sizeof(int16_t));
        return;
    }
    std::lock_guard<std::mutex> lk(g_lg_mu);
    legacy_init();
    DeviceModel *dm = legacy_model(pt_inst, nullptr, nullptr, -1);
    LegacyIO *io = g_lg.h_io;
    io->mode = LG_NET;
    io->nn_id = -1;
    io->numlayers_run = layers;
    memcpy(io->ctx, input, sizeof io->ctx);
    gather_hc(pt_inst, io);
    legacy_run(dm);
    scatter_hc(pt_inst, io, layers);
    legacy_net_outputs(pt_inst, io, layers, output);
}

/* ---- NNSPClass -------------------------------------------------------------------------------------- */
int NNSPClass_init(NNSPClass *pt_inst, void *pt_net, void *pt_feat, char nn_id, const int32_t *pt_mean,
                   const int32_t *pt_stdR, int16_t *pt_thresh_prob, int16_t *pt_th_count_trigger)
{
    pt_inst->nn_id = nn_id;
    pt_inst->pt_feat = pt_feat;
    pt_inst->pt_net = pt_net;
    FeatureClass_construct((FeatureClass *)pt_feat, pt_mean, pt_stdR, ((NeuralNetClass *)pt_net)->qbit_input[0]);
    pt_inst->num_dnsmpl = 2;
    pt_inst->pt_thresh_prob = pt_thresh_prob;
    pt_inst->pt_th_count_trigger = pt_th_count_trigger;
    NeuralNetClass_init((NeuralNetClass *)pt_net);
    return 0;
}

int NNSPClass_reset(NNSPClass *pt_inst)                                   /* nn_speech.c:57-72 */
{
    FeatureClass_setDefault((FeatureClass *)pt_inst->pt_feat);
    NeuralNetClass_setDefault((NeuralNetClass *)pt_inst->pt_net);
    pt_inst->slides = 1;
    pt_inst->trigger = 0;
    for (int i = 0; i < DIM_INTENTS; i++) pt_inst->counts_category[i] = 0;
    for (int i = 0; i < 3; i++) pt_inst->outputs[i] = 0;
    pt_inst->argmax_last = 0;
    return 0;
}

int16_t NNSPClass_exec(NNSPClass *pt_inst, int16_t *rawPCM)               /* nn_speech.c:74-127, one fused launch */
{
    std::lock_guard<std::mutex> lk(g_lg_mu);
    legacy_init();
    FeatureClass *feat = (FeatureClass *)pt_inst->pt_feat;
    NeuralNetClass *net = (NeuralNetClass *)pt_inst->pt_net;
    DeviceModel *dm = legacy_model(net, feat->pt_norm_mean, feat->pt_norm_stdR, pt_inst->nn_id);
    LegacyIO *io = g_lg.h_io;
    const bool run_nn = (pt_inst->slides == 1);
    io->mode = LG_FEATURE | (run_nn ? (LG_NET | LG_POST) : 0);
    io->nn_id = pt_inst->nn_id;
    io->numlayers_run = net->numlayers;
    io->thresh_prob = *pt_inst->pt_thresh_prob;
    io->th_count = *pt_inst->pt_th_count_trigger;
    legacy_stage_feature(feat, rawPCM, io);
    gather_hc(net, io);
    io->scal[SC_TRIGGER] = pt_inst->trigger;
    for (int i = 0; i < 3; i++) io->scal[SC_OUT0 + i] = pt_inst->outputs[i];
    for (int i = 0; i < 8; i++) io->scal[SC_CNT0 + i] = pt_inst->counts_category[i];
    io->scal[SC_ARGMAX_LAST] = pt_inst->argmax_last;
    io->scal[SC_SLIDES] = pt_inst->slides;
    legacy_run(dm);
    memcpy(feat->normFeatContext, io->ctx, sizeof io->ctx);
    memcpy(feat->feature, io->logmel, sizeof io->logmel);
    if (run_nn) {
        scatter_hc(net, io, net->numlayers);
        pt_inst->trigger = io->scal[SC_TRIGGER];
        for (int i = 0; i < 3; i++) pt_inst->outputs[i] = io->scal[SC_OUT0 + i];
        for (int i = 0; i < 8; i++) pt_inst->counts_category[i] = io->scal[SC_CNT0 + i];
        pt_inst->argmax_last = io->scal[SC_ARGMAX_LAST];
    }
    pt_inst->slides = (int8_t)((pt_inst->slides + 1) % 2);                /* nn_speech.c:125 */
    return pt_inst->trigger;
}

}  /* extern "C" */
