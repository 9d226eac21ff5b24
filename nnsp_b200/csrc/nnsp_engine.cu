/* nnsp_engine.cu -- kernels and host driver of the batched NNSPClass path.
 *
 * Two kernels per exec call:
 *   feat_kernel : log-mel of every (stream, frame) of the call; frames are independent, so the
 *                 grid covers S*T frames with one half-warp each (nnsp_feat.cuh); it also writes
 *                 the last two PCM frames into the next call's history, for its windows
 *   nn_kernel   : per stream (one warp), the T frames in order: standardise the new row into
 *                 the 6x40 context, every 2nd frame run the network and the post-processing,
 *                 update the NNSPClass scalars and LSTM state (nnsp_net.cuh)
 * sm_100a only; no CPU path exists. */
#include <cuda_runtime.h>
#include <mutex>
#include <new>
#include <stdlib.h>
#include <string.h>
#include <utility>

#include "nnsp_feat.cuh"
#include "nnsp_host.h"
#include "nnsp_net.cuh"
#include "nnsp_tma.cuh"

namespace nnsp {

std::atomic<long long> g_launches{0}, g_tc5_launches{0};
std::atomic<long long> g_cascade_net_launches[3] = {};
std::atomic<long long> g_scan_launches[6] = {};

/* ======================================================================================== */
/* device bookkeeping                                                                         */
/* ======================================================================================== */
static std::mutex g_mu;
static DevTables *g_dev_tables[64] = { nullptr };
static int g_sm_count[64] = { 0 };

int select_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        nnsp_set_error("no CUDA device available (%s); nnsp-b200 has no CPU fallback", cudaGetErrorString(e));
        return NNSP_B200_ERR_CUDA;
    }
    if (device < 0 || device >= n || device >= 64) { nnsp_set_error("device %d out of range (have %d)", device, n); return NNSP_B200_ERR_ARG; }
    NNSP_CUDA(cudaSetDevice(device));
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_sm_count[device]) {
        cudaDeviceProp p;
        NNSP_CUDA(cudaGetDeviceProperties(&p, device));
        if (p.major < 10) {
            nnsp_set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, p.major, p.minor);
            return NNSP_B200_ERR_CUDA;
        }
        g_sm_count[device] = p.multiProcessorCount;
    }
    return NNSP_B200_OK;
}
int sm_count(int device) { return g_sm_count[device] ? g_sm_count[device] : 148; }

static bool fill_dev_tables(const nnsp_tables *t, DevTables *d)
{
    bool ok = true;
    memset(d, 0, sizeof *d);
    for (int p = 0; p < 240; p++) d->win2[p] = make_int2((int)t->stft_win[2 * p], (int)t->stft_win[2 * p + 1]);
    auto unpack = [](int32_t w) { return make_int2((int)(int16_t)(w & 0xffff), (int)(w >> 16)); };   /* COMPLEX16: lo = re, hi = im */
    for (int a = 0; a < 4; a++)
        for (int n = 0; n < 3; n++)
            for (int L = 0; L < 16; L++) d->tw0[a][n][L] = unpack(t->fft_tw[4 * (L + 16 * a) + 1 + n]);
    for (int n = 0; n < 3; n++)
        for (int L = 0; L < 16; L++) d->tw1[n][L] = unpack(t->fft_tw[16 * L + 1 + n]);
    for (int m = 0; m < 4; m++)
        for (int n = 0; n < 3; n++) d->tw2[m][n] = unpack(t->fft_tw[64 * m + 1 + n]);
    {   /* the shapes frame_logmel compiles in for stage 2 (nnsp_feat.cuh, cmul_tw) */
        auto one = [](int2 w) { return w.x == 0x7fff && w.y == 0; };
        auto diag = [](int2 w) { return w.x == w.y; };
        auto adiag = [](int2 w) { return w.y == -(w.x + 1); };
        if (!(one(d->tw2[0][0]) && one(d->tw2[0][1]) && one(d->tw2[0][2]) && adiag(d->tw2[1][0]) &&
              d->tw2[2][0].x == 0 && d->tw2[2][0].y == -32768 && adiag(d->tw2[2][1]) && diag(d->tw2[2][2]) && diag(d->tw2[3][0])))
            ok = false;
    }
    for (int k = 0; k < 256; k++) d->rtw[k] = unpack(t->rfft_tw[k]);
    d->rtw[256] = make_int2(0, 0);
    {   /* regroup the filterbank: per band, aligned groups of 4 bins with zero taps outside [start, end] */
        int g = 0;
        for (int b = 0; b < 40; b++) {
            const int s0 = t->mel_start[b], e0 = t->mel_end[b], bin0 = s0 & ~3, ng = ((e0 | 3) - bin0 + 1) / 4;
            d->mel_meta[b] = (uint32_t)g | ((uint32_t)ng << 8) | ((uint32_t)bin0 << 16);
            if (ng > (b >= 24 ? MEL_MAXG0 : (b >= 8 ? MEL_MAXG1 : MEL_MAXG2)) || g + ng > MEL_GROUPS) ok = false;
            for (int i = 0; i < ng; i++, g++) {
                int w[4];
                for (int k = 0; k < 4; k++) {
                    const int bin = bin0 + 4 * i + k;
                    w[k] = (bin >= s0 && bin <= e0) ? (int)t->mel_taps[t->mel_off[b] + bin - s0] : 0;
                }
                if (g < MEL_GROUPS) d->mel_tap4[g] = make_int4(w[0], w[1], w[2], w[3]);
            }
        }
    }
    memcpy(d->log_lut, t->log_lut, sizeof d->log_lut);
    memcpy(d->tanh_lut, t->tanh_lut, sizeof d->tanh_lut);
    /* the folded tanh table: half-segments of 512 (the original segments start at 512 + 1024 k, the clamp region is
     * [0, 512), the saturation starts at 320 * 512), slope = the segment's, constant = any value of the interval that
     * makes all 512 points of the half-segment exact. An empty interval would mean coeffs_tanh is not the table this
     * was derived for: refuse to run rather than approximate. */
    auto tanh_def = [&](int64_t xi) -> int64_t {                 /* activation.c:31-69 for xi = |x| */
        if (xi >= (5 << 15)) return 0x7fff;
        int64_t kx = (xi - 512) >> 10;
        kx = kx < 0 ? 0 : kx;
        const int64_t v = (int64_t)t->tanh_lut[2 * kx] + (((xi - 512 - (kx << 10)) * (int64_t)t->tanh_lut[2 * kx + 1]) >> 15);
        return v > 0 ? v : 0;
    };
    for (int w = 0; w < 320; w++) {
        const int64_t k = w >= 1 ? (w - 1) >> 1 : 0, s = t->tanh_lut[2 * k + 1];
        int64_t lo = INT64_MIN, hi = INT64_MAX;
        for (int64_t dd = 0; dd < 512; dd++) {
            const int64_t y = tanh_def(512 * w + dd);
            lo = std::max(lo, y * 32768 - dd * s);
            hi = std::min(hi, (y + 1) * 32768 - dd * s);
        }
        if (lo >= hi || lo < 0 || lo + 511 * s > INT32_MAX) ok = false;
        d->tanh2[w] = make_int2((int)s, (int)lo);
    }
    d->tanh2[320] = make_int2(0, 0x7fff << 15);
    for (int64_t xi = 0; xi < (5 << 15) + 2048 && ok; xi++) {
        const int64_t w = std::min<int64_t>(xi >> 9, 320), dd = xi - (w << 9);
        if (((dd * d->tanh2[w].x + d->tanh2[w].y) >> 15) != tanh_def(xi)) ok = false;
    }
    return ok;
}

int get_device_tables(int device, const DevTables **out)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_dev_tables[device]) {
        const nnsp_tables *t = nnsp_tables_get();
        if (!t) { nnsp_set_error("constant-table self check failed (fingerprint mismatch)"); return NNSP_B200_ERR_ARG; }
        DevTables h;
        if (!fill_dev_tables(t, &h)) { nnsp_set_error("constant tables do not have the structure the kernels compile in (mel group bounds, stage-2 twiddles, folded tanh table)"); return NNSP_B200_ERR_ARG; }
        DevTables *d = nullptr;
        NNSP_CUDA(cudaMalloc(&d, sizeof h));
        NNSP_CUDA(cudaMemcpy(d, &h, sizeof h, cudaMemcpyHostToDevice));
        NNSP_CUDA(cudaDeviceSynchronize());      /* pageable source: returned once staged; the engine's streams are non-blocking */
        g_dev_tables[device] = d;
    }
    *out = g_dev_tables[device];
    return NNSP_B200_OK;
}

/* ---- model upload: canonical row-major int8 -> K-major packed words ----------------------- */
static void pack_matrix(uint32_t *dst, const int8_t *w, int nrows, int nrows_pad, int cols, int k4)
{
    for (int k = 0; k < k4; k++)
        for (int r = 0; r < nrows_pad; r++) {
            uint32_t word = 0;
            for (int b = 0; b < 4; b++) {
                const int c = 4 * k + b;
                const uint8_t v = (r < nrows && c < cols) ? (uint8_t)w[(size_t)r * cols + c] : 0;
                word |= (uint32_t)v << (8 * b);
            }
            dst[(size_t)k * nrows_pad + r] = word;
        }
}

int upload_model(const nnsp_b200_model *m, DeviceModel *out)
{
    DevModel &D = out->h;
    memset(&D, 0, sizeof D);
    D.nn_id = m->nn_id;
    D.numlayers = m->numlayers;
    D.n_out = m->size_layer[m->numlayers];
    D.feat_rshift = 30 - m->layer[0].qi;
    memcpy(D.mean, m->mean, sizeof D.mean);
    memcpy(D.stdR, m->stdR, sizeof D.stdR);
    for (int i = 0; i < 40; i++) {          /* feature_module.c:32-37, LOG10_2POW_N15_Q15 = -147963 (:9) */
        int64_t t = ((int64_t)-147963 - (int64_t)m->mean[i]) * (int64_t)m->stdR[i];
        t >>= D.feat_rshift;
        t = t > 32767 ? 32767 : (t < -32768 ? -32768 : t);
        D.silence[i] = (int16_t)t;
    }
    int woff = 0, boff = 0;
    for (int i = 0; i < m->numlayers; i++) {
        const nnsp_layer &L = m->layer[i];
        DevLayer &G = D.layer[i];
        G.type = L.type; G.act = L.act; G.rows = L.rows; G.cols = L.cols; G.acc32 = L.acc32;
        G.nrows = (L.type == NNSP_LAYER_LSTM) ? 4 * L.rows : L.rows;
        G.nrows_pad = (G.nrows + 31) & ~31;
        G.k4 = (L.cols + 3) / 4;
        G.k4rec = (L.type == NNSP_LAYER_LSTM) ? (L.rows + 3) / 4 : 0;
        /* the affine that produces the output: for lstm it is the recurrent half, whose input
         * Q-format is qbit_input_rec (affine.c:387-393) */
        const int qi_out = (L.type == NNSP_LAYER_LSTM) ? L.qi_next : L.qi;
        const int qs = (qi_out + L.qk) > 15 ? (qi_out + L.qk) : 15;     /* affine.c:69-72 (bias present) */
        G.sh_x = (L.type == NNSP_LAYER_LSTM) ? (L.qi_next - L.qi) : 0;
        G.sh_bias = qs - L.qb;
        G.sh_out = 15 - qs;
        G.w_off = woff; woff += G.k4 * G.nrows_pad;
        G.wrec_off = woff; woff += G.k4rec * G.nrows_pad;
        G.bias_off = boff; boff += G.nrows_pad;
        if (i < m->numlayers - 1) D.act_stride += L.rows;
        if (L.type == NNSP_LAYER_LSTM) D.h_stride += L.rows;
        if (L.cols > 480) { nnsp_set_error("layer %d: %d inputs exceed the exact-int32 dot-product bound (480)", i, L.cols); return NNSP_B200_ERR_UNSUPPORTED; }
    }
    if (D.h_stride > NNSP_B200_MAX_WIDTH) { nnsp_set_error("total LSTM state %d exceeds %d", D.h_stride, NNSP_B200_MAX_WIDTH); return NNSP_B200_ERR_UNSUPPORTED; }
    D.weight_words = (woff + 3) & ~3;      /* 16-byte multiple for the bulk copy */
    D.bias_count = (boff + 7) & ~7;
    uint32_t *hw = (uint32_t *)calloc((size_t)D.weight_words + 4, 4);
    int16_t *hb = (int16_t *)calloc((size_t)D.bias_count + 8, 2);
    if (!hw || !hb) { free(hw); free(hb); return NNSP_B200_ERR_NOMEM; }
    for (int i = 0; i < m->numlayers; i++) {
        const nnsp_layer &L = m->layer[i];
        const DevLayer &G = D.layer[i];
        pack_matrix(hw + G.w_off, L.w, G.nrows, G.nrows_pad, L.cols, G.k4);
        if (L.type == NNSP_LAYER_LSTM) pack_matrix(hw + G.wrec_off, L.wrec, G.nrows, G.nrows_pad, L.rows, G.k4rec);
        memcpy(hb + G.bias_off, L.bias, (size_t)G.nrows * 2);
    }
    cudaError_t e1 = cudaMalloc(&out->wimg, (size_t)D.weight_words * 4);
    cudaError_t e2 = cudaMalloc(&out->bimg, (size_t)D.bias_count * 2);
    cudaError_t e3 = cudaMalloc(&out->d, sizeof D);
    if (e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess) {
        e1 = cudaMemcpy(out->wimg, hw, (size_t)D.weight_words * 4, cudaMemcpyHostToDevice);
        e2 = cudaMemcpy(out->bimg, hb, (size_t)D.bias_count * 2, cudaMemcpyHostToDevice);
        e3 = cudaMemcpy(out->d, &D, sizeof D, cudaMemcpyHostToDevice);
    }
    free(hw);
    free(hb);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
        nnsp_set_error("model upload failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
        free_model(out);
        return NNSP_B200_ERR_CUDA;
    }
    return NNSP_B200_OK;
}

void free_model(DeviceModel *dm)
{
    if (dm->wimg) cudaFree(dm->wimg);
    if (dm->bimg) cudaFree(dm->bimg);
    if (dm->d) cudaFree(dm->d);
    dm->wimg = nullptr; dm->bimg = nullptr; dm->d = nullptr;
}

/* ======================================================================================== */
/* feature kernel                                                                             */
/* ======================================================================================== */
#ifndef FEAT_WARPS_PER_CTA
#define FEAT_WARPS_PER_CTA 8
#endif
constexpr int FEAT_WARPS = FEAT_WARPS_PER_CTA;   /* two frames in flight per warp */
constexpr int FEAT_THREADS = FEAT_WARPS * 32;
#ifndef FEAT_CTAS_PER_SM
#define FEAT_CTAS_PER_SM 3
#endif
#ifndef FEAT_ITERS
#define FEAT_ITERS 8
#endif

struct FeatSmem {
    FeatSmemTables tb;
    FrameScratch fs[FEAT_WARPS * 2];
    int32_t norm[84];              /* mean[40], stdR[40], rshift: only when the kernel standardises */
};

/* RAGGED (a ragged cascade call, nfr != null): stream s has stream_frames(nfr, s, T) frames; a later frame reads no PCM
 * and writes no row, and a warp whose two frames are both past their streams' counts skips the pair. The uniform
 * instantiation is the kernel as it was before ragged calls existed, instruction for instruction. */
template <bool RAGGED>
__global__ void __launch_bounds__(FEAT_THREADS, FEAT_CTAS_PER_SM)
feat_kernel(const DevTables *__restrict__ tables, const int16_t *__restrict__ pcm, long long stride,
            const int16_t *__restrict__ hist, int hist_frames, int s0, int ns, int T,
            int32_t *__restrict__ logmel, const int32_t *__restrict__ norm, int16_t *__restrict__ feat16,
            const int32_t *__restrict__ nfr, int16_t *__restrict__ hist_out, const int32_t *__restrict__ lm_hist,
            int32_t *__restrict__ lm_out, int lm_rows)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FeatSmem &sm = *reinterpret_cast<FeatSmem *>(smem_raw);
    load_feat_tables(&sm.tb, tables, threadIdx.x, FEAT_THREADS);
    if (norm && threadIdx.x < 81) sm.norm[threadIdx.x] = norm[threadIdx.x];
    const int32_t *snorm = norm ? sm.norm : nullptr;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, half = lane >> 4, L = lane & 15;
    FrameScratch &fs = sm.fs[warp * 2 + half];
    const long long F = (long long)ns * T;
    const int hist_len = hist_frames * NNSP_B200_FRAME;
    for (long long f0 = ((long long)blockIdx.x * FEAT_WARPS + warp) * 2; f0 < F; f0 += (long long)gridDim.x * FEAT_WARPS * 2) {
        const long long f = f0 + half;
        bool valid = f < F;
        const long long fc = valid ? f : 0;
        const int s = s0 + (int)(fc / T), t = (int)(fc % T);
        const int Ts = RAGGED ? stream_frames(nfr, s, T) : T;               /* frames of stream s in this call */
        if (RAGGED) {
            valid = valid && t < Ts;
            if (!__any_sync(0xffffffffu, valid)) continue;              /* warp-uniform: neither frame is live */
        }
        /* the 480-sample window starts two frames back: word L + 16a of it comes from this call's PCM or, for
         * the first two frames, from the carried history (both 4-byte aligned; immediates after unrolling) */
        const int base = (t - 2) * NNSP_B200_FRAME;                        /* first sample of the window */
        const unsigned int *pw = reinterpret_cast<const unsigned int *>(pcm + (long long)s * stride + base) + L;
        const unsigned int *hw = reinterpret_cast<const unsigned int *>(hist + (long long)s * hist_len + hist_len + base) + L;
        const int pth = (2 - t) * (NNSP_B200_FRAME / 2);                   /* pairs below pth precede the call */
        /* hist_out: a frame among the stream's newest hist_frames also goes into the next call's PCM history, at frame
         * hist_frames - (Ts - t). Its own 160 samples are window words 160..239 (a = 10..14), which always come from this
         * call's PCM. */
        unsigned int *ho = nullptr;
        if (hist_out && valid && t >= Ts - hist_frames)
            ho = reinterpret_cast<unsigned int *>(hist_out + (long long)s * hist_len + hist_len + base - Ts * NNSP_B200_FRAME) + L;
        auto load_pair = [&](int a, int p) -> uint32_t {
            if (RAGGED && !valid) return 0u;
            const uint32_t v = (p < pth) ? __ldg(hw + 16 * a) : __ldg(pw + 16 * a);
            if (a >= 10 && ho) ho[16 * a] = v;
            return v;
        };
        /* lm_out: the same for the log-mel row, into the next call's lm_rows-row log-mel history (row lm_rows - (Ts - t)) */
        int32_t *lo = nullptr;
        if (lm_out && valid && t >= Ts - lm_rows) lo = lm_out + ((long long)s * lm_rows + lm_rows - (Ts - t)) * NNSP_B200_NMEL;
        const long long row = ((long long)s * T + t) * NNSP_B200_NMEL;
        frame_logmel<false>(sm.tb, fs, L, load_pair, logmel + row, valid, FeatDump{}, snorm, feat16 + row, lo);
    }
    /* the frames of an old history that stay among a stream's newest `frames` (it has fewer frames in this call):
     * out frames [0, frames - Ts) <- in frames [Ts, frames), frames of wpf words, a warp per stream */
    auto keep_old = [&](const void *in, void *out, int frames, int wpf) {
        const int words = frames * wpf;
        for (int w = blockIdx.x * FEAT_WARPS + warp; w < ns; w += gridDim.x * FEAT_WARPS) {
            const long long s = s0 + w;
            const int Ts = RAGGED ? stream_frames(nfr, s, T) : T;
            const unsigned int *hi = static_cast<const unsigned int *>(in) + s * words + Ts * wpf;
            unsigned int *ho = static_cast<unsigned int *>(out) + s * words;
            for (int i = lane; i < words - Ts * wpf; i += 32) ho[i] = hi[i];
        }
    };
    if (hist_out && (RAGGED || T < hist_frames)) keep_old(hist, hist_out, hist_frames, NNSP_B200_FRAME / 2);
    if (lm_out && (RAGGED || T < lm_rows)) keep_old(lm_hist, lm_out, lm_rows, NNSP_B200_NMEL);
}

int launch_feature(const DevTables *tb, const FeatLaunch &a, int device, cudaStream_t st)
{
    static bool attr_set[64] = { false };
    static std::mutex attr_mu;                         /* host threads may drive separate handles on one device */
    std::unique_lock<std::mutex> attr_lk(attr_mu);
    if (!attr_set[device]) {
        NNSP_CUDA(cudaFuncSetAttribute(feat_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FeatSmem)));
        NNSP_CUDA(cudaFuncSetAttribute(feat_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FeatSmem)));
        attr_set[device] = true;
    }
    attr_lk.unlock();
    const long long F = (long long)a.ns * a.T;
    if (F <= 0) return NNSP_B200_OK;
    long long blocks = (F + FEAT_WARPS * 2 - 1) / (FEAT_WARPS * 2);
    /* at least one resident wave; beyond that a CTA takes FEAT_ITERS rounds of 16 frames and retires, so that the
     * (higher-priority, latency-bound) network kernels of the previous call find room on every SM while this
     * kernel streams through (the table prologue is ~2 % of such a CTA) */
    const long long cap = (long long)sm_count(device) * FEAT_CTAS_PER_SM;
    /* rounds per CTA: FEAT_ITERS for about eight waves, up to four times that on larger calls (the table prologue
     * amortises further: S2I x 32 768 -0.6 %; 8 is best for the 4 096-stream call) */
    long long iters = blocks / (cap * 8);
    iters = iters < FEAT_ITERS ? FEAT_ITERS : (iters > 4 * FEAT_ITERS ? 4 * FEAT_ITERS : iters);
    static const int iters_env = [] { const char *e = getenv("NNSP_B200_FEAT_ITERS"); return e ? atoi(e) : 0; }();   /* measurement knob */
    if (iters_env > 0) iters = iters_env;
    const long long chunked = (blocks + iters - 1) / iters;
    /* a whole number of resident waves: every CTA slot then runs the same number of CTAs and the slots finish within one
     * round of each other instead of one CTA lifetime (3 200 CTAs on 444 slots left the last wave 20 % full) */
    if (blocks > cap) blocks = chunked > cap ? ((chunked + cap / 2) / cap) * cap : cap;
    static const int pad = [] { const char *e = getenv("NNSP_B200_FEAT_SMEM_PAD"); return e ? atoi(e) : 0; }();   /* measurement knob: fewer resident CTAs */
    if (pad > 0) {
        static bool pad_set[64] = { false };
        if (!pad_set[device]) {
            NNSP_CUDA(cudaFuncSetAttribute(feat_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FeatSmem) + pad));
            NNSP_CUDA(cudaFuncSetAttribute(feat_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FeatSmem) + pad));
            pad_set[device] = true;
        }
    }
    const size_t smem = sizeof(FeatSmem) + (pad > 0 ? pad : 0);
    if (a.nfr)
        feat_kernel<true><<<(unsigned)blocks, FEAT_THREADS, smem, st>>>(tb, a.pcm, a.stride, a.hist, a.hist_frames, a.s0, a.ns, a.T,
                                                                       a.logmel, a.norm, a.feat16, a.nfr, a.hist_out, a.lm_hist, a.lm_out, a.lm_rows);
    else
        feat_kernel<false><<<(unsigned)blocks, FEAT_THREADS, smem, st>>>(tb, a.pcm, a.stride, a.hist, a.hist_frames, a.s0, a.ns, a.T,
                                                                        a.logmel, a.norm, a.feat16, nullptr, a.hist_out, a.lm_hist, a.lm_out, a.lm_rows);
    NNSP_LAUNCH_CHECK();
    return NNSP_B200_OK;
}

/* ======================================================================================== */
/* network + post-processing kernel                                                           */
/* ======================================================================================== */
constexpr int NN_WARPS = 16;
constexpr int NN_THREADS = NN_WARPS * 32;

struct NNArgs {
    const DevModel *model;
    const uint32_t *wimg;
    const int16_t  *bimg;
    const DevTables *tables;
    StreamState st;
    const int32_t *logmel;          /* [S][T][40] */
    int s0, ns, T;
    nnsp_b200_result *results;      /* [S][T] or null */
    nnsp_b200_taps taps;
    int16_t thresh_prob, th_count;
    int raw_ctx;                    /* nnsp_b200_net_eval: the stored context IS the network input (no slide, no new row) */
};

struct NNSmemLayout { size_t bar, w, b, lut, model, scratch, total; };
static inline size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }
static NNSmemLayout nn_layout(const DevModel &D)
{
    NNSmemLayout l;
    l.bar = 0;
    l.w = 16;
    l.b = l.w + (size_t)D.weight_words * 4;
    l.lut = align16(l.b + (size_t)D.bias_count * 2);
    l.model = align16(l.lut + 384 * 2);
    l.scratch = align16(l.model + sizeof(DevModel));
    l.total = l.scratch + sizeof(WarpScratch) * NN_WARPS;
    return l;
}

__global__ void __launch_bounds__(NN_THREADS, 1)
nn_kernel(NNArgs a, int off_b, int off_lut, int off_model, int off_scratch)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    uint32_t *wimg = reinterpret_cast<uint32_t *>(smem_raw + 16);
    int16_t *bimg = reinterpret_cast<int16_t *>(smem_raw + off_b);
    int16_t *lut = reinterpret_cast<int16_t *>(smem_raw + off_lut);
    DevModel &M = *reinterpret_cast<DevModel *>(smem_raw + off_model);
    WarpScratch *wsa = reinterpret_cast<WarpScratch *>(smem_raw + off_scratch);

    {   /* descriptor, bias, LUT by plain loads; the weight image by TMA */
        const int *src = reinterpret_cast<const int *>(a.model);
        int *dst = reinterpret_cast<int *>(&M);
        for (int i = threadIdx.x; i < (int)(sizeof(DevModel) / 4); i += NN_THREADS) dst[i] = src[i];
        for (int i = threadIdx.x; i < 384; i += NN_THREADS) lut[i] = a.tables->tanh_lut[i];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < M.bias_count; i += NN_THREADS) bimg[i] = a.bimg[i];
    tma_stage_weights(wimg, a.wimg, (uint32_t)M.weight_words * 4u, bar);
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpScratch *ws = &wsa[warp];
    const int T = a.T, HS = M.h_stride, AS = M.act_stride, NO = M.n_out;

    for (int si = blockIdx.x * NN_WARPS + warp; si < a.ns; si += gridDim.x * NN_WARPS) {
        const int s = a.s0 + si;
        /* load the stream's state */
        for (int i = lane; i < 240; i += 32) ws->ctx[i] = a.st.ctx[(long long)s * 240 + i];
        for (int i = lane; i < HS; i += 32) { ws->h[i] = a.st.h[(long long)s * HS + i]; ws->c[i] = a.st.c[(long long)s * HS + i]; }
        if (lane < SC_N) ws->scal[lane] = a.st.scal[(long long)s * SC_N + lane];
        __syncwarp();
        const int32_t *lm = a.logmel + (long long)s * T * NNSP_B200_NMEL;
        int32_t lm0 = 0, lm1 = 0;
        if (!a.raw_ctx) { lm0 = lm[lane]; lm1 = (lane < 8) ? lm[32 + lane] : 0; }
        for (int t = 0; t < T; t++) {
            const long long ft = (long long)s * T + t;
            /* FeatureClass_execute tail: slide the context (feature_module.c:54-57), standardise (:67-73) */
            if (!a.raw_ctx) {
                int16_t mv[7];
#pragma unroll
                for (int j = 0; j < 7; j++) { const int i = lane + 32 * j; mv[j] = (i < 200) ? ws->ctx[i + 40] : (int16_t)0; }
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 7; j++) { const int i = lane + 32 * j; if (i < 200) ws->ctx[i] = mv[j]; }
                const int16_t f0 = standardise(lm0, M.mean[lane], M.stdR[lane], M.feat_rshift);
                ws->ctx[200 + lane] = f0;
                int16_t f1 = 0;
                if (lane < 8) { f1 = standardise(lm1, M.mean[32 + lane], M.stdR[32 + lane], M.feat_rshift); ws->ctx[232 + lane] = f1; }
                if (a.taps.logmel) { a.taps.logmel[ft * 40 + lane] = lm0; if (lane < 8) a.taps.logmel[ft * 40 + 32 + lane] = lm1; }
                if (a.taps.feat) { a.taps.feat[ft * 40 + lane] = f0; if (lane < 8) a.taps.feat[ft * 40 + 32 + lane] = f1; }
                if (t + 1 < T) { lm0 = lm[(t + 1) * 40 + lane]; lm1 = (lane < 8) ? lm[(t + 1) * 40 + 32 + lane] : 0; }   /* prefetch */
            }
            __syncwarp();
            const bool ran = (ws->scal[SC_SLIDES] == 1);                                  /* nn_speech.c:84 */
            if (ran) {
                net_forward(M, wimg, bimg, lut, ws, lane,
                            a.taps.act ? a.taps.act + ft * AS : nullptr,
                            a.taps.logits ? a.taps.logits + ft * NO : nullptr);
                if (lane == 0) {
                    if (M.nn_id == NNSP_B200_ID_S2I) post_s2i(ws->scal, ws->logits, a.th_count);   /* nn_speech.c:97-119 */
                    else post_binary(ws->scal, ws->logits, a.thresh_prob, a.th_count);
                }
            } else {
                if (a.taps.act) for (int i = lane; i < AS; i += 32) a.taps.act[ft * AS + i] = 0;
                if (a.taps.logits) for (int i = lane; i < NO; i += 32) a.taps.logits[ft * NO + i] = 0;
            }
            if (lane == 0) {
                ws->scal[SC_SLIDES] = (int16_t)((ws->scal[SC_SLIDES] + 1) % 2);            /* nn_speech.c:125 */
                if (a.results) {
                    nnsp_b200_result r;
                    r.trigger = ws->scal[SC_TRIGGER];
                    r.outputs[0] = ws->scal[SC_OUT0]; r.outputs[1] = ws->scal[SC_OUT0 + 1]; r.outputs[2] = ws->scal[SC_OUT0 + 2];
                    a.results[ft] = r;
                }
            }
            __syncwarp();
            if (a.taps.hstate) for (int i = lane; i < HS; i += 32) a.taps.hstate[ft * HS + i] = ws->h[i];
            if (a.taps.cstate) for (int i = lane; i < HS; i += 32) a.taps.cstate[ft * HS + i] = ws->c[i];
            if (a.taps.post && lane < SC_N) {
                int16_t v = ws->scal[lane];
                if (lane == SC_RAN) v = ran ? 1 : 0;
                if (lane == SC_STAGE) v = (int16_t)M.nn_id;
                a.taps.post[ft * SC_N + lane] = v;
            }
        }
        /* store the stream's state */
        __syncwarp();
        for (int i = lane; i < 240; i += 32) a.st.ctx[(long long)s * 240 + i] = ws->ctx[i];
        for (int i = lane; i < HS; i += 32) { a.st.h[(long long)s * HS + i] = ws->h[i]; a.st.c[(long long)s * HS + i] = ws->c[i]; }
        if (lane < SC_N) a.st.scal[(long long)s * SC_N + lane] = ws->scal[lane];
        __syncwarp();
    }
}

/* NNSPClass_reset for every stream (nn_speech.c:57-72, feature_module.c:26-45, neural_nets.c:27-42) */
__global__ void reset_kernel(const DevModel *__restrict__ M, StreamState st, int S, int hist_words)
{
    const int s = blockIdx.x;
    if (s >= S) return;
    const int HS = M->h_stride;
    /* FeatureClass_setDefault pre-fills rows 0..4 only (feature_module.c:39-42); row 5 keeps whatever the
     * previous activation left there and is shifted into row 4 by the first execute -- reproduced */
    for (int i = threadIdx.x; i < 200; i += blockDim.x) st.ctx[(long long)s * 240 + i] = M->silence[i % 40];
    for (int i = threadIdx.x; i < HS; i += blockDim.x) { st.h[(long long)s * HS + i] = 0; st.c[(long long)s * HS + i] = 0; }
    for (int i = threadIdx.x; i < SC_N; i += blockDim.x) st.scal[(long long)s * SC_N + i] = (i == SC_SLIDES) ? 1 : 0;
    unsigned int *h = reinterpret_cast<unsigned int *>(st.hist) + (long long)s * hist_words;
    for (int i = threadIdx.x; i < hist_words; i += blockDim.x) h[i] = 0;                  /* spectrogram_module.c:25-31 */
}

/* The application's PCM conditioning in front of the path (evb/src/main_nnsp.cc:58-65): the AUDADC delivers one
 * 32-bit word per sample, the 12-bit sample sits in bits 4..15 (`& 0x0000FFF0`, kept as int16), and sample 3 of
 * every 160-sample frame is replaced by the mean of its neighbours (sample-glitch workaround, :61-64).
 * One thread converts 8 samples (two 128-bit loads, one 128-bit store); frames are 20 such groups, so the
 * glitch fix (samples 2, 3, 4) is local to the thread that owns group 0 of a frame. HBM-bound: 6 B per sample. */
__global__ void __launch_bounds__(256) ingest_audadc_kernel(const uint4 *__restrict__ raw, uint4 *__restrict__ pcm, long long n_groups)
{
    for (long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x; gidx < n_groups; gidx += (long long)gridDim.x * blockDim.x) {
        const uint4 a = __ldg(raw + 2 * gidx), b = __ldg(raw + 2 * gidx + 1);
        uint32_t s0 = a.x & 0xfff0u, s1 = a.y & 0xfff0u, s2 = a.z & 0xfff0u, s3 = a.w & 0xfff0u;
        const uint32_t s4 = b.x & 0xfff0u, s5 = b.y & 0xfff0u, s6 = b.z & 0xfff0u, s7 = b.w & 0xfff0u;
        if (gidx % (NNSP_B200_FRAME / 8) == 0)
            s3 = (uint32_t)(((int32_t)(int16_t)s2 + (int32_t)(int16_t)s4) >> 1) & 0xffffu;
        uint4 o;
        o.x = s0 | (s1 << 16); o.y = s2 | (s3 << 16); o.z = s4 | (s5 << 16); o.w = s6 | (s7 << 16);
        pcm[gidx] = o;
    }
}

int launch_ingest(const uint32_t *raw_dev, int16_t *pcm_dev, long long n_frames, int device, cudaStream_t st)
{
    if (n_frames <= 0) return NNSP_B200_OK;
    const long long groups = n_frames * (NNSP_B200_FRAME / 8);
    long long blocks = (groups + 255) / 256;
    const long long cap = (long long)sm_count(device) * 8;
    if (blocks > cap) blocks = cap;
    ingest_audadc_kernel<<<(unsigned)blocks, 256, 0, st>>>((const uint4 *)raw_dev, (uint4 *)pcm_dev, groups);
    NNSP_LAUNCH_CHECK();
    return NNSP_B200_OK;
}

/* integer-pipe peaks: 8 independent register chains per thread, 16 operations per chain-iteration
 *   mode 0: IMAD (32-bit multiply-add)          mode 1: IMAD + independent ALU ops (add / shift / xor), 1:1
 *   mode 2: IMAD.WIDE (32x32 -> 64 accumulate)  mode 3: IDP.2A (two int16 x int8 MACs per instruction) */
__global__ void __launch_bounds__(256) int_peak_kernel(int *sink, int iters, int mode)
{
    int a[8], b[8];
    long long w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { a[i] = threadIdx.x * 7 + i * 13 + blockIdx.x; b[i] = a[i] ^ 0x55; w[i] = a[i]; }
    const int m = (int)threadIdx.x | 1, c = blockIdx.x + 3;
    if (mode == 0) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int i = 0; i < 8; i++) { a[i] = a[i] * m + c; a[i] = a[i] * c + m; }
        }
    } else if (mode == 1) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int i = 0; i < 8; i++) { a[i] = a[i] * m + c; b[i] = (b[i] >> 1) ^ it; }
#pragma unroll
            for (int i = 0; i < 8; i++) { a[i] = a[i] * c + m; b[i] = b[i] + (it | c); }
        }
    } else if (mode == 2) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int i = 0; i < 8; i++) { w[i] += (long long)a[i] * m; w[i] += (long long)b[i] * c; }
        }
    } else {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int i = 0; i < 8; i++) { a[i] = __dp2a_lo(m, c, a[i]); a[i] = __dp2a_hi(c, m, a[i]); }
        }
    }
    int r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r ^= a[i] ^ b[i] ^ (int)w[i] ^ (int)(w[i] >> 32);
    if (r == 0x7fffffff) sink[threadIdx.x] = r;      /* keeps the chains alive, (almost) never stores */
}

/* stage-by-stage tap of the front end (parity tool, nnsp_b200_feature_stages) */
__global__ void __launch_bounds__(FEAT_THREADS)
feat_stages_kernel(const DevTables *__restrict__ tables, const int16_t *__restrict__ windows, int n,
                   int32_t *fft_in, int32_t *spec, int32_t *pspec, int32_t *mel, int32_t *logmel)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FeatSmem &sm = *reinterpret_cast<FeatSmem *>(smem_raw);
    load_feat_tables(&sm.tb, tables, threadIdx.x, FEAT_THREADS);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, half = lane >> 4, L = lane & 15;
    FrameScratch &fs = sm.fs[warp * 2 + half];
    for (int f0 = (blockIdx.x * FEAT_WARPS + warp) * 2; f0 < n; f0 += gridDim.x * FEAT_WARPS * 2) {
        const int f = f0 + half;
        const bool valid = f < n;
        const int fc = valid ? f : 0;
        const int16_t *w = windows + (long long)fc * 480;
        auto load_pair = [&](int a, int p) -> uint32_t { return *reinterpret_cast<const unsigned int *>(w + 2 * p); };
        FeatDump d;
        d.fft_in = fft_in ? fft_in + (long long)fc * 512 : nullptr;
        d.spec = spec ? spec + (long long)fc * 514 : nullptr;
        d.pspec = pspec ? pspec + (long long)fc * 257 : nullptr;
        d.mel = mel ? mel + (long long)fc * 40 : nullptr;
        frame_logmel<true>(sm.tb, fs, L, load_pair, logmel + (long long)fc * 40, valid, d);
    }
}

}  // namespace nnsp

/* ======================================================================================== */
/* C ABI: batched NNSPClass                                                                   */
/* ======================================================================================== */
using namespace nnsp;

#define HOST_RING 4

struct nnsp_b200_batch {
    int device = 0, S = 0;
    cudaStream_t stream = nullptr;          /* device-buffer API */
    cudaStream_t xs[4] = { nullptr, nullptr, nullptr, nullptr };   /* host-buffer API pipeline */
    const DevTables *tables = nullptr;
    DeviceModel dm;
    MmaDeviceModel mm;
    bool mma_ok = false, split_ok = false;
    int nn_path = 0;                        /* 0 auto, 1 dp2a warp-per-stream, 2 IMMA 16-streams-per-warp, 3 scan-split */
    int slides = 1;                         /* host mirror of NNSPClass.slides (nn_speech.c:62,125): uniform over the batch */
    uint8_t *sp_planes[2] = { nullptr, nullptr };  /* scan-split activation planes [tile][inference][hi|lo][16][pa] */
    int32_t *sp_dec = nullptr;              /* decision records [S][inference] */
    long long sp_cap_inf = 0;
    int16_t *feat16[2] = { nullptr, nullptr }; long long feat16_frames = 0;   /* scan-split: standardised rows [S][T][40], double buffered */
    /* device-buffer calls on the scan-split path are pipelined over two CUDA streams: the front end of call N+1
     * (throughput-bound, `stream`) overlaps the latency-bound network kernels of call N (`nn_stream`) */
    cudaStream_t nn_stream = nullptr;
    cudaEvent_t ev_feat[2] = { nullptr, nullptr }, ev_nn[2] = { nullptr, nullptr }, ev_nn0 = nullptr;
    bool nn_pending[2] = { false, false }, last_piped = false;
    unsigned pipe = 0;
    int32_t *norm_dev = nullptr;            /* mean[40], stdR[40], rshift for feat_kernel's standardising mode */
    StreamState st{};
    int16_t *hist2 = nullptr;               /* the next PCM history: every front end writes it, and the two swap after each call */
    int16_t thresh_prob = 0, th_count = 0;
    int32_t *logmel = nullptr; long long logmel_frames = 0;       /* capacity in frames per stream */
    int16_t *d_pcm = nullptr; long long d_pcm_frames = 0;
    nnsp_b200_result *d_res = nullptr; long long d_res_frames = 0;
    NNSmemLayout lay{};
    int nn_ctas_per_sm = 1;
    cudaEvent_t ev[3] = { nullptr, nullptr, nullptr };
    bool ev_valid = false;
    /* asynchronous host-buffer calls: one completion event per pipeline stream, a ring of HOST_RING calls */
    cudaEvent_t host_ev[HOST_RING][4] = {};
    long long host_seq = 0;                 /* ticket of the latest asynchronous host call */
    bool host_inflight = false;
    int host_last_T = 0;                    /* frames per stream of the latest host-buffer call */
    int host_fmt = NNSP_B200_HOST_PCM16;    /* what the host-buffer calls are handed: int16 PCM or raw 32-bit AUDADC words */
    uint32_t *d_raw = nullptr;              /* staging of the raw words, [S][T*160] */
};

static int batch_nn_path(const nnsp_b200_batch *b);

static int batch_ensure_logmel(nnsp_b200_batch *b, int T)
{
    if (batch_nn_path(b) == 3) {                       /* the scan-split path consumes standardised int16 rows */
        if (T <= b->feat16_frames) return NNSP_B200_OK;
        NNSP_CUDA(cudaStreamSynchronize(b->stream)); NNSP_CUDA(cudaStreamSynchronize(b->nn_stream));
        for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
        for (auto &f : b->feat16) { if (f) cudaFree(f); f = nullptr; }
        for (auto &f : b->feat16) NNSP_CUDA(cudaMalloc(&f, (size_t)b->S * T * NNSP_B200_NMEL * sizeof(int16_t)));
        b->feat16_frames = T;
        return NNSP_B200_OK;
    }
    if (T <= b->logmel_frames) return NNSP_B200_OK;
    if (b->logmel) { NNSP_CUDA(cudaStreamSynchronize(b->stream)); for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s)); cudaFree(b->logmel); b->logmel = nullptr; }
    NNSP_CUDA(cudaMalloc(&b->logmel, (size_t)b->S * T * NNSP_B200_NMEL * sizeof(int32_t)));
    b->logmel_frames = T;
    return NNSP_B200_OK;
}

static int batch_nn_path(const nnsp_b200_batch *b)
{
    if (b->nn_path) return b->nn_path;
    return b->split_ok ? 3 : (b->mma_ok ? 2 : 1);
}

/* inference frames of a call of T frames that starts with NNSPClass.slides == slides0 (nn_speech.c:84,125) */
static void inference_frames(int slides0, int T, int *first, int *n_inf)
{
    *first = (slides0 == 1) ? 0 : 1;
    *n_inf = (T > *first) ? (T - *first + 1) / 2 : 0;
}

static int batch_ensure_split(nnsp_b200_batch *b, int n_inf)
{
    if (batch_nn_path(b) != 3 || n_inf <= b->sp_cap_inf) return NNSP_B200_OK;
    NNSP_CUDA(cudaStreamSynchronize(b->stream));
    NNSP_CUDA(cudaStreamSynchronize(b->nn_stream));
    for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    for (auto &p : b->sp_planes) { if (p) cudaFree(p); p = nullptr; }
    if (b->sp_dec) { cudaFree(b->sp_dec); b->sp_dec = nullptr; }
    b->sp_cap_inf = 0;
    const size_t pb = split_plane_bytes(b->mm, b->S, n_inf);
    for (auto &p : b->sp_planes) { NNSP_CUDA(cudaMalloc(&p, pb)); NNSP_CUDA(cudaMemset(p, 0, pb)); }   /* columns no layer writes are read (against zero weights) */
    NNSP_CUDA(cudaMalloc(&b->sp_dec, (size_t)((b->S + 15) & ~15) * n_inf * sizeof(int32_t)));
    b->sp_cap_inf = n_inf;
    return NNSP_B200_OK;
}

/* st: stream of the front end (and of everything else unless st_nn is given); st_nn + ev_feat: the network kernels go
 * to st_nn once ev_feat (recorded on st behind the front end) has fired. The front end writes the next PCM history into
 * b->hist2; the caller swaps it with b->st.hist once per call. */
static int batch_launch(nnsp_b200_batch *b, const int16_t *pcm, long long stride, int T, int s0, int ns,
                        nnsp_b200_result *results, const nnsp_b200_taps *taps, cudaStream_t st, bool timed,
                        int fbuf = 0, cudaStream_t st_nn = nullptr, cudaEvent_t ev_feat = nullptr)
{
    const int path = batch_nn_path(b);
    int16_t *feat16 = b->feat16[fbuf];
    FeatLaunch fl{ pcm, stride, b->st.hist, 2, s0, ns, T, b->logmel };
    fl.hist_out = b->hist2;
    if (path == 3) { fl.logmel = nullptr; fl.norm = b->norm_dev; fl.feat16 = feat16; }
    if (timed) NNSP_CUDA(cudaEventRecord(b->ev[0], st));
    int rc = launch_feature(b->tables, fl, b->device, st);
    if (rc) return rc;
    if (timed) NNSP_CUDA(cudaEventRecord(b->ev[1], st));
    const bool piped = st_nn != nullptr;
    if (piped) {
        NNSP_CUDA(cudaEventRecord(ev_feat, st));
        NNSP_CUDA(cudaStreamWaitEvent(st_nn, ev_feat, 0));
        st = st_nn;
        if (timed) NNSP_CUDA(cudaEventRecord(b->ev_nn0, st));
    }
    if (path == 3 && taps && taps->logmel) {            /* debug tap: a second, log-mel pass straight into the tap */
        FeatLaunch ft{ pcm, stride, b->st.hist, 2, s0, ns, T, taps->logmel };
        if ((rc = launch_feature(b->tables, ft, b->device, st))) return rc;
    }
    if (path == 3) {
        if (!b->split_ok) { nnsp_set_error("this model has no scan-split formulation"); return NNSP_B200_ERR_UNSUPPORTED; }
        int first, n_inf;
        inference_frames(b->slides, T, &first, &n_inf);
        NNLaunch l{};
        l.tables = b->tables; l.st = b->st; l.logmel = b->logmel; l.s0 = s0; l.ns = ns; l.T = T; l.results = results;
        if (taps) l.taps = *taps;
        l.thresh_prob = b->thresh_prob; l.th_count = b->th_count;
        if ((rc = launch_nn_split(b->mm, l, feat16, first, n_inf, b->sp_planes[0], b->sp_planes[1], b->sp_dec, (int)b->sp_cap_inf, b->device, st))) return rc;
    } else if (path == 2) {
        if (!b->mma_ok) { nnsp_set_error("this model has no IMMA formulation"); return NNSP_B200_ERR_UNSUPPORTED; }
        NNLaunch l{};
        l.tables = b->tables; l.st = b->st; l.logmel = b->logmel; l.s0 = s0; l.ns = ns; l.T = T; l.results = results;
        if (taps) l.taps = *taps;
        l.thresh_prob = b->thresh_prob; l.th_count = b->th_count;
        if ((rc = launch_nn_mma(b->mm, l, b->device, st))) return rc;
    } else {
        NNArgs a{};
        a.model = b->dm.d; a.wimg = b->dm.wimg; a.bimg = b->dm.bimg; a.tables = b->tables; a.st = b->st;
        a.logmel = b->logmel; a.s0 = s0; a.ns = ns; a.T = T; a.results = results;
        if (taps) a.taps = *taps;
        a.thresh_prob = b->thresh_prob; a.th_count = b->th_count;
        int blocks = (ns + NN_WARPS - 1) / NN_WARPS;
        const int cap = sm_count(b->device) * b->nn_ctas_per_sm;
        if (blocks > cap) blocks = cap;
        nn_kernel<<<blocks, NN_THREADS, b->lay.total, st>>>(a, (int)b->lay.b, (int)b->lay.lut, (int)b->lay.model, (int)b->lay.scratch);
        NNSP_LAUNCH_CHECK();
    }
    if (timed) {
        NNSP_CUDA(cudaEventRecord(b->ev[2], st));
        b->ev_valid = true; b->last_piped = piped;
    }
    return NNSP_B200_OK;
}

/* everything the network stream still has in flight must be over before `st` touches the stream state */
static int batch_join_nn(nnsp_b200_batch *b, cudaStream_t st)
{
    for (int i = 0; i < 2; i++)
        if (b->nn_pending[i]) { NNSP_CUDA(cudaStreamWaitEvent(st, b->ev_nn[i], 0)); b->nn_pending[i] = false; }
    return NNSP_B200_OK;
}

/* asynchronous host-buffer calls leave work on the pipeline streams: everything else waits for it first */
static int batch_drain_host(nnsp_b200_batch *b)
{
    if (!b->host_inflight) return NNSP_B200_OK;
    for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    b->host_inflight = false;
    return NNSP_B200_OK;
}

static int batch_enqueue_host(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride, int n_frames,
                              nnsp_b200_result *results);

extern "C" {

const char *nnsp_b200_version(void) { return "nnsp-b200 0.1 (sm_100a)"; }
long long nnsp_b200_kernel_launches(void) { return g_launches.load(); }
long long nnsp_b200_tc5_launches(void) { return g_tc5_launches.load(); }
long long nnsp_b200_cascade_kernel_launches(int kind) { return (kind >= 0 && kind < 3) ? g_cascade_net_launches[kind].load() : -1; }
long long nnsp_b200_scan_kernel_launches(int kind) { return (kind >= 0 && kind < 6) ? g_scan_launches[kind].load() : -1; }

int nnsp_b200_device_count(void)
{
    int n = 0;
    return (cudaGetDeviceCount(&n) == cudaSuccess) ? n : 0;
}

int nnsp_b200_device_pci_bus_id(int device, char *buf, int len)
{
    if (!buf || len < 16) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaDeviceGetPCIBusId(buf, len, device));
    return NNSP_B200_OK;
}

int nnsp_b200_batch_create(const nnsp_b200_model *m, int n_streams, int device, int16_t thresh_prob,
                           int16_t th_count_trigger, nnsp_b200_batch **out)
{
    if (!m || !out || n_streams <= 0) return NNSP_B200_ERR_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    nnsp_b200_batch *b = new (std::nothrow) nnsp_b200_batch();
    if (!b) return NNSP_B200_ERR_NOMEM;
    b->device = device; b->S = n_streams; b->thresh_prob = thresh_prob; b->th_count = th_count_trigger;
    auto fail = [&](int code) { nnsp_b200_batch_destroy(b); return code; };
    if ((rc = get_device_tables(device, &b->tables))) return fail(rc);
    if ((rc = upload_model(m, &b->dm))) return fail(rc);
    rc = upload_model_mma(m, &b->mm);
    if (rc == NNSP_B200_OK) { b->mma_ok = true; b->split_ok = split_supported(b->mm) != 0; }
    else if (rc != NNSP_B200_ERR_UNSUPPORTED) return fail(rc);
    b->lay = nn_layout(b->dm.h);
    if (b->lay.total > 227 * 1024) { nnsp_set_error("model needs %zu bytes of shared memory (> 227 KB)", b->lay.total); return fail(NNSP_B200_ERR_UNSUPPORTED); }
    b->nn_ctas_per_sm = (int)((227 * 1024) / b->lay.total);
    if (b->nn_ctas_per_sm > 4) b->nn_ctas_per_sm = 4;
    if (b->nn_ctas_per_sm < 1) b->nn_ctas_per_sm = 1;
    const int HS = b->dm.h.h_stride > 0 ? b->dm.h.h_stride : 1;
    const size_t S = (size_t)n_streams;
#define TRY(x) do { if ((x) != cudaSuccess) { nnsp_set_error("%s failed: %s", #x, cudaGetErrorString(cudaGetLastError())); return fail(NNSP_B200_ERR_CUDA); } } while (0)
    TRY(cudaFuncSetAttribute(nn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->lay.total > 48 * 1024 ? 227 * 1024 : 48 * 1024));
    TRY(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    for (auto &s : b->xs) TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    {
        int lo = 0, hi = 0;                                /* the network stream outranks the front-end stream */
        TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        TRY(cudaStreamCreateWithPriority(&b->nn_stream, cudaStreamNonBlocking, hi));
    }
    for (auto &e : b->ev) TRY(cudaEventCreate(&e));
    TRY(cudaEventCreate(&b->ev_nn0));
    for (auto &e : b->ev_feat) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : b->ev_nn) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &r : b->host_ev) for (auto &e : r) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    TRY(cudaMalloc(&b->st.ctx, S * 240 * sizeof(int16_t)));
    TRY(cudaMemset(b->st.ctx, 0, S * 240 * sizeof(int16_t)));
    TRY(cudaMalloc(&b->st.h, S * HS * sizeof(int16_t)));
    TRY(cudaMalloc(&b->st.c, S * HS * sizeof(int32_t)));
    TRY(cudaMalloc(&b->st.scal, S * SC_N * sizeof(int16_t)));
    TRY(cudaMalloc(&b->st.hist, S * 2 * NNSP_B200_FRAME * sizeof(int16_t)));
    TRY(cudaMalloc(&b->hist2, S * 2 * NNSP_B200_FRAME * sizeof(int16_t)));
    {
        int32_t norm[84] = { 0 };
        memcpy(norm, b->dm.h.mean, 160);
        memcpy(norm + 40, b->dm.h.stdR, 160);
        norm[80] = b->dm.h.feat_rshift;
        TRY(cudaMalloc(&b->norm_dev, sizeof norm));
        TRY(cudaMemcpy(b->norm_dev, norm, sizeof norm, cudaMemcpyHostToDevice));
    }
#undef TRY
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(NNSP_B200_ERR_CUDA);   /* model / table uploads went through the default stream */
    if ((rc = nnsp_b200_batch_reset(b))) return fail(rc);
    *out = b;
    return NNSP_B200_OK;
}

int nnsp_b200_batch_reset(nnsp_b200_batch *b)
{
    if (!b) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(b->device));
    for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    b->host_inflight = false;
    if (b->nn_stream) NNSP_CUDA(cudaStreamSynchronize(b->nn_stream));
    b->nn_pending[0] = b->nn_pending[1] = false;
    reset_kernel<<<b->S, 128, 0, b->stream>>>(b->dm.d, b->st, b->S, NNSP_B200_FRAME);
    NNSP_LAUNCH_CHECK();
    NNSP_CUDA(cudaStreamSynchronize(b->stream));
    b->slides = 1;                                                      /* nn_speech.c:62 */
    return NNSP_B200_OK;
}

static int check_pcm_args(const void *pcm, long long stride, int T)
{
    if (!pcm || T <= 0) { nnsp_set_error("null PCM pointer or n_frames <= 0"); return NNSP_B200_ERR_ARG; }
    if ((stride & 1) || ((uintptr_t)pcm & 3) || stride < (long long)T * NNSP_B200_FRAME) {
        nnsp_set_error("PCM must be 4-byte aligned with an even stream_stride >= n_frames*160");
        return NNSP_B200_ERR_ARG;
    }
    return NNSP_B200_OK;
}

int nnsp_b200_batch_exec(nnsp_b200_batch *b, const int16_t *pcm_dev, long long stream_stride, int n_frames,
                         nnsp_b200_result *results_dev, const nnsp_b200_taps *taps)
{
    if (!b) return NNSP_B200_ERR_ARG;
    int rc = check_pcm_args(pcm_dev, stream_stride, n_frames);
    if (rc) return rc;
    NNSP_CUDA(cudaSetDevice(b->device));
    if ((rc = batch_drain_host(b))) return rc;
    if ((rc = batch_ensure_logmel(b, n_frames))) return rc;
    if ((rc = batch_ensure_split(b, (n_frames + 1) / 2))) return rc;
    if (batch_nn_path(b) == 3 && !taps) {
        /* pipelined: front end of this call on `stream` while the network kernels of the previous call still run on
         * `nn_stream`; the feature buffer alternates, a buffer is rewritten only after its network pass (two calls ago) */
        const int i = (int)(b->pipe++ & 1u);
        if (b->nn_pending[i]) NNSP_CUDA(cudaStreamWaitEvent(b->stream, b->ev_nn[i], 0));
        rc = batch_launch(b, pcm_dev, stream_stride, n_frames, 0, b->S, results_dev, nullptr, b->stream, true, i, b->nn_stream, b->ev_feat[i]);
        if (rc == NNSP_B200_OK) { NNSP_CUDA(cudaEventRecord(b->ev_nn[i], b->nn_stream)); b->nn_pending[i] = true; }
    } else {
        if ((rc = batch_join_nn(b, b->stream))) return rc;
        rc = batch_launch(b, pcm_dev, stream_stride, n_frames, 0, b->S, results_dev, taps, b->stream, true);
    }
    if (rc == NNSP_B200_OK) {
        b->slides = (b->slides + n_frames) % 2;
        std::swap(b->st.hist, b->hist2);
    }
    return rc;
}

int nnsp_b200_batch_exec_host(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride, int n_frames,
                              nnsp_b200_result *results)
{
    if (!b) return NNSP_B200_ERR_ARG;
    int rc = batch_enqueue_host(b, pcm, stream_stride, n_frames, results);
    if (rc) return rc;
    for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    b->host_inflight = false;
    return NNSP_B200_OK;
}

int nnsp_b200_batch_exec_host_async(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride, int n_frames,
                                    nnsp_b200_result *results, long long *ticket)
{
    if (!b) return NNSP_B200_ERR_ARG;
    int rc = batch_enqueue_host(b, pcm, stream_stride, n_frames, results);
    if (rc) return rc;
    const long long t = ++b->host_seq;
    for (int j = 0; j < 4; j++) NNSP_CUDA(cudaEventRecord(b->host_ev[t % HOST_RING][j], b->xs[j]));
    if (ticket) *ticket = t;
    return NNSP_B200_OK;
}

int nnsp_b200_batch_wait_host(nnsp_b200_batch *b, long long ticket)
{
    if (!b || ticket <= 0 || ticket > b->host_seq) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(b->device));
    /* a slot that has been reused holds the events of a later call on the same streams: waiting for those covers it */
    for (int j = 0; j < 4; j++) NNSP_CUDA(cudaEventSynchronize(b->host_ev[ticket % HOST_RING][j]));
    if (ticket == b->host_seq) b->host_inflight = false;
    return NNSP_B200_OK;
}

} /* extern "C" */

/* one host-buffer call queued on the four pipeline streams; nothing here waits for it. Slice k always goes to stream
 * k % 4, so consecutive calls are ordered slice by slice (staging buffers, stream state, result staging) by stream
 * order alone, and the H2D of call N+1 starts while the last slices of call N are still in their kernels */
static int batch_enqueue_host(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride, int n_frames,
                              nnsp_b200_result *results)
{
    int rc = check_pcm_args(pcm, stream_stride, n_frames);
    if (rc) return rc;
    NNSP_CUDA(cudaSetDevice(b->device));
    const int T = n_frames;
    if ((rc = batch_ensure_logmel(b, T))) return rc;
    if ((rc = batch_ensure_split(b, (T + 1) / 2))) return rc;
    if (T > b->d_pcm_frames) {
        NNSP_CUDA(cudaDeviceSynchronize());
        if (b->d_pcm) cudaFree(b->d_pcm);
        if (b->d_res) cudaFree(b->d_res);
        if (b->d_raw) cudaFree(b->d_raw);
        b->d_pcm = nullptr; b->d_res = nullptr; b->d_raw = nullptr;
        NNSP_CUDA(cudaMalloc(&b->d_pcm, (size_t)b->S * T * NNSP_B200_FRAME * sizeof(int16_t)));
        NNSP_CUDA(cudaMalloc(&b->d_res, (size_t)b->S * T * sizeof(nnsp_b200_result)));
        b->d_pcm_frames = T; b->d_res_frames = T;
    }
    NNSP_CUDA(cudaStreamSynchronize(b->stream));
    NNSP_CUDA(cudaStreamSynchronize(b->nn_stream));
    b->nn_pending[0] = b->nn_pending[1] = false;
    /* The per-call scratch (feature rows, staged PCM, result records) is laid out [stream][T]: a slice owns the same bytes
     * in consecutive calls only while T stays the same. When T changes and an asynchronous call is still in flight, every
     * pipeline stream first waits for ALL streams of that call (stream order alone covers equal-length calls; the
     * inference-dependent buffers are strided by their capacity and never move). */
    if (b->host_inflight && b->host_seq > 0 && b->host_last_T != T)
        for (int j = 0; j < 4; j++)
            for (int k = 0; k < 4; k++) NNSP_CUDA(cudaStreamWaitEvent(b->xs[j], b->host_ev[b->host_seq % HOST_RING][k], 0));
    b->host_last_T = T;
    if (b->host_fmt == NNSP_B200_HOST_AUDADC && !b->d_raw) {
        NNSP_CUDA(cudaDeviceSynchronize());
        NNSP_CUDA(cudaMalloc(&b->d_raw, (size_t)b->S * b->d_pcm_frames * NNSP_B200_FRAME * sizeof(uint32_t)));
    }
    /* slices of streams pipelined over four CUDA streams: H2D(k+1) overlaps kernels(k) overlaps D2H(k-1). The call
     * is bound by the host link (320 B of PCM per stream-frame), so slices are small enough that the work left
     * after the last H2D -- one slice of kernels and its D2H -- is short, and large enough to fill the GPU */
    const long long dstride = (long long)T * NNSP_B200_FRAME;
    b->host_inflight = true;
    int nsl = b->S / 256;
    nsl = nsl < 1 ? 1 : (nsl > 16 ? 16 : nsl);
    for (int k = 0; k < nsl; k++) {
        /* slice boundaries on 16-stream tiles (the tensor-core paths work on tiles) */
        const int s0 = (int)(((long long)b->S * k / nsl) & ~15LL);
        const int s1 = (k == nsl - 1) ? b->S : (int)(((long long)b->S * (k + 1) / nsl) & ~15LL);
        if (s1 <= s0) continue;
        cudaStream_t st = b->xs[k % 4];
        if (b->host_fmt == NNSP_B200_HOST_AUDADC) {
            /* the application's ingest in front of the path: raw 32-bit words over the link, conditioned on the device
             * (mask to the 12-bit sample, sample-3 glitch fix: main_nnsp.cc:58-65), then the same kernels */
            const uint32_t *raw = reinterpret_cast<const uint32_t *>(pcm);
            NNSP_CUDA(cudaMemcpy2DAsync(b->d_raw + (size_t)s0 * dstride, dstride * sizeof(uint32_t),
                                        raw + (size_t)s0 * stream_stride, stream_stride * sizeof(uint32_t),
                                        dstride * sizeof(uint32_t), (size_t)(s1 - s0), cudaMemcpyHostToDevice, st));
            if ((rc = launch_ingest(b->d_raw + (size_t)s0 * dstride, b->d_pcm + (size_t)s0 * dstride, (long long)(s1 - s0) * T, b->device, st))) return rc;
        } else if (stream_stride == dstride) {
            NNSP_CUDA(cudaMemcpyAsync(b->d_pcm + (size_t)s0 * dstride, pcm + (size_t)s0 * stream_stride,
                                      (size_t)(s1 - s0) * dstride * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        } else {
            NNSP_CUDA(cudaMemcpy2DAsync(b->d_pcm + (size_t)s0 * dstride, dstride * sizeof(int16_t),
                                        pcm + (size_t)s0 * stream_stride, stream_stride * sizeof(int16_t),
                                        dstride * sizeof(int16_t), (size_t)(s1 - s0), cudaMemcpyHostToDevice, st));
        }
        rc = batch_launch(b, b->d_pcm, dstride, T, s0, s1 - s0, results ? b->d_res : nullptr, nullptr, st, false);
        if (rc) return rc;
        if (results)
            NNSP_CUDA(cudaMemcpyAsync(results + (size_t)s0 * T, b->d_res + (size_t)s0 * T,
                                      (size_t)(s1 - s0) * T * sizeof(nnsp_b200_result), cudaMemcpyDeviceToHost, st));
    }
    b->slides = (b->slides + T) % 2;
    std::swap(b->st.hist, b->hist2);                    /* once per call: every slice reads the same buffer */
    return NNSP_B200_OK;
}

extern "C" {

int nnsp_b200_batch_sync(nnsp_b200_batch *b)
{
    if (!b) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(b->device));
    NNSP_CUDA(cudaStreamSynchronize(b->stream));
    NNSP_CUDA(cudaStreamSynchronize(b->nn_stream));
    for (auto s : b->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    b->host_inflight = false;
    return NNSP_B200_OK;
}

int nnsp_b200_batch_last_kernel_ms(nnsp_b200_batch *b, float ms[3])
{
    if (!b || !ms) return NNSP_B200_ERR_ARG;
    ms[0] = ms[1] = ms[2] = 0.f;
    if (!b->ev_valid) return NNSP_B200_OK;
    NNSP_CUDA(cudaSetDevice(b->device));
    NNSP_CUDA(cudaEventSynchronize(b->ev[2]));
    NNSP_CUDA(cudaEventElapsedTime(&ms[0], b->ev[0], b->ev[1]));
    NNSP_CUDA(cudaEventElapsedTime(&ms[1], b->last_piped ? b->ev_nn0 : b->ev[1], b->ev[2]));
    return NNSP_B200_OK;
}

int nnsp_b200_batch_dims(const nnsp_b200_batch *b, int *n_streams, int *act_stride, int *h_stride, int *n_out)
{
    if (!b) return NNSP_B200_ERR_ARG;
    if (n_streams) *n_streams = b->S;
    if (act_stride) *act_stride = b->dm.h.act_stride;
    if (h_stride) *h_stride = b->dm.h.h_stride;
    if (n_out) *n_out = b->dm.h.n_out;
    return NNSP_B200_OK;
}

void *nnsp_b200_batch_stream(nnsp_b200_batch *b) { return b ? (void *)b->stream : nullptr; }

int nnsp_b200_batch_set_nn_path(nnsp_b200_batch *b, int path)
{
    if (!b || path < 0 || path > 3) return NNSP_B200_ERR_ARG;
    if (path == 2 && !b->mma_ok) { nnsp_set_error("this model has no IMMA formulation"); return NNSP_B200_ERR_UNSUPPORTED; }
    if (path == 3 && !b->split_ok) { nnsp_set_error("this model has no scan-split formulation"); return NNSP_B200_ERR_UNSUPPORTED; }
    b->nn_path = path;
    return NNSP_B200_OK;
}

int nnsp_b200_batch_get_nn_path(const nnsp_b200_batch *b) { return b ? batch_nn_path(b) : NNSP_B200_ERR_ARG; }

int nnsp_b200_batch_set_host_format(nnsp_b200_batch *b, int fmt)
{
    if (!b || (fmt != NNSP_B200_HOST_PCM16 && fmt != NNSP_B200_HOST_AUDADC)) return NNSP_B200_ERR_ARG;
    int rc = nnsp_b200_batch_sync(b);
    if (rc) return rc;
    b->host_fmt = fmt;
    return NNSP_B200_OK;
}

void nnsp_b200_batch_destroy(nnsp_b200_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    cudaDeviceSynchronize();
    free_model(&b->dm);
    free_model_mma(&b->mm);
    cudaFree(b->st.ctx); cudaFree(b->st.h); cudaFree(b->st.c); cudaFree(b->st.scal); cudaFree(b->st.hist); cudaFree(b->hist2);
    cudaFree(b->logmel); cudaFree(b->d_pcm); cudaFree(b->d_res); cudaFree(b->d_raw);
    cudaFree(b->sp_planes[0]); cudaFree(b->sp_planes[1]); cudaFree(b->sp_dec);
    cudaFree(b->feat16[0]); cudaFree(b->feat16[1]); cudaFree(b->norm_dev);
    if (b->nn_stream) cudaStreamDestroy(b->nn_stream);
    if (b->ev_nn0) cudaEventDestroy(b->ev_nn0);
    for (auto e : b->ev_feat) if (e) cudaEventDestroy(e);
    for (auto e : b->ev_nn) if (e) cudaEventDestroy(e);
    if (b->stream) cudaStreamDestroy(b->stream);
    for (auto s : b->xs) if (s) cudaStreamDestroy(s);
    for (auto e : b->ev) if (e) cudaEventDestroy(e);
    for (auto &r : b->host_ev) for (auto e : r) if (e) cudaEventDestroy(e);
    delete b;
}

/* ---- one network evaluation on explicit inputs and explicit LSTM state (parity tool) ------------------ */
/* NeuralNetClass_exe (neural_nets.c:44-168) for n independent (input, state) pairs on the network kernels of the chosen
 * path: the stored context / the staged feature rows are loaded with x as it stands, no front end runs. */
int nnsp_b200_net_eval(const nnsp_b200_model *m, int device, int nn_path, int n, const int16_t *x, const int16_t *h0,
                       const int32_t *c0, int16_t *act, int32_t *logits, int16_t *h1, int32_t *c1)
{
    if (!m || !x || n <= 0 || nn_path < 0 || nn_path > 3) { nnsp_set_error("net_eval: bad arguments"); return NNSP_B200_ERR_ARG; }
    nnsp_b200_batch *b = nullptr;
    int rc = nnsp_b200_batch_create(m, n, device, 16383, 4, &b);
    if (rc) return rc;
    int16_t *t_act = nullptr, *t_h = nullptr, *xs = nullptr;
    int32_t *t_logits = nullptr, *t_c = nullptr;
    auto done = [&](int code) {
        cudaFree(t_act); cudaFree(t_logits); cudaFree(t_h); cudaFree(t_c);
        free(xs);
        nnsp_b200_batch_destroy(b);
        return code;
    };
#define NE_CUDA(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { nnsp_set_error("%s failed: %s", #expr, cudaGetErrorString(e__)); return done(NNSP_B200_ERR_CUDA); } } while (0)
    if (nn_path && (rc = nnsp_b200_batch_set_nn_path(b, nn_path))) return done(rc);
    const int path = batch_nn_path(b);
    const DevModel &D = b->dm.h;
    const int HS = D.h_stride, AS = D.act_stride > 0 ? D.act_stride : 1, NO = D.n_out;
    const size_t N = (size_t)n;
    NE_CUDA(cudaMalloc(&t_act, N * AS * sizeof(int16_t)));
    NE_CUDA(cudaMalloc(&t_logits, N * NO * sizeof(int32_t)));
    NE_CUDA(cudaMalloc(&t_h, N * (HS > 0 ? HS : 1) * sizeof(int16_t)));
    NE_CUDA(cudaMalloc(&t_c, N * (HS > 0 ? HS : 1) * sizeof(int32_t)));
    NE_CUDA(cudaMemset(t_act, 0, N * AS * sizeof(int16_t)));
    if (HS > 0) {
        if (h0) NE_CUDA(cudaMemcpy(b->st.h, h0, N * HS * sizeof(int16_t), cudaMemcpyHostToDevice));
        if (c0) NE_CUDA(cudaMemcpy(b->st.c, c0, N * HS * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    nnsp_b200_taps tp{};
    tp.act = t_act; tp.logits = t_logits;
    if (HS > 0) { tp.hstate = t_h; tp.cstate = t_c; }
    if (path == 3) {
        /* the scan-split kernels take the window as (context rows 1..5 carried, row of frame 0 staged): feed x that way */
        if ((rc = batch_ensure_logmel(b, 1)) || (rc = batch_ensure_split(b, 1))) return done(rc);
        xs = (int16_t *)calloc(N * 240 + N * 40, sizeof(int16_t));
        if (!xs) return done(NNSP_B200_ERR_NOMEM);
        int16_t *row5 = xs + N * 240;
        for (size_t i = 0; i < N; i++) {
            memcpy(xs + i * 240 + 40, x + i * 240, 200 * sizeof(int16_t));
            memcpy(row5 + i * 40, x + i * 240 + 200, 40 * sizeof(int16_t));
        }
        NE_CUDA(cudaMemcpy(b->st.ctx, xs, N * 240 * sizeof(int16_t), cudaMemcpyHostToDevice));
        NE_CUDA(cudaMemcpy(b->feat16[0], row5, N * 40 * sizeof(int16_t), cudaMemcpyHostToDevice));
        NE_CUDA(cudaDeviceSynchronize());
        NNLaunch l{};
        l.tables = b->tables; l.st = b->st; l.s0 = 0; l.ns = n; l.T = 1; l.taps = tp;
        l.thresh_prob = b->thresh_prob; l.th_count = b->th_count;
        if ((rc = launch_nn_split(b->mm, l, b->feat16[0], 0, 1, b->sp_planes[0], b->sp_planes[1], b->sp_dec, (int)b->sp_cap_inf, b->device, b->stream))) return done(rc);
    } else {
        NE_CUDA(cudaMemcpy(b->st.ctx, x, N * 240 * sizeof(int16_t), cudaMemcpyHostToDevice));
        NE_CUDA(cudaDeviceSynchronize());
        if (path == 2) {
            NNLaunch l{};
            l.tables = b->tables; l.st = b->st; l.s0 = 0; l.ns = n; l.T = 1; l.taps = tp; l.raw_ctx = 1;
            l.thresh_prob = b->thresh_prob; l.th_count = b->th_count;
            if ((rc = launch_nn_mma(b->mm, l, b->device, b->stream))) return done(rc);
        } else {
            NNArgs a{};
            a.model = b->dm.d; a.wimg = b->dm.wimg; a.bimg = b->dm.bimg; a.tables = b->tables; a.st = b->st;
            a.s0 = 0; a.ns = n; a.T = 1; a.taps = tp; a.raw_ctx = 1;
            a.thresh_prob = b->thresh_prob; a.th_count = b->th_count;
            int blocks = (n + NN_WARPS - 1) / NN_WARPS;
            const int cap = sm_count(b->device) * b->nn_ctas_per_sm;
            if (blocks > cap) blocks = cap;
            nn_kernel<<<blocks, NN_THREADS, b->lay.total, b->stream>>>(a, (int)b->lay.b, (int)b->lay.lut, (int)b->lay.model, (int)b->lay.scratch);
            g_launches.fetch_add(1);
            NE_CUDA(cudaGetLastError());
        }
    }
    NE_CUDA(cudaStreamSynchronize(b->stream));
    if (act && D.act_stride > 0) NE_CUDA(cudaMemcpy(act, t_act, N * D.act_stride * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (logits) NE_CUDA(cudaMemcpy(logits, t_logits, N * NO * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (h1 && HS > 0) NE_CUDA(cudaMemcpy(h1, t_h, N * HS * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (c1 && HS > 0) NE_CUDA(cudaMemcpy(c1, t_c, N * HS * sizeof(int32_t), cudaMemcpyDeviceToHost));
#undef NE_CUDA
    return done(NNSP_B200_OK);
}

/* ---- stage-by-stage front-end tap -------------------------------------------------------- */

int nnsp_b200_feature_stages(int device, const int16_t *windows, int n, int32_t *fft_in, int32_t *spec,
                             int32_t *pspec, int32_t *mel, int32_t *logmel)
{
    if (!windows || n <= 0) return NNSP_B200_ERR_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    const DevTables *tb;
    if ((rc = get_device_tables(device, &tb))) return rc;
    int16_t *dw = nullptr;
    int32_t *dbuf = nullptr;
    const size_t per = 512 + 514 + 257 + 40 + 40;
    NNSP_CUDA(cudaMalloc(&dw, (size_t)n * 480 * 2));
    NNSP_CUDA(cudaMalloc(&dbuf, (size_t)n * per * 4));
    NNSP_CUDA(cudaMemcpy(dw, windows, (size_t)n * 480 * 2, cudaMemcpyHostToDevice));
    NNSP_CUDA(cudaDeviceSynchronize());
    int32_t *d_fi = dbuf, *d_sp = d_fi + (size_t)n * 512, *d_ps = d_sp + (size_t)n * 514, *d_me = d_ps + (size_t)n * 257, *d_lm = d_me + (size_t)n * 40;
    NNSP_CUDA(cudaFuncSetAttribute(feat_stages_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FeatSmem)));
    int blocks = (n + FEAT_WARPS * 2 - 1) / (FEAT_WARPS * 2);
    if (blocks > 1024) blocks = 1024;
    feat_stages_kernel<<<blocks, FEAT_THREADS, sizeof(FeatSmem)>>>(tb, dw, n, d_fi, d_sp, d_ps, d_me, d_lm);
    NNSP_LAUNCH_CHECK();
    NNSP_CUDA(cudaDeviceSynchronize());
    if (fft_in) NNSP_CUDA(cudaMemcpy(fft_in, d_fi, (size_t)n * 512 * 4, cudaMemcpyDeviceToHost));
    if (spec) NNSP_CUDA(cudaMemcpy(spec, d_sp, (size_t)n * 514 * 4, cudaMemcpyDeviceToHost));
    if (pspec) NNSP_CUDA(cudaMemcpy(pspec, d_ps, (size_t)n * 257 * 4, cudaMemcpyDeviceToHost));
    if (mel) NNSP_CUDA(cudaMemcpy(mel, d_me, (size_t)n * 40 * 4, cudaMemcpyDeviceToHost));
    if (logmel) NNSP_CUDA(cudaMemcpy(logmel, d_lm, (size_t)n * 40 * 4, cudaMemcpyDeviceToHost));
    cudaFree(dw);
    cudaFree(dbuf);
    return NNSP_B200_OK;
}

int nnsp_b200_ingest_audadc(int device, const uint32_t *raw_dev, int16_t *pcm_dev, long long n_frames, void *stream)
{
    if (!raw_dev || !pcm_dev || n_frames < 0 || ((uintptr_t)raw_dev & 15) || ((uintptr_t)pcm_dev & 15)) {
        nnsp_set_error("ingest: null or not 16-byte aligned buffers");
        return NNSP_B200_ERR_ARG;
    }
    int rc = select_device(device);
    if (rc) return rc;
    return launch_ingest(raw_dev, pcm_dev, n_frames, device, (cudaStream_t)stream);
}

int nnsp_b200_table(const char *name, const void **data, int *elem_bytes)
{
    const nnsp_tables *t = nnsp_tables_get();
    if (!t || !name || !data || !elem_bytes) return NNSP_B200_ERR_ARG;
    struct { const char *n; const void *p; int eb, cnt; } tab[] = {
        { "stft_win", t->stft_win, 2, 480 }, { "fft_tw", t->fft_tw, 4, 256 }, { "rfft_tw", t->rfft_tw, 4, 256 },
        { "bitrev", t->bitrev, 2, 256 }, { "mel", t->mel, 2, 534 }, { "log_lut", t->log_lut, 2, 256 },
        { "tanh_lut", t->tanh_lut, 2, 384 },
    };
    for (auto &e : tab)
        if (!strcmp(e.n, name)) { *data = e.p; *elem_bytes = e.eb; return e.cnt; }
    return NNSP_B200_ERR_ARG;
}

/* ---- events and the integer-pipe microbenchmark --------------------------------------------- */
int nnsp_b200_event_create(int device, void **event)
{
    int rc = select_device(device);
    if (rc) return rc;
    cudaEvent_t e;
    NNSP_CUDA(cudaEventCreate(&e));
    *event = (void *)e;
    return NNSP_B200_OK;
}
int nnsp_b200_event_record(void *event, void *stream) { NNSP_CUDA(cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream)); return NNSP_B200_OK; }
int nnsp_b200_event_elapsed_ms(void *start, void *stop, float *ms)
{
    NNSP_CUDA(cudaEventSynchronize((cudaEvent_t)stop));
    NNSP_CUDA(cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop));
    return NNSP_B200_OK;
}
int nnsp_b200_event_destroy(void *event) { NNSP_CUDA(cudaEventDestroy((cudaEvent_t)event)); return NNSP_B200_OK; }

int nnsp_b200_int_peak(int device, double gops[4])
{
    int rc = select_device(device);
    if (rc) return rc;
    if (!gops) return NNSP_B200_ERR_ARG;
    int *sink = nullptr;
    NNSP_CUDA(cudaMalloc(&sink, 1 << 20));
    const int blocks = sm_count(device) * 8, threads = 256, iters = 4096;
    cudaEvent_t e0, e1;
    NNSP_CUDA(cudaEventCreate(&e0));
    NNSP_CUDA(cudaEventCreate(&e1));
    for (int mode = 0; mode < 4; mode++) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {
            NNSP_CUDA(cudaEventRecord(e0));
            int_peak_kernel<<<blocks, threads>>>(sink, iters, mode);
            NNSP_LAUNCH_CHECK();
            NNSP_CUDA(cudaEventRecord(e1));
            NNSP_CUDA(cudaEventSynchronize(e1));
            float ms;
            NNSP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        /* instructions per thread per iteration: 16 (modes 0, 2, 3) or 32 (mode 1) */
        gops[mode] = (double)blocks * threads * (double)iters * (mode == 1 ? 32.0 : 16.0) / (best * 1e-3) * 1e-9;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    return NNSP_B200_OK;
}

/* ---- device utilities ---------------------------------------------------------------------- */
int nnsp_b200_dev_alloc(int device, size_t nbytes, void **ptr)
{
    int rc = select_device(device);
    if (rc) return rc;
    NNSP_CUDA(cudaMalloc(ptr, nbytes));
    return NNSP_B200_OK;
}
int nnsp_b200_dev_free(int device, void *ptr) { NNSP_CUDA(cudaSetDevice(device)); NNSP_CUDA(cudaFree(ptr)); return NNSP_B200_OK; }
int nnsp_b200_host_alloc_pinned(size_t nbytes, void **ptr) { NNSP_CUDA(cudaMallocHost(ptr, nbytes)); return NNSP_B200_OK; }
int nnsp_b200_host_free_pinned(void *ptr) { NNSP_CUDA(cudaFreeHost(ptr)); return NNSP_B200_OK; }
/* The engine's streams are cudaStreamNonBlocking, i.e. NOT ordered against the legacy default stream these helpers
 * use -- and cudaMemcpy from pageable memory returns once the data is staged, cudaMemset is asynchronous to the host.
 * So each helper drains the default stream before returning: on return the bytes ARE in place for any stream. */
int nnsp_b200_memcpy_h2d(int device, void *dst, const void *src, size_t n)
{
    NNSP_CUDA(cudaSetDevice(device));
    NNSP_CUDA(cudaMemcpy(dst, src, n, cudaMemcpyHostToDevice));
    NNSP_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
    return NNSP_B200_OK;
}
int nnsp_b200_memcpy_d2h(int device, void *dst, const void *src, size_t n) { NNSP_CUDA(cudaSetDevice(device)); NNSP_CUDA(cudaMemcpy(dst, src, n, cudaMemcpyDeviceToHost)); return NNSP_B200_OK; }
int nnsp_b200_memset(int device, void *dst, int value, size_t n)
{
    NNSP_CUDA(cudaSetDevice(device));
    NNSP_CUDA(cudaMemset(dst, value, n));
    NNSP_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
    return NNSP_B200_OK;
}

}  /* extern "C" */
