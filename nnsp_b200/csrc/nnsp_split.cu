/* nnsp_split.cu -- "scan-split" network path: NeuralNetClass_exe reorganised around its only recurrence.
 *
 * Reference semantics (unchanged, bit for bit): NeuralNetClass_exe (neural_nets.c:44-168) runs the layer
 * list once per inference; fc_8x16 (affine.c:409-490), lstm_8x16 (lstm.c:15-214) -> rc_Krows_8x16
 * (affine.c:348-407), activations (activation.c:6-86), then s2i_post_proc / binary_post_proc
 * (nn_speech.c:146-227) and the stride-2 gate of NNSPClass_exec (nn_speech.c:84,125).
 *
 * Observation: within one exec call of T frames only the LSTM's recurrent half and the post-processing
 * counters depend on the previous inference. Everything else is a function of data that is known for all
 * T frames up front, so it is computed for every (stream, inference) row at once:
 *
 *   seg_kernel<feat>   layers before the LSTM (layer 0: 240 -> H0) for all rows. The A operand of row
 *                      (s, t) is the 6x40 context window = 240 consecutive bytes of the stream's
 *                      standardised feature rows, so 16 consecutive inferences share one 36-row plane.
 *   scan_kernel        the LSTM, one CTA per 16-stream tile, one warp per 8-unit group, sequential over the
 *                      inferences: input planes arrive by TMA bulk copies through a 4-deep mbarrier ring,
 *                      Wx.x of step k+1 is issued between arriving on and waiting for the h barrier of step k,
 *                      cell state and biases live in registers, h goes back to HBM by one TMA bulk store per step.
 *   seg_kernel<planes> layers after the LSTM for all rows, logits -> per-row decision record
 *                      (argmax triple or the softmax-threshold flag of binary_post_proc).
 *   post_kernel        the NNSPClass counters / trigger / outputs over the decision records, per stream.
 *   ctx_kernel         normFeatContext for the next call (feature_module.c:54-73).
 * feat_kernel runs in its standardising mode for this path: it writes the int16 feature row of every frame
 * (feature_module.c:67-73) instead of the int32 log-mel row.
 *
 * The contraction itself is the exact hi/lo byte-plane IMMA of nnsp_mma.cuh (16 streams x 8 units x 32 k per
 * mma.sync.m16n8k32, s8/u8 x s8, int32). Activation planes between kernels: [tile][inference][hi|lo][16][pa]
 * bytes, so one tile-step is a contiguous, 16-byte aligned block (bulk-copyable, conflict-free as A operand).
 * Only models whose every layer has the exact 32-bit finish (MmaLayer.fast) take this path.
 * The kernels work on a stream selection (StreamSel): a contiguous range for the batched NNSPClass, or a device-side
 * list for the cascade, whose stage-sorted pass (nnsp_cascade.cu) runs them once per (model, phase) group. */
#include <cuda_runtime.h>
#include <mutex>
#include <stdlib.h>
#include <string.h>

#include "nnsp_host.h"
#include "nnsp_mma.cuh"
#include "nnsp_tma.cuh"

namespace nnsp {

#ifndef NNSP_SEG_WARPS
#define NNSP_SEG_WARPS 8
#endif
constexpr int SEG_WARPS = NNSP_SEG_WARPS;
constexpr int SEG_THREADS = SEG_WARPS * 32;
constexpr int SEG_KC = 16;                          /* inferences per work item                          */
constexpr int SEG_FROWS = 2 * SEG_KC + 4;           /* feature rows covering 16 windows of 6, stride 2   */
constexpr int SEG_PC = SEG_FROWS * 40 + 16;         /* plane pitch: 364 words = 12 mod 32, conflict-free */
constexpr int SCAN_NST = 4;                         /* depth of the input ring of the scan               */
constexpr int SPLIT_MAX_DYN_SMEM = 227 * 1024 - 512;   /* the kernels also hold up to 276 B of static shared memory */
constexpr int LUT2_N = 321;                         /* half-segments of coeffs_tanh up to the saturation + the saturated entry (DevTables.tanh2) */
__host__ __device__ constexpr int lut2_bytes(int copies) { return (LUT2_N * 8 * copies + 127) & ~127; }   /* what follows it in shared memory stays 128-byte aligned */
/* The LUT is indexed by data, so lanes of a warp collide on banks (ncu: 58 % of the scan's LUT wavefronts were excess).
 * It can be replicated: copy c of entry k sits at [k * COPIES + c] and lane l reads copy l % COPIES, i.e. always the same
 * bank pair -- with 16 copies a 64-bit load of a half-warp touches every bank exactly once. */
#ifndef NNSP_LUT2_COPIES_SCAN
#define NNSP_LUT2_COPIES_SCAN 1
#endif
constexpr int LUT2_COPIES_SCAN = NNSP_LUT2_COPIES_SCAN;                 /* measured: 16 copies remove the conflicts but not a microsecond (the scan is
                                                       latency-bound), and the extra shared memory costs seg_kernel a resident CTA */
constexpr int LUT2_COPIES_SEG = 1;

static_assert((SEG_PC % 16) == 0 && ((SEG_PC / 4) % 8) == 4, "feature plane pitch");

/* ---- tanh LUT as (slope, constant) pairs: one 64-bit shared load and 11 instructions per evaluation ------------ */
/* tanh_fix, activation.c:31-69, on the folded table DevTables.tanh2: w = min(|x| >> 9, 320), d = |x| - 512 w,
 * y = (d * slope_w + const_w) >> 15. The reference's value + ((dx * slope) >> 15), its clamp at 0 (which only fires at
 * x = 0) and the saturation from |x| = 5.0 on are all in the constants (checked for every |x| when the tables are built).
 * x == INT32_MIN as in nnsp_device.cuh (-0x7fff): |x| = 2^31 as unsigned lands in the saturated entry, whose slope is 0.
 * Branch-free so that the evaluations of one epilogue interleave.
 * lut2: the calling lane's copy, i.e. base + (lane % COPIES); stride = COPIES */
template <int COPIES>
__device__ __forceinline__ int32_t tanh_q15v(int32_t x, const int2 *__restrict__ lut2)
{
    const uint32_t xi = (x < 0) ? (0u - (uint32_t)x) : (uint32_t)x;
    const uint32_t w = min(xi >> 9, (uint32_t)(LUT2_N - 1));
    const int2 e = lut2[w * COPIES];
    const int32_t v = (int32_t)((xi - (w << 9)) * (uint32_t)e.x + (uint32_t)e.y) >> 15;
    return x < 0 ? -v : v;
}
template <int COPIES>
__device__ __forceinline__ int32_t sigmoid_q15v(int32_t x, const int2 *__restrict__ lut2)     /* activation.c:72-86 */
{
    return (tanh_q15v<COPIES>(x >> 1, lut2) >> 1) + 16384;
}
template <int COPIES>
__device__ __forceinline__ void fill_lut2(int2 *lut2, const DevTables *__restrict__ tb, int tid, int nthr)
{
    for (int i = tid; i < LUT2_N * COPIES; i += nthr) {
        const int k = i / COPIES;
        lut2[i] = tb->tanh2[k];
    }
}

/* ---- decision records: the part of the post-processing that does not depend on earlier frames ---------- */
/* binary_post_proc, nn_speech.c:191-227 up to the comparison; 1 when this frame counts towards the streak */
__device__ __forceinline__ int binary_flag(int32_t l0, int32_t l1, int16_t thresh_prob)
{
    const int32_t mx = l0 > l1 ? l0 : l1;
    int32_t est[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int32_t val = (int32_t)((uint32_t)(i ? l1 : l0) - (uint32_t)mx);
        const int64_t ref = ((int64_t)val * 0xB8AA) >> 15;
        est[i] = pwr2_q15(sat32_dev(ref));
    }
    const int32_t den = (int32_t)((uint32_t)est[0] + (uint32_t)est[1]);
    const int32_t thresh = 32768 - (int32_t)thresh_prob;
    const int32_t tmp = (int32_t)(((int64_t)thresh * (int64_t)den) >> 15);
    return est[0] <= tmp ? 1 : 0;
}
/* NNSPClass scalars of one stream in registers (no dynamically indexed array: the counters are updated by
 * compare-and-add over the seven categories) */
struct PostRegs {
    int trig, out0, out1, out2, last, slides;
    int cnt[8];
};
__device__ __forceinline__ void apply_binary(PostRegs &r, int flag, int th_count)
{
    const int cnt = flag ? (int)(int16_t)(r.cnt[0] + 1) : 0;
    r.cnt[0] = cnt;
    r.trig = (cnt >= th_count) ? 1 : 0;
}
/* s2i_post_proc, nn_speech.c:146-189, on (argmax intent, argmax slot0, argmax slot1) */
__device__ __forceinline__ void apply_s2i(PostRegs &r, int dec, int th_count)
{
    const int ai = dec & 0xff;
    r.trig = 0; r.out0 = 0; r.out1 = 0; r.out2 = 0;
    if (r.last == 0 || r.last == ai) {
        int hit = 0;
#pragma unroll
        for (int i = 1; i < 7; i++) {
            const int c = (int)(int16_t)(r.cnt[i] + 1);
            if (ai == i) { r.cnt[i] = c; hit = c > th_count; }
        }
        if (hit) {
            r.trig = 1;
            r.out0 = ai;
            r.out1 = (dec >> 8) & 0xff;
            r.out2 = (dec >> 16) & 0xff;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 7; i++) r.cnt[i] = 0;
    }
    r.last = ai;
}

/* ======================================================================================================== */
/* seg_kernel: a run of fc layers [l0, l1) for every (16-stream tile, inference) row block                   */
/* ======================================================================================================== */
/* Which streams a launch works on: a contiguous range (batched NNSPClass: s0 .. s0+ns-1) or a device-side list
 * (cascade: the streams whose live instance runs this model with this inference phase; list, its length and its
 * first plane tile are produced on the device by the classify kernels, so no host round trip sizes the launch). */
struct StreamSel {
    const int *list;
    const int *count;
    const int *tile_off;
    int s0, ns;
    int tile0;                      /* plane tile of s0 (range) / first tile of the slice's plane region (list) */
};
__device__ __forceinline__ int sel_count(const StreamSel &q) { return q.list ? *q.count : q.ns; }
__device__ __forceinline__ size_t sel_tile_base(const StreamSel &q) { return (size_t)q.tile0 + (q.list ? (size_t)*q.tile_off : 0); }
__device__ __forceinline__ int sel_sid(const StreamSel &q, int tile, int row) { return q.list ? q.list[16 * tile + row] : q.s0 + 16 * tile + row; }

}   /* namespace nnsp */
#include "nnsp_tc5.cuh"
namespace nnsp {

struct SegArgs {
    const MmaModel *model;
    const uint2 *frag;              /* fragment image of the whole model */
    const int32_t *bias32;
    const DevTables *tables;
    int l0, l1;
    int w_base, w_bytes;            /* fragments of layers [l0, l1): uint2 offset in the image, byte count */
    int off_bias, off_lut, off_w, off_fp, off_row, off_wb, off_log, nbuf;   /* shared-memory layout (seg_layout) */
    StreamSel sel;
    int T, first, n_inf, nchunks;
    long long tile_bytes;           /* bytes of one tile's plane region (>= n_inf * 32 * pa) */
    int dec_stride;                 /* decision records per stream */
    const int16_t *feat16;          /* [S][T][40] standardised rows of this call (MODE 1) */
    const int32_t *logmel;          /* [S][T][40] log-mel rows of this call      (MODE 2) */
    const int32_t *lmhist;          /* [S][dmax][40] log-mel rows before the call (MODE 2) */
    int dmax, dback;                /* rows in lmhist; look-back of this model: frame t reads row t - dback (MODE 2) */
    const int16_t *ctx;             /* [S][240] context before the call          (MODE 1, 2) */
    const uint8_t *in_planes;       /* [tile][n_inf][2][16][pa]                  (MODE 0) */
    uint8_t *out_planes;            /* same layout, when l1 < numlayers */
    int32_t *dec;                   /* [S][dec_stride], when l1 == numlayers */
    int16_t *tap_act;               /* [S][T][act_stride] or null */
    int32_t *tap_logits;            /* [S][T][n_out] or null */
    int ao0;                        /* offset of layer l0's output inside an act row */
    int16_t thresh_prob;
    const int16_t *thr_prob; int thr_stride;   /* per-stream thresholds (cascade), else null */
    const int *tstart, *tb, *age0;  /* cascade rounds: per-stream first inference frame, life begin, age there (SplitGroup) */
    const int32_t *lmfix;           /* [S][2][40] log-mel rows of an instance's first two frames */
    const int32_t *nfr;             /* ragged cascade call: per-stream end frame (SplitGroup) */
};

/* Where the outputs of one fc layer of one (tile, inference) row block go. */
struct FcOut {
    uint8_t *oh, *ol;               /* output planes [16][pa] (not written by the model's last layer) */
    int32_t *wlog;                  /* logits rows [16][nop] (linear layers and the model's last layer) */
    const int2 *lut2;
    int pa, nop, rs, act;
    bool last;
};

/* NC (1..4) column tiles of 8 units starting at unit 8*n0 for the warp's 16 rows: both byte-plane products, then the
 * layer's finish. Everything that depends on NC or the lane is resolved at compile time or hoisted, the activation is
 * chosen once per group, so the 4*NC evaluations of a group are straight-line code that interleaves.
 * exact 32-bit finish (MmaLayer.fast): affine.c:190-249 without reachable clamps; the bias (pre-shifted) rides in the
 * low-plane accumulator; units past the layer's rows are computed too (zero weights) and only ever meet zero weights. */
template <int NC, int KT>           /* KT: k-steps of the layer when known at compile time (fully unrolled), 0 = run-time kt */
__device__ __forceinline__ void fc_group(int kt_rt, const uint2 *__restrict__ wf, uint32_t ah, uint32_t al,
                                         const int32_t *__restrict__ B, int n0, int g, int q, const FcOut &o)
{
    const int kt = KT ? KT : kt_rt;
    int ch[NC][4], cl[NC][4];
    {                                                                       /* k-step 0 starts the accumulators */
        uint32_t fh[4], fl[4];
        load_a_ldm(ah, fh);
        load_a_ldm(al, fl);
#pragma unroll
        for (int j = 0; j < NC; j++) {
            const int2 bias = *reinterpret_cast<const int2 *>(B + (n0 + j) * 8 + 2 * q);
            const uint2 b = wf[(j * kt) * 32];
            imma_s8s8_first(ch[j], fh, b);
            imma_u8s8_first(cl[j], fl, b, bias.x, bias.y);
        }
    }
    if (KT) {
#pragma unroll
        for (int ks = 1; ks < (KT ? KT : 1); ks++) {
            uint32_t fh[4], fl[4];
            load_a_ldm(ah + 32 * ks, fh);
            load_a_ldm(al + 32 * ks, fl);
#pragma unroll
            for (int j = 0; j < NC; j++) {
                const uint2 b = wf[(j * KT + ks) * 32];
                imma_s8s8(ch[j], fh, b);
                imma_u8s8(cl[j], fl, b);
            }
        }
    } else {
#pragma unroll 1
        for (int ks = 1; ks < kt; ks++) {
            uint32_t fh[4], fl[4];
            load_a_ldm(ah + 32 * ks, fh);
            load_a_ldm(al + 32 * ks, fl);
#pragma unroll
            for (int j = 0; j < NC; j++) {
                const uint2 b = wf[(j * kt + ks) * 32];
                imma_s8s8(ch[j], fh, b);
                imma_u8s8(cl[j], fl, b);
            }
        }
    }
    /* relu6_fix (activation.c:6-17) starts with x >> 3: two arithmetic right shifts compose exactly, so its layers shift once */
    const int rs = o.rs + (o.act == ACT_RELU6 ? 3 : 0);
    int32_t v[NC][4];
#pragma unroll
    for (int j = 0; j < NC; j++)
#pragma unroll
        for (int e = 0; e < 4; e++) v[j][e] = (int32_t)(((uint32_t)ch[j][e] << 8) + (uint32_t)cl[j][e]) >> rs;
    const int r0 = g * o.pa + n0 * 8 + 2 * q, r1 = r0 + 8 * o.pa;           /* plane bytes of rows g, g+8 */
    int32_t *w0 = o.wlog + g * o.nop + n0 * 8 + 2 * q, *w1 = w0 + 8 * o.nop;  /* logits words of rows g, g+8 */
    if (o.act == ACT_LINEAR) {                                              /* activation.c:19-29: int32 stays */
#pragma unroll
        for (int j = 0; j < NC; j++) {
            *reinterpret_cast<int2 *>(w0 + 8 * j) = make_int2(v[j][0], v[j][1]);
            *reinterpret_cast<int2 *>(w1 + 8 * j) = make_int2(v[j][2], v[j][3]);
            if (!o.last) { store_pair(o.oh, o.ol, r0 + 8 * j, 0, 0); store_pair(o.oh, o.ol, r1 + 8 * j, 0, 0); }
        }
        return;
    }
    if (o.act == ACT_RELU6) {
#pragma unroll
        for (int j = 0; j < NC; j++)
#pragma unroll
            for (int e = 0; e < 4; e++) v[j][e] = min(max(v[j][e], 0), 6 << 12);
    } else if (o.act == ACT_TANH) {
#pragma unroll
        for (int j = 0; j < NC; j++)
#pragma unroll
            for (int e = 0; e < 4; e++) v[j][e] = tanh_q15v<LUT2_COPIES_SEG>(v[j][e], o.lut2);
    } else {
#pragma unroll
        for (int j = 0; j < NC; j++)
#pragma unroll
            for (int e = 0; e < 4; e++) v[j][e] = sigmoid_q15v<LUT2_COPIES_SEG>(v[j][e], o.lut2);
    }
    if (o.last) {                                                           /* neural_nets.c:160-166 */
#pragma unroll
        for (int j = 0; j < NC; j++) {
            *reinterpret_cast<int2 *>(w0 + 8 * j) = make_int2(v[j][0], v[j][1]);
            *reinterpret_cast<int2 *>(w1 + 8 * j) = make_int2(v[j][2], v[j][3]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < NC; j++) {
            store_pair(o.oh, o.ol, r0 + 8 * j, v[j][0], v[j][1]);
            store_pair(o.oh, o.ol, r1 + 8 * j, v[j][2], v[j][3]);
        }
    }
}

/* all nt column tiles of one fc layer for the warp's 16 rows, in groups of four */
template <int KT>
__device__ __forceinline__ void fc_layer(int kt, int nt, const uint2 *__restrict__ wl, uint32_t ah, uint32_t al,
                                         const int32_t *__restrict__ B, int g, int q, const FcOut &o)
{
    int n0 = 0;
    for (; n0 + 4 <= nt; n0 += 4) fc_group<4, KT>(kt, wl + n0 * kt * 32, ah, al, B, n0, g, q, o);
    switch (nt - n0) {
    case 3: fc_group<3, KT>(kt, wl + n0 * kt * 32, ah, al, B, n0, g, q, o); break;
    case 2: fc_group<2, KT>(kt, wl + n0 * kt * 32, ah, al, B, n0, g, q, o); break;
    case 1: fc_group<1, KT>(kt, wl + n0 * kt * 32, ah, al, B, n0, g, q, o); break;
    default: break;
    }
}

/* MODE 0: input = activation planes; 1: input = feat16 rows (batched NNSPClass); 2: input = log-mel rows with
 * look-back, standardised while staging (cascade) */
template <int MODE>
#ifndef SEG_MINB
#define SEG_MINB 2
#endif
#ifdef SEG_MAXNREG            /* register cap instead of a residency target: a CTA that fits the hole one retiring feat_kernel CTA leaves */
__global__ void __maxnreg__(SEG_MAXNREG)
#else
__global__ void __launch_bounds__(SEG_THREADS, SEG_MINB)
#endif
seg_kernel(SegArgs a)
{
    constexpr bool FROM_FEAT = MODE != 0;
    __shared__ int sids[16], s_ts[16], s_te[16], s_tb[16], s_ag[16], s_ninf;
    extern __shared__ __align__(128) unsigned char smem[];
    const bool per_row = a.tstart != nullptr;                     /* cascade rounds: every row has its own start frame */
    {   /* nothing selected (a later round of the cascade, an empty group) or more CTAs than work items: leave before the prologue */
        const int nsel0 = sel_count(a.sel);
        if ((int)blockIdx.x >= ((nsel0 + 15) >> 4) * a.nchunks) return;
    }
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem);
    MmaModel &M = *reinterpret_cast<MmaModel *>(smem + 16);
    int32_t *bias32 = reinterpret_cast<int32_t *>(smem + a.off_bias);
    int2 *lut2_all = reinterpret_cast<int2 *>(smem + a.off_lut);
    const int2 *lut2 = lut2_all + (threadIdx.x & (LUT2_COPIES_SEG - 1));
    const uint2 *wsm = reinterpret_cast<const uint2 *>(smem + a.off_w);
    uint8_t *fplanes = smem + a.off_fp;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;

    /* once per (persistent) CTA: descriptor, biases, LUT by plain loads; the segment's weight fragments by TMA */
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        const int *src = reinterpret_cast<const int *>(a.model);
        int *dst = reinterpret_cast<int *>(&M);
        for (int i = tid; i < (int)(sizeof(MmaModel) / 4); i += SEG_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    if (tid == 0) {
        const unsigned char *wsrc = reinterpret_cast<const unsigned char *>(a.frag + a.w_base);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"((uint32_t)a.w_bytes) : "memory");
        for (int o = 0; o < a.w_bytes; o += 32768) {
            const uint32_t n = (uint32_t)min(32768, a.w_bytes - o);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(smem + a.off_w + o)), "l"(wsrc + o), "r"(n), "r"(smem_u32(bar)) : "memory");
        }
    }
    const int XB = 32 * M.pa;                                    /* bytes of one tile-step: [hi|lo][16][pa] */
    uint8_t *wb = smem + a.off_wb + (size_t)warp * a.nbuf * XB;
    const int NOP = M.no + 4;                                     /* logits row pitch: (no + 4) words keeps the 8 rows of a store on distinct banks */
    const int pa = M.pa, nlayers = M.numlayers, act_stride = M.act_stride;
    int32_t *wlog = reinterpret_cast<int32_t *>(smem + a.off_log) + warp * 16 * NOP;
    {   /* activation planes start zeroed: padded k columns must hold defined bytes (they meet zero weights) */
        uint32_t *z = reinterpret_cast<uint32_t *>(smem + a.off_wb);
        for (int i = tid; i < SEG_WARPS * a.nbuf * XB / 4; i += SEG_THREADS) z[i] = 0;
    }
    for (int i = tid; i < M.bias_count; i += SEG_THREADS) bias32[i] = a.bias32[i];
    fill_lut2<LUT2_COPIES_SEG>(lut2_all, a.tables, tid, SEG_THREADS);
    if (FROM_FEAT)
        for (int e = tid; e < 32 * 4; e += SEG_THREADS)              /* k-step over-read behind the last window */
            *reinterpret_cast<uint32_t *>(fplanes + (e >> 2) * SEG_PC + SEG_FROWS * 40 + (e & 3) * 4) = 0;
    {
        uint32_t done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(smem_u32(bar)) : "memory");
    }
    const int T = a.T;
    const int nsel = sel_count(a.sel);
    const int nitems = ((nsel + 15) >> 4) * a.nchunks;
    const size_t tile_base = sel_tile_base(a.sel);
    /* MODE 2 staging: 16-byte pieces of 8 features as in MODE 1. Thread (px, pj, pr) stages features 8 px .. 8 px + 7 of
     * rows j = pj, pj + JP, ... of tile row pr, so it standardises with the same 8 (mean, stdR) pairs throughout; consecutive
     * threads write consecutive pieces of a row, then the next row. */
    constexpr int JP = SEG_THREADS / 80;
    static_assert(JP >= 1 && SEG_FROWS % JP == 0, "staging threads");
    const int px = tid % 5, pr = tid / (5 * JP), pj = tid / 5 - pr * JP;
    __syncthreads();

    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        /* chunk-major order: the last chunk of every tile is a short one (n_inf = 50: 16, 16, 16, 2), and with the tile-major
         * order a CTA met the same chunk index over and over (grid 296 is a multiple of 4 chunks): a quarter of the CTAs
         * got nothing but short items. Now every CTA walks through all chunk indices and the short items come last. */
        const int ntl = (nsel + 15) >> 4;
        const int chunk = item / ntl, tile = item - chunk * ntl;
        const int k0 = chunk * SEG_KC;
        const int nvalid = min(16, nsel - 16 * tile);
        const size_t tile_abs = tile_base + tile;
        int ninf_tile = a.n_inf;
        if (FROM_FEAT || per_row) {
            __syncthreads();                                         /* planes of the previous item are free */
            if (tid < 16) {
                const int sid = (tid < nvalid) ? sel_sid(a.sel, tile, tid) : 0;
                int ts = a.first, tbv = 0, ag = 2;
                if (per_row && tid < nvalid) { ts = a.tstart[sid]; tbv = a.tb[sid]; ag = a.age0[sid]; }
                sids[tid] = sid; s_ts[tid] = ts; s_tb[tid] = tbv; s_ag[tid] = ag;
                const int Ts = per_row && tid < nvalid ? stream_frames(a.nfr, sid, T) : T;
                s_te[tid] = Ts;
                int ni = (tid < nvalid) ? (per_row ? (ts < Ts ? (Ts - ts + 1) >> 1 : 0) : a.n_inf) : 0;
                for (int o = 8; o; o >>= 1) ni = max(ni, __shfl_xor_sync(0x0000ffffu, ni, o));
                if (tid == 0) s_ninf = ni;
            }
            __syncthreads();
            ninf_tile = s_ninf;                                      /* most inferences any row of the tile has */
        }
        if (k0 >= ninf_tile) continue;
        if (FROM_FEAT) {
            /* standardised rows of frames f_first .. f_first+35 as byte planes; frames before the call are the
             * carried context rows 1..5 (feature_module.c:54-57); loads of a batch are issued before its stores */
            const int f_first = a.first + 2 * k0 - 5;
            if (MODE == 1) {
                constexpr int NQ = 16 * SEG_FROWS * 5;               /* 16-byte pieces: 8 features each */
                for (int e0 = 0; e0 < NQ; e0 += 4 * SEG_THREADS) {
                    uint4 v[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * SEG_THREADS + tid;
                        v[u] = make_uint4(0, 0, 0, 0);
                        if (e < NQ) {
                            const int r = e / (SEG_FROWS * 5), rem = e - r * (SEG_FROWS * 5), j = rem / 5, x = rem - j * 5;
                            const int f = f_first + j;
                            if (r < nvalid) {
                                const long long s = sids[r];
                                if (f < 0) v[u] = *reinterpret_cast<const uint4 *>(a.ctx + s * 240 + (6 + f) * 40 + x * 8);
                                else if (f < T) v[u] = __ldg(reinterpret_cast<const uint4 *>(a.feat16 + (s * T + f) * NNSP_B200_NMEL + x * 8));
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * SEG_THREADS + tid;
                        if (e < NQ) {
                            const int r = e / (SEG_FROWS * 5), rem = e - r * (SEG_FROWS * 5), j = rem / 5, x = rem - j * 5;
                            uint2 hi, lo;
                            lo.x = __byte_perm(v[u].x, v[u].y, 0x6420); hi.x = __byte_perm(v[u].x, v[u].y, 0x7531);
                            lo.y = __byte_perm(v[u].z, v[u].w, 0x6420); hi.y = __byte_perm(v[u].z, v[u].w, 0x7531);
                            *reinterpret_cast<uint2 *>(fplanes + r * SEG_PC + j * 40 + x * 8) = hi;
                            *reinterpret_cast<uint2 *>(fplanes + (16 + r) * SEG_PC + j * 40 + x * 8) = lo;
                        }
                    }
                }
            } else {
                /* cascade: frame f of the instance is raw frame f - dback (PcmBufClass_getData look-back,
                 * PcmBufClass.c:38-85): its log-mel row comes from this call or from the carried history and is
                 * standardised with this model's statistics (feature_module.c:67-73). The source of each staged row is
                 * resolved once per item: a log-mel row (int32), a stored context row (int16, already standardised,
                 * tagged by bit 0) or none (0: the row stages as zeros) */
                uintptr_t *s_row = reinterpret_cast<uintptr_t *>(smem + a.off_row);    /* [16][SEG_FROWS] */
                for (int j = tid >> 4; j < SEG_FROWS; j += SEG_THREADS >> 4) {
                    const int r = tid & 15;
                    uintptr_t src = 0;
                    if (r < nvalid) {
                        const long long s = sids[r];
                        const int f = s_ts[r] + 2 * k0 - 5 + j;                      /* frame of the call */
                        const int life = f - s_tb[r];                                /* frames since the instance's life in this call began */
                        if (life < 0) {                                              /* before that: the instance's stored context rows 1..5 */
                            src = reinterpret_cast<uintptr_t>(a.ctx + s * 240 + (6 + life) * 40) | 1;
                        } else if (f < s_te[r]) {                                    /* frames past the row's own end stage as zeros */
                            const int la = life + s_ag[r], fr = f - a.dback;
                            src = reinterpret_cast<uintptr_t>((la < 2) ? a.lmfix + (s * 2 + la) * NNSP_B200_NMEL   /* STFT buffer still partly zero */
                                                            : (fr >= 0) ? a.logmel + (s * T + fr) * NNSP_B200_NMEL
                                                                        : a.lmhist + (s * a.dmax + a.dmax + fr) * NNSP_B200_NMEL);
                        }
                    }
                    s_row[r * SEG_FROWS + j] = src;
                }
                __syncthreads();
                if (tid < 80 * JP) {
                    int32_t mn[8], sd[8];                                    /* the thread's features: registers, not a shared load per value */
#pragma unroll
                    for (int c = 0; c < 8; c++) { mn[c] = M.mean[8 * px + c]; sd[c] = M.stdR[8 * px + c]; }
                    const int rs = M.feat_rshift;
                    const uintptr_t *rows = s_row + pr * SEG_FROWS + pj;
                    uint8_t *dst = fplanes + pr * SEG_PC + pj * 40 + px * 8;
                    constexpr int NP = SEG_FROWS / JP;                       /* pieces per thread */
#pragma unroll 1
                    for (int m0 = 0; m0 < NP; m0 += 4) {
                        int4 v[4][2];                                        /* log-mel values */
                        uint4 w[4];                                          /* 8 int16 features, pairwise: context rows, zeros */
                        bool lm[4];
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const bool in = NP % 4 == 0 || m0 + u < NP;
                            const uintptr_t src = in ? rows[(m0 + u) * JP] : 0;
                            const bool cx = src & 1;
                            const int4 *p = reinterpret_cast<const int4 *>(src & ~(uintptr_t)1) + (cx ? px : 2 * px);
                            lm[u] = src && !cx;
                            v[u][0] = lm[u] ? __ldg(p) : make_int4(0, 0, 0, 0);
                            v[u][1] = lm[u] ? __ldg(p + 1) : make_int4(0, 0, 0, 0);
                            w[u] = cx ? __ldg(reinterpret_cast<const uint4 *>(p)) : make_uint4(0, 0, 0, 0);
                        }
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            if (NP % 4 != 0 && m0 + u >= NP) break;
                            if (lm[u]) {
                                const int32_t e[8] = { v[u][0].x, v[u][0].y, v[u][0].z, v[u][0].w, v[u][1].x, v[u][1].y, v[u][1].z, v[u][1].w };
                                int32_t z[8];
#pragma unroll
                                for (int c = 0; c < 8; c++) z[c] = standardise(e[c], mn[c], sd[c], rs);
                                w[u].x = __byte_perm(z[0], z[1], 0x5410); w[u].y = __byte_perm(z[2], z[3], 0x5410);
                                w[u].z = __byte_perm(z[4], z[5], 0x5410); w[u].w = __byte_perm(z[6], z[7], 0x5410);
                            }
                            uint2 hi, lo;
                            lo.x = __byte_perm(w[u].x, w[u].y, 0x6420); hi.x = __byte_perm(w[u].x, w[u].y, 0x7531);
                            lo.y = __byte_perm(w[u].z, w[u].w, 0x6420); hi.y = __byte_perm(w[u].z, w[u].w, 0x7531);
                            *reinterpret_cast<uint2 *>(dst + (m0 + u) * JP * 40) = hi;
                            *reinterpret_cast<uint2 *>(dst + 16 * SEG_PC + (m0 + u) * JP * 40) = lo;
                        }
                    }
                }
            }
            __syncthreads();
        }

        for (int i = warp; i < SEG_KC; i += SEG_WARPS) {
            const int k = k0 + i;
            if (k >= ninf_tile) break;
            const int t = a.first + 2 * k;                               /* frame of this inference */
            const uint8_t *in_hi, *in_lo;
            int in_pitch;
            if (FROM_FEAT) {
                in_hi = fplanes + 80 * i; in_lo = in_hi + 16 * SEG_PC; in_pitch = SEG_PC;
            } else {
                const uint4 *src = reinterpret_cast<const uint4 *>(a.in_planes + tile_abs * (size_t)a.tile_bytes + (size_t)k * XB);
                uint4 *dst = reinterpret_cast<uint4 *>(wb + XB);
                for (int x = lane; x < XB / 16; x += 32) dst[x] = __ldg(src + x);
                __syncwarp();
                in_hi = wb + XB; in_lo = in_hi + 16 * M.pa; in_pitch = M.pa;
            }
            int pp = 0, ao = a.ao0;
            for (int li = a.l0; li < a.l1; li++) {
                const MmaLayer &L = M.layer[li];
                const int kt = L.kt, nt = L.nt, rows = L.rows;
                const int32_t *B = bias32 + L.bias_off;
                FcOut out;
                out.oh = wb + pp * XB; out.ol = out.oh + 16 * pa; out.wlog = wlog; out.lut2 = lut2;
                out.pa = pa; out.nop = NOP; out.rs = -L.sh_out; out.act = L.act; out.last = (li == nlayers - 1);
                const uint32_t ah = ldm_lane_addr(in_hi, in_pitch, lane), al = ldm_lane_addr(in_lo, in_pitch, lane);
                const uint2 *wl = wsm + (L.w_off - a.w_base) + lane;
                switch (kt) {                                             /* the shipped models: 1 (VAD), 2 (KWS), 3 and 8 (S2I, layer 0) */
                case 1: fc_layer<1>(kt, nt, wl, ah, al, B, g, q, out); break;
                case 2: fc_layer<2>(kt, nt, wl, ah, al, B, g, q, out); break;
                case 3: fc_layer<3>(kt, nt, wl, ah, al, B, g, q, out); break;
                case 8: fc_layer<8>(kt, nt, wl, ah, al, B, g, q, out); break;
                default: fc_layer<0>(kt, nt, wl, ah, al, B, g, q, out); break;
                }
                __syncwarp();
                if (a.tap_act && !out.last && out.act != ACT_LINEAR) {        /* debug tap: the layer's int16 outputs back from the planes */
                    for (int x = lane; x < nvalid * rows; x += 32) {
                        const int row = x / rows, n = x - row * rows;
                        a.tap_act[((long long)sel_sid(a.sel, tile, row) * T + t) * act_stride + ao + n] =
                            (int16_t)(((int)(int8_t)out.oh[row * pa + n] << 8) | out.ol[row * pa + n]);
                    }
                }
                in_hi = out.oh; in_lo = out.ol; in_pitch = pa;
                pp ^= 1;
                if (!out.last) ao += rows;
            }
            if (a.l1 < M.numlayers) {
                const uint4 *src = reinterpret_cast<const uint4 *>(wb + (pp ^ 1) * XB);
                uint4 *dst = reinterpret_cast<uint4 *>(a.out_planes + tile_abs * (size_t)a.tile_bytes + (size_t)k * XB);
                for (int x = lane; x < XB / 16; x += 32) dst[x] = src[x];
            } else {
                if (lane < nvalid) {
                    const int32_t *lg = wlog + lane * NOP;
                    int d;
                    if (M.nn_id == NNSP_B200_ID_S2I)
                        d = argmax_last_wins(lg, 7) | (argmax_last_wins(lg + 7, 17) << 8) | (argmax_last_wins(lg + 24, 17) << 16);
                    else
                        d = binary_flag(lg[0], lg[1], a.thr_prob ? a.thr_prob[(size_t)sel_sid(a.sel, tile, lane) * a.thr_stride] : a.thresh_prob);
                    a.dec[(size_t)sel_sid(a.sel, tile, lane) * a.dec_stride + k] = d;
                }
                if (a.tap_logits)
                    for (int x = lane; x < 16 * M.n_out; x += 32) {
                        const int row = x / M.n_out, n = x - row * M.n_out;
                        if (row < nvalid) a.tap_logits[((long long)sel_sid(a.sel, tile, row) * T + t) * M.n_out + n] = wlog[row * NOP + n];
                    }
            }
            __syncwarp();
        }
    }
}

/* ======================================================================================================== */
/* scan_kernel: one LSTM layer over the inferences of a 16-stream tile                                       */
/* ======================================================================================================== */
struct ScanArgs {
    const uint2 *frag;              /* fragment image; the layer's Wx tiles at w_off, Wh tiles right behind */
    const int32_t *bias32;
    const DevTables *tables;
    int H, kt, ktr, nt, rs, w_off, bias_off, pa;
    int ho, hs, ao, act_stride, tap_out;   /* state offset / stride, act-row offset, 1: layer output is tapped */
    StreamSel sel;
    int T, first, n_inf;
    long long tile_bytes;           /* bytes of one tile's plane region */
    const uint8_t *xin;             /* [tile][n_inf][2][16][pa] */
    uint8_t *hout;                  /* same layout */
    int16_t *h;                     /* [S][hs] */
    int32_t *c;
    int16_t *tap_act, *tap_h;
    int32_t *tap_c;
    const int *tstart;              /* cascade rounds: per-stream first inference frame (null: every row has n_inf inferences) */
    const int32_t *nfr;             /* ragged cascade call: per-stream end frame (SplitGroup) */
};

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/* one half of a gate pre-activation for the warp's four gate tiles (rc_Krows_8x16, affine.c:348-407): acc (+)= W . plane.
 * NK = k-steps when known at compile time (0 = run time); FIRST: the accumulators start here, from the bias (low plane)
 * and zero (high plane), handed to the first k-step as its C operand */
template <int NK, bool FIRST>
__device__ __forceinline__ void scan_half(int nk_rt, const uint8_t *plane, int pa, int lane, const uint2 *__restrict__ w,
                                          int (&ach)[4][4], int (&acl)[4][4], const int32_t (&bz)[4][2])
{
    const int nk = NK ? NK : nk_rt;
    const uint32_t ah = ldm_lane_addr(plane, pa, lane), al = ah + 16 * pa;
    if (FIRST) {
        uint32_t fh[4], fl[4];
        load_a_ldm(ah, fh);
        load_a_ldm(al, fl);
#pragma unroll
        for (int gt = 0; gt < 4; gt++) {
            const uint2 b = w[(gt * nk) * 32];
            imma_s8s8_first(ach[gt], fh, b);
            imma_u8s8_first(acl[gt], fl, b, bz[gt][0], bz[gt][1]);
        }
    }
    if (NK) {
#pragma unroll
        for (int ks = FIRST ? 1 : 0; ks < (NK ? NK : 1); ks++) {
            uint32_t fh[4], fl[4];
            load_a_ldm(ah + 32 * ks, fh);
            load_a_ldm(al + 32 * ks, fl);
#pragma unroll
            for (int gt = 0; gt < 4; gt++) {
                const uint2 b = w[(gt * NK + ks) * 32];
                imma_s8s8(ach[gt], fh, b);
                imma_u8s8(acl[gt], fl, b);
            }
        }
    } else {
#pragma unroll 1
        for (int ks = FIRST ? 1 : 0; ks < nk; ks++) {
            uint32_t fh[4], fl[4];
            load_a_ldm(ah + 32 * ks, fh);
            load_a_ldm(al + 32 * ks, fl);
#pragma unroll
            for (int gt = 0; gt < 4; gt++) {
                const uint2 b = w[(gt * nk + ks) * 32];
                imma_s8s8(ach[gt], fh, b);
                imma_u8s8(acl[gt], fl, b);
            }
        }
    }
}

/* NW = warps per CTA (>= unit groups of the layer), MINB = CTAs per SM the register budget is sized for;
 * KT = k-steps of both the input and the recurrent half when they are equal and known (0 = run time) */
template <int NW, int MINB, int KT>
__global__ void __launch_bounds__(32 * NW, MINB)
scan_kernel(ScanArgs a)
{
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);             /* [0..NST) input ring, [NST] weights, [NST+1] h */
    uint64_t *hbar = bars + SCAN_NST + 1;
    const int WB = 4 * a.nt * (a.kt + a.ktr) * 256, XB = 32 * a.pa;
    const uint2 *wsm = reinterpret_cast<const uint2 *>(smem + 64);
    int2 *lut2_all = reinterpret_cast<int2 *>(smem + 64 + WB);
    const int2 *lut2 = lut2_all + (threadIdx.x & (LUT2_COPIES_SCAN - 1));
    uint8_t *xs = smem + 64 + WB + lut2_bytes(LUT2_COPIES_SCAN);
    uint8_t *hb = xs + SCAN_NST * XB;
    const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;
    __shared__ int sids[16], s_last[16], s_ninf;
    const int tile = blockIdx.x;
    const int nsel = sel_count(a.sel);
    if (16 * tile >= nsel) return;                                   /* (list launches are sized for the worst case) */
    const int nvalid = min(16, nsel - 16 * tile);
    const size_t tile_abs = sel_tile_base(a.sel) + tile;
    const uint8_t *xg = a.xin + tile_abs * (size_t)a.tile_bytes;
    uint8_t *hg = a.hout + tile_abs * (size_t)a.tile_bytes;
    const bool per_row = a.tstart != nullptr;
    if (threadIdx.x < 16) {
        const int r = threadIdx.x;
        const int sid = (r < nvalid) ? sel_sid(a.sel, tile, r) : 0;
        sids[r] = sid;
        /* inferences of this row: the tile runs as many steps as its longest row; a row's state is final after its own
         * last step and is stored right there (cascade rounds start streams at different frames) */
        int ni = 0;
        if (r < nvalid) {
            ni = a.n_inf;
            if (per_row) { const int ts = a.tstart[sid], Ts = stream_frames(a.nfr, sid, a.T); ni = ts < Ts ? (Ts - ts + 1) >> 1 : 0; }
        }
        s_last[r] = ni - 1;
        for (int o = 8; o; o >>= 1) ni = max(ni, __shfl_xor_sync(0x0000ffffu, ni, o));
        if (r == 0) s_ninf = ni;
    }
    __syncthreads();
    const int H = a.H, pa = a.pa, HS = a.hs, T = a.T, n_inf = s_ninf, rs = a.rs;
    if (n_inf <= 0) return;

    if (tid == 0) {
        for (int i = 0; i <= SCAN_NST; i++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bars + i)));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(hbar)), "r"(a.nt));   /* one arrival per active warp */
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 3 * XB / 4; i += nthr) reinterpret_cast<uint32_t *>(hb)[i] = 0;
    fill_lut2<LUT2_COPIES_SCAN>(lut2_all, a.tables, tid, nthr);
    __syncthreads();
    uint8_t *h2 = hb + 2 * XB;                                       /* h before the first inference */
    for (int idx = tid; idx < 16 * H; idx += nthr) {
        const int r = idx / H, u = idx - r * H;
        const int v = (r < nvalid) ? (int)a.h[(long long)sids[r] * HS + a.ho + u] : 0;
        h2[r * pa + u] = (uint8_t)(v >> 8);
        h2[(16 + r) * pa + u] = (uint8_t)v;
    }
    if (tid == 0) {
        const unsigned char *wsrc = reinterpret_cast<const unsigned char *>(a.frag + a.w_off);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bars + SCAN_NST)), "r"((uint32_t)WB) : "memory");
        for (int o = 0; o < WB; o += 32768) {
            const uint32_t n = (uint32_t)min(32768, WB - o);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(smem + 64 + o)), "l"(wsrc + o), "r"(n), "r"(smem_u32(bars + SCAN_NST)) : "memory");
        }
        for (int m = 0; m < SCAN_NST && m < n_inf; m++) bulk_load(xs + m * XB, xg + (size_t)m * XB, XB, bars + m);
    }
    /* the lane's cells: rows g, g+8 x units u0, u0+1 of group `warp`; their biases and cell state stay in registers.
     * Units past H (last group) have zero weights and biases: they are computed like the rest and never stored. */
    const int u0 = 8 * warp + 2 * q;
    int32_t bz[4][2], cst[4];
#pragma unroll
    for (int gt = 0; gt < 4; gt++)
#pragma unroll
        for (int cc = 0; cc < 2; cc++) bz[gt][cc] = (u0 + cc < H) ? a.bias32[a.bias_off + gt * H + u0 + cc] : 0;
#pragma unroll
    for (int e = 0; e < 4; e++) {
        const int row = g + 8 * (e >> 1), u = u0 + (e & 1);
        cst[e] = (row < nvalid && u < H) ? a.c[(long long)sids[row] * HS + a.ho + u] : 0;
    }
    __syncthreads();
    mbar_wait(bars + SCAN_NST, 0);

    const bool active = warp < a.nt;                                  /* spare warps only help with copies and barriers */
    const uint2 *wx = wsm + (size_t)warp * 4 * a.kt * 32 + lane;
    const uint2 *wh = wsm + (size_t)a.nt * 4 * a.kt * 32 + (size_t)warp * 4 * a.ktr * 32 + lane;
    int ach[4][4], acl[4][4];
    auto tap_state = [&](const uint8_t *hp, int t) {                         /* debug taps only */
        if (a.tap_h)
            for (int idx = tid; idx < nvalid * H; idx += nthr) {
                const int r = idx / H, u = idx - r * H;
                a.tap_h[((long long)sids[r] * T + t) * HS + a.ho + u] = (int16_t)(((int)(int8_t)hp[r * pa + u] << 8) | hp[(16 + r) * pa + u]);
            }
        if (a.tap_c && active) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const int row = g + 8 * (e >> 1), u = u0 + (e & 1);
                if (row < nvalid && u < H) a.tap_c[((long long)sids[row] * T + t) * HS + a.ho + u] = cst[e];
            }
        }
    };

    mbar_wait(bars + 0, 0);
    if (active) scan_half<KT, true>(a.kt, xs, pa, lane, wx, ach, acl, bz);   /* b + Wx . x of inference 0 */
    if (a.first == 1) tap_state(h2, 0);                               /* frame 0 ran no inference */

    /* per inference: recurrent half + cell on the accumulators that already hold Wx.x + b; the warp then ARRIVES
     * on the h barrier, issues Wx.x of the next inference (independent of the recurrence), and only then WAITS
     * for the other warps' h slices: the barrier latency hides behind tensor work */
    for (int k = 0; k < n_inf; k++) {
        const uint8_t *hp = hb + ((k + 2) % 3) * XB;                  /* h of the previous inference */
        uint8_t *hn = hb + (k % 3) * XB;
        const int t = a.first + 2 * k;
        if (active) {
            scan_half<KT, false>(a.ktr, hp, pa, lane, wh, ach, acl, bz);   /* + Wh . h_old (lstm.c:54-104 all read the old h) */
            int32_t gate[4][4];
#pragma unroll
            for (int gt = 0; gt < 4; gt++)
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int32_t pre = (int32_t)(((uint32_t)ach[gt][e] << 8) + (uint32_t)acl[gt][e]) >> rs;
                    gate[gt][e] = (gt == 1) ? tanh_q15v<LUT2_COPIES_SCAN>(pre, lut2) : sigmoid_q15v<LUT2_COPIES_SCAN>(pre, lut2);      /* lstm.c:65,78,91,104 */
                }
            int32_t y[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const int64_t tt = ((int64_t)gate[0][e] * (int64_t)gate[1][e] + (int64_t)gate[2][e] * (int64_t)cst[e]) >> 15;   /* lstm.c:108-109 */
                const int32_t cn = sat32_dev(tt);
                cst[e] = cn;
                int32_t o = (tanh_q15v<LUT2_COPIES_SCAN>(cn, lut2) * gate[3][e]) >> 15;                               /* lstm.c:111-115 */
                o = o > 32767 ? 32767 : (o < -32768 ? -32768 : o);
                y[e] = o;
            }
            store_pair(hn, hn + 16 * pa, g * pa + u0, y[0], y[1]);
            store_pair(hn, hn + 16 * pa, (g + 8) * pa + u0, y[2], y[3]);
            if (per_row) {                                            /* a row's last own step: its state goes home now */
#pragma unroll
                for (int rr = 0; rr < 2; rr++) {
                    if (k == s_last[g + 8 * rr]) {                    /* (rows past nvalid have last = -1) */
                        const long long o = (long long)sids[g + 8 * rr] * HS + a.ho + u0;
                        if (u0 < H) { a.h[o] = (int16_t)y[2 * rr]; a.c[o] = cst[2 * rr]; }
                        if (u0 + 1 < H) { a.h[o + 1] = (int16_t)y[2 * rr + 1]; a.c[o + 1] = cst[2 * rr + 1]; }
                    }
                }
            }
            if (a.tap_out && a.tap_act) {
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int row = g + 8 * (e >> 1), u = u0 + (e & 1);
                    if (row < nvalid && u < H) a.tap_act[((long long)sids[row] * T + t) * a.act_stride + a.ao + u] = (int16_t)y[e];
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  /* h slice -> visible to the bulk store */
            __syncwarp();
            if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   /* buffer of step k-2 is free again */
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(hbar)) : "memory");
            if (k + 1 < n_inf) {                                      /* Wx . x of the next inference, off the recurrence */
                mbar_wait(bars + ((k + 1) % SCAN_NST), (uint32_t)(((k + 1) / SCAN_NST) & 1));
                scan_half<KT, true>(a.kt, xs + ((k + 1) % SCAN_NST) * XB, pa, lane, wx, ach, acl, bz);
            }
        }
        mbar_wait(hbar, (uint32_t)(k & 1));                           /* every slice of h(k) is in hn */
        if (tid == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(hg + (size_t)k * XB), "r"(smem_u32(hn)), "r"((uint32_t)XB) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            /* x(k) was consumed before anyone arrived for step k - 1 .. k: its slot takes x(k + NST) */
            const int m = k + SCAN_NST;
            if (m < n_inf) bulk_load(xs + (k % SCAN_NST) * XB, xg + (size_t)m * XB, XB, bars + (k % SCAN_NST));
        }
        if (a.tap_h || a.tap_c) {
            tap_state(hn, t);
            if (t + 1 < T) tap_state(hn, t + 1);
        }
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (per_row) return;                                             /* every row stored its state after its own last step */
    /* state for the next call */
    const uint8_t *hf = hb + ((n_inf + 2) % 3) * XB;
    for (int idx = tid; idx < nvalid * H; idx += nthr) {
        const int r = idx / H, u = idx - r * H;
        a.h[(long long)sids[r] * HS + a.ho + u] = (int16_t)(((int)(int8_t)hf[r * pa + u] << 8) | hf[(16 + r) * pa + u]);
    }
    if (active) {
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int row = g + 8 * (e >> 1), u = u0 + (e & 1);
            if (row < nvalid && u < H) a.c[(long long)sids[row] * HS + a.ho + u] = cst[e];
        }
    }
}

/* ======================================================================================================== */
/* post_kernel / ctx_kernel / feat_tap_kernel                                                                */
/* ======================================================================================================== */
constexpr int POST_THREADS = 64;                    /* streams per CTA */
constexpr int POST_KCH = 64;                        /* decision records staged per round */

struct PostArgs {
    int nn_id, s0, ns, T, first, n_inf, dec_stride;
    const int32_t *dec;
    int16_t *scal;
    nnsp_b200_result *results;
    int16_t *tap_post;
    int16_t th_count;
};

/* the NNSPClass state machine of every stream over the call's frames (nn_speech.c:84-125); one thread per stream,
 * decision records staged through shared memory so that the loop has no dependent global load */
__global__ void __launch_bounds__(POST_THREADS) post_kernel(PostArgs a)
{
    __shared__ int32_t dsm[POST_THREADS][POST_KCH + 1];
    const int si0 = blockIdx.x * POST_THREADS, si = si0 + threadIdx.x;
    const bool valid = si < a.ns;
    const long long s = a.s0 + (valid ? si : 0);
    PostRegs r;
    {
        int16_t sc[SC_N];
        const uint4 *p = reinterpret_cast<const uint4 *>(a.scal + s * SC_N);
        *reinterpret_cast<uint4 *>(&sc[0]) = p[0];
        *reinterpret_cast<uint4 *>(&sc[8]) = p[1];
        r.trig = sc[SC_TRIGGER]; r.out0 = sc[SC_OUT0]; r.out1 = sc[SC_OUT0 + 1]; r.out2 = sc[SC_OUT0 + 2];
#pragma unroll
        for (int i = 0; i < 8; i++) r.cnt[i] = sc[SC_CNT0 + i];
        r.last = sc[SC_ARGMAX_LAST]; r.slides = sc[SC_SLIDES];
    }
    const int th = a.th_count;
    const int nstr = min(POST_THREADS, a.ns - si0);
    auto emit = [&](int t, bool ran) {                                /* frame t is over: result record (+ tap) */
        r.slides ^= 1;                                                /* nn_speech.c:125 */
        if (a.results) {
            uint2 w;
            w.x = (uint32_t)(uint16_t)r.trig | ((uint32_t)(uint16_t)r.out0 << 16);
            w.y = (uint32_t)(uint16_t)r.out1 | ((uint32_t)(uint16_t)r.out2 << 16);
            *reinterpret_cast<uint2 *>(a.results + s * a.T + t) = w;
        }
        if (a.tap_post) {
            int16_t *o = a.tap_post + (s * a.T + t) * SC_N;
            o[SC_TRIGGER] = (int16_t)r.trig; o[SC_OUT0] = (int16_t)r.out0; o[SC_OUT0 + 1] = (int16_t)r.out1; o[SC_OUT0 + 2] = (int16_t)r.out2;
#pragma unroll
            for (int i = 0; i < 8; i++) o[SC_CNT0 + i] = (int16_t)r.cnt[i];
            o[SC_ARGMAX_LAST] = (int16_t)r.last; o[SC_SLIDES] = (int16_t)r.slides;
            o[SC_RAN] = ran ? 1 : 0; o[SC_STAGE] = (int16_t)a.nn_id;
        }
    };
    if (valid && a.first == 1) emit(0, false);                        /* frame 0 ran no inference (nn_speech.c:84) */
    for (int kc = 0; kc < a.n_inf; kc += POST_KCH) {
        const int nk = min(POST_KCH, a.n_inf - kc);
        __syncthreads();
        for (int e = threadIdx.x; e < nstr * nk; e += POST_THREADS) {
            const int rr = e / nk, kk = e - rr * nk;
            dsm[rr][kk] = a.dec[(size_t)(a.s0 + si0 + rr) * a.dec_stride + kc + kk];
        }
        __syncthreads();
        if (valid) {
            for (int kk = 0; kk < nk; kk++) {
                const int t = a.first + 2 * (kc + kk);
                const int dv = dsm[threadIdx.x][kk];
                if (a.nn_id == NNSP_B200_ID_S2I) apply_s2i(r, dv, th);                        /* nn_speech.c:97-119 */
                else apply_binary(r, dv, th);
                emit(t, true);
                if (t + 1 < a.T) emit(t + 1, false);
            }
        }
    }
    if (valid) {
        int16_t sc[SC_N];
        sc[SC_TRIGGER] = (int16_t)r.trig; sc[SC_OUT0] = (int16_t)r.out0; sc[SC_OUT0 + 1] = (int16_t)r.out1; sc[SC_OUT0 + 2] = (int16_t)r.out2;
#pragma unroll
        for (int i = 0; i < 8; i++) sc[SC_CNT0 + i] = (int16_t)r.cnt[i];
        sc[SC_ARGMAX_LAST] = (int16_t)r.last; sc[SC_SLIDES] = (int16_t)r.slides;
        sc[SC_RAN] = 0; sc[SC_STAGE] = 0;
        uint4 *p = reinterpret_cast<uint4 *>(a.scal + s * SC_N);
        p[0] = *reinterpret_cast<uint4 *>(&sc[0]);
        p[1] = *reinterpret_cast<uint4 *>(&sc[8]);
    }
}

/* normFeatContext after the call: the newest 6 rows of (old rows ++ this call's standardised rows); a warp per stream */
__global__ void __launch_bounds__(256) ctx_kernel(const int16_t *__restrict__ feat16, int16_t *ctx, int s0, int ns, int T)
{
    const int si = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (si >= ns) return;
    const long long s = s0 + si;
    uint4 *c4 = reinterpret_cast<uint4 *>(ctx + s * 240);                /* 30 pieces of 8 features */
    uint4 v = make_uint4(0, 0, 0, 0);
    if (lane < 30) {
        const int j = lane / 5, x = lane - j * 5, f = T - 6 + j;         /* new row j <- frame f of this call, or old row j + T */
        v = (f >= 0) ? __ldg(reinterpret_cast<const uint4 *>(feat16 + (s * T + f) * NNSP_B200_NMEL) + x) : c4[(j + T) * 5 + x];
    }
    __syncwarp();
    if (lane < 30) c4[lane] = v;
}

/* debug taps of the front end: standardised row and (from a second, log-mel pass of feat_kernel) the log-mel row */
__global__ void feat_tap_kernel(const int16_t *__restrict__ feat16, int16_t *feat, long long base, long long n)
{
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        feat[base + e] = feat16[base + e];
}

/* ======================================================================================================== */
/* host                                                                                                      */
/* ======================================================================================================== */
struct SegLayout { int off_bias, off_lut, off_w, off_fp, off_row, off_wb, off_log, nbuf, w_base, w_bytes; size_t total; };

/* row_tab: the per-item source table of the log-mel staging (seg_kernel<2>) */
static SegLayout seg_layout(const MmaModel *D, int l0, int l1, bool from_feat, bool row_tab)
{
    SegLayout s{};
    auto a16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    size_t off = a16(16 + sizeof(MmaModel));
    s.off_bias = (int)off; off = a16(off + (size_t)D->bias_count * 4);
    s.off_lut = (int)off; off += lut2_bytes(LUT2_COPIES_SEG);
    s.w_base = D->layer[l0].w_off;
    long long cnt = 0;
    for (int i = l0; i < l1; i++) cnt += (long long)D->layer[i].nt * D->layer[i].kt * 32;
    s.w_bytes = (int)(cnt * 8);
    off = (off + 127) & ~(size_t)127;
    s.off_w = (int)off; off += (size_t)s.w_bytes;
    s.off_fp = (int)off; if (from_feat) off += 2 * 16 * SEG_PC;
    s.off_row = (int)off; if (row_tab) off += 16 * SEG_FROWS * sizeof(uintptr_t);
    s.nbuf = (from_feat && l1 - l0 == 1) ? 1 : 2;
    s.off_wb = (int)off; off += (size_t)SEG_WARPS * s.nbuf * 32 * D->pa;
    s.off_log = (int)off; if (l1 == D->numlayers) off += (size_t)SEG_WARPS * 16 * (D->no + 4) * 4;
    s.total = off;
    return s;
}
static size_t scan_smem(const MmaModel *D, const MmaLayer &L)
{
    return 64 + (size_t)4 * L.nt * (L.kt + L.ktr) * 256 + lut2_bytes(LUT2_COPIES_SCAN) + (size_t)(SCAN_NST + 3) * 32 * D->pa;   /* 64: 6 mbarriers */
}

int split_supported(const MmaDeviceModel &mm)
{
    const MmaModel *D = mm.h;
    if (!D || D->numlayers < 1) return 0;
    if (D->layer[0].type != LAYER_FC || D->layer[D->numlayers - 1].type != LAYER_FC) return 0;
    if (D->nn_id == NNSP_B200_ID_S2I ? D->n_out < 41 : D->n_out < 2) return 0;
    for (int i = 0; i < D->numlayers; i++) {
        const MmaLayer &L = D->layer[i];
        if (!L.fast) return 0;
        if (L.type == LAYER_FC && L.act == ACT_LINEAR && i != D->numlayers - 1) return 0;
        if (L.type == LAYER_LSTM && (L.nt > 16 || scan_smem(D, L) > (size_t)SPLIT_MAX_DYN_SMEM)) return 0;
        if (L.type == LAYER_LSTM && L.wh_off != L.w_off + 4 * L.nt * L.kt * 32) return 0;
    }
    for (int l0 = 0; l0 < D->numlayers;) {                           /* every fc run must fit shared memory */
        int l1 = l0;
        while (l1 < D->numlayers && D->layer[l1].type == LAYER_FC) l1++;
        /* with the staging table: any model may run in a cascade */
        if (l1 > l0 && seg_layout(D, l0, l1, l0 == 0, l0 == 0).total > (size_t)SPLIT_MAX_DYN_SMEM) return 0;
        l0 = (l1 > l0) ? l1 : l0 + 1;
    }
    return 1;
}

size_t split_plane_bytes(const MmaDeviceModel &mm, int n_streams, int n_inf)
{
    return (size_t)((n_streams + 15) / 16) * (size_t)n_inf * 32 * mm.h->pa;
}

/* kind: the index nnsp_b200_scan_kernel_launches counts this specialisation under */
template <int NW, int MINB, int KT>
static int launch_scan(int kind, const ScanArgs &a, int ntiles, size_t smem, int device, cudaStream_t st)
{
    static bool attr_done[64] = { false };
    static std::mutex attr_mu;                         /* host threads may drive separate handles on one device */
    std::unique_lock<std::mutex> attr_lk(attr_mu);
    if (!attr_done[device]) {
        NNSP_CUDA(cudaFuncSetAttribute(scan_kernel<NW, MINB, KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SPLIT_MAX_DYN_SMEM));
        NNSP_CUDA(cudaFuncSetAttribute(scan_kernel<NW, MINB, KT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_done[device] = true;
    }
    attr_lk.unlock();
    scan_kernel<NW, MINB, KT><<<ntiles, 32 * NW, smem, st>>>(a);
    NNSP_LAUNCH_CHECK();
    g_scan_launches[kind].fetch_add(1, std::memory_order_relaxed);
    return NNSP_B200_OK;
}

/* The tcgen05 layer-0 kernel works on tiles of 2 streams x 64 inference slots; a call with few inferences per stream fills
 * few of the slots (a 2-frame call: 1 of 64) and the mma.sync kernel, whose cost follows the rows, is faster -- measured
 * break-even near half-full tiles (4 096 streams x 2 frames: 59 vs 48 us per call; 100-frame calls: 240 vs 395 us).
 * NNSP_B200_TC5: 0 = never, 2 = whenever the layer qualifies (tests), otherwise by that rule. */
/* The window rows of a cascade round, once per stream instead of once per 16-inference work item: row v of stream s is
 * frame tstart[s] - 5 + v of the call, for v < 2 * (its inferences) + 4. Sources exactly as seg_kernel<2> stages them:
 * frames before the instance's life in this call began are its stored context rows (already standardised); later ones are
 * log-mel rows -- of the instance's first two frames (lmfix), of this call, or of the carried history, by the model's
 * look-back (PcmBufClass_getData, PcmBufClass.c:38-85) -- standardised with the model's statistics
 * (feature_module.c:67-73). One thread per (stream, row, 4 features). */
struct VseqArgs {
    const MmaModel *model;
    const int *list, *count;
    const int *tstart, *tb, *age0;
    const int32_t *logmel, *lmhist, *lmfix;
    const int16_t *ctx;
    int T, dmax, dback, rows;
    int16_t *vseq;
    const int32_t *nfr;
};
__global__ void __launch_bounds__(256) vseq_kernel(VseqArgs a)
{
    const int nsel = *a.count;
    const long long total = (long long)nsel * a.rows * 10;
    const MmaModel &M = *a.model;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int p = (int)(e / (a.rows * 10)), rem = (int)(e - (long long)p * a.rows * 10), v = rem / 10, x = rem - v * 10;
        const long long s = a.list[p];
        const int ts = a.tstart[s], Ts = stream_frames(a.nfr, s, a.T);
        const int ninf = ts < Ts ? (Ts - ts + 1) >> 1 : 0;
        if (v >= 2 * ninf + 4 || ninf == 0) continue;
        const int f = ts - 5 + v, life = f - a.tb[s];
        int16_t w[4] = { 0, 0, 0, 0 };
        if (life < 0) {
            const uint2 c = *reinterpret_cast<const uint2 *>(a.ctx + s * 240 + (6 + life) * 40 + x * 4);
            *reinterpret_cast<uint2 *>(w) = c;
        } else if (f < a.T) {
            const int la = life + a.age0[s], fr = f - a.dback;
            const int32_t *row = (la < 2) ? a.lmfix + (s * 2 + la) * NNSP_B200_NMEL
                               : (fr >= 0) ? a.logmel + (s * a.T + fr) * NNSP_B200_NMEL
                                           : a.lmhist + (s * a.dmax + a.dmax + fr) * NNSP_B200_NMEL;
            const int4 q = __ldg(reinterpret_cast<const int4 *>(row + x * 4));
            const int32_t u[4] = { q.x, q.y, q.z, q.w };
#pragma unroll
            for (int c = 0; c < 4; c++) w[c] = standardise(u[c], M.mean[4 * x + c], M.stdR[4 * x + c], M.feat_rshift);
        }
        *reinterpret_cast<uint2 *>(a.vseq + (s * a.rows + v) * NNSP_B200_NMEL + x * 4) = *reinterpret_cast<const uint2 *>(w);
    }
}

/* debug tap of a tcgen05 layer 0 (batched NNSPClass): its int16 outputs back from the byte planes it wrote, decoded like
 * the tap of seg_kernel. Runs right behind seg0_tc5_kernel, before anything reuses that plane buffer. */
__global__ void tc5_tap_kernel(const uint8_t *planes, long long tile_bytes, int pa, int tile0, int s0, int ns, int T,
                               int first, int n_inf, int H, int act_stride, int16_t *tap_act)
{
    const long long n = (long long)ns * n_inf * H;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int u = (int)(i % H);
        const long long pk = i / H;
        const int k = (int)(pk % n_inf), p = (int)(pk / n_inf);
        const uint8_t *x = planes + (size_t)(tile0 + (p >> 4)) * (size_t)tile_bytes + (size_t)k * 32 * pa + (p & 15) * pa + u;
        tap_act[((long long)(s0 + p) * T + first + 2 * k) * act_stride + u] = (int16_t)(((int)(int8_t)x[0] << 8) | x[16 * pa]);
    }
}

static bool tc5_wanted(int n_inf)
{
    const char *e = getenv("NNSP_B200_TC5");
    if (e && e[0] == '0') return false;
    if (e && e[0] == '2') return true;
    const int nchunks = (n_inf + TC5_KC - 1) / TC5_KC;
    return 20 * n_inf >= 9 * nchunks * TC5_SLOTS;                 /* slots in use >= 45 % */
}

/* the fc runs and lstm scans of one model over one stream selection (launch_nn_split: a range of a batch;
 * cascade: a device-side list). mode: 1 = feat16 input, 2 = log-mel input with look-back. Returns through *dec. */
int launch_split_layers(const MmaDeviceModel &mm, const SplitGroup &q, int device, cudaStream_t st)
{
    const MmaModel *D = mm.h;
    static bool attr_done[64] = { false };
    static std::mutex attr_mu;                         /* host threads may drive separate handles on one device */
    std::unique_lock<std::mutex> attr_lk(attr_mu);
    if (!attr_done[device]) {
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SPLIT_MAX_DYN_SMEM));
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SPLIT_MAX_DYN_SMEM));
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SPLIT_MAX_DYN_SMEM));
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<0>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        NNSP_CUDA(cudaFuncSetAttribute(seg_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        NNSP_CUDA(cudaFuncSetAttribute(seg0_tc5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Tc5Smem) + 1024));
        attr_done[device] = true;
    }
    attr_lk.unlock();
    if (q.n_inf <= 0 || q.max_streams <= 0) return NNSP_B200_OK;
    StreamSel sel{};
    sel.list = q.list; sel.count = q.count; sel.tile_off = q.tile_off; sel.s0 = q.s0; sel.ns = q.ns; sel.tile0 = q.tile0;
    const int ntiles = (q.max_streams + 15) / 16, nchunks = (q.n_inf + SEG_KC - 1) / SEG_KC;
    const long long tile_bytes = q.tile_bytes ? q.tile_bytes : (long long)q.n_inf * 32 * D->pa;
    const nnsp_b200_taps &tp = q.taps;
    uint8_t *cur_in = nullptr, *bufs[2] = { q.planes0, q.planes1 };
    int which = 0, li = 0, ao = 0, ho = 0, rc;
    bool from_feat = true;
    while (li < D->numlayers) {
        int l1 = li;
        while (l1 < D->numlayers && D->layer[l1].type == LAYER_FC) l1++;
        const bool tc5_batch = q.mode == 1 && !q.list && !q.tstart;                       /* the batched NNSPClass */
        const bool tc5_round = q.mode == 2 && q.list && q.tstart && q.vseq && !tp.act;     /* first round of the cascade (never tapped: cascade_use_split) */
        /* a tapped batch call takes the same layer-0 kernel as an untapped one: tc5_tap_kernel reads its outputs back */
        if (l1 > li && from_feat && l1 == 1 && (tc5_batch || tc5_round) && mm.tc5 && D->pa <= TC5_PAMAX && tc5_wanted(q.n_inf)) {
            /* layer 0 on the tcgen05 tensor cores (nnsp_tc5.cuh) */
            if (tc5_round) {
                VseqArgs v{};
                v.model = mm.d; v.list = q.list; v.count = q.count; v.tstart = q.tstart; v.tb = q.tb; v.age0 = q.age0;
                v.logmel = q.logmel; v.lmhist = q.lmhist; v.lmfix = q.lmfix; v.ctx = q.ctx;
                v.T = q.T; v.dmax = q.dmax; v.dback = q.dback; v.rows = q.vseq_rows; v.vseq = q.vseq; v.nfr = q.nfr;
                long long work = (long long)q.max_streams * q.vseq_rows * 10;
                int grid = (int)((work + 255) / 256);
                grid = grid < 1 ? 1 : (grid > 8 * sm_count(device) ? 8 * sm_count(device) : grid);
                vseq_kernel<<<grid, 256, 0, st>>>(v);
                NNSP_LAUNCH_CHECK();
            }
            Tc5Args a{};
            a.img = mm.tc5; a.tables = q.tables; a.np = mm.tc5_np; a.rs = -D->layer[0].sh_out;
            a.s0 = q.s0; a.ns = q.ns; a.tile0 = q.tile0;
            a.T = q.T; a.first = q.first; a.n_inf = q.n_inf; a.nchunks = (q.n_inf + TC5_KC - 1) / TC5_KC;
            a.pa = D->pa; a.tile_bytes = tile_bytes;
            a.feat16 = q.feat16; a.ctx = q.ctx; a.out_planes = bufs[which];
            if (tc5_round) { a.list = q.list; a.count = q.count; a.tile_off = q.tile_off; a.tstart = q.tstart; a.vseq = q.vseq; a.vf = q.vseq_rows; a.nfr = q.nfr; }
            const int nitems = (((tc5_round ? q.max_streams : q.ns) + 1) / 2) * a.nchunks;
            const int grid = nitems < sm_count(device) ? nitems : sm_count(device);
            seg0_tc5_kernel<<<grid, TC5_THREADS, sizeof(Tc5Smem) + 1024, st>>>(a);
            NNSP_LAUNCH_CHECK();
            g_tc5_launches.fetch_add(1, std::memory_order_relaxed);
            if (tp.act) {
                const long long n = (long long)q.ns * q.n_inf * D->layer[0].rows;
                const int tgrid = (int)((n + 255) / 256 < 4 * sm_count(device) ? (n + 255) / 256 : 4 * sm_count(device));
                tc5_tap_kernel<<<tgrid, 256, 0, st>>>(bufs[which], tile_bytes, D->pa, q.tile0, q.s0, q.ns, q.T, q.first, q.n_inf,
                                                      D->layer[0].rows, D->act_stride, tp.act);
                NNSP_LAUNCH_CHECK();
            }
            ao += D->layer[0].rows;
            cur_in = bufs[which]; which ^= 1;
            from_feat = false;
            li = l1;
        } else
        if (l1 > li) {                                           /* a run of fc layers */
            const SegLayout lay = seg_layout(D, li, l1, from_feat, from_feat && q.mode == 2);
            SegArgs a{};
            a.model = mm.d; a.frag = (const uint2 *)mm.frag; a.bias32 = mm.bias32; a.tables = q.tables;
            a.l0 = li; a.l1 = l1; a.w_base = lay.w_base; a.w_bytes = lay.w_bytes;
            a.off_bias = lay.off_bias; a.off_lut = lay.off_lut; a.off_w = lay.off_w; a.off_fp = lay.off_fp; a.off_row = lay.off_row;
            a.off_wb = lay.off_wb; a.off_log = lay.off_log; a.nbuf = lay.nbuf;
            a.sel = sel; a.T = q.T; a.first = q.first; a.n_inf = q.n_inf; a.nchunks = nchunks;
            a.tile_bytes = tile_bytes; a.dec_stride = q.dec_stride;
            a.feat16 = q.feat16; a.logmel = q.logmel; a.lmhist = q.lmhist; a.dmax = q.dmax; a.dback = q.dback;
            a.ctx = q.ctx; a.in_planes = cur_in;
            a.out_planes = (l1 < D->numlayers) ? bufs[which] : nullptr;
            a.dec = q.dec; a.tap_act = tp.act; a.tap_logits = tp.logits; a.ao0 = ao; a.thresh_prob = q.thresh_prob; a.thr_prob = q.thr_prob; a.thr_stride = q.thr_stride;
            a.tstart = q.tstart; a.tb = q.tb; a.age0 = q.age0; a.lmfix = q.lmfix; a.nfr = q.nfr;
            int per_sm = (int)((227 * 1024) / (lay.total + 1024));
            per_sm = per_sm < 1 ? 1 : (per_sm > SEG_MINB ? SEG_MINB : per_sm);     /* __launch_bounds__(256, SEG_MINB) */
            int grid = sm_count(device) * per_sm;
            if (grid > nchunks * ntiles) grid = nchunks * ntiles;
            if (!from_feat) seg_kernel<0><<<grid, SEG_THREADS, lay.total, st>>>(a);
            else if (q.mode == 2) seg_kernel<2><<<grid, SEG_THREADS, lay.total, st>>>(a);
            else seg_kernel<1><<<grid, SEG_THREADS, lay.total, st>>>(a);
            NNSP_LAUNCH_CHECK();
            for (int i = li; i < l1; i++) if (i < D->numlayers - 1) ao += D->layer[i].rows;
            if (l1 < D->numlayers) { cur_in = bufs[which]; which ^= 1; }
            from_feat = false;
            li = l1;
        }
        if (li < D->numlayers) {                                 /* an lstm layer */
            const MmaLayer &L = D->layer[li];
            ScanArgs a{};
            a.frag = (const uint2 *)mm.frag; a.bias32 = mm.bias32; a.tables = q.tables;
            a.H = L.rows; a.kt = L.kt; a.ktr = L.ktr; a.nt = L.nt; a.rs = -L.sh_out; a.w_off = L.w_off; a.bias_off = L.bias_off; a.pa = D->pa;
            a.ho = ho; a.hs = q.h_stride; a.ao = ao; a.act_stride = D->act_stride; a.tap_out = (li < D->numlayers - 1);
            a.sel = sel; a.T = q.T; a.first = q.first; a.n_inf = q.n_inf; a.tile_bytes = tile_bytes;
            a.xin = cur_in; a.hout = bufs[which]; a.h = q.h; a.c = q.c;
            a.tap_act = tp.act; a.tap_h = tp.hstate; a.tap_c = tp.cstate; a.tstart = q.tstart; a.nfr = q.nfr;
            const size_t smem = scan_smem(D, L);
            /* the shipped layers get their k-step counts compiled in: VAD 28 -> 28 (1 k-step), KWS 64 -> 64 (2), S2I 72 -> 72 (3) */
            const int kq = (L.kt == L.ktr) ? L.kt : 0;
            if (L.nt <= 4) rc = (kq == 1) ? launch_scan<4, 4, 1>(0, a, ntiles, smem, device, st) : launch_scan<4, 4, 0>(1, a, ntiles, smem, device, st);
            /* 64-unit layers (KWS): eight unit groups take eight warps, not nine (-2 % of the network time; capping the
             * registers for three CTAs per SM spills and gains nothing: profiles/r2_cascade_overlap.txt) */
            else if (L.nt <= 8 && kq == 2) rc = launch_scan<8, 2, 2>(2, a, ntiles, smem, device, st);
            /* kq is 3 or 0 here: nt 9 is H in 65..72 (ktr 3), and H in 33..64 with kq 2 took the branch above */
            else if (L.nt <= 9) rc = (kq == 3) ? launch_scan<9, 2, 3>(3, a, ntiles, smem, device, st) : launch_scan<9, 2, 0>(4, a, ntiles, smem, device, st);
            else rc = launch_scan<16, 1, 0>(5, a, ntiles, smem, device, st);
            if (rc) return rc;
            cur_in = bufs[which]; which ^= 1;
            ao += L.rows; ho += L.rows;
            li++;
        }
    }
    return NNSP_B200_OK;
}

int launch_nn_split(const MmaDeviceModel &mm, const NNLaunch &l, const int16_t *feat16, int first, int n_inf,
                    uint8_t *planes0, uint8_t *planes1, int32_t *dec, int cap_inf, int device, cudaStream_t st)
{
    /* cap_inf: the inference capacity the plane / decision buffers were allocated for. Strides follow the capacity, not
     * this call's n_inf, so that a stream slice owns the same bytes in every call (calls of different lengths may be in
     * flight on different CUDA streams of the host-buffer pipeline) */
    if (cap_inf < n_inf) cap_inf = n_inf;
    const MmaModel *D = mm.h;
    if (l.ns <= 0 || l.T <= 0) return NNSP_B200_OK;
    if ((l.s0 & 15) != 0) { nnsp_set_error("stream slices of the split path must start at a multiple of 16"); return NNSP_B200_ERR_ARG; }
    const int T = l.T;
    const nnsp_b200_taps &tp = l.taps;
    int rc;
    if (tp.feat) {
        const long long fbase = (long long)l.s0 * T * NNSP_B200_NMEL, fcount = (long long)l.ns * T * NNSP_B200_NMEL;
        const long long nb = (fcount + 255) / 256;
        feat_tap_kernel<<<(unsigned)(nb > 4096 ? 4096 : nb), 256, 0, st>>>(feat16, tp.feat, fbase, fcount);
        NNSP_LAUNCH_CHECK();
    }
    if (tp.act) NNSP_CUDA(cudaMemsetAsync(tp.act + (long long)l.s0 * T * D->act_stride, 0, (size_t)l.ns * T * D->act_stride * 2, st));
    if (tp.logits) NNSP_CUDA(cudaMemsetAsync(tp.logits + (long long)l.s0 * T * D->n_out, 0, (size_t)l.ns * T * D->n_out * 4, st));

    if (n_inf > 0) {
        SplitGroup q{};
        q.tables = l.tables; q.s0 = l.s0; q.ns = l.ns; q.tile0 = l.s0 >> 4; q.max_streams = l.ns;
        q.T = T; q.first = first; q.n_inf = n_inf; q.mode = 1; q.feat16 = feat16; q.ctx = l.st.ctx;
        q.h = l.st.h; q.c = l.st.c; q.h_stride = D->h_stride; q.planes0 = planes0; q.planes1 = planes1;
        q.dec = dec; q.dec_stride = cap_inf; q.tile_bytes = (long long)cap_inf * 32 * D->pa; q.thresh_prob = l.thresh_prob; q.taps = tp;
        if ((rc = launch_split_layers(mm, q, device, st))) return rc;
    } else if ((tp.hstate || tp.cstate) && D->h_stride > 0) {
        /* a call without any inference (one frame, slides == 0): the state taps repeat the stored state */
        for (int si = 0; si < l.ns; si++) {
            const long long s = l.s0 + si;
            if (tp.hstate) NNSP_CUDA(cudaMemcpyAsync(tp.hstate + s * T * D->h_stride, l.st.h + s * D->h_stride, (size_t)D->h_stride * 2, cudaMemcpyDeviceToDevice, st));
            if (tp.cstate) NNSP_CUDA(cudaMemcpyAsync(tp.cstate + s * T * D->h_stride, l.st.c + s * D->h_stride, (size_t)D->h_stride * 4, cudaMemcpyDeviceToDevice, st));
        }
    }
    {
        PostArgs p{};
        p.nn_id = D->nn_id; p.s0 = l.s0; p.ns = l.ns; p.T = T; p.first = first; p.n_inf = n_inf; p.dec_stride = cap_inf;
        p.dec = dec; p.scal = l.st.scal; p.results = l.results; p.tap_post = tp.post; p.th_count = l.th_count;
        post_kernel<<<(l.ns + POST_THREADS - 1) / POST_THREADS, POST_THREADS, 0, st>>>(p);
        NNSP_LAUNCH_CHECK();
    }
    ctx_kernel<<<(l.ns * 32 + 255) / 256, 256, 0, st>>>(feat16, l.st.ctx, l.s0, l.ns, T);
    NNSP_LAUNCH_CHECK();
    return NNSP_B200_OK;
}

}  // namespace nnsp
