/* nnsp_cascade.cu -- batched nnCntrlClass: the VAD -> KWS -> S2I gated cascade, one controller per
 * stream (evb/src/nnCntrlClass.c:56-272, PcmBufClass.c:10-85, ParamsNNCntrl.h:8-21).
 *
 * What the reference keeps per stream: three NNSPClass instances (own FeatureClass, own LSTM state),
 * a 100-frame PCM ring with look-back, two timeout counters and the sequence position. Exactly one
 * instance runs per frame, and an instance is always reset when the controller leaves it, so the
 * engine keeps ONE live instance state per stream plus what survives a reset in the reference:
 * context row 5 of every instance (feature_module.c:39-42 refills rows 0..4 only).
 *
 * Per exec call:
 *   feat_kernel    : log-mel of every raw (undelayed) frame of the call, full 3-frame window; also the
 *                    newest d_max+2 PCM frames and d_max log-mel rows, the next call's histories
 *   cascade_kernel : per stream (one warp), frame by frame: pick the active model and its look-back d,
 *                    take the log-mel row of frame t-d (this call or the log-mel history), or -- for the
 *                    first two frames after an activation, whose window is partly the zeroed
 *                    dataBuffer -- recompute it on the spot; standardise, network, post-processing,
 *                    controller transition, reset-on-exit */
#include <algorithm>
#include <cstdlib>
#include <cuda_runtime.h>
#include <vector>
#include <new>
#include <string.h>

#include "nnsp_feat.cuh"
#include "nnsp_host.h"
#include "nnsp_mma.cuh"
#include "nnsp_net.cuh"
#include "nnsp_tma.cuh"

namespace nnsp {

/* Two shapes of the sequential kernel. WIDE: any model the engine accepts, 8 warps per CTA, a front-end scratch per warp.
 * NARROW (all models at most 80 wide, 48 outputs -- the shipped three): the per-stream scratch shrinks to 2.1 KB and the
 * front-end scratch, needed only for the two frames after an instance reset, is a pool of 4 per CTA behind a lock, so
 * 16 warps fit next to the three weight images. The kernel is latency-bound (one warp walks one stream), so the
 * resident warps are what it runs on. */
struct CsWide   { using WS = WarpScratch;            static constexpr int WARPS = 8,  NFS = 8; static constexpr bool POOL = false; };
struct CsNarrow { using WS = WarpScratchT<80, 48>;   static constexpr int WARPS = 16, NFS = 4; static constexpr bool POOL = true;  };
constexpr int CS_MAXSEQ = 3;
constexpr int LOGMEL_OF_ZERO = 0x2688 * -15;     /* log10_q15(0): fixlog10.c:39-47 with x -> 1 */

/* ParamCntrlClass is a member of every nnCntrlClass instance (nnCntrlClass.h:12-29), i.e. per stream: the thresholds and
 * time-outs of a stream live in a 16-byte device record (nnsp_b200_cascade_set_stream_params); the look-back depths size
 * the history buffers and stay per handle (CascadeDev.P). prob / cnts are indexed by NNSP id. */
struct CascThr { int16_t prob[3], cnts[3], timeout_kws, timeout_s2i; };
static_assert(sizeof(CascThr) == 16, "one 128-bit load per stream");

struct CascadeDev {                   /* small, by value in kernel params */
    int seq[CS_MAXSEQ], len_seq;
    nnsp_b200_cascade_params P;       /* look-back depths; the thresholds of a stream are thr[stream] */
    const CascThr *thr;
    int dmax;                         /* max look-back frames over the ids in seq */
    int wbytes[3], woff_words[3], boff[3];   /* per id: weight bytes, word offset of its image in smem, bias offset */
};

struct CascadeArgs {
    const DevModel *model[3];
    const uint32_t *wimg[3];
    const int16_t *bimg[3];
    const DevTables *tables;
    StreamState st;                   /* ctx/h/c/scal of the live instance, hist, lmhist, casc */
    int16_t *stale;                   /* [S][3][40] context row 5 left behind by each instance */
    const int16_t *pcm; long long stride;
    const int32_t *logmel;            /* [S][T][40] of this call */
    int s0, ns, T;
    nnsp_b200_cascade_result *results;
    nnsp_b200_taps taps;
    CascadeDev cd;
    const int *t0;                    /* per stream: first frame this kernel still has to process (null: 0) */
    const int *replay_list;           /* with t0: the streams that still have frames left, handed out dynamically ... */
    int *replay_ctl;                  /* ... [0] = how many, [1] = cursor                                         */
    const int32_t *nfr;               /* ragged call: stream s runs frames [0, stream_frames(nfr, s, T)) (null: all T) */
};

/* frames [Ts, T) of stream s in a ragged call: "no frame" records -- stage_id -1, every other field 0 -- by the threads
 * i0, i0 + step, ... (12-byte records, written as 4-byte words) */
__device__ __forceinline__ void write_no_frames(nnsp_b200_cascade_result *results, long long s, int Ts, int T, int i0, int step)
{
    uint32_t *out = reinterpret_cast<uint32_t *>(results + s * T);
    for (int i = 3 * Ts + i0; i < 3 * T; i += step) out[i] = (i % 3 == 0) ? 0xffu : 0u;
}

__device__ __forceinline__ CascThr load_thr(const CascadeDev &cd, long long s)
{
    CascThr t;
    *reinterpret_cast<int4 *>(&t) = __ldg(reinterpret_cast<const int4 *>(cd.thr + s));
    return t;
}

template <class V>
struct CascadeSmem {
    FeatSmemTables ft;
    int16_t tanh_lut[384];
    DevModel model[3];
    FrameScratch fs[V::NFS];
    typename V::WS ws[V::WARPS];
    int fs_lock[V::NFS];
};

template <class V>
__global__ void __launch_bounds__(32 * V::WARPS, 1)
cascade_kernel(CascadeArgs a, int off_w, int off_b)
{
    constexpr int CS_WARPS = V::WARPS, CS_THREADS = 32 * V::WARPS;
    using WS = typename V::WS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    CascadeSmem<V> &sm = *reinterpret_cast<CascadeSmem<V> *>(smem_raw + 16);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    uint32_t *wimg = reinterpret_cast<uint32_t *>(smem_raw + off_w);
    int16_t *bimg = reinterpret_cast<int16_t *>(smem_raw + off_b);
    const CascadeDev &cd = a.cd;
    if (a.replay_list && a.replay_ctl[0] == 0) return;            /* fallback after the stage-sorted rounds: nothing left */

    load_feat_tables(&sm.ft, a.tables, threadIdx.x, CS_THREADS);
    for (int i = threadIdx.x; i < 384; i += CS_THREADS) sm.tanh_lut[i] = a.tables->tanh_lut[i];
    if (threadIdx.x < V::NFS) sm.fs_lock[threadIdx.x] = 0;
    for (int k = 0; k < cd.len_seq; k++) {
        const int id = cd.seq[k];
        const int *src = reinterpret_cast<const int *>(a.model[id]);
        int *dst = reinterpret_cast<int *>(&sm.model[id]);
        for (int i = threadIdx.x; i < (int)(sizeof(DevModel) / 4); i += CS_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    for (int k = 0; k < cd.len_seq; k++) {
        const int id = cd.seq[k];
        for (int i = threadIdx.x; i < sm.model[id].bias_count; i += CS_THREADS) bimg[cd.boff[id] + i] = a.bimg[id][i];
    }
    /* all weight images by TMA bulk copies on one mbarrier */
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
        for (int k = 0; k < cd.len_seq; k++) total += (uint32_t)cd.wbytes[cd.seq[k]];
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(total) : "memory");
        for (int k = 0; k < cd.len_seq; k++) {
            const int id = cd.seq[k];
            uint32_t off = 0;
            const uint32_t bytes = (uint32_t)cd.wbytes[id];
            while (off < bytes) {
                const uint32_t n = (bytes - off) > 32768u ? 32768u : (bytes - off);
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(smem_u32((char *)(wimg + cd.woff_words[id]) + off)), "l"((const char *)a.wimg[id] + off), "r"(n), "r"(smem_u32(bar)) : "memory");
                off += n;
            }
        }
    }
    {
        uint32_t done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(smem_u32(bar)) : "memory");
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, L16 = lane & 15;
    WS *ws = &sm.ws[warp];
    const int T = a.T, HS = NNSP_B200_MAX_WIDTH, HW = WS::WIDTH;      /* HS: stride of the state in global memory, HW: what the scratch holds */
    const int hist_frames = cd.dmax + 2, hist_len = hist_frames * NNSP_B200_FRAME;

    for (int it = 0;; it++) {
        int s;
        if (a.replay_list) {                                          /* replay after the stage-sorted pass: dynamic hand-out */
            int idx = 0;
            if (lane == 0) idx = atomicAdd(a.replay_ctl + 1, 1);
            idx = __shfl_sync(0xffffffffu, idx, 0);
            if (idx >= a.replay_ctl[0]) break;
            s = a.replay_list[idx];
        } else {
            const int si = blockIdx.x * CS_WARPS + warp + it * gridDim.x * CS_WARPS;
            if (si >= a.ns) break;
            s = a.s0 + si;
        }
        const int Ts = stream_frames(a.nfr, s, T);                    /* this stream's frames [0, Ts) of the call */
        if (!a.replay_list && Ts < T) {                               /* ragged call: nothing for the frames past them */
            if (a.results) write_no_frames(a.results, s, Ts, T, lane, 32);
            const long long f0 = (long long)s * T + Ts, nf = T - Ts;
            if (a.taps.logmel) for (long long i = lane; i < nf * 40; i += 32) a.taps.logmel[f0 * 40 + i] = 0;
            if (a.taps.feat) for (long long i = lane; i < nf * 40; i += 32) a.taps.feat[f0 * 40 + i] = 0;
            if (a.taps.hstate) for (long long i = lane; i < nf * HS; i += 32) a.taps.hstate[f0 * HS + i] = 0;
            if (a.taps.cstate) for (long long i = lane; i < nf * HS; i += 32) a.taps.cstate[f0 * HS + i] = 0;
            if (a.taps.post) for (long long i = lane; i < nf * SC_N; i += 32) a.taps.post[f0 * SC_N + i] = 0;
        }
        const int t_begin = a.t0 ? a.t0[s] : 0;                       /* frames before it were done by the stage-sorted pass */
        if (t_begin >= Ts) continue;
        for (int i = lane; i < 240; i += 32) ws->ctx[i] = a.st.ctx[(long long)s * 240 + i];
        for (int i = lane; i < HW; i += 32) { ws->h[i] = a.st.h[(long long)s * HS + i]; ws->c[i] = a.st.c[(long long)s * HS + i]; }
        if (lane < SC_N) ws->scal[lane] = a.st.scal[(long long)s * SC_N + lane];
        int pos = a.st.casc[(long long)s * CS_N + CS_POS];
        int cnt_kws = a.st.casc[(long long)s * CS_N + CS_CNT_KWS], cnt_s2i = a.st.casc[(long long)s * CS_N + CS_CNT_S2I];
        int age = a.st.casc[(long long)s * CS_N + CS_AGE];
        const CascThr thr = load_thr(cd, s);
        __syncwarp();
        const int16_t *ps = a.pcm + (long long)s * a.stride;
        const int16_t *hs = a.st.hist + (long long)s * hist_len + hist_len;                 /* hs[g], g < 0 */
        const int32_t *lm_now = a.logmel + (long long)s * T * NNSP_B200_NMEL;
        const int32_t *lm_old = a.st.lmhist + ((long long)s * cd.dmax + cd.dmax) * NNSP_B200_NMEL;   /* lm_old[r*40], r < 0 */

        for (int t = t_begin; t < Ts; t++) {
            const long long ft = (long long)s * T + t;
            const int id = cd.seq[pos];
            const DevModel &M = sm.model[id];
            const int d = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? cd.P.frs_vbufBk_kws : cd.P.frs_vbufBk_s2i);
            const int tf = t - d;                                        /* raw frame fed to the instance (PcmBufClass_getData look-back) */
            /* ---- FeatureClass_execute of the live instance ------------------------------------------ */
            int32_t lm0, lm1;
            if (age >= 2) {
                const int32_t *row = (tf >= 0) ? (lm_now + (long long)tf * NNSP_B200_NMEL) : (lm_old + (long long)tf * NNSP_B200_NMEL);
                lm0 = row[lane];
                lm1 = (lane < 8) ? row[32 + lane] : 0;
            } else {
                /* the instance's dataBuffer still holds zeros from its reset (spectrogram_module.c:25-31):
                 * window = [0, (age ? frame tf-1 : 0), frame tf]; both half-warps compute the same frame */
                const int base = (tf - 2) * NNSP_B200_FRAME;
                const int first_live = (2 - age) * NNSP_B200_FRAME;
                auto load_pair = [&](int, int p) -> uint32_t {
                    if (2 * p < first_live) return 0u;
                    const int g = base + 2 * p;
                    const int16_t *q = (g < 0) ? (hs + g) : (ps + g);
                    return *reinterpret_cast<const unsigned int *>(q);
                };
                int slot = warp;
                if (V::POOL) {                                       /* borrow a front-end scratch from the CTA's pool */
                    slot = -1;
                    if (lane == 0) {
                        for (int probe = warp; slot < 0; probe++)
                            if (atomicCAS(&sm.fs_lock[probe % V::NFS], 0, 1) == 0) slot = probe % V::NFS;
                        __threadfence_block();
                    }
                    slot = __shfl_sync(0xffffffffu, slot, 0);
                }
                frame_logmel<false>(sm.ft, sm.fs[slot], L16, load_pair, ws->logits, lane < 16, FeatDump{});   /* logits[] doubles as a 40-int scratch row */
                __syncwarp();
                if (V::POOL && lane == 0) { __threadfence_block(); atomicExch(&sm.fs_lock[slot], 0); }
                lm0 = ws->logits[lane];
                lm1 = (lane < 8) ? ws->logits[32 + lane] : 0;
                __syncwarp();
            }
            int16_t mv[7];
#pragma unroll
            for (int j = 0; j < 7; j++) { const int i = lane + 32 * j; mv[j] = (i < 200) ? ws->ctx[i + 40] : (int16_t)0; }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 7; j++) { const int i = lane + 32 * j; if (i < 200) ws->ctx[i] = mv[j]; }
            const int16_t f0 = standardise(lm0, M.mean[lane], M.stdR[lane], M.feat_rshift);
            ws->ctx[200 + lane] = f0;
            if (lane < 8) ws->ctx[232 + lane] = standardise(lm1, M.mean[32 + lane], M.stdR[32 + lane], M.feat_rshift);
            if (a.taps.logmel) { a.taps.logmel[ft * 40 + lane] = lm0; if (lane < 8) a.taps.logmel[ft * 40 + 32 + lane] = lm1; }
            __syncwarp();
            /* ---- NNSPClass_exec tail ------------------------------------------------------------------ */
            const bool ran = (ws->scal[SC_SLIDES] == 1);
            const int16_t th_prob = thr.prob[id], th_cnt = thr.cnts[id];
            if (ran) {
                net_forward(M, wimg + cd.woff_words[id], bimg + cd.boff[id], sm.tanh_lut, ws, lane, nullptr, nullptr);
                if (lane == 0) {
                    if (id == NNSP_B200_ID_S2I) post_s2i(ws->scal, ws->logits, th_cnt);
                    else post_binary(ws->scal, ws->logits, th_prob, th_cnt);
                }
            }
            if (lane == 0) ws->scal[SC_SLIDES] = (int16_t)((ws->scal[SC_SLIDES] + 1) % 2);
            __syncwarp();
            /* ---- controller (nnCntrlClass.c:172-269), evaluated redundantly by every lane ------------- */
            const int detected = ws->scal[SC_TRIGGER];
            int next_pos = pos, do_reset = 0, cnt_out = 0;
            if (id == NNSP_B200_ID_S2I) {
                cnt_s2i = (cnt_s2i + 1) % thr.timeout_s2i;
                if (detected || cnt_s2i == thr.timeout_s2i - 1) {
                    next_pos = (pos + 1) % cd.len_seq;
                    if (detected || cd.seq[next_pos] != id) { cnt_s2i = 0; do_reset = 1; }
                }
                cnt_out = cnt_s2i;
            } else if (id == NNSP_B200_ID_KWS) {
                cnt_kws = (cnt_kws + 1) % thr.timeout_kws;
                if (detected || cnt_kws == thr.timeout_kws - 1) {
                    if (detected) next_pos = (pos + 1) % cd.len_seq;
                    else { next_pos = (pos - 1) % cd.len_seq; if (next_pos < 0) next_pos += cd.len_seq; }
                    if (detected || cd.seq[next_pos] != id) { cnt_kws = 0; do_reset = 1; }
                }
                cnt_out = cnt_kws;
            } else if (detected) {
                next_pos = (pos + 1) % cd.len_seq;
                do_reset = 1;
            }
            if (lane == 0 && a.results) {
                nnsp_b200_cascade_result r;
                r.stage_id = (int8_t)id; r.pos_after = (int8_t)next_pos; r.detected = (int16_t)detected;
                r.outputs[0] = ws->scal[SC_OUT0]; r.outputs[1] = ws->scal[SC_OUT0 + 1]; r.outputs[2] = ws->scal[SC_OUT0 + 2];
                r.cnt_timeout = (uint16_t)cnt_out;
                a.results[ft] = r;
            }
            /* taps of the instance that ran; zero-filled when the controller reset it this frame */
            if (a.taps.feat) { a.taps.feat[ft * 40 + lane] = do_reset ? (int16_t)0 : ws->ctx[200 + lane]; if (lane < 8) a.taps.feat[ft * 40 + 32 + lane] = do_reset ? (int16_t)0 : ws->ctx[232 + lane]; }
            if (a.taps.hstate) for (int i = lane; i < HS; i += 32) a.taps.hstate[ft * HS + i] = (do_reset || i >= M.h_stride) ? (int16_t)0 : ws->h[i];
            if (a.taps.cstate) for (int i = lane; i < HS; i += 32) a.taps.cstate[ft * HS + i] = (do_reset || i >= M.h_stride) ? 0 : ws->c[i];
            if (a.taps.post && lane < SC_N) {
                int16_t v = do_reset ? (int16_t)0 : ws->scal[lane];
                if (lane == SC_RAN) v = do_reset ? (int16_t)0 : (int16_t)(ran ? 1 : 0);
                if (lane == SC_STAGE) v = (int16_t)id;
                a.taps.post[ft * SC_N + lane] = v;
            }
            __syncwarp();
            if (do_reset) {
                /* NNSPClass_reset of the instance we leave: its context row 5 stays behind ... */
                int16_t *stale = a.stale + ((long long)s * 3 + id) * 40;
                stale[lane] = ws->ctx[200 + lane];
                if (lane < 8) stale[32 + lane] = ws->ctx[232 + lane];
                __syncwarp();
                /* ... and the instance we enter starts from ITS reset state plus ITS stale row 5 */
                const int nid = cd.seq[next_pos];
                reset_stream_scratch(sm.model[nid], ws, lane);
                const int16_t *st2 = a.stale + ((long long)s * 3 + nid) * 40;
                ws->ctx[200 + lane] = st2[lane];
                if (lane < 8) ws->ctx[232 + lane] = st2[32 + lane];
                age = 0;
            } else {
                age = age < 2 ? age + 1 : 2;
            }
            pos = next_pos;
            __syncwarp();
        }
        __syncwarp();
        for (int i = lane; i < 240; i += 32) a.st.ctx[(long long)s * 240 + i] = ws->ctx[i];
        for (int i = lane; i < HW; i += 32) { a.st.h[(long long)s * HS + i] = ws->h[i]; a.st.c[(long long)s * HS + i] = ws->c[i]; }
        if (lane < SC_N) a.st.scal[(long long)s * SC_N + lane] = ws->scal[lane];
        if (lane == 0) {
            a.st.casc[(long long)s * CS_N + CS_POS] = (uint16_t)pos;
            a.st.casc[(long long)s * CS_N + CS_CNT_KWS] = (uint16_t)cnt_kws;
            a.st.casc[(long long)s * CS_N + CS_CNT_S2I] = (uint16_t)cnt_s2i;
            a.st.casc[(long long)s * CS_N + CS_AGE] = (uint16_t)age;
        }
        __syncwarp();
    }
}


/* ======================================================================================================== */
/* cascade_replay_kernel: what is left after the stage-sorted rounds, NNSP_CR_GW (two) warps per stream          */
/* ======================================================================================================== */
/* Same per-frame semantics as cascade_kernel (see there for the reference lines), narrow models only, no taps (a call
 * with taps never takes the stage-sorted pass). The replay lasts as long as its longest remainder, so the chain per
 * stream is what counts: a group of NNSP_CR_GW warps (two; four leave too few streams in flight) shares one stream
 * (net_forward_group), 16 / NNSP_CR_GW groups per CTA next to the three weight images; streams are handed out to groups
 * dynamically, longest remainder first. */
#ifndef NNSP_CR_GW
#define NNSP_CR_GW 2
#endif
constexpr int CR_GW = NNSP_CR_GW, CR_GT = 32 * CR_GW, CR_GROUPS = 16 / CR_GW, CR_THREADS = 512;   /* warps, threads per group */
struct ReplaySmem {
    FeatSmemTables ft;
    int16_t tanh_lut[384];
    DevModel model[3];
    FrameScratch fs[CR_GROUPS];
    CsNarrow::WS ws[CR_GROUPS];
    int slot[CR_GROUPS];
};
/* both kernels stage the same weight images behind their structs: every cascade the narrow sequential kernel takes fits
 * the replay kernel, so cascade_kernel<CsNarrow> replays only when NNSP_B200_REPLAY_COOP=0 asks for it */
static_assert(sizeof(ReplaySmem) <= sizeof(CascadeSmem<CsNarrow>), "the replay kernel must fit wherever the narrow kernel does");

__global__ void __launch_bounds__(CR_THREADS, 1)
cascade_replay_kernel(CascadeArgs a, int off_w, int off_b)
{
    using WS = CsNarrow::WS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ReplaySmem &sm = *reinterpret_cast<ReplaySmem *>(smem_raw + 16);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    uint32_t *wimg = reinterpret_cast<uint32_t *>(smem_raw + off_w);
    int16_t *bimg = reinterpret_cast<int16_t *>(smem_raw + off_b);
    const CascadeDev &cd = a.cd;
    if (a.replay_ctl[0] == 0) return;                             /* nothing left after the stage-sorted rounds */

    load_feat_tables(&sm.ft, a.tables, threadIdx.x, CR_THREADS);
    for (int i = threadIdx.x; i < 384; i += CR_THREADS) sm.tanh_lut[i] = a.tables->tanh_lut[i];
    for (int k = 0; k < cd.len_seq; k++) {
        const int id = cd.seq[k];
        const int *src = reinterpret_cast<const int *>(a.model[id]);
        int *dst = reinterpret_cast<int *>(&sm.model[id]);
        for (int i = threadIdx.x; i < (int)(sizeof(DevModel) / 4); i += CR_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    for (int k = 0; k < cd.len_seq; k++) {
        const int id = cd.seq[k];
        for (int i = threadIdx.x; i < sm.model[id].bias_count; i += CR_THREADS) bimg[cd.boff[id] + i] = a.bimg[id][i];
    }
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
        for (int k = 0; k < cd.len_seq; k++) total += (uint32_t)cd.wbytes[cd.seq[k]];
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(total) : "memory");
        for (int k = 0; k < cd.len_seq; k++) {
            const int id = cd.seq[k];
            uint32_t off = 0;
            const uint32_t bytes = (uint32_t)cd.wbytes[id];
            while (off < bytes) {
                const uint32_t n = (bytes - off) > 32768u ? 32768u : (bytes - off);
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(smem_u32((char *)(wimg + cd.woff_words[id]) + off)), "l"((const char *)a.wimg[id] + off), "r"(n), "r"(smem_u32(bar)) : "memory");
                off += n;
            }
        }
    }
    {
        uint32_t done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(smem_u32(bar)) : "memory");
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, L16 = lane & 15;
    const int grp = warp / CR_GW, wg = warp % CR_GW, gt = threadIdx.x % CR_GT, bid = 1 + grp;      /* barrier 0 is __syncthreads */
    WS *ws = &sm.ws[grp];
    FrameScratch &fs = sm.fs[grp];
    const int T = a.T, HS = NNSP_B200_MAX_WIDTH, HW = WS::WIDTH;
    const int hist_frames = cd.dmax + 2, hist_len = hist_frames * NNSP_B200_FRAME;

    for (;;) {
        if (gt == 0) sm.slot[grp] = atomicAdd(a.replay_ctl + 1, 1);
        group_sync<CR_GW>(bid);
        const int idx = sm.slot[grp];
        group_sync<CR_GW>(bid);                                              /* everyone has read the slot before it is rewritten */
        if (idx >= a.replay_ctl[0]) break;
        const int s = a.replay_list[idx];
        const int t_begin = a.t0[s], Ts = stream_frames(a.nfr, s, T);
        if (t_begin >= Ts) continue;
        for (int i = gt; i < 240; i += CR_GT) ws->ctx[i] = a.st.ctx[(long long)s * 240 + i];
        for (int i = gt; i < HW; i += CR_GT) { ws->h[i] = a.st.h[(long long)s * HS + i]; ws->c[i] = a.st.c[(long long)s * HS + i]; }
        if (gt < SC_N) ws->scal[gt] = a.st.scal[(long long)s * SC_N + gt];
        int pos = a.st.casc[(long long)s * CS_N + CS_POS];
        int cnt_kws = a.st.casc[(long long)s * CS_N + CS_CNT_KWS], cnt_s2i = a.st.casc[(long long)s * CS_N + CS_CNT_S2I];
        int age = a.st.casc[(long long)s * CS_N + CS_AGE];
        const CascThr thr = load_thr(cd, s);
        group_sync<CR_GW>(bid);
        const int16_t *ps = a.pcm + (long long)s * a.stride;
        const int16_t *hs = a.st.hist + (long long)s * hist_len + hist_len;
        const int32_t *lm_now = a.logmel + (long long)s * T * NNSP_B200_NMEL;
        const int32_t *lm_old = a.st.lmhist + ((long long)s * cd.dmax + cd.dmax) * NNSP_B200_NMEL;

        for (int t = t_begin; t < Ts; t++) {
            const long long ft = (long long)s * T + t;
            const int id = cd.seq[pos];
            const DevModel &M = sm.model[id];
            const int d = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? cd.P.frs_vbufBk_kws : cd.P.frs_vbufBk_s2i);
            const int tf = t - d;
            /* ---- FeatureClass_execute of the live instance: log-mel value of feature gt (gt < 40) ---- */
            int32_t lmv = 0;
            if (age >= 2) {
                const int32_t *row = (tf >= 0) ? (lm_now + (long long)tf * NNSP_B200_NMEL) : (lm_old + (long long)tf * NNSP_B200_NMEL);
                if (gt < 40) lmv = row[gt];
            } else {
                if (wg == 0) {                                       /* the first warp recomputes the frame (zeros in the STFT buffer) */
                    const int base = (tf - 2) * NNSP_B200_FRAME;
                    const int first_live = (2 - age) * NNSP_B200_FRAME;
                    auto load_pair = [&](int, int p) -> uint32_t {
                        if (2 * p < first_live) return 0u;
                        const int g = base + 2 * p;
                        const int16_t *q = (g < 0) ? (hs + g) : (ps + g);
                        return *reinterpret_cast<const unsigned int *>(q);
                    };
                    frame_logmel<false>(sm.ft, fs, L16, load_pair, ws->logits, lane < 16, FeatDump{});
                }
                group_sync<CR_GW>(bid);
                if (gt < 40) lmv = ws->logits[gt];
                group_sync<CR_GW>(bid);
            }
            /* context rows up by one, the new row standardised with the instance's statistics */
            constexpr int NMV = (200 + CR_GT - 1) / CR_GT;
            int16_t mv[NMV];
#pragma unroll
            for (int j = 0; j < NMV; j++) { const int i = gt + CR_GT * j; mv[j] = (i < 200) ? ws->ctx[i + 40] : (int16_t)0; }
            group_sync<CR_GW>(bid);
#pragma unroll
            for (int j = 0; j < NMV; j++) { const int i = gt + CR_GT * j; if (i < 200) ws->ctx[i] = mv[j]; }
            if (gt < 40) ws->ctx[200 + gt] = standardise(lmv, M.mean[gt], M.stdR[gt], M.feat_rshift);
            group_sync<CR_GW>(bid);
            /* ---- NNSPClass_exec tail ------------------------------------------------------------------ */
            const bool ran = (ws->scal[SC_SLIDES] == 1);
            const int16_t th_prob = thr.prob[id], th_cnt = thr.cnts[id];
            group_sync<CR_GW>(bid);                                          /* everyone has read slides before it changes */
            if (ran) {
                net_forward_group<CR_GW>(M, wimg + cd.woff_words[id], bimg + cd.boff[id], sm.tanh_lut, ws, wg, lane, bid);
                if (gt == 0) {
                    if (id == NNSP_B200_ID_S2I) post_s2i(ws->scal, ws->logits, th_cnt);
                    else post_binary(ws->scal, ws->logits, th_prob, th_cnt);
                }
            }
            if (gt == 0) ws->scal[SC_SLIDES] = (int16_t)((ws->scal[SC_SLIDES] + 1) % 2);
            group_sync<CR_GW>(bid);
            /* ---- controller (nnCntrlClass.c:172-269), evaluated redundantly by every thread of the group ---- */
            const int detected = ws->scal[SC_TRIGGER];
            int next_pos = pos, do_reset = 0, cnt_out = 0;
            if (id == NNSP_B200_ID_S2I) {
                cnt_s2i = (cnt_s2i + 1) % thr.timeout_s2i;
                if (detected || cnt_s2i == thr.timeout_s2i - 1) {
                    next_pos = (pos + 1) % cd.len_seq;
                    if (detected || cd.seq[next_pos] != id) { cnt_s2i = 0; do_reset = 1; }
                }
                cnt_out = cnt_s2i;
            } else if (id == NNSP_B200_ID_KWS) {
                cnt_kws = (cnt_kws + 1) % thr.timeout_kws;
                if (detected || cnt_kws == thr.timeout_kws - 1) {
                    if (detected) next_pos = (pos + 1) % cd.len_seq;
                    else { next_pos = (pos - 1) % cd.len_seq; if (next_pos < 0) next_pos += cd.len_seq; }
                    if (detected || cd.seq[next_pos] != id) { cnt_kws = 0; do_reset = 1; }
                }
                cnt_out = cnt_kws;
            } else if (detected) {
                next_pos = (pos + 1) % cd.len_seq;
                do_reset = 1;
            }
            if (gt == 0 && a.results) {
                nnsp_b200_cascade_result r;
                r.stage_id = (int8_t)id; r.pos_after = (int8_t)next_pos; r.detected = (int16_t)detected;
                r.outputs[0] = ws->scal[SC_OUT0]; r.outputs[1] = ws->scal[SC_OUT0 + 1]; r.outputs[2] = ws->scal[SC_OUT0 + 2];
                r.cnt_timeout = (uint16_t)cnt_out;
                a.results[ft] = r;
            }
            group_sync<CR_GW>(bid);
            if (do_reset) {
                int16_t *stale = a.stale + ((long long)s * 3 + id) * 40;
                if (gt < 40) stale[gt] = ws->ctx[200 + gt];
                group_sync<CR_GW>(bid);
                const int nid = cd.seq[next_pos];
                const DevModel &N = sm.model[nid];
                for (int i = gt; i < 200; i += CR_GT) ws->ctx[i] = N.silence[i % 40];             /* reset_stream_scratch, group-wide */
                for (int i = gt; i < HW; i += CR_GT) { ws->h[i] = 0; ws->c[i] = 0; }
                if (gt < SC_N) ws->scal[gt] = (gt == SC_SLIDES) ? 1 : 0;
                const int16_t *st2 = a.stale + ((long long)s * 3 + nid) * 40;
                if (gt < 40) ws->ctx[200 + gt] = st2[gt];
                age = 0;
            } else {
                age = age < 2 ? age + 1 : 2;
            }
            pos = next_pos;
            group_sync<CR_GW>(bid);
        }
        for (int i = gt; i < 240; i += CR_GT) a.st.ctx[(long long)s * 240 + i] = ws->ctx[i];
        for (int i = gt; i < HW; i += CR_GT) { a.st.h[(long long)s * HS + i] = ws->h[i]; a.st.c[(long long)s * HS + i] = ws->c[i]; }
        if (gt < SC_N) a.st.scal[(long long)s * SC_N + gt] = ws->scal[gt];
        if (gt == 0) {
            a.st.casc[(long long)s * CS_N + CS_POS] = (uint16_t)pos;
            a.st.casc[(long long)s * CS_N + CS_CNT_KWS] = (uint16_t)cnt_kws;
            a.st.casc[(long long)s * CS_N + CS_CNT_S2I] = (uint16_t)cnt_s2i;
            a.st.casc[(long long)s * CS_N + CS_AGE] = (uint16_t)age;
        }
        group_sync<CR_GW>(bid);
    }
}

/* ======================================================================================================== */
/* stage-sorted rounds: the scan-split network kernels (nnsp_split.cu) over the streams of each live model      */
/* ======================================================================================================== */
/* Within a call most streams stay in the stage they are in. Round 0 sorts the streams by live model on the device,
 * runs every group through the batched scan-split kernels as if nothing changed, and cascade_post_kernel then walks
 * every stream's frames through the controller (nnCntrlClass.c:172-269). At the first frame where the controller
 * leaves the instance, that instance is reset -- which is all the reference keeps of it (plus context row 5) -- the
 * speculative rest is dropped, and the stream is queued for the NEXT ROUND with the instance it enters: round r + 1 is
 * the same three kernels over the queued streams, each starting at its own frame (tstart[s]; the kernels take per-row
 * start frames and inference counts). A stream takes one round per stage change inside the call; what is still queued
 * after the last round (CS_MAX_ROUNDS) goes to the sequential kernel. The first two frames of a fresh instance see a
 * partly zero STFT buffer (spectrogram_module.c:25-31): cascade_fix_kernel computes those log-mel rows on the side. */
constexpr int CG_GROUPS = 6;                        /* plane tiles reserved per slice beyond S/16 (one partial tile per group + slack) */
constexpr int CPOST_WARPS = 8;                      /* streams per CTA of the controller walk */
constexpr int CS_MAX_ROUNDS = 4;
/* per-slice control block (ints, zeroed at the start of a call): round r at CTL_ROUND * r */
constexpr int CTL_ROUND = 12;                       /* [0..2] group sizes by model id, [3..5] first plane tile of the group, */
constexpr int CTL_NEXT = 6, CTL_FIX = 7;            /* [6] streams queued for the next round, [7] streams that need fix rows */
constexpr int CTL_REPLAY = CTL_ROUND * CS_MAX_ROUNDS;   /* [0] streams left for the sequential kernel, [1] its cursor          */
constexpr int CTL_INTS = 64;

struct RoundArrays {                  /* per stream, valid during one call */
    int *t0;                          /* -1: live in the current round; T + 1: lived through the call (context rebuild);
                                         else: first frame the sequential kernel still has to process                   */
    int *tstart, *tb, *age0;          /* see SplitGroup */
    int32_t *lmfix;                   /* [S][2][40] */
};

__global__ void cascade_classify_kernel(StreamState st, CascadeDev cd, int s0, int ns, int S, int *list, int *ctl, RoundArrays ra,
                                        int *fix_list, const int32_t *nfr, int T)
{
    const int si = blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= ns) return;
    const long long s = s0 + si;
    const int pos = st.casc[s * CS_N + CS_POS], age = st.casc[s * CS_N + CS_AGE];
    const int id = cd.seq[pos];
    ra.tb[s] = 0;
    ra.tstart[s] = (st.scal[s * SC_N + SC_SLIDES] == 1) ? 0 : 1;     /* nn_speech.c:84: the stride-2 gate */
    ra.age0[s] = age;
    ra.t0[s] = -1;
    if (stream_frames(nfr, s, T) == 0) return;                       /* ragged call, idle stream: in no group */
    list[(long long)id * S + s0 + atomicAdd(&ctl[id], 1)] = (int)s;
    if (age < 2) fix_list[s0 + atomicAdd(&ctl[CTL_FIX], 1)] = (int)s;
}
__global__ void cascade_offsets_kernel(int *ctl)
{
    int o = 0;
    for (int g = 0; g < 3; g++) { ctl[3 + g] = o; o += (ctl[g] + 15) >> 4; }
}

/* round r >= 1: the streams queued by the previous round's walk, sorted by (model they entered, frames left) so that a
 * 16-stream tile holds streams of similar length; one CTA, counting sort over 3 x 256 buckets. The key T - (frames left)
 * is the start frame unless the call is ragged. */
constexpr int CSORT_THREADS = 1024, CSORT_BUCKETS = 1024, CRG_NB = 256;
__global__ void __launch_bounds__(CSORT_THREADS) cascade_regroup_kernel(StreamState st, CascadeDev cd, const int *__restrict__ pend,
                                                                       const int *__restrict__ ctl_prev, int *ctl, int *list, int S, int s0,
                                                                       RoundArrays ra, int T, const int32_t *nfr)
{
    __shared__ int hist[3 * CRG_NB];
    __shared__ int gstart[4];
    const int n = ctl_prev[CTL_NEXT];
    if (n == 0) return;                                               /* (ctl of this round stays zero: every kernel of the round leaves at once) */
    for (int i = threadIdx.x; i < 3 * CRG_NB; i += CSORT_THREADS) hist[i] = 0;
    __syncthreads();
    auto bucket = [&](int s) {
        const int id = cd.seq[st.casc[(long long)s * CS_N + CS_POS]];
        const long long b = (long long)(ra.tstart[s] + T - stream_frames(nfr, s, T)) * CRG_NB / (T + 1);
        return id * CRG_NB + (int)(b < 0 ? 0 : (b >= CRG_NB ? CRG_NB - 1 : b));
    };
    for (int i = threadIdx.x; i < n; i += CSORT_THREADS) atomicAdd(&hist[bucket(pend[i])], 1);
    __syncthreads();
    if (threadIdx.x < 32) {                                            /* exclusive scan of the 768 counts by one warp */
        int carry = 0;
        for (int base = 0; base < 3 * CRG_NB; base += 32) {
            if ((base % CRG_NB) == 0 && threadIdx.x == 0) gstart[base / CRG_NB] = carry;
            const int v = hist[base + threadIdx.x];
            int x = v;
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if ((int)threadIdx.x >= o) x += y; }
            hist[base + threadIdx.x] = carry + x - v;
            carry += __shfl_sync(0xffffffffu, x, 31);
        }
        if (threadIdx.x == 0) {
            gstart[3] = carry;
            int o = 0;
            for (int g = 0; g < 3; g++) { const int c = gstart[g + 1] - gstart[g]; ctl[g] = c; ctl[3 + g] = o; o += (c + 15) >> 4; }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += CSORT_THREADS) {
        const int s = pend[i], b = bucket(s), id = b / CRG_NB;
        list[(long long)id * S + s0 + (atomicAdd(&hist[b], 1) - gstart[id])] = s;
    }
}

/* log-mel rows of the first two frames of a fresh instance: window = [0, (second frame ? raw frame tf-1 : 0), raw frame tf]
 * with tf = t - look-back. One half-warp per (stream, life frame); streams from a device-side list. */
struct FixArgs {
    const DevTables *tables;
    StreamState st;
    const int16_t *pcm; long long stride;
    const int *list, *count;
    RoundArrays ra;
    CascadeDev cd;
    int T;
    const int32_t *nfr;              /* ragged call: no row past the stream's own frames */
};
struct FixSmem { FeatSmemTables ft; FrameScratch fs[16]; };
__global__ void __launch_bounds__(256) cascade_fix_kernel(FixArgs a)
{
    __shared__ FixSmem sm;
    const int n = *a.count;
    if ((int)blockIdx.x * 8 >= n) return;                             /* a warp takes both life frames of one stream */
    load_feat_tables(&sm.ft, a.tables, threadIdx.x, 256);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, la = lane >> 4, L = lane & 15;
    const CascadeDev &cd = a.cd;
    const int hist_len = (cd.dmax + 2) * NNSP_B200_FRAME;
    for (int i = blockIdx.x * 8 + warp; i < n; i += gridDim.x * 8) {
        const long long s = a.list[i];
        const int id = cd.seq[a.st.casc[s * CS_N + CS_POS]];
        const int d = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? cd.P.frs_vbufBk_kws : cd.P.frs_vbufBk_s2i);
        const int t = a.ra.tb[s] + la - a.ra.age0[s];                 /* frame of the call with life index la */
        const bool valid = la >= a.ra.age0[s] && t < stream_frames(a.nfr, s, a.T);
        const int tf = t - d, base = (tf - 2) * NNSP_B200_FRAME, first_live = (2 - la) * NNSP_B200_FRAME;
        const int16_t *ps = a.pcm + s * a.stride;
        const int16_t *hs = a.st.hist + s * hist_len + hist_len;       /* hs[g], g < 0: frames before the call */
        auto load_pair = [&](int, int p) -> uint32_t {
            if (!valid || 2 * p < first_live) return 0u;
            const int g = base + 2 * p;
            return *reinterpret_cast<const unsigned int *>((g < 0) ? (hs + g) : (ps + g));
        };
        frame_logmel<false>(sm.ft, sm.fs[warp * 2 + la], L, load_pair, a.ra.lmfix + (s * 2 + la) * NNSP_B200_NMEL, valid, FeatDump{});
    }
}

/* The replay is latency-bound -- one warp walks one stream frame by frame, so the kernel lasts at least as long as the
 * longest remainder. Handing the streams out longest-first (earliest t0 first; in a ragged call, least T - frames left)
 * keeps a long one from being started last: a counting sort of the list, one CTA. */
__global__ void __launch_bounds__(CSORT_THREADS) cascade_sort_replay_kernel(const int *__restrict__ list_in, int *__restrict__ list_out,
                                                                           const int *__restrict__ count_in, int *__restrict__ ctl_out,
                                                                           const int *__restrict__ t0, int T, const int32_t *__restrict__ nfr)
{
    __shared__ int hist[CSORT_BUCKETS];
    const int n = *count_in;
    if (threadIdx.x == 0) { ctl_out[0] = n; ctl_out[1] = 0; }
    if (n == 0) return;
    for (int i = threadIdx.x; i < CSORT_BUCKETS; i += CSORT_THREADS) hist[i] = 0;
    __syncthreads();
    auto bucket = [&](int s) {
        const long long b = (long long)(t0[s] + T - stream_frames(nfr, s, T)) * CSORT_BUCKETS / (T + 1);
        return (int)(b < 0 ? 0 : (b >= CSORT_BUCKETS ? CSORT_BUCKETS - 1 : b));
    };
    for (int i = threadIdx.x; i < n; i += CSORT_THREADS) atomicAdd(&hist[bucket(list_in[i])], 1);
    __syncthreads();
    if (threadIdx.x < 32) {                                            /* exclusive scan of 1024 counts by one warp */
        int carry = 0;
        for (int base = 0; base < CSORT_BUCKETS; base += 32) {
            const int v = hist[base + threadIdx.x];
            int x = v;
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if ((int)threadIdx.x >= o) x += y; }
            hist[base + threadIdx.x] = carry + x - v;
            carry += __shfl_sync(0xffffffffu, x, 31);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += CSORT_THREADS) { const int s = list_in[i]; list_out[atomicAdd(&hist[bucket(s)], 1)] = s; }
}

struct CascadePostArgs {
    const MmaModel *model[3];        /* statistics and silence rows of each model */
    StreamState st;
    int16_t *stale;
    const int32_t *logmel;
    const int32_t *dec;
    int dec_stride;
    RoundArrays ra;
    const int *list, *count;         /* the round's streams (null: the range s0 .. s0 + ns - 1, round 0) */
    int *next_list, *next_count;     /* streams that change stage are queued here for the next round */
    int s0, ns, T;
    nnsp_b200_cascade_result *results;
    CascadeDev cd;
    const int32_t *nfr;              /* ragged call: stream s ends at frame stream_frames(nfr, s, T) */
};

/* log-mel row the instance of stream s reads at frame f of the call (f >= its tb): a fix row during its first two frames */
__device__ __forceinline__ const int32_t *cascade_lm_row(const CascadePostArgs &a, long long s, int f, int d, int tb, int age0)
{
    const int la = f - tb + age0, fr = f - d;
    if (la < 2) return a.ra.lmfix + (s * 2 + la) * NNSP_B200_NMEL;
    return (fr >= 0) ? a.logmel + (s * a.T + fr) * NNSP_B200_NMEL
                     : a.st.lmhist + (s * a.cd.dmax + a.cd.dmax + fr) * NNSP_B200_NMEL;
}

/* The controller walk of one round, a warp per stream. Between two stage changes the per-frame work of
 * nnCntrlClass_exec (nnCntrlClass.c:172-269) is closed-form: the time-out counter is (c0 + frames) mod time-out, and no
 * frame before the exit frame can carry a detection (every detection resets the instance, i.e. IS the exit). So the warp
 * (every lane redundantly, on broadcast decision records) only steps through the INFERENCES of the round to find the
 * first detection -- s2i_post_proc / binary_post_proc on the decision records, nn_speech.c:146-227 -- takes the earlier of
 * that and the first time-out that leaves the instance, and then writes all result records of the round in parallel. */
template <bool RAGGED>                                                 /* RAGGED: a.nfr != null; false: the uniform call's code */
__global__ void __launch_bounds__(32 * CPOST_WARPS) cascade_post_kernel(CascadePostArgs a)
{
    const CascadeDev &cd = a.cd;
    const int nsel = a.list ? *a.count : a.ns;
    const int lane = threadIdx.x & 31;
    const int si = blockIdx.x * CPOST_WARPS + (threadIdx.x >> 5);
    if (si >= nsel) return;
    const long long s = a.list ? a.list[si] : (long long)a.s0 + si;
    const int T = a.T, Ts = RAGGED ? stream_frames(a.nfr, s, T) : T;  /* the stream's frames of the call: [0, Ts) */
    if (RAGGED) {
        if (!a.list && a.results && Ts < T) write_no_frames(a.results, s, Ts, T, lane, 32);   /* round 0 */
        if (Ts == 0) return;                                          /* idle stream: its state stays as it is */
    }
    const int tb = a.ra.tb[s], ts = a.ra.tstart[s], age0 = a.ra.age0[s];
    const int pos = a.st.casc[s * CS_N + CS_POS];
    int cnt_kws = a.st.casc[s * CS_N + CS_CNT_KWS], cnt_s2i = a.st.casc[s * CS_N + CS_CNT_S2I];
    const int id = cd.seq[pos];
    const int d = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? cd.P.frs_vbufBk_kws : cd.P.frs_vbufBk_s2i);
    const CascThr thr = load_thr(cd, s);
    const int th_cnt = thr.cnts[id];
    /* NNSPClass scalars in registers (counters updated by compare-and-add, no dynamically indexed array) */
    int trig, out0, out1, out2, last, slides, cnt[8];
    {
        int16_t sc[SC_N];
        const uint4 *p = reinterpret_cast<const uint4 *>(a.st.scal + s * SC_N);
        *reinterpret_cast<uint4 *>(&sc[0]) = p[0];
        *reinterpret_cast<uint4 *>(&sc[8]) = p[1];
        trig = sc[SC_TRIGGER]; out0 = sc[SC_OUT0]; out1 = sc[SC_OUT0 + 1]; out2 = sc[SC_OUT0 + 2];
#pragma unroll
        for (int i = 0; i < 8; i++) cnt[i] = sc[SC_CNT0 + i];
        last = sc[SC_ARGMAX_LAST]; slides = sc[SC_SLIDES];
    }
    const int st_o0 = out0, st_o1 = out1, st_o2 = out2;              /* outputs[] as the round finds them (binary models never touch them) */
    /* ---- time-outs (nnCntrlClass.c:186-206, 222-242): the counter of the live model is (c0 + n) mod time-out after n frames */
    const bool has_to = id != NNSP_B200_ID_VAD;
    const int timeout = (id == NNSP_B200_ID_S2I) ? thr.timeout_s2i : thr.timeout_kws;
    const int c0 = (id == NNSP_B200_ID_S2I) ? cnt_s2i : cnt_kws;
    int to_next = pos, t_to = Ts;                                     /* first frame whose counter reads time-out - 1 */
    bool to_exit = false;
    if (has_to) {
        int n = (timeout - 1 - c0) % timeout;                          /* c0 may exceed a time-out that was shortened at run time */
        if (n < 1) n += timeout;
        t_to = tb + n - 1;
        if (id == NNSP_B200_ID_S2I) to_next = (pos + 1) % cd.len_seq;
        else { to_next = (pos - 1) % cd.len_seq; if (to_next < 0) to_next += cd.len_seq; }
        to_exit = cd.seq[to_next] != id;                              /* otherwise the time-out changes nothing (:198, :234) */
    }
    const int t_lim = (to_exit && t_to < Ts) ? t_to : Ts - 1;         /* last frame this instance can see in this call */
    /* ---- first detection: a stale trigger on the frame before the first inference, else the first inference that fires */
    int t_det = -1;
    if (ts > tb && tb <= t_lim && trig) t_det = tb;                   /* nn_speech.c:126: odd frames return the previous trigger */
    if (t_det < 0 && ts <= t_lim) {
        const int k_lim = ((t_lim - ts) >> 1) + 1;                    /* inferences at frames ts, ts + 2, ... <= t_lim */
        const int32_t *dec = a.dec + (size_t)s * a.dec_stride;
        for (int kb = 0; kb < k_lim && t_det < 0; kb += 32) {
            const int dchunk = (kb + lane < k_lim) ? dec[kb + lane] : 0;
            const int nk = min(32, k_lim - kb);
            for (int j = 0; j < nk; j++) {
                const int dv = __shfl_sync(0xffffffffu, dchunk, j);
                if (id == NNSP_B200_ID_S2I) {                                               /* s2i_post_proc, nn_speech.c:146-189 */
                    const int ai = dv & 0xff;
                    trig = 0; out0 = 0; out1 = 0; out2 = 0;
                    if (last == 0 || last == ai) {
                        int hit = 0;
#pragma unroll
                        for (int i = 1; i < 7; i++) {
                            const int c1 = (int)(int16_t)(cnt[i] + 1);
                            if (ai == i) { cnt[i] = c1; hit = c1 > th_cnt; }
                        }
                        if (hit) { trig = 1; out0 = ai; out1 = (dv >> 8) & 0xff; out2 = (dv >> 16) & 0xff; }
                    } else {
#pragma unroll
                        for (int i = 0; i < 7; i++) cnt[i] = 0;
                    }
                    last = ai;
                } else {                                                                    /* binary_post_proc, nn_speech.c:219-226 */
                    const int cc = dv ? (int)(int16_t)(cnt[0] + 1) : 0;
                    cnt[0] = cc;
                    trig = (cc >= th_cnt) ? 1 : 0;
                }
                if (trig) { t_det = ts + 2 * (kb + j); break; }
            }
        }
    }
    /* ---- where the round ends for this stream */
    int t_exit = -1, next_pos_exit = pos;
    bool by_det = false;
    if (t_det >= 0) { t_exit = t_det; by_det = true; next_pos_exit = (pos + 1) % cd.len_seq; }   /* :189-205, :224-228, :256-266 */
    else if (to_exit && t_to < Ts) { t_exit = t_to; next_pos_exit = to_next; }
    const int t_last = (t_exit >= 0) ? t_exit : Ts - 1;
    /* ---- result records of frames tb .. t_last, in parallel */
    if (a.results) {
        uint32_t *out = reinterpret_cast<uint32_t *>(a.results + s * T);                   /* 12-byte records, 4-byte aligned */
        const bool zero_outs = id == NNSP_B200_ID_S2I;                                      /* s2i_post_proc clears outputs[] at every inference */
        for (int t = tb + lane; t <= t_last; t += 32) {
            const bool ex = t == t_exit;
            const int det = (ex && by_det) ? trig : 0;
            int o0 = st_o0, o1 = st_o1, o2 = st_o2;
            if (zero_outs && t >= ts) { o0 = 0; o1 = 0; o2 = 0; }
            if (ex && by_det && t >= ts) { o0 = out0; o1 = out1; o2 = out2; }
            const int ct = (!has_to || ex) ? 0 : (c0 + (t - tb + 1)) % timeout;
            const int pa = ex ? next_pos_exit : pos;
            out[3 * t + 0] = (uint32_t)(uint8_t)id | ((uint32_t)(uint8_t)pa << 8) | ((uint32_t)(uint16_t)det << 16);
            out[3 * t + 1] = (uint32_t)(uint16_t)o0 | ((uint32_t)(uint16_t)o1 << 16);
            out[3 * t + 2] = (uint32_t)(uint16_t)o2 | ((uint32_t)(uint16_t)ct << 16);
        }
    }
    const MmaModel &M = *a.model[id];
    int16_t *ctx = a.st.ctx + s * 240;
    if (t_exit >= 0) {
        /* NNSPClass_reset of the instance the controller leaves (nn_speech.c:57-72): its newest context row stays
         * behind as that instance's stale row 5 (feature_module.c:39-42) ... */
        const int32_t *row = cascade_lm_row(a, s, t_exit, d, tb, age0);
        int16_t *stale = a.stale + (s * 3 + id) * 40;
        for (int i = lane; i < 40; i += 32) stale[i] = standardise(row[i], M.mean[i], M.stdR[i], M.feat_rshift);
        __syncwarp();
        /* ... and the instance entered starts from ITS reset state plus ITS stale row */
        const int nid = cd.seq[next_pos_exit];
        const MmaModel &N = *a.model[nid];
        const int16_t *st2 = a.stale + (s * 3 + nid) * 40;
        for (int i = lane; i < 240; i += 32) ctx[i] = (i < 200) ? N.silence[i % 40] : st2[i - 200];
        for (int i = lane; i < NNSP_B200_MAX_WIDTH; i += 32) { a.st.h[s * NNSP_B200_MAX_WIDTH + i] = 0; a.st.c[s * NNSP_B200_MAX_WIDTH + i] = 0; }
        trig = out0 = out1 = out2 = last = 0; slides = 1;
#pragma unroll
        for (int i = 0; i < 8; i++) cnt[i] = 0;
        if (id == NNSP_B200_ID_S2I) cnt_s2i = 0; else if (id == NNSP_B200_ID_KWS) cnt_kws = 0;
        if (lane == 0) {
            a.st.casc[s * CS_N + CS_POS] = (uint16_t)next_pos_exit;
            a.st.casc[s * CS_N + CS_AGE] = 0;
            a.ra.t0[s] = t_exit + 1;
            a.ra.tb[s] = t_exit + 1; a.ra.tstart[s] = t_exit + 1; a.ra.age0[s] = 0;   /* a fresh instance: slides == 1 (nn_speech.c:62) */
            if (t_exit + 1 < Ts) a.next_list[a.s0 + atomicAdd(a.next_count, 1)] = (int)s;   /* at Ts - 1: next call */
        }
    } else {
        const int n = Ts - tb;                                         /* frames the instance lived in this call */
        if (has_to) { const int c = (c0 + n) % timeout; if (id == NNSP_B200_ID_S2I) cnt_s2i = c; else cnt_kws = c; }
        slides ^= n & 1;                                               /* nn_speech.c:125 */
        if (lane == 0) {
            a.ra.t0[s] = T + 1;                    /* lived through the call: cascade_ctx_kernel rebuilds its context */
            const int age = age0 + n;
            a.st.casc[s * CS_N + CS_AGE] = (uint16_t)(age < 2 ? age : 2);
        }
    }
    if (lane == 0) {
        a.st.casc[s * CS_N + CS_CNT_KWS] = (uint16_t)cnt_kws;
        a.st.casc[s * CS_N + CS_CNT_S2I] = (uint16_t)cnt_s2i;
        int16_t sc[SC_N];
        sc[SC_TRIGGER] = (int16_t)trig; sc[SC_OUT0] = (int16_t)out0; sc[SC_OUT0 + 1] = (int16_t)out1; sc[SC_OUT0 + 2] = (int16_t)out2;
#pragma unroll
        for (int i = 0; i < 8; i++) sc[SC_CNT0 + i] = (int16_t)cnt[i];
        sc[SC_ARGMAX_LAST] = (int16_t)last; sc[SC_SLIDES] = (int16_t)slides; sc[SC_RAN] = 0; sc[SC_STAGE] = 0;
        uint4 *p = reinterpret_cast<uint4 *>(a.st.scal + s * SC_N);
        p[0] = *reinterpret_cast<uint4 *>(&sc[0]);
        p[1] = *reinterpret_cast<uint4 *>(&sc[8]);
    }
}

/* context of the instances that lived through the call (t0 == T + 1): the newest six standardised rows of (the rows the
 * instance had when its life in this call began ++ the rows of its frames tb .. Ts-1, read with its look-back); a warp
 * per stream */
__global__ void __launch_bounds__(256) cascade_ctx_kernel(CascadePostArgs a)
{
    const int si = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (si >= a.ns) return;
    const long long s = a.s0 + si;
    const int T = a.T;
    if (a.ra.t0[s] != T + 1) return;
    const CascadeDev &cd = a.cd;
    const int id = cd.seq[a.st.casc[s * CS_N + CS_POS]];
    const int d = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? cd.P.frs_vbufBk_kws : cd.P.frs_vbufBk_s2i);
    const int tb = a.ra.tb[s], age0 = a.ra.age0[s], Ts = stream_frames(a.nfr, s, T);
    const MmaModel &M = *a.model[id];
    int16_t *ctx = a.st.ctx + s * 240;
    int16_t v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int e = lane + 32 * k;
        v[k] = 0;
        if (e < 240) {
            const int j = e / 40, i = e - j * 40, f = Ts - 6 + j;
            v[k] = (f >= tb) ? standardise(cascade_lm_row(a, s, f, d, tb, age0)[i], M.mean[i], M.stdR[i], M.feat_rshift)
                             : ctx[(6 + f - tb) * 40 + i];
        }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; k++) { const int e = lane + 32 * k; if (e < 240) ctx[e] = v[k]; }
}

struct ResetModels { const DevModel *m[3]; int seq[CS_MAXSEQ]; };

/* A stream's record (nnsp_b200_cascade_export_streams): the 64-byte nnsp_b200_stream_header, then the state at these
 * byte offsets, every part a multiple of 8 bytes at an 8-byte aligned offset; the PCM ring (hist_words 32-bit words)
 * at REC_RING, the log-mel history (lm_words) behind it. In the records a call stages for its imports, the header's
 * `reserved` word holds the destination stream instead (REC_DEST). */
constexpr int REC_DEST = 56, REC_SCAL = 64, REC_CASC = 96, REC_PAD = 104, REC_CTX = 112, REC_H = 592, REC_C = 848,
              REC_STALE = 1360, REC_RING = 1600;
static_assert(REC_H == REC_CTX + 240 * 2 && REC_C == REC_H + NNSP_B200_MAX_WIDTH * 2 &&
              REC_STALE == REC_C + NNSP_B200_MAX_WIDTH * 4 && REC_RING == REC_STALE + 120 * 2, "record layout");
__host__ __device__ constexpr long long rec_bytes_of(int hist_words, int lm_words) { return REC_RING + 4LL * (hist_words + lm_words); }

__device__ __forceinline__ void copy8(void *dst, const void *src, int nbytes)
{
    uint2 *d = reinterpret_cast<uint2 *>(dst);
    const uint2 *q = reinterpret_cast<const uint2 *>(src);
    for (int i = threadIdx.x; i < nbytes / 8; i += blockDim.x) d[i] = q[i];
}

/* Entries of a device list of pending operations: (stream << 2 | op) for the resets, (record << 2 | op) for the ops that
 * load a staged record, which names its stream at REC_DEST. OP_INSTANCE / OP_FRESH are NNSP_B200_RESET_INSTANCE / _FRESH. */
constexpr int OP_INSTANCE = 0, OP_FRESH = 1, OP_LOAD = 2, OP_LOAD_INSTANCE = 3;

/* nnCntrlClass_reset (nnCntrlClass.c:130-150): every instance reset, ring cleared, timeout counters
 * zeroed; current_pos_seq is NOT rewound (only nnCntrlClass_init sets it, :125) and every instance keeps
 * its context row 5. fresh != 0 (create = init + reset on zeroed structs) also rewinds and clears those.
 * list == null: streams 0 .. S-1, one per CTA, all with `fresh`; else the entries list[0 .. gridDim.x) (OP_*):
 * OP_LOAD writes the record recs[entry >> 2] into its stream, OP_LOAD_INSTANCE does that and then the reset.
 * `parts` says what is written: the histories (PCM ring and log-mel rows), which the front end reads and rewrites, and
 * the controller / instance state, which the chain reads -- a pipelined call resets them on different streams. */
constexpr int RESET_HIST = 1, RESET_STATE = 2;
__global__ void cascade_reset_kernel(ResetModels rm, StreamState st, int16_t *stale, int S,
                                     int hist_words, int lm_words, int fresh, const int *list, int parts, const uint8_t *recs)
{
    int s = blockIdx.x, op = fresh;
    const uint8_t *rec = nullptr;
    if (list) {
        const int e = list[blockIdx.x];
        op = e & 3;
        if (op & OP_LOAD) { rec = recs + (e >> 2) * rec_bytes_of(hist_words, lm_words); s = *reinterpret_cast<const int *>(rec + REC_DEST); }
        else s = e >> 2;
    }
    if (s >= S) return;
    const int HS = NNSP_B200_MAX_WIDTH;
    if ((parts & RESET_STATE) && rec) {
        copy8(st.scal + (long long)s * SC_N, rec + REC_SCAL, SC_N * 2);
        copy8(st.casc + (long long)s * CS_N, rec + REC_CASC, CS_N * 2);
        copy8(st.ctx + (long long)s * 240, rec + REC_CTX, 240 * 2);
        copy8(st.h + (long long)s * HS, rec + REC_H, HS * 2);
        copy8(st.c + (long long)s * HS, rec + REC_C, HS * 4);
        copy8(stale + (long long)s * 120, rec + REC_STALE, 120 * 2);
    }
    if ((parts & RESET_STATE) && op != OP_LOAD) {
        const bool fresh = op == OP_FRESH;
        __syncthreads();                                                  /* the position a load just wrote */
        const int pos = fresh ? 0 : st.casc[(long long)s * CS_N + CS_POS];
        const DevModel *M = rm.m[rm.seq[pos]];
        __syncthreads();
        for (int i = threadIdx.x; i < 200; i += blockDim.x) st.ctx[(long long)s * 240 + i] = M->silence[i % 40];
        if (fresh) {
            for (int i = threadIdx.x; i < 40; i += blockDim.x) st.ctx[(long long)s * 240 + 200 + i] = 0;
            for (int i = threadIdx.x; i < 120; i += blockDim.x) stale[(long long)s * 120 + i] = 0;
        }
        for (int i = threadIdx.x; i < HS; i += blockDim.x) { st.h[(long long)s * HS + i] = 0; st.c[(long long)s * HS + i] = 0; }
        for (int i = threadIdx.x; i < SC_N; i += blockDim.x) st.scal[(long long)s * SC_N + i] = (i == SC_SLIDES) ? 1 : 0;
        for (int i = threadIdx.x; i < CS_N; i += blockDim.x) st.casc[(long long)s * CS_N + i] = (i == CS_POS) ? (uint16_t)pos : (uint16_t)0;
    }
    if (parts & RESET_HIST) {                   /* OP_LOAD_INSTANCE: the reset overwrites all the load would write here */
        unsigned int *h = reinterpret_cast<unsigned int *>(st.hist) + (long long)s * hist_words;
        int32_t *lm = st.lmhist + (long long)s * lm_words;
        if (op == OP_LOAD) {
            copy8(h, rec + REC_RING, hist_words * 4);
            copy8(lm, rec + REC_RING + 4LL * hist_words, lm_words * 4);
        } else {
            for (int i = threadIdx.x; i < hist_words; i += blockDim.x) h[i] = 0;              /* PcmBufClass_reset, PcmBufClass.c:19-28 */
            for (int i = threadIdx.x; i < lm_words; i += blockDim.x) lm[i] = LOGMEL_OF_ZERO;  /* log-mel of an all-zero window */
        }
    }
}

/* the records of the streams ids[0 .. gridDim.x), one per CTA, into out: header `hdr`, then the state (REC_*) */
__global__ void cascade_export_kernel(StreamState st, const int16_t *stale, const int *ids, uint8_t *out, int hist_words,
                                      int lm_words, nnsp_b200_stream_header hdr)
{
    const long long s = ids[blockIdx.x];
    const int HS = NNSP_B200_MAX_WIDTH;
    uint8_t *rec = out + blockIdx.x * rec_bytes_of(hist_words, lm_words);
    copy8(rec, &hdr, (int)sizeof hdr);
    if (threadIdx.x == 0) *reinterpret_cast<uint2 *>(rec + REC_PAD) = make_uint2(0, 0);
    copy8(rec + REC_SCAL, st.scal + s * SC_N, SC_N * 2);
    copy8(rec + REC_CASC, st.casc + s * CS_N, CS_N * 2);
    copy8(rec + REC_CTX, st.ctx + s * 240, 240 * 2);
    copy8(rec + REC_H, st.h + s * HS, HS * 2);
    copy8(rec + REC_C, st.c + s * HS, HS * 4);
    copy8(rec + REC_STALE, stale + s * 120, 120 * 2);
    copy8(rec + REC_RING, st.hist + s * hist_words * 2, hist_words * 4);
    copy8(rec + REC_RING + 4LL * hist_words, st.lmhist + s * lm_words, lm_words * 4);
}

}  // namespace nnsp

using namespace nnsp;

#define CS_HOST_RING 4

struct nnsp_b200_cascade {
    int device = 0, S = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t xs[3] = { nullptr, nullptr, nullptr };
    const DevTables *tables = nullptr;
    DeviceModel dm[3];
    bool have[3] = { false, false, false };
    CascadeDev cd{};
    CascThr *thr = nullptr;              /* [S] thresholds and time-outs of every stream (device); cd.thr points here */
    StreamState st{};
    int16_t *stale = nullptr;
    int32_t *logmel = nullptr; long long logmel_frames = 0;
    int16_t *d_pcm = nullptr; long long d_pcm_frames = 0;   /* host-buffer calls: staged PCM, two buffers of [S][d_pcm_frames][160] used alternately */
    /* The H2D copies of host-buffer calls go through their own stream, all slices of a call back to back, so that the host
     * link never waits for a slice's kernels (it bounds the end-to-end rate: 262 MB per 100-frame call of 8 192 streams).
     * ev_h2d[buffer][slice]: the slice's PCM has arrived; ev_read[buffer][slice]: the kernels that read it are done. */
    cudaStream_t h2d_stream = nullptr;
    cudaEvent_t ev_h2d[2][8] = {}, ev_read[2][8] = {};
    bool read_valid[2][8] = {};
    long long host_calls = 0;
    nnsp_b200_cascade_result *d_res = nullptr;
    size_t smem_total = 0; int off_w = 0, off_b = 0;
    bool narrow = false;                      /* which shape of the sequential kernel (CsNarrow / CsWide) */
    bool replay_coop = true;                  /* what the rounds leave goes to cascade_replay_kernel (NNSP_CR_GW warps per stream); NNSP_B200_REPLAY_COOP=0: one warp per stream */
    size_t smem_replay = 0; int off_w_replay = 0;
    /* CUDA events around the front end and around the controller / network chain of the last CS_TL device-buffer calls:
     * [0] front end starts, [1] front end done, [2] chain starts, [3] chain done (nnsp_b200_cascade_timeline) */
    cudaEvent_t tl[8][4] = {};
    long long tl_count = 0;
    bool ev_valid = false;
    /* stage-sorted pass (scan-split kernels per (model, phase) group + replay) */
    MmaDeviceModel mm[3];
    bool split_ok = false;
    int path = 0;                              /* 0 auto, 1 sequential kernel only, 2 stage-sorted pass + replay */
    int pa_max = 0;
    int *grp_list = nullptr, *ctl = nullptr, *fix_list = nullptr, *pend[2] = { nullptr, nullptr }, *replay_sorted = nullptr;
    RoundArrays ra{};
    int rounds = 3;                            /* stage-sorted rounds per call (1 .. CS_MAX_ROUNDS); NNSP_B200_CASCADE_ROUNDS */
    uint8_t *planes[2] = { nullptr, nullptr };
    int16_t *vseq = nullptr; int vseq_rows = 0;   /* [S][vseq_rows][40]: the standardised window rows of round 1 (vseq_kernel), input of the tcgen05 layer-0 kernel */
    int32_t *dec = nullptr;
    long long split_cap_T = 0;
    cudaStream_t gs[4][3] = {};                /* per pipeline stream (3 host-call streams + the device-call stream): one per model group */
    /* device-buffer calls are pipelined like the batched path: front end of call N+1 on `stream`, controller / network
     * work of call N on `nn_stream`; log-mel rows are double buffered */
    cudaStream_t nn_stream = nullptr;
    cudaEvent_t ev_feat[2] = { nullptr, nullptr }, ev_nn[2] = { nullptr, nullptr };
    bool nn_pending[2] = { false, false }, last_piped = false;
    unsigned pipe = 0;
    int32_t *logmel2 = nullptr;                /* second log-mel buffer */
    /* Every call's front end writes the next PCM and log-mel histories into hist2 / lmhist2, and the three buffers of
     * each rotate once per call (cascade_next_hist). Three, because a pipelined call N+1's front end then writes the
     * buffers that call N-1's chain read, which it waits for anyway (for its log-mel rows), while call N's chain may
     * still read the ones call N read. */
    int16_t *hist2 = nullptr, *hist3 = nullptr;       /* the next PCM history, the spare */
    int32_t *lmhist2 = nullptr, *lmhist3 = nullptr;   /* the same for the log-mel history */
    cudaEvent_t ev_fork[4] = {}, ev_join[4][3] = {};
    /* asynchronous host-buffer calls: one completion event per pipeline stream, a ring of CS_HOST_RING calls */
    cudaEvent_t host_ev[CS_HOST_RING][3] = {};
    long long host_seq = 0;
    bool host_inflight = false;
    int host_last_T = 0;                       /* frames per stream of the latest host-buffer call */
    int host_fmt = NNSP_B200_HOST_PCM16;       /* int16 PCM or raw 32-bit AUDADC words (conditioned on the device) */
    uint32_t *d_raw = nullptr;
    int32_t *d_nfr = nullptr;                  /* ragged host-buffer calls: the per-stream counts, two buffers of [S] like d_pcm */
    /* nnsp_b200_cascade_reset_streams: the pending mode of every stream (-1: none) and the streams that have one. The next
     * call takes them as a list sorted by stream, entries (stream << 1 | fresh), written into pinned staging rs_host[b]
     * and copied to rs_dev[...] on the stream that reads it. Both staging buffers alternate between the calls that carry
     * resets; rs_copied[b][j] marks the end of the copies out of rs_host[b] on pipeline stream j (0: c->stream for device
     * calls). A device-buffer call uses rs_dev[its pipe index] (rewritten after the chain two calls back, like the log-mel
     * rows); a host-buffer call puts slice [s0, s1)'s entries at rs_dev[0] + s0, always on the slice's own stream. */
    std::vector<int8_t> rs_mode;               /* OP_* or -1 */
    std::vector<int> rs_ids;
    std::vector<int> rs_taken, rs_taken_loads; /* the latest take: its streams in list order, loads before each entry (+ total) */
    int *rs_host[2] = { nullptr, nullptr }, *rs_dev[2] = { nullptr, nullptr };
    cudaEvent_t rs_copied[2][3] = {};
    bool rs_copy_valid[2][3] = {};
    unsigned rs_flushes = 0;
    /* nnsp_b200_cascade_import_streams: the pending record of a stream whose mode is OP_LOAD / OP_LOAD_INSTANCE sits at
     * slot ip_slot[s] of ip_pool (a stream imported and then reset FRESH keeps its slot, unused, until the take; every
     * pending stream's slot is released when the pool is emptied). The call that takes it packs the records of its loads, in list order, into pinned
     * rp_host[b] (b as rs_host) and copies them to rp_dev[b] on the streams of the kernels that read them; rp_read[b][j]
     * marks the end of those kernels on pipeline stream j (0..2: c->stream / the host slices' streams, 3: nn_stream), and
     * both buffers of b are rewritten only after them. Capacities in records, grown on demand. */
    std::vector<uint8_t> ip_pool;
    std::vector<int> ip_slot;
    uint8_t *rp_host[2] = { nullptr, nullptr }, *rp_dev[2] = { nullptr, nullptr };
    int rp_cap[2] = { 0, 0 };
    cudaEvent_t rp_read[2][4] = {};
    bool rp_read_valid[2][4] = {};
    int *ex_ids = nullptr; uint8_t *ex_dev = nullptr; long long ex_cap = 0;   /* export: device ids and records, grown on demand */
    nnsp_b200_stream_header hdr{};             /* the header of this handle's records */
    long long rec_bytes = 0;
};

constexpr int CS_MAX_SLICES = 8;

static bool cascade_use_split(const nnsp_b200_cascade *c, const nnsp_b200_taps *taps)
{
    if (c->path == 1 || !c->split_ok) return false;
    if (taps && (taps->logmel || taps->feat || taps->act || taps->logits || taps->hstate || taps->cstate || taps->post))
        return false;                          /* the debug taps are produced by the sequential kernel */
    return true;
}

/* Layer 0 of the first round (which holds nearly all streams) on the tcgen05 kernel: vseq_kernel writes every stream's
 * standardised window rows once, seg0_tc5_kernel contracts them (nnsp_split.cu, nnsp_tc5.cuh). Bit-exact and tested, but
 * OFF unless NNSP_B200_TC5=2: its CTA needs a whole SM's shared memory, so unlike seg_kernel<2> it cannot share SMs with
 * the next call's front end, and the call is no faster (8 192 streams x 100 frames: 1.441 vs 1.430 ms back to back). */
static bool cascade_tc5_round()
{
    const char *e = getenv("NNSP_B200_TC5");
    return e && e[0] == '2';
}

static int cascade_ensure_split(nnsp_b200_cascade *c, int T)
{
    if (!c->split_ok || c->path == 1 || T <= c->split_cap_T) return NNSP_B200_OK;
    NNSP_CUDA(cudaDeviceSynchronize());
    for (auto &p : c->planes) { if (p) cudaFree(p); p = nullptr; }
    if (c->dec) { cudaFree(c->dec); c->dec = nullptr; }
    if (c->vseq) { cudaFree(c->vseq); c->vseq = nullptr; }
    c->split_cap_T = 0;
    const size_t n_inf_max = (size_t)(T + 1) / 2, tiles = (size_t)c->S / 16 + (size_t)(CG_GROUPS + 1) * CS_MAX_SLICES + 2;
    for (auto &p : c->planes) NNSP_CUDA(cudaMalloc(&p, tiles * n_inf_max * 32 * c->pa_max));
    NNSP_CUDA(cudaMalloc(&c->dec, ((size_t)c->S + 16) * n_inf_max * sizeof(int32_t)));
    if (cascade_tc5_round()) {
        c->vseq_rows = (int)(2 * n_inf_max + 4);
        NNSP_CUDA(cudaMalloc(&c->vseq, (size_t)c->S * c->vseq_rows * NNSP_B200_NMEL * sizeof(int16_t)));
    }
    c->split_cap_T = T;
    return NNSP_B200_OK;
}

static int cascade_ensure_logmel(nnsp_b200_cascade *c, int T)
{
    if (T <= c->logmel_frames) return NNSP_B200_OK;
    NNSP_CUDA(cudaDeviceSynchronize());
    if (c->logmel) cudaFree(c->logmel);
    if (c->logmel2) cudaFree(c->logmel2);
    c->logmel = nullptr; c->logmel2 = nullptr;
    NNSP_CUDA(cudaMalloc(&c->logmel, (size_t)c->S * T * NNSP_B200_NMEL * sizeof(int32_t)));
    NNSP_CUDA(cudaMalloc(&c->logmel2, (size_t)c->S * T * NNSP_B200_NMEL * sizeof(int32_t)));
    c->logmel_frames = T;
    return NNSP_B200_OK;
}

static int cascade_hist_words(const nnsp_b200_cascade *c) { return (c->cd.dmax + 2) * (NNSP_B200_FRAME / 2); }
static int cascade_lm_words(const nnsp_b200_cascade *c) { return (c->cd.dmax > 0 ? c->cd.dmax : 1) * NNSP_B200_NMEL; }

/* cascade_reset_kernel over every stream (list null, all `fresh`) or over the n entries of the device list, whose
 * loads read the device records `recs` */
static int cascade_launch_reset(nnsp_b200_cascade *c, const int *list, int n, int fresh, int parts, cudaStream_t st,
                                const uint8_t *recs = nullptr)
{
    ResetModels rm{};
    for (int i = 0; i < 3; i++) rm.m[i] = c->dm[i].d;
    for (int i = 0; i < c->cd.len_seq; i++) rm.seq[i] = c->cd.seq[i];
    cascade_reset_kernel<<<list ? n : c->S, 128, 0, st>>>(rm, c->st, c->stale, c->S, cascade_hist_words(c), cascade_lm_words(c),
                                                          fresh, list, parts, recs);
    NNSP_LAUNCH_CHECK();
    return NNSP_B200_OK;
}

/* The pending resets and imports as a list sorted by stream in the pinned staging buffer of this call (*list, *n, *b =
 * which one; n == 0: none), the records of its *loads in rp_host[*b], and the pending set cleared. The buffers were
 * last written by the call before last that carried any: the host waits until the device has run that call's list
 * copies -- and, when this call loads records, the kernels that read that call's records -- the only host waits these
 * functions add. Those sit in stream order behind what was queued before them on their stream -- on a pipelined device
 * call the wait for the chain two calls back (a record's reader: one call back), on a host call the same slice of the
 * ticket before -- so a caller that resets before every call runs at most about two calls ahead of the device; calls
 * without pending operations never wait here. */
static int cascade_take_resets(nnsp_b200_cascade *c, const int **list, int *n, int *b, int *loads)
{
    *n = (int)c->rs_ids.size();
    *loads = 0;
    if (*n == 0) return NNSP_B200_OK;
    *b = (int)(c->rs_flushes++ & 1u);
    for (int j = 0; j < 3; j++)
        if (c->rs_copy_valid[*b][j]) { NNSP_CUDA(cudaEventSynchronize(c->rs_copied[*b][j])); c->rs_copy_valid[*b][j] = false; }
    std::sort(c->rs_ids.begin(), c->rs_ids.end());
    c->rs_taken.swap(c->rs_ids);
    c->rs_ids.clear();
    c->rs_taken_loads.resize((size_t)*n + 1);
    for (int k = 0; k < *n; k++) {
        c->rs_taken_loads[(size_t)k] = *loads;
        if (c->rs_mode[(size_t)c->rs_taken[(size_t)k]] & OP_LOAD) ++*loads;
    }
    c->rs_taken_loads[(size_t)*n] = *loads;
    if (*loads) {
        for (int j = 0; j < 4; j++)
            if (c->rp_read_valid[*b][j]) { NNSP_CUDA(cudaEventSynchronize(c->rp_read[*b][j])); c->rp_read_valid[*b][j] = false; }
        if (*loads > c->rp_cap[*b]) {                                  /* nothing reads either buffer any more */
            if (c->rp_host[*b]) NNSP_CUDA(cudaFreeHost(c->rp_host[*b]));
            if (c->rp_dev[*b]) NNSP_CUDA(cudaFree(c->rp_dev[*b]));
            c->rp_host[*b] = nullptr; c->rp_dev[*b] = nullptr; c->rp_cap[*b] = 0;
            NNSP_CUDA(cudaHostAlloc(&c->rp_host[*b], (size_t)*loads * c->rec_bytes, cudaHostAllocDefault));
            NNSP_CUDA(cudaMalloc(&c->rp_dev[*b], (size_t)*loads * c->rec_bytes));
            c->rp_cap[*b] = *loads;
        }
    }
    int *h = c->rs_host[*b];
    for (int k = 0, l = 0; k < *n; k++) {
        const int s = c->rs_taken[(size_t)k], op = c->rs_mode[(size_t)s];
        if (op & OP_LOAD) {
            uint8_t *r = c->rp_host[*b] + (size_t)l * c->rec_bytes;
            memcpy(r, c->ip_pool.data() + (size_t)c->ip_slot[(size_t)s] * c->rec_bytes, (size_t)c->rec_bytes);
            memcpy(r + REC_DEST, &s, sizeof s);
            h[k] = (l++ << 2) | op;
        } else
            h[k] = (s << 2) | op;
        c->rs_mode[(size_t)s] = -1;
        c->ip_slot[(size_t)s] = -1;            /* also a slot whose import a FRESH reset replaced: the pool is emptied */
    }
    c->ip_pool.clear();
    *list = h;
    return NNSP_B200_OK;
}

/* what a call applies before its kernels read the state: the device list, the device records of its loads (null:
 * none) and the events to record behind the kernels that read those records on the front-end stream and the chain's */
struct PendingOps {
    const int *list; int n;
    const uint8_t *recs;
    cudaEvent_t read_hist, read_state;
};

/* The front end writes the next PCM and log-mel histories of streams s0 .. s0+ns-1 out of place into c->hist2 /
 * c->lmhist2 (the caller rotates the buffers once per call: cascade_next_hist).
 * st_nn (with ev_feat): pipelined call -- everything behind the front end goes to st_nn.
 * ops (null: none): streams reset or loaded before the call -- the histories on st before the front end reads them, the
 * rest on the stream of the chain before the chain reads it. */
static int cascade_launch(nnsp_b200_cascade *c, const int16_t *pcm, long long stride, int T, int s0, int ns,
                          nnsp_b200_cascade_result *results, const nnsp_b200_taps *taps, cudaStream_t st, bool timed,
                          int slice = 0, int32_t *logmel = nullptr, cudaStream_t st_nn = nullptr, cudaEvent_t ev_feat = nullptr,
                          const int32_t *nfr = nullptr, const PendingOps *ops = nullptr)
{
    if (!logmel) logmel = c->logmel;
    const bool piped = st_nn != nullptr;
    int rc;
    if (ops) {
        if ((rc = cascade_launch_reset(c, ops->list, ops->n, 0, piped ? RESET_HIST : RESET_HIST | RESET_STATE, st, ops->recs))) return rc;
        if (ops->recs) NNSP_CUDA(cudaEventRecord(ops->read_hist, st));
    }
    FeatLaunch fl{ pcm, stride, c->st.hist, c->cd.dmax + 2, s0, ns, T, logmel };
    fl.nfr = nfr;
    fl.hist_out = c->hist2;
    if (c->cd.dmax > 0) { fl.lm_hist = c->st.lmhist; fl.lm_out = c->lmhist2; fl.lm_rows = c->cd.dmax; }
    cudaEvent_t *tl = c->tl[c->tl_count % 8];
    if (timed) NNSP_CUDA(cudaEventRecord(tl[0], st));
    rc = launch_feature(c->tables, fl, c->device, st);
    if (rc) return rc;
    if (timed) NNSP_CUDA(cudaEventRecord(tl[1], st));
    if (piped) {
        NNSP_CUDA(cudaEventRecord(ev_feat, st));
        NNSP_CUDA(cudaStreamWaitEvent(st_nn, ev_feat, 0));
        st = st_nn;
        if (timed) NNSP_CUDA(cudaEventRecord(tl[2], st));
        /* behind the previous call's chain (stream order) and this call's front end (ev_feat), before anything reads it */
        if (ops) {
            if ((rc = cascade_launch_reset(c, ops->list, ops->n, 0, RESET_STATE, st, ops->recs))) return rc;
            if (ops->recs) NNSP_CUDA(cudaEventRecord(ops->read_state, st));
        }
    }
    CascadeArgs a{};
    for (int i = 0; i < 3; i++) { a.model[i] = c->dm[i].d; a.wimg[i] = c->dm[i].wimg; a.bimg[i] = c->dm[i].bimg; }
    a.tables = c->tables; a.st = c->st; a.stale = c->stale; a.pcm = pcm; a.stride = stride; a.logmel = logmel;
    a.s0 = s0; a.ns = ns; a.T = T; a.results = results; a.cd = c->cd; a.nfr = nfr;
    if (taps) a.taps = *taps;
    if (cascade_use_split(c, taps)) {
        /* stage-sorted rounds (see the kernels above). Everything is sized for the worst case and reads its true size
         * from the slice's control block on the device: no host round trip between the rounds. */
        int *ctl = c->ctl + slice * CTL_INTS;
        const int lane_set = piped ? 3 : slice % 3;     /* group streams / events of this pipeline stream */
        const int n_inf_max = (T + 1) / 2;
        const int cap = sm_count(c->device);
        NNSP_CUDA(cudaMemsetAsync(ctl, 0, CTL_INTS * sizeof(int), st));
        cascade_classify_kernel<<<(ns + 255) / 256, 256, 0, st>>>(c->st, c->cd, s0, ns, c->S, c->grp_list, ctl, c->ra, c->fix_list, nfr, T);
        NNSP_LAUNCH_CHECK();
        cascade_offsets_kernel<<<1, 1, 0, st>>>(ctl);
        NNSP_LAUNCH_CHECK();
        CascadePostArgs p{};
        for (int i = 0; i < 3; i++) p.model[i] = c->mm[i].d;
        p.st = c->st; p.stale = c->stale; p.logmel = logmel; p.dec = c->dec; p.dec_stride = n_inf_max; p.ra = c->ra;
        p.s0 = s0; p.ns = ns; p.T = T; p.results = results; p.cd = c->cd; p.nfr = nfr;
        for (int r = 0; r < c->rounds; r++) {
            int *ctl_r = ctl + CTL_ROUND * r, *ctl_prev = ctl + CTL_ROUND * (r - 1);
            const int *queued = r ? c->pend[r & 1] + s0 : nullptr;        /* streams the previous round's walk queued */
            if (r) {
                cascade_regroup_kernel<<<1, CSORT_THREADS, 0, st>>>(c->st, c->cd, queued, ctl_prev, ctl_r, c->grp_list, c->S, s0, c->ra, T, nfr);
                NNSP_LAUNCH_CHECK();
            }
            {   /* log-mel rows of the first two frames of fresh instances */
                FixArgs f{};
                f.tables = c->tables; f.st = c->st; f.pcm = pcm; f.stride = stride; f.ra = c->ra; f.cd = c->cd; f.T = T; f.nfr = nfr;
                f.list = r ? queued : c->fix_list + s0;
                f.count = r ? ctl_prev + CTL_NEXT : ctl + CTL_FIX;
                int fb = (ns + 7) / 8;
                if (fb > 4 * cap) fb = 4 * cap;
                cascade_fix_kernel<<<fb, 256, 0, st>>>(f);
                NNSP_LAUNCH_CHECK();
            }
            /* every model's group through the scan-split kernels, side by side on their own CUDA streams (independent
             * chains, and the scans are latency-bound) */
            NNSP_CUDA(cudaEventRecord(c->ev_fork[lane_set], st));
            for (int k = 0; k < c->cd.len_seq; k++) {
                const int id = c->cd.seq[k];
                SplitGroup q{};
                q.tables = c->tables;
                q.list = c->grp_list + (size_t)id * c->S + s0; q.count = ctl_r + id; q.tile_off = ctl_r + 3 + id;
                q.tile0 = (s0 >> 4) + (CG_GROUPS + 1) * slice; q.max_streams = ns;
                q.tile_bytes = (long long)n_inf_max * 32 * c->pa_max;
                q.T = T; q.first = 0; q.n_inf = n_inf_max;
                q.mode = 2; q.logmel = logmel; q.lmhist = c->st.lmhist; q.dmax = c->cd.dmax;
                q.dback = (id == NNSP_B200_ID_VAD) ? 0 : (id == NNSP_B200_ID_KWS ? c->cd.P.frs_vbufBk_kws : c->cd.P.frs_vbufBk_s2i);
                q.ctx = c->st.ctx; q.h = c->st.h; q.c = c->st.c; q.h_stride = NNSP_B200_MAX_WIDTH;
                q.planes0 = c->planes[0]; q.planes1 = c->planes[1];
                q.dec = c->dec; q.dec_stride = n_inf_max;
                q.thresh_prob = 0; q.thr_prob = &c->thr->prob[id]; q.thr_stride = (int)(sizeof(CascThr) / sizeof(int16_t));   /* per stream: thr[s].prob[id] */
                q.tstart = c->ra.tstart; q.tb = c->ra.tb; q.age0 = c->ra.age0; q.lmfix = c->ra.lmfix; q.nfr = nfr;
                if (r == 0 && c->vseq) { q.vseq = c->vseq; q.vseq_rows = c->vseq_rows; }
                cudaStream_t gs = c->gs[lane_set][k];
                NNSP_CUDA(cudaStreamWaitEvent(gs, c->ev_fork[lane_set], 0));
                if ((rc = launch_split_layers(c->mm[id], q, c->device, gs))) return rc;
                NNSP_CUDA(cudaEventRecord(c->ev_join[lane_set][k], gs));
                NNSP_CUDA(cudaStreamWaitEvent(st, c->ev_join[lane_set][k], 0));
            }
            /* walk the controller over the decisions; a stream that changes stage is cut there and queued for the next round */
            p.list = queued; p.count = r ? ctl_prev + CTL_NEXT : nullptr;
            p.next_list = c->pend[(r + 1) & 1]; p.next_count = ctl_r + CTL_NEXT;
            if (nfr) cascade_post_kernel<true><<<(ns + CPOST_WARPS - 1) / CPOST_WARPS, 32 * CPOST_WARPS, 0, st>>>(p);
            else cascade_post_kernel<false><<<(ns + CPOST_WARPS - 1) / CPOST_WARPS, 32 * CPOST_WARPS, 0, st>>>(p);
            NNSP_LAUNCH_CHECK();
        }
        cascade_ctx_kernel<<<(ns * 32 + 255) / 256, 256, 0, st>>>(p);
        NNSP_LAUNCH_CHECK();
        /* what is still queued after the last round goes to the sequential kernel, longest remainder first */
        a.t0 = c->ra.t0;
        cascade_sort_replay_kernel<<<1, CSORT_THREADS, 0, st>>>(c->pend[c->rounds & 1] + s0, c->replay_sorted + s0,
                                                                ctl + CTL_ROUND * (c->rounds - 1) + CTL_NEXT, ctl + CTL_REPLAY, c->ra.t0, T, nfr);
        NNSP_LAUNCH_CHECK();
        a.replay_list = c->replay_sorted + s0; a.replay_ctl = ctl + CTL_REPLAY;
    }
    const int cs_warps = c->narrow ? CsNarrow::WARPS : CsWide::WARPS;
    int blocks = (ns + cs_warps - 1) / cs_warps;
    const int cap = sm_count(c->device);
    if (blocks > cap) blocks = cap;
    int kind;                                   /* nnsp_b200_cascade_kernel_launches */
    if (a.replay_list && c->narrow && c->replay_coop) {
        /* NNSP_CR_GW warps per stream; as many CTAs as the worst case needs (ns streams), at most one per SM */
        int rb = (ns + CR_GROUPS - 1) / CR_GROUPS;
        if (rb > cap) rb = cap;
        cascade_replay_kernel<<<rb, CR_THREADS, c->smem_replay, st>>>(a, c->off_w_replay, c->off_w_replay + (c->off_b - c->off_w));
        kind = 2;
    } else if (c->narrow) { cascade_kernel<CsNarrow><<<blocks, 32 * CsNarrow::WARPS, c->smem_total, st>>>(a, c->off_w, c->off_b); kind = 0; }
    else { cascade_kernel<CsWide><<<blocks, 32 * CsWide::WARPS, c->smem_total, st>>>(a, c->off_w, c->off_b); kind = 1; }
    g_cascade_net_launches[kind].fetch_add(1, std::memory_order_relaxed);
    NNSP_LAUNCH_CHECK();
    if (timed) {
        if (!piped) NNSP_CUDA(cudaEventRecord(tl[2], st));      /* one stream: the chain starts where the front end ended */
        NNSP_CUDA(cudaEventRecord(tl[3], st));
        c->ev_valid = true; c->last_piped = piped; c->tl_count++;
    }
    return NNSP_B200_OK;
}

/* after a call (never per slice: every slice of a host call reads the same buffers, and slice k always covers the same
 * streams on the same CUDA stream): the histories its front end wrote are the live ones. Without a look-back the
 * one-row log-mel history is never written and does not rotate. */
static void cascade_next_hist(nnsp_b200_cascade *c)
{
    int16_t *t = c->st.hist; c->st.hist = c->hist2; c->hist2 = c->hist3; c->hist3 = t;
    if (c->cd.dmax > 0) { int32_t *u = c->st.lmhist; c->st.lmhist = c->lmhist2; c->lmhist2 = c->lmhist3; c->lmhist3 = u; }
}

static int cascade_join_nn(nnsp_b200_cascade *c, cudaStream_t st)
{
    for (int i = 0; i < 2; i++)
        if (c->nn_pending[i]) { NNSP_CUDA(cudaStreamWaitEvent(st, c->ev_nn[i], 0)); c->nn_pending[i] = false; }
    return NNSP_B200_OK;
}

extern "C" {

void nnsp_b200_cascade_default_params(nnsp_b200_cascade_params *p)     /* ParamsNNCntrl.h:8-21 */
{
    if (!p) return;
    p->thresh_prob_vad = 32767 >> 1; p->thresh_cnts_vad = 4;
    p->frs_vbufBk_s2i = 80; p->thresh_timeout_s2i = 1000; p->thresh_prob_s2i = 32767 >> 1; p->thresh_cnts_s2i = 4;
    p->frs_vbufBk_kws = 80; p->thresh_timeout_kws = 1000; p->thresh_prob_kws = 32767 >> 1; p->thresh_cnts_kws = 4;
}

int nnsp_b200_cascade_create(const nnsp_b200_model *const models[3], const int *seq, int len_seq,
                             const nnsp_b200_cascade_params *params, int n_streams, int device,
                             nnsp_b200_cascade **out)
{
    if (!models || !seq || !out || n_streams <= 0 || len_seq < 1 || len_seq > CS_MAXSEQ) {
        nnsp_set_error("cascade_create: bad arguments (sequence length must be 1..%d)", CS_MAXSEQ);
        return NNSP_B200_ERR_ARG;
    }
    bool seen[3] = { false, false, false };
    for (int i = 0; i < len_seq; i++) {
        if (seq[i] < 0 || seq[i] > 2 || !models[seq[i]]) { nnsp_set_error("cascade_create: seq[%d]=%d has no model", i, seq[i]); return NNSP_B200_ERR_ARG; }
        if (seen[seq[i]]) { nnsp_set_error("cascade_create: id %d appears twice in the sequence (unsupported)", seq[i]); return NNSP_B200_ERR_UNSUPPORTED; }
        if (models[seq[i]]->nn_id != seq[i]) { nnsp_set_error("cascade_create: models[%d] carries nn_id %d", seq[i], models[seq[i]]->nn_id); return NNSP_B200_ERR_ARG; }
        seen[seq[i]] = true;
    }
    int rc = select_device(device);
    if (rc) return rc;
    nnsp_b200_cascade *c = new (std::nothrow) nnsp_b200_cascade();
    if (!c) return NNSP_B200_ERR_NOMEM;
    c->device = device; c->S = n_streams;
    auto fail = [&](int code) { nnsp_b200_cascade_destroy(c); return code; };
    if (params) c->cd.P = *params; else nnsp_b200_cascade_default_params(&c->cd.P);
    const nnsp_b200_cascade_params &P = c->cd.P;
    if (P.thresh_timeout_kws < 1 || P.thresh_timeout_s2i < 1 || P.frs_vbufBk_kws < 0 || P.frs_vbufBk_s2i < 0 ||
        P.frs_vbufBk_kws > 99 || P.frs_vbufBk_s2i > 99) {      /* PcmBufClass ring holds NUM_FRS_VBUF = 100 frames (PcmBufClass.c:6) */
        nnsp_set_error("cascade_create: look-back must be 0..99 frames and timeouts >= 1");
        return fail(NNSP_B200_ERR_ARG);
    }
    c->cd.len_seq = len_seq;
    for (int i = 0; i < len_seq; i++) c->cd.seq[i] = seq[i];
    c->cd.dmax = 0;
    if (seen[NNSP_B200_ID_KWS] && P.frs_vbufBk_kws > c->cd.dmax) c->cd.dmax = P.frs_vbufBk_kws;
    if (seen[NNSP_B200_ID_S2I] && P.frs_vbufBk_s2i > c->cd.dmax) c->cd.dmax = P.frs_vbufBk_s2i;
    if ((rc = get_device_tables(device, &c->tables))) return fail(rc);
    size_t wtot = 0, btot = 0;
    for (int id = 0; id < 3; id++) {
        if (!seen[id]) continue;
        if ((rc = upload_model(models[id], &c->dm[id]))) return fail(rc);
        c->have[id] = true;
        c->cd.woff_words[id] = (int)(wtot / 4); c->cd.wbytes[id] = c->dm[id].h.weight_words * 4; wtot += (size_t)c->cd.wbytes[id];
        c->cd.boff[id] = (int)btot; btot += (size_t)c->dm[id].h.bias_count;
    }
    c->split_ok = true;
    for (int id = 0; id < 3; id++) {
        if (!seen[id]) continue;
        rc = upload_model_mma(models[id], &c->mm[id]);
        if (rc == NNSP_B200_ERR_UNSUPPORTED) { c->split_ok = false; continue; }
        if (rc) return fail(rc);
        if (!split_supported(c->mm[id])) c->split_ok = false;
        if (c->mm[id].h && c->mm[id].h->pa > c->pa_max) c->pa_max = c->mm[id].h->pa;
    }
    /* the narrow shape of the sequential kernel when every model fits its scratch */
    c->narrow = true;
    for (int id = 0; id < 3; id++) {
        if (!seen[id]) continue;
        const DevModel &D = c->dm[id].h;
        if (D.h_stride > CsNarrow::WS::WIDTH || D.n_out > 48) c->narrow = false;
        for (int i = 0; i < D.numlayers; i++)
            if (D.layer[i].rows > CsNarrow::WS::WIDTH || (i > 0 && ((D.layer[i].cols + 3) & ~3) > CsNarrow::WS::WIDTH)) c->narrow = false;
    }
    { const char *e = getenv("NNSP_B200_CASCADE_WIDE"); if (e && e[0] == '1') c->narrow = false; }   /* A/B switch for measurements */
    const size_t smem_struct = c->narrow ? sizeof(CascadeSmem<CsNarrow>) : sizeof(CascadeSmem<CsWide>);
    c->off_w = (int)((16 + smem_struct + 127) & ~(size_t)127);
    c->off_b = (int)(c->off_w + wtot);
    c->smem_total = (size_t)c->off_b + btot * 2 + 16;
    c->off_w_replay = (int)((16 + sizeof(ReplaySmem) + 127) & ~(size_t)127);
    c->smem_replay = (size_t)c->off_w_replay + wtot + btot * 2 + 16;
    { const char *e = getenv("NNSP_B200_REPLAY_COOP"); c->replay_coop = !(e && e[0] == '0'); }        /* A/B switch for measurements */
    if (c->smem_replay > 227 * 1024) c->replay_coop = false;      /* the one-warp-per-stream shape fits whenever create succeeds */
    { const char *e = getenv("NNSP_B200_CASCADE_ROUNDS"); if (e && e[0] >= '1' && e[0] <= '0' + CS_MAX_ROUNDS) c->rounds = e[0] - '0'; }
    if (c->smem_total > 227 * 1024) { nnsp_set_error("cascade needs %zu bytes of shared memory (> 227 KB)", c->smem_total); return fail(NNSP_B200_ERR_UNSUPPORTED); }
    const size_t S = (size_t)n_streams, HS = NNSP_B200_MAX_WIDTH;
    const int hist_frames = c->cd.dmax + 2, lm_rows = c->cd.dmax > 0 ? c->cd.dmax : 1;
#define TRY(x) do { if ((x) != cudaSuccess) { nnsp_set_error("%s failed: %s", #x, cudaGetErrorString(cudaGetLastError())); return fail(NNSP_B200_ERR_CUDA); } } while (0)
    TRY(cudaFuncSetAttribute(cascade_kernel<CsWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    TRY(cudaFuncSetAttribute(cascade_kernel<CsNarrow>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    TRY(cudaFuncSetAttribute(cascade_replay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (auto &s : c->xs) TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto &r : c->host_ev) for (auto &e : r) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    TRY(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
    for (auto &r : c->ev_h2d) for (auto &e : r) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &r : c->ev_read) for (auto &e : r) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &row : c->tl) for (auto &e : row) TRY(cudaEventCreate(&e));
    {
        int lo = 0, hi = 0;                                /* the controller / network chain outranks the front-end stream */
        TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        TRY(cudaStreamCreateWithPriority(&c->nn_stream, cudaStreamNonBlocking, hi));
        const char *e = getenv("NNSP_B200_GS_PRIO");       /* measurement knob: 0 = group streams at the default priority */
        const int gp = (e && e[0] == '0') ? lo : hi;
        for (auto &row : c->gs) for (auto &g : row) TRY(cudaStreamCreateWithPriority(&g, cudaStreamNonBlocking, gp));
    }
    for (auto &e : c->ev_feat) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : c->ev_nn) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : c->ev_fork) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &row : c->ev_join) for (auto &e : row) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    TRY(cudaMalloc(&c->st.ctx, S * 240 * sizeof(int16_t)));
    TRY(cudaMalloc(&c->st.h, S * HS * sizeof(int16_t)));
    TRY(cudaMalloc(&c->st.c, S * HS * sizeof(int32_t)));
    TRY(cudaMalloc(&c->st.scal, S * SC_N * sizeof(int16_t)));
    TRY(cudaMalloc(&c->st.casc, S * CS_N * sizeof(uint16_t)));
    TRY(cudaMalloc(&c->st.hist, S * hist_frames * NNSP_B200_FRAME * sizeof(int16_t)));
    TRY(cudaMalloc(&c->hist2, S * hist_frames * NNSP_B200_FRAME * sizeof(int16_t)));
    TRY(cudaMalloc(&c->hist3, S * hist_frames * NNSP_B200_FRAME * sizeof(int16_t)));
    TRY(cudaMalloc(&c->st.lmhist, S * lm_rows * NNSP_B200_NMEL * sizeof(int32_t)));
    TRY(cudaMalloc(&c->lmhist2, S * lm_rows * NNSP_B200_NMEL * sizeof(int32_t)));
    TRY(cudaMalloc(&c->lmhist3, S * lm_rows * NNSP_B200_NMEL * sizeof(int32_t)));
    TRY(cudaMalloc(&c->stale, S * 120 * sizeof(int16_t)));
    TRY(cudaMalloc(&c->thr, S * sizeof(CascThr)));
    c->cd.thr = c->thr;
    {
        std::vector<nnsp_b200_cascade_params> all(S, c->cd.P);              /* every stream starts with the handle's parameters */
        if ((rc = nnsp_b200_cascade_set_stream_params(c, 0, (int)S, all.data()))) return fail(rc);
    }
    TRY(cudaMalloc(&c->grp_list, (size_t)3 * S * sizeof(int)));
    TRY(cudaMalloc(&c->ctl, CS_MAX_SLICES * CTL_INTS * sizeof(int)));
    TRY(cudaMalloc(&c->fix_list, S * sizeof(int)));
    for (auto &q : c->pend) TRY(cudaMalloc(&q, S * sizeof(int)));
    TRY(cudaMalloc(&c->replay_sorted, S * sizeof(int)));
    TRY(cudaMalloc(&c->ra.t0, S * sizeof(int)));
    TRY(cudaMalloc(&c->ra.tstart, S * sizeof(int)));
    TRY(cudaMalloc(&c->ra.tb, S * sizeof(int)));
    TRY(cudaMalloc(&c->ra.age0, S * sizeof(int)));
    TRY(cudaMalloc(&c->ra.lmfix, S * 2 * NNSP_B200_NMEL * sizeof(int32_t)));
    TRY(cudaMemset(c->ra.lmfix, 0, S * 2 * NNSP_B200_NMEL * sizeof(int32_t)));
    for (int b = 0; b < 2; b++) {
        TRY(cudaHostAlloc(&c->rs_host[b], S * sizeof(int), cudaHostAllocDefault));
        TRY(cudaMalloc(&c->rs_dev[b], S * sizeof(int)));
        for (auto &e : c->rs_copied[b]) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto &e : c->rp_read[b]) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
#undef TRY
    c->rs_mode.assign(S, (int8_t)-1);
    c->ip_slot.assign(S, -1);
    c->rec_bytes = rec_bytes_of(cascade_hist_words(c), cascade_lm_words(c));
    nnsp_b200_stream_header &H = c->hdr;
    H.magic = NNSP_B200_STREAM_MAGIC; H.version = NNSP_B200_STREAM_VERSION; H.record_bytes = (uint32_t)c->rec_bytes;
    H.len_seq = len_seq; H.frs_vbufBk_kws = P.frs_vbufBk_kws; H.frs_vbufBk_s2i = P.frs_vbufBk_s2i;
    for (int k = 0; k < 3; k++) {
        H.seq[k] = k < len_seq ? seq[k] : -1;
        if (k >= len_seq) continue;
        size_t nb = 0;
        if ((rc = nnsp_b200_model_to_blob(models[seq[k]], nullptr, 0, &nb))) return fail(rc);
        std::vector<unsigned char> blob(nb);
        if ((rc = nnsp_b200_model_to_blob(models[seq[k]], blob.data(), nb, &nb))) return fail(rc);
        uint64_t f = 0xcbf29ce484222325ull;                              /* FNV-1a, 64 bits */
        for (unsigned char x : blob) f = (f ^ x) * 0x100000001b3ull;
        H.model_fnv1a[k] = f;
    }
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(NNSP_B200_ERR_CUDA);   /* uploads went through the default stream */
    if ((rc = cascade_launch_reset(c, nullptr, 0, 1, RESET_HIST | RESET_STATE, c->stream))) return fail(rc);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) { nnsp_set_error("cascade reset kernel failed: %s", cudaGetErrorString(cudaGetLastError())); return fail(NNSP_B200_ERR_CUDA); }
    *out = c;
    return NNSP_B200_OK;
}

/* ParamCntrlClass of individual streams (nnCntrlClass.h:12-29 is a member of every controller instance). Thresholds and
 * time-outs take effect with the next call; a counter that already reads beyond a shortened time-out wraps as the
 * reference's `(cnt + 1) % timeout` does. The look-back depths size the history buffers and cannot differ from the handle's. */
int nnsp_b200_cascade_set_stream_params(nnsp_b200_cascade *c, int first_stream, int n_streams, const nnsp_b200_cascade_params *params)
{
    if (!c || !params || first_stream < 0 || n_streams < 0 || (long long)first_stream + n_streams > c->S) {
        nnsp_set_error("cascade_set_stream_params: bad stream range");
        return NNSP_B200_ERR_ARG;
    }
    std::vector<CascThr> h((size_t)n_streams);
    for (int i = 0; i < n_streams; i++) {
        const nnsp_b200_cascade_params &P = params[i];
        if (P.thresh_timeout_kws < 1 || P.thresh_timeout_s2i < 1 || P.frs_vbufBk_kws != c->cd.P.frs_vbufBk_kws || P.frs_vbufBk_s2i != c->cd.P.frs_vbufBk_s2i) {
            nnsp_set_error("cascade_set_stream_params: stream %d: time-outs must be >= 1 and the look-back depths those of the handle (%d, %d)",
                           first_stream + i, (int)c->cd.P.frs_vbufBk_kws, (int)c->cd.P.frs_vbufBk_s2i);
            return NNSP_B200_ERR_ARG;
        }
        CascThr &t = h[(size_t)i];
        t.prob[NNSP_B200_ID_S2I] = P.thresh_prob_s2i; t.prob[NNSP_B200_ID_VAD] = P.thresh_prob_vad; t.prob[NNSP_B200_ID_KWS] = P.thresh_prob_kws;
        t.cnts[NNSP_B200_ID_S2I] = P.thresh_cnts_s2i; t.cnts[NNSP_B200_ID_VAD] = P.thresh_cnts_vad; t.cnts[NNSP_B200_ID_KWS] = P.thresh_cnts_kws;
        t.timeout_kws = P.thresh_timeout_kws; t.timeout_s2i = P.thresh_timeout_s2i;
    }
    NNSP_CUDA(cudaSetDevice(c->device));
    NNSP_CUDA(cudaDeviceSynchronize());                          /* calls in flight still read the old records */
    if (n_streams) NNSP_CUDA(cudaMemcpy(c->thr + first_stream, h.data(), (size_t)n_streams * sizeof(CascThr), cudaMemcpyHostToDevice));
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_reset(nnsp_b200_cascade *c)
{
    if (!c) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(c->device));
    NNSP_CUDA(cudaDeviceSynchronize());
    c->nn_pending[0] = c->nn_pending[1] = false;
    c->host_inflight = false;
    /* resets still pending stay pending: applied at the next call, after this one, they leave what they would have left
     * before it (a reset stream's state does not depend on the state it had). A pending import is followed by this
     * reset: it becomes load-then-reset. */
    for (int s : c->rs_ids)
        if (c->rs_mode[(size_t)s] == OP_LOAD) c->rs_mode[(size_t)s] = OP_LOAD_INSTANCE;
    const int rc = cascade_launch_reset(c, nullptr, 0, 0, RESET_HIST | RESET_STATE, c->stream);
    if (rc) return rc;
    NNSP_CUDA(cudaStreamSynchronize(c->stream));
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_reset_streams(nnsp_b200_cascade *c, const int32_t *streams, int n, int mode)
{
    if (!c || n < 0 || (n > 0 && !streams) || (mode != NNSP_B200_RESET_INSTANCE && mode != NNSP_B200_RESET_FRESH)) {
        nnsp_set_error("cascade_reset_streams: bad arguments (n = %d, mode = %d)", n, mode);
        return NNSP_B200_ERR_ARG;
    }
    for (int i = 0; i < n; i++)                                       /* checked before anything is recorded */
        if (streams[i] < 0 || streams[i] >= c->S) {
            nnsp_set_error("cascade_reset_streams: streams[%d] = %d is outside [0, %d)", i, (int)streams[i], c->S);
            return NNSP_B200_ERR_ARG;
        }
    for (int i = 0; i < n; i++) {
        int8_t &m = c->rs_mode[(size_t)streams[i]];
        if (m < 0) c->rs_ids.push_back(streams[i]);
        if (m >= OP_LOAD) m = (int8_t)(mode == OP_FRESH ? OP_FRESH : OP_LOAD_INSTANCE);   /* an import, then this reset */
        else if (m < mode) m = (int8_t)mode;                          /* FRESH after or before INSTANCE leaves FRESH */
    }
    return NNSP_B200_OK;
}

size_t nnsp_b200_cascade_stream_state_bytes(const nnsp_b200_cascade *c) { return c ? (size_t)c->rec_bytes : 0; }

/* A record that may go to the device: its header matches this handle's, and every body field a kernel uses as an
 * index or a loop bound is in range (the readers of casc / scal in nnsp_cascade.cu and nnsp_split.cu: cd.seq[pos],
 * the fix rows of ages 0 and 1, the frame a time-out falls on, the first inference frame, the S2I argmax). */
int nnsp_cascade_check_records(const nnsp_b200_cascade *c, const void *records, int n)
{
    if (n > 0 && !records) { nnsp_set_error("stream records: null pointer"); return NNSP_B200_ERR_ARG; }
    for (int i = 0; i < n; i++) {
        const unsigned char *r = static_cast<const unsigned char *>(records) + (size_t)i * c->rec_bytes;
        nnsp_b200_stream_header h;
        memcpy(&h, r, sizeof h);
        const char *bad = nullptr;
        if (h.magic != NNSP_B200_STREAM_MAGIC) bad = "bad magic";
        else if (h.version != NNSP_B200_STREAM_VERSION) bad = "unknown version";
        else if (h.record_bytes != (uint32_t)c->rec_bytes) bad = "record size differs from this handle's";
        else if (h.len_seq != c->hdr.len_seq || memcmp(h.seq, c->hdr.seq, sizeof h.seq)) bad = "cascade sequence differs from this handle's";
        else if (h.frs_vbufBk_kws != c->hdr.frs_vbufBk_kws || h.frs_vbufBk_s2i != c->hdr.frs_vbufBk_s2i) bad = "look-back depths differ from this handle's";
        else if (memcmp(h.model_fnv1a, c->hdr.model_fnv1a, sizeof h.model_fnv1a)) bad = "model fingerprints differ from this handle's";
        if (!bad) {
            uint16_t cs[CS_N];
            int16_t sc[SC_N];
            memcpy(cs, r + REC_CASC, sizeof cs);
            memcpy(sc, r + REC_SCAL, sizeof sc);
            if (cs[CS_POS] >= c->cd.len_seq) bad = "sequence position out of range";
            else if (cs[CS_AGE] > 2) bad = "instance age out of range";
            else if (cs[CS_CNT_KWS] >= 32767 || cs[CS_CNT_S2I] >= 32767) bad = "time-out counter out of range";
            else if (sc[SC_SLIDES] != 0 && sc[SC_SLIDES] != 1) bad = "NNSPClass.slides out of range";
            else if (sc[SC_ARGMAX_LAST] < 0 || sc[SC_ARGMAX_LAST] > 6) bad = "last S2I argmax out of range";
        }
        if (bad) { nnsp_set_error("stream record %d: %s", i, bad); return NNSP_B200_ERR_ARG; }
    }
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_import_streams(nnsp_b200_cascade *c, const int32_t *streams, int n, const void *records)
{
    if (!c || n < 0 || (n > 0 && !streams)) { nnsp_set_error("cascade_import_streams: bad arguments (n = %d)", n); return NNSP_B200_ERR_ARG; }
    std::vector<char> seen;
    for (int i = 0; i < n; i++) {                                     /* checked before anything is recorded */
        if (streams[i] < 0 || streams[i] >= c->S) {
            nnsp_set_error("cascade_import_streams: streams[%d] = %d is outside [0, %d)", i, (int)streams[i], c->S);
            return NNSP_B200_ERR_ARG;
        }
        if (seen.empty()) seen.assign((size_t)c->S, 0);
        if (seen[(size_t)streams[i]]++) { nnsp_set_error("cascade_import_streams: stream %d listed twice", (int)streams[i]); return NNSP_B200_ERR_ARG; }
    }
    int rc = nnsp_cascade_check_records(c, records, n);
    if (rc) return rc;
    for (int i = 0; i < n; i++) {
        const size_t s = (size_t)streams[i];
        if (c->rs_mode[s] < 0) c->rs_ids.push_back(streams[i]);
        c->rs_mode[s] = OP_LOAD;                                      /* whatever was pending before: the last import wins */
        if (c->ip_slot[s] < 0) {
            c->ip_slot[s] = (int)(c->ip_pool.size() / (size_t)c->rec_bytes);
            c->ip_pool.resize(c->ip_pool.size() + (size_t)c->rec_bytes);
        }
        memcpy(c->ip_pool.data() + (size_t)c->ip_slot[s] * c->rec_bytes, static_cast<const unsigned char *>(records) + (size_t)i * c->rec_bytes,
               (size_t)c->rec_bytes);
    }
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_export_streams(nnsp_b200_cascade *c, const int32_t *streams, int n, void *records)
{
    if (!c || n < 0 || (n > 0 && (!streams || !records))) { nnsp_set_error("cascade_export_streams: bad arguments (n = %d)", n); return NNSP_B200_ERR_ARG; }
    for (int i = 0; i < n; i++)
        if (streams[i] < 0 || streams[i] >= c->S) {
            nnsp_set_error("cascade_export_streams: streams[%d] = %d is outside [0, %d)", i, (int)streams[i], c->S);
            return NNSP_B200_ERR_ARG;
        }
    if (n == 0) return NNSP_B200_OK;
    int rc = nnsp_b200_cascade_sync(c);                               /* every call issued, host tickets included */
    if (rc) return rc;
    /* the device is idle: the pending resets and imports, both parts at once, on c->stream */
    const int *rl = nullptr;
    int rn = 0, rb = 0, loads = 0;
    if ((rc = cascade_take_resets(c, &rl, &rn, &rb, &loads))) return rc;
    if (rn) {
        NNSP_CUDA(cudaMemcpyAsync(c->rs_dev[0], rl, (size_t)rn * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        NNSP_CUDA(cudaEventRecord(c->rs_copied[rb][0], c->stream));
        c->rs_copy_valid[rb][0] = true;
        if (loads) NNSP_CUDA(cudaMemcpyAsync(c->rp_dev[rb], c->rp_host[rb], (size_t)loads * c->rec_bytes, cudaMemcpyHostToDevice, c->stream));
        if ((rc = cascade_launch_reset(c, c->rs_dev[0], rn, 0, RESET_HIST | RESET_STATE, c->stream, loads ? c->rp_dev[rb] : nullptr))) return rc;
        if (loads) { NNSP_CUDA(cudaEventRecord(c->rp_read[rb][0], c->stream)); c->rp_read_valid[rb][0] = true; }
    }
    if (n > c->ex_cap) {
        cudaFree(c->ex_ids); cudaFree(c->ex_dev);
        c->ex_ids = nullptr; c->ex_dev = nullptr; c->ex_cap = 0;
        NNSP_CUDA(cudaMalloc(&c->ex_ids, (size_t)n * sizeof(int)));
        NNSP_CUDA(cudaMalloc(&c->ex_dev, (size_t)n * c->rec_bytes));
        c->ex_cap = n;
    }
    NNSP_CUDA(cudaMemcpyAsync(c->ex_ids, streams, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    cascade_export_kernel<<<n, 128, 0, c->stream>>>(c->st, c->stale, c->ex_ids, c->ex_dev, cascade_hist_words(c), cascade_lm_words(c), c->hdr);
    NNSP_LAUNCH_CHECK();
    NNSP_CUDA(cudaMemcpyAsync(records, c->ex_dev, (size_t)n * c->rec_bytes, cudaMemcpyDeviceToHost, c->stream));
    NNSP_CUDA(cudaStreamSynchronize(c->stream));
    return NNSP_B200_OK;
}

static int cascade_check_pcm(const void *pcm, long long stride, int T)
{
    if (!pcm || T <= 0) { nnsp_set_error("null PCM pointer or n_frames <= 0"); return NNSP_B200_ERR_ARG; }
    if ((stride & 1) || ((uintptr_t)pcm & 3) || stride < (long long)T * NNSP_B200_FRAME) {
        nnsp_set_error("PCM must be 4-byte aligned with an even stream_stride >= n_frames*160");
        return NNSP_B200_ERR_ARG;
    }
    return NNSP_B200_OK;
}

/* nfr: per-stream frame counts on the device (ragged call), or null */
static int cascade_exec_dev(nnsp_b200_cascade *c, const int16_t *pcm_dev, long long stream_stride, int n_frames,
                            const int32_t *nfr, nnsp_b200_cascade_result *results_dev, const nnsp_b200_taps *taps)
{
    if (!c) return NNSP_B200_ERR_ARG;
    int rc = cascade_check_pcm(pcm_dev, stream_stride, n_frames);
    if (rc) return rc;
    NNSP_CUDA(cudaSetDevice(c->device));
    if (c->host_inflight) {                             /* asynchronous host-buffer calls still on the pipeline streams */
        for (auto s : c->xs) NNSP_CUDA(cudaStreamSynchronize(s));
        c->host_inflight = false;
    }
    if ((rc = cascade_ensure_logmel(c, n_frames))) return rc;
    if ((rc = cascade_ensure_split(c, n_frames))) return rc;
    const int *rl = nullptr;                            /* pending resets and imports: uploaded on c->stream behind the waits below */
    int rn = 0, rb = 0, loads = 0;
    PendingOps ops{};
    auto upload_resets = [&](int *dst, bool piped) -> int {
        NNSP_CUDA(cudaMemcpyAsync(dst, rl, (size_t)rn * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        NNSP_CUDA(cudaEventRecord(c->rs_copied[rb][0], c->stream));
        c->rs_copy_valid[rb][0] = true;
        ops.list = dst; ops.n = rn;
        if (loads) {
            NNSP_CUDA(cudaMemcpyAsync(c->rp_dev[rb], c->rp_host[rb], (size_t)loads * c->rec_bytes, cudaMemcpyHostToDevice, c->stream));
            ops.recs = c->rp_dev[rb];
            ops.read_hist = c->rp_read[rb][0]; c->rp_read_valid[rb][0] = true;
            if (piped) { ops.read_state = c->rp_read[rb][3]; c->rp_read_valid[rb][3] = true; }
        }
        return NNSP_B200_OK;
    };
    if ((rc = cascade_take_resets(c, &rl, &rn, &rb, &loads))) return rc;
    if (cascade_use_split(c, taps)) {
        const int i = (int)(c->pipe++ & 1u);
        if (c->nn_pending[i]) NNSP_CUDA(cudaStreamWaitEvent(c->stream, c->ev_nn[i], 0));   /* log-mel buffer i / the histories written next: in use two calls ago */
        if (rn && (rc = upload_resets(c->rs_dev[i], true))) return rc;    /* rs_dev[i] too: its last readers ran in that chain */
        rc = cascade_launch(c, pcm_dev, stream_stride, n_frames, 0, c->S, results_dev, nullptr, c->stream, true, 0,
                            i ? c->logmel2 : c->logmel, c->nn_stream, c->ev_feat[i], nfr, rn ? &ops : nullptr);
        if (rc) return rc;
        NNSP_CUDA(cudaEventRecord(c->ev_nn[i], c->nn_stream));
        c->nn_pending[i] = true;
    } else {
        if ((rc = cascade_join_nn(c, c->stream))) return rc;
        if (rn && (rc = upload_resets(c->rs_dev[0], false))) return rc;
        rc = cascade_launch(c, pcm_dev, stream_stride, n_frames, 0, c->S, results_dev, taps, c->stream, true, 0, nullptr, nullptr,
                            nullptr, nfr, rn ? &ops : nullptr);
        if (rc) return rc;
    }
    cascade_next_hist(c);
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_exec(nnsp_b200_cascade *c, const int16_t *pcm_dev, long long stream_stride, int n_frames,
                           nnsp_b200_cascade_result *results_dev, const nnsp_b200_taps *taps)
{
    return cascade_exec_dev(c, pcm_dev, stream_stride, n_frames, nullptr, results_dev, taps);
}

int nnsp_b200_cascade_exec_ragged(nnsp_b200_cascade *c, const int16_t *pcm_dev, long long stream_stride, int max_frames,
                                  const int32_t *n_frames_dev, nnsp_b200_cascade_result *results_dev, const nnsp_b200_taps *taps)
{
    if (!n_frames_dev) { nnsp_set_error("cascade_exec_ragged: null n_frames"); return NNSP_B200_ERR_ARG; }
    return cascade_exec_dev(c, pcm_dev, stream_stride, max_frames, n_frames_dev, results_dev, taps);
}

/* one host-buffer call queued on the pipeline streams (slice k always on stream k % 3: consecutive calls are ordered
 * slice by slice by stream order alone); nothing here waits for it */
static int cascade_enqueue_host(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride, int n_frames,
                                nnsp_b200_cascade_result *results, const int32_t *nfr = nullptr)
{
    int rc = cascade_check_pcm(pcm, stream_stride, n_frames);
    if (rc) return rc;
    NNSP_CUDA(cudaSetDevice(c->device));
    const int T = n_frames;
    if ((rc = cascade_ensure_logmel(c, T))) return rc;
    if ((rc = cascade_ensure_split(c, T))) return rc;
    if (T > c->d_pcm_frames) {
        NNSP_CUDA(cudaDeviceSynchronize());
        if (c->d_pcm) cudaFree(c->d_pcm);
        if (c->d_res) cudaFree(c->d_res);
        if (c->d_raw) cudaFree(c->d_raw);
        c->d_pcm = nullptr; c->d_res = nullptr; c->d_raw = nullptr;
        NNSP_CUDA(cudaMalloc(&c->d_pcm, (size_t)2 * c->S * T * NNSP_B200_FRAME * sizeof(int16_t)));
        for (auto &r : c->read_valid) for (auto &v : r) v = false;
        NNSP_CUDA(cudaMalloc(&c->d_res, (size_t)c->S * T * sizeof(nnsp_b200_cascade_result)));
        c->d_pcm_frames = T;
    }
    NNSP_CUDA(cudaStreamSynchronize(c->stream));
    NNSP_CUDA(cudaStreamSynchronize(c->nn_stream));
    c->nn_pending[0] = c->nn_pending[1] = false;
    /* every per-call scratch array is laid out [stream][T] (or by n_inf_max = (T + 1) / 2): a slice owns the same bytes in
     * consecutive calls only while T stays the same. When it changes with an asynchronous call still in flight, every
     * pipeline stream first waits for all streams of that call. */
    if (c->host_inflight && c->host_seq > 0 && c->host_last_T != T) {
        for (int j = 0; j < 3; j++)
            for (int k = 0; k < 3; k++) NNSP_CUDA(cudaStreamWaitEvent(c->xs[j], c->host_ev[c->host_seq % CS_HOST_RING][k], 0));
        /* ... and the copy stream: with another T the slices of the staged PCM are other byte ranges, the per-slice read
         * events of the earlier calls no longer say when they are free */
        for (int k = 0; k < 3; k++) NNSP_CUDA(cudaStreamWaitEvent(c->h2d_stream, c->host_ev[c->host_seq % CS_HOST_RING][k], 0));
    }
    c->host_last_T = T;
    const long long dstride = (long long)T * NNSP_B200_FRAME;
    if (c->host_fmt == NNSP_B200_HOST_AUDADC && !c->d_raw) {
        NNSP_CUDA(cudaDeviceSynchronize());
        NNSP_CUDA(cudaMalloc(&c->d_raw, (size_t)c->S * c->d_pcm_frames * NNSP_B200_FRAME * sizeof(uint32_t)));
    }
    if (nfr && !c->d_nfr) {
        NNSP_CUDA(cudaDeviceSynchronize());
        NNSP_CUDA(cudaMalloc(&c->d_nfr, (size_t)2 * c->S * sizeof(int32_t)));
    }
    const int *rl = nullptr;                                          /* pending resets and imports, sorted by stream */
    int rn = 0, rb = 0, loads = 0;
    if ((rc = cascade_take_resets(c, &rl, &rn, &rb, &loads))) return rc;
    c->host_inflight = true;
    const int nsl = c->S >= 4096 ? 8 : (c->S >= 256 ? 4 : 1);
    const int buf = (int)(c->host_calls++ & 1);
    int16_t *dpcm = c->d_pcm + (size_t)buf * c->S * c->d_pcm_frames * NNSP_B200_FRAME;
    int32_t *dnfr = nfr ? c->d_nfr + (size_t)buf * c->S : nullptr;     /* the counts of a ragged call, buffered like the PCM */
    auto slice = [&](int k, int *s0, int *s1) {
        *s0 = (int)(((long long)c->S * k / nsl) & ~15LL);
        *s1 = (k == nsl - 1) ? c->S : (int)(((long long)c->S * (k + 1) / nsl) & ~15LL);
    };
    if (c->host_fmt != NNSP_B200_HOST_AUDADC)
        for (int k = 0; k < nsl; k++) {                             /* all copies of the call, in slice order, on the copy stream */
            int s0, s1;
            slice(k, &s0, &s1);
            if (s1 <= s0) continue;
            if (c->read_valid[buf][k]) NNSP_CUDA(cudaStreamWaitEvent(c->h2d_stream, c->ev_read[buf][k], 0));   /* the call before last has read this buffer */
            if (stream_stride == dstride)
                NNSP_CUDA(cudaMemcpyAsync(dpcm + (size_t)s0 * dstride, pcm + (size_t)s0 * stream_stride,
                                          (size_t)(s1 - s0) * dstride * sizeof(int16_t), cudaMemcpyHostToDevice, c->h2d_stream));
            else
                NNSP_CUDA(cudaMemcpy2DAsync(dpcm + (size_t)s0 * dstride, dstride * sizeof(int16_t),
                                            pcm + (size_t)s0 * stream_stride, stream_stride * sizeof(int16_t),
                                            dstride * sizeof(int16_t), (size_t)(s1 - s0), cudaMemcpyHostToDevice, c->h2d_stream));
            if (dnfr)
                NNSP_CUDA(cudaMemcpyAsync(dnfr + s0, nfr + s0, (size_t)(s1 - s0) * sizeof(int32_t), cudaMemcpyHostToDevice, c->h2d_stream));
            NNSP_CUDA(cudaEventRecord(c->ev_h2d[buf][k], c->h2d_stream));
        }
    for (int k = 0; k < nsl; k++) {
        int s0, s1;
        slice(k, &s0, &s1);
        if (s1 <= s0) continue;
        cudaStream_t st = c->xs[k % 3];
        if (c->host_fmt == NNSP_B200_HOST_AUDADC) {                 /* the application's ingest (main_nnsp.cc:58-65) on the device */
            const uint32_t *raw = reinterpret_cast<const uint32_t *>(pcm);
            NNSP_CUDA(cudaMemcpy2DAsync(c->d_raw + (size_t)s0 * dstride, dstride * sizeof(uint32_t),
                                        raw + (size_t)s0 * stream_stride, stream_stride * sizeof(uint32_t),
                                        dstride * sizeof(uint32_t), (size_t)(s1 - s0), cudaMemcpyHostToDevice, st));
            if ((rc = launch_ingest(c->d_raw + (size_t)s0 * dstride, dpcm + (size_t)s0 * dstride, (long long)(s1 - s0) * T, c->device, st))) return rc;
            if (dnfr)
                NNSP_CUDA(cudaMemcpyAsync(dnfr + s0, nfr + s0, (size_t)(s1 - s0) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        } else
            NNSP_CUDA(cudaStreamWaitEvent(st, c->ev_h2d[buf][k], 0));
        /* the slice's own resets, at rs_dev[0] + s0: only this slice's kernels, all on st, ever use those entries; its
         * records, p0 .. p1 - 1 of the call's, at the same place in rp_dev[rb] */
        const int *taken = c->rs_taken.data();
        const int r0 = rn ? (int)(std::lower_bound(taken, taken + rn, s0) - taken) : 0;
        const int r1 = rn ? (int)(std::lower_bound(taken, taken + rn, s1) - taken) : 0;
        PendingOps ops{ c->rs_dev[0] + s0, r1 - r0, nullptr, nullptr, nullptr };
        if (r1 > r0) {
            NNSP_CUDA(cudaMemcpyAsync(c->rs_dev[0] + s0, rl + r0, (size_t)(r1 - r0) * sizeof(int), cudaMemcpyHostToDevice, st));
            NNSP_CUDA(cudaEventRecord(c->rs_copied[rb][k % 3], st));   /* re-recorded by later slices on st: the last copy */
            c->rs_copy_valid[rb][k % 3] = true;
            const int p0 = c->rs_taken_loads[(size_t)r0], p1 = c->rs_taken_loads[(size_t)r1];
            if (p1 > p0) {
                NNSP_CUDA(cudaMemcpyAsync(c->rp_dev[rb] + (size_t)p0 * c->rec_bytes, c->rp_host[rb] + (size_t)p0 * c->rec_bytes,
                                          (size_t)(p1 - p0) * c->rec_bytes, cudaMemcpyHostToDevice, st));
                ops.recs = c->rp_dev[rb];
                ops.read_hist = c->rp_read[rb][k % 3];
                c->rp_read_valid[rb][k % 3] = true;
            }
        }
        rc = cascade_launch(c, dpcm, dstride, T, s0, s1 - s0, results ? c->d_res : nullptr, nullptr, st, false, k,
                            nullptr, nullptr, nullptr, dnfr, r1 > r0 ? &ops : nullptr);
        if (rc) return rc;
        NNSP_CUDA(cudaEventRecord(c->ev_read[buf][k], st));         /* every reader of the slice's PCM has joined st by now */
        c->read_valid[buf][k] = true;
        if (results)
            NNSP_CUDA(cudaMemcpyAsync(results + (size_t)s0 * T, c->d_res + (size_t)s0 * T,
                                      (size_t)(s1 - s0) * T * sizeof(nnsp_b200_cascade_result), cudaMemcpyDeviceToHost, st));
    }
    cascade_next_hist(c);
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_exec_host(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride, int n_frames,
                                nnsp_b200_cascade_result *results)
{
    if (!c) return NNSP_B200_ERR_ARG;
    int rc = cascade_enqueue_host(c, pcm, stream_stride, n_frames, results);
    if (rc) return rc;
    for (auto s : c->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    c->host_inflight = false;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_exec_host_async(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride, int n_frames,
                                      nnsp_b200_cascade_result *results, long long *ticket)
{
    if (!c) return NNSP_B200_ERR_ARG;
    int rc = cascade_enqueue_host(c, pcm, stream_stride, n_frames, results);
    if (rc) return rc;
    const long long t = ++c->host_seq;
    for (int j = 0; j < 3; j++) NNSP_CUDA(cudaEventRecord(c->host_ev[t % CS_HOST_RING][j], c->xs[j]));
    if (ticket) *ticket = t;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_exec_host_ragged_async(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride, int max_frames,
                                             const int32_t *n_frames, nnsp_b200_cascade_result *results, long long *ticket)
{
    if (!c) return NNSP_B200_ERR_ARG;
    if (!n_frames) { nnsp_set_error("cascade_exec_host_ragged_async: null n_frames"); return NNSP_B200_ERR_ARG; }
    for (int s = 0; s < c->S; s++)                                   /* checked before anything is queued */
        if (n_frames[s] < 0 || n_frames[s] > max_frames) {
            nnsp_set_error("cascade_exec_host_ragged_async: n_frames[%d] = %d is outside [0, %d]", s, (int)n_frames[s], max_frames);
            return NNSP_B200_ERR_ARG;
        }
    int rc = cascade_enqueue_host(c, pcm, stream_stride, max_frames, results, n_frames);
    if (rc) return rc;
    const long long t = ++c->host_seq;
    for (int j = 0; j < 3; j++) NNSP_CUDA(cudaEventRecord(c->host_ev[t % CS_HOST_RING][j], c->xs[j]));
    if (ticket) *ticket = t;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_wait_host(nnsp_b200_cascade *c, long long ticket)
{
    if (!c || ticket <= 0 || ticket > c->host_seq) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(c->device));
    /* a reused slot holds the events of a later call on the same streams: waiting for those covers the older one */
    for (int j = 0; j < 3; j++) NNSP_CUDA(cudaEventSynchronize(c->host_ev[ticket % CS_HOST_RING][j]));
    if (ticket == c->host_seq) c->host_inflight = false;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_sync(nnsp_b200_cascade *c)
{
    if (!c) return NNSP_B200_ERR_ARG;
    NNSP_CUDA(cudaSetDevice(c->device));
    NNSP_CUDA(cudaStreamSynchronize(c->stream));
    NNSP_CUDA(cudaStreamSynchronize(c->nn_stream));
    NNSP_CUDA(cudaStreamSynchronize(c->h2d_stream));
    for (auto s : c->xs) NNSP_CUDA(cudaStreamSynchronize(s));
    c->host_inflight = false;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_last_kernel_ms(nnsp_b200_cascade *c, float ms[3])
{
    if (!c || !ms) return NNSP_B200_ERR_ARG;
    ms[0] = ms[1] = ms[2] = 0.f;
    if (!c->ev_valid) return NNSP_B200_OK;
    NNSP_CUDA(cudaSetDevice(c->device));
    cudaEvent_t *tl = c->tl[(c->tl_count - 1) % 8];
    NNSP_CUDA(cudaEventSynchronize(tl[3]));
    NNSP_CUDA(cudaEventElapsedTime(&ms[0], tl[0], tl[1]));
    NNSP_CUDA(cudaEventElapsedTime(&ms[1], c->last_piped ? tl[2] : tl[1], tl[3]));
    return NNSP_B200_OK;
}

/* When, on the device, the front end and the controller / network chain of the last calls ran: for each of the last
 * n <= 8 device-buffer calls (oldest first) ms[k][0..3] = front end starts / done, chain starts / done, in milliseconds
 * after the oldest call's front end started. Synchronises the handle. Shows how far consecutive calls overlap. */
int nnsp_b200_cascade_timeline(nnsp_b200_cascade *c, float *ms, int *n_calls)
{
    if (!c || !ms || !n_calls) return NNSP_B200_ERR_ARG;
    int rc = nnsp_b200_cascade_sync(c);
    if (rc) return rc;
    const int n = (int)(c->tl_count < 8 ? c->tl_count : 8);
    *n_calls = n;
    if (n == 0) return NNSP_B200_OK;
    const long long first = c->tl_count - n;
    for (int k = 0; k < n; k++)
        for (int j = 0; j < 4; j++)
            NNSP_CUDA(cudaEventElapsedTime(&ms[4 * k + j], c->tl[first % 8][0], c->tl[(first + k) % 8][j]));
    return NNSP_B200_OK;
}

void *nnsp_b200_cascade_stream(nnsp_b200_cascade *c) { return c ? (void *)c->stream : nullptr; }

int nnsp_b200_cascade_set_host_format(nnsp_b200_cascade *c, int fmt)
{
    if (!c || (fmt != NNSP_B200_HOST_PCM16 && fmt != NNSP_B200_HOST_AUDADC)) return NNSP_B200_ERR_ARG;
    int rc = nnsp_b200_cascade_sync(c);
    if (rc) return rc;
    c->host_fmt = fmt;
    return NNSP_B200_OK;
}

int nnsp_b200_cascade_set_path(nnsp_b200_cascade *c, int path)
{
    if (!c || path < 0 || path > 2) return NNSP_B200_ERR_ARG;
    if (path == 2 && !c->split_ok) { nnsp_set_error("a model of this cascade has no scan-split formulation"); return NNSP_B200_ERR_UNSUPPORTED; }
    c->path = path;
    return NNSP_B200_OK;
}

void nnsp_b200_cascade_destroy(nnsp_b200_cascade *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 3; i++) if (c->have[i]) free_model(&c->dm[i]);
    cudaFree(c->st.ctx); cudaFree(c->st.h); cudaFree(c->st.c); cudaFree(c->st.scal); cudaFree(c->st.casc);
    cudaFree(c->st.hist); cudaFree(c->st.lmhist); cudaFree(c->stale); cudaFree(c->thr); cudaFree(c->vseq);
    cudaFree(c->logmel); cudaFree(c->logmel2); cudaFree(c->hist2); cudaFree(c->hist3); cudaFree(c->lmhist2); cudaFree(c->lmhist3); cudaFree(c->d_pcm); cudaFree(c->d_res); cudaFree(c->d_raw); cudaFree(c->d_nfr);
    if (c->nn_stream) cudaStreamDestroy(c->nn_stream);
    for (auto e : c->ev_feat) if (e) cudaEventDestroy(e);
    for (auto e : c->ev_nn) if (e) cudaEventDestroy(e);
    for (int i = 0; i < 3; i++) free_model_mma(&c->mm[i]);
    cudaFree(c->replay_sorted); cudaFree(c->grp_list); cudaFree(c->ctl); cudaFree(c->fix_list); cudaFree(c->pend[0]); cudaFree(c->pend[1]);
    cudaFree(c->ra.t0); cudaFree(c->ra.tstart); cudaFree(c->ra.tb); cudaFree(c->ra.age0); cudaFree(c->ra.lmfix);
    cudaFree(c->planes[0]); cudaFree(c->planes[1]); cudaFree(c->dec);
    if (c->stream) cudaStreamDestroy(c->stream);
    for (auto s : c->xs) if (s) cudaStreamDestroy(s);
    for (auto &r : c->host_ev) for (auto e : r) if (e) cudaEventDestroy(e);
    if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
    for (auto &r : c->ev_h2d) for (auto e : r) if (e) cudaEventDestroy(e);
    for (auto &r : c->ev_read) for (auto e : r) if (e) cudaEventDestroy(e);
    for (auto &row : c->tl) for (auto e : row) if (e) cudaEventDestroy(e);
    for (auto &row : c->gs) for (auto g : row) if (g) cudaStreamDestroy(g);
    for (auto e : c->ev_fork) if (e) cudaEventDestroy(e);
    for (auto &row : c->ev_join) for (auto e : row) if (e) cudaEventDestroy(e);
    for (int b = 0; b < 2; b++) {
        if (c->rs_host[b]) cudaFreeHost(c->rs_host[b]);
        cudaFree(c->rs_dev[b]);
        for (auto e : c->rs_copied[b]) if (e) cudaEventDestroy(e);
        if (c->rp_host[b]) cudaFreeHost(c->rp_host[b]);
        cudaFree(c->rp_dev[b]);
        for (auto e : c->rp_read[b]) if (e) cudaEventDestroy(e);
    }
    cudaFree(c->ex_ids); cudaFree(c->ex_dev);
    delete c;
}

}  /* extern "C" */
