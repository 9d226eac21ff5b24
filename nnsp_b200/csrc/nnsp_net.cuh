/* nnsp_net.cuh -- NeuralNetClass_exe + NNSPClass post-processing for one stream, by one warp.
 *
 * Reference path: NeuralNetClass_exe (neural_nets.c:44-168) -> fc_8x16 (affine.c:409-490) /
 * lstm_8x16 (lstm.c:15-214) -> affine_Krows_8x16 ARM variant (affine.c:12-259) and
 * rc_Krows_8x16 (affine.c:348-407), or their _acc32b twins (affine_acc32b.c, lstm.c:216-415)
 * -> activation.c; then s2i_post_proc / binary_post_proc (nn_speech.c:146-227).
 *
 * Mapping: the whole weight image of the model sits in shared memory (staged once per CTA by
 * a TMA bulk copy), K-major, one 32-bit word = four consecutive-K int8 weights of one row.
 * Lane l accumulates rows l, l+32, ... with dp2a (two int16 x int8 MACs per instruction,
 * int32 accumulator). For 64-bit-accumulator models the int32 dot product is exact because
 * cols <= 480 bounds |sum| by 480 * 128 * 32768 < 2^31; everything after the dot product
 * (Q-format alignment, bias, output shift, saturation) is done in 64 bits like the reference.
 * For ACC32BIT_OPT models the same dot product wraps modulo 2^32, which is what __SMLAD does. */
#pragma once
#include "nnsp_device.cuh"
#include "nnsp_engine.cuh"

namespace nnsp {

/* One stream's working set in shared memory. W = widest layer / LSTM state it can hold, NOUT = widest final layer;
 * the functions below take any instantiation (the cascade uses a narrow one to fit twice the warps per CTA). */
template <int W, int NOUT>
struct WarpScratchT {
    static constexpr int WIDTH = W;
    alignas(16) int16_t ctx[240];      /* normFeatContext, 6 rows x 40 (feature_module.h:12)      */
    alignas(16) int16_t buf[2][W];     /* ping-pong layer I/O (neural_nets.c:9-10)                */
    alignas(16) int16_t h[W];
    int32_t c[W];
    int16_t gates[4 * W];
    int32_t logits[NOUT];
    int16_t scal[SC_N];
};
using WarpScratch = WarpScratchT<NNSP_B200_MAX_WIDTH, NNSP_B200_MAX_OUT>;

/* acc[i] += W[row r0 + 32 i] . x for NR rows per lane; x is int16, 8-byte aligned */
template <int NR>
__device__ __forceinline__ void dot_rows(const uint32_t *__restrict__ W, int nrows_pad, int k4n,
                                         const int16_t *__restrict__ x, int r0, int32_t (&acc)[4])
{
    const uint2 *x2 = reinterpret_cast<const uint2 *>(x);
    const uint32_t *w = W + r0;
#pragma unroll 4
    for (int k = 0; k < k4n; k++) {
        const uint2 xx = x2[k];
#pragma unroll
        for (int i = 0; i < NR; i++) {
            const int wv = (int)w[32 * i];
            acc[i] = __dp2a_lo((int)xx.x, wv, acc[i]);
            acc[i] = __dp2a_hi((int)xx.y, wv, acc[i]);
        }
        w += nrows_pad;
    }
}

__device__ __forceinline__ void dot_rows_n(int nr, const uint32_t *W, int nrows_pad, int k4n,
                                           const int16_t *x, int r0, int32_t (&acc)[4])
{
    switch (nr) {
    case 4: dot_rows<4>(W, nrows_pad, k4n, x, r0, acc); break;
    case 3: dot_rows<3>(W, nrows_pad, k4n, x, r0, acc); break;
    case 2: dot_rows<2>(W, nrows_pad, k4n, x, r0, acc); break;
    default: dot_rows<1>(W, nrows_pad, k4n, x, r0, acc); break;
    }
}

/* accumulator -> 32-bit pre-activation: bias alignment + add (affine.c:190-217), output shift
 * and saturation (affine.c:242-249); acc32: wrapping adds, no saturation (affine_acc32b.c:249).
 * Quirk Q1: the accumulator is NOT re-aligned to the bias Q-format (affine.c:186-187 is dead). */
template <class LT>
__device__ __forceinline__ int32_t finish_fc(const LT &L, int32_t acc, int32_t bias)
{
    if (L.acc32) {
        const uint32_t b = (L.sh_bias >= 0) ? ((uint32_t)bias << L.sh_bias) : (uint32_t)(bias >> (-L.sh_bias));
        return shift32_dev((int32_t)((uint32_t)acc + b), L.sh_out);
    }
    int64_t a = (int64_t)acc;
    a += (L.sh_bias >= 0) ? (int64_t)((uint64_t)(int64_t)bias << L.sh_bias) : ((int64_t)bias >> (-L.sh_bias));
    return sat32_dev(shift64_dev(a, L.sh_out));
}
/* rc_Krows_8x16: input half, rescale by qbit_input_rec - qbit_input (affine.c:371,384), recurrent half */
template <class LT>
__device__ __forceinline__ int32_t finish_gate(const LT &L, int32_t acc_x, int32_t acc_h, int32_t bias)
{
    if (L.acc32) {
        const uint32_t a = (uint32_t)shift32_dev(acc_x, L.sh_x) + (uint32_t)acc_h;
        const uint32_t b = (L.sh_bias >= 0) ? ((uint32_t)bias << L.sh_bias) : (uint32_t)(bias >> (-L.sh_bias));
        return shift32_dev((int32_t)(a + b), L.sh_out);
    }
    int64_t a = shift64_dev((int64_t)acc_x, L.sh_x) + (int64_t)acc_h;
    a += (L.sh_bias >= 0) ? (int64_t)((uint64_t)(int64_t)bias << L.sh_bias) : ((int64_t)bias >> (-L.sh_bias));
    return sat32_dev(shift64_dev(a, L.sh_out));
}

__device__ __forceinline__ int32_t activate16(int act, int32_t pre, const int16_t *lut)
{
    switch (act) {
    case ACT_TANH: return tanh_q15(pre, lut);
    case ACT_SIGMOID: return sigmoid_q15(pre, lut);
    default: return relu6_q12(pre);
    }
}

/* dot_rows reads the old h of an LSTM as 8-byte words from ws->h + ho. A second LSTM behind a first one whose width is
 * not a multiple of 4 starts at an offset that is not, and its rounded-up last word may reach past ws->h. Such a layer
 * reads a copy instead: its old h in `row` (the layer's output buffer, which the cell loop writes only after every gate
 * product), zero-padded to the k4rec words read. A caller syncs the threads that share `row` before reading it. */
__device__ __forceinline__ void stage_h_row(int16_t *row, const int16_t *h, int rows, int k4rec, int t, int nt)
{
    for (int k = t; k < 4 * k4rec; k += nt) row[k] = (k < rows) ? h[k] : (int16_t)0;
}

/* One network evaluation for the warp's stream. ws->ctx is the input; LSTM state in ws->h/c.
 * tap_act / tap_logits (global, may be null) receive the layer outputs of this frame. */
template <class WS>
__device__ __forceinline__ void net_forward(const DevModel &M, const uint32_t *__restrict__ wimg,
                                            const int16_t *__restrict__ bimg,
                                            const int16_t *__restrict__ tanh_lut, WS *ws,
                                            int lane, int16_t *tap_act, int32_t *tap_logits)
{
    const int16_t *x = ws->ctx;
    int pp = 0, ho = 0, ao = 0;
    for (int li = 0; li < M.numlayers; li++) {
        const DevLayer &L = M.layer[li];
        int16_t *y = ws->buf[pp];
        const uint32_t *W = wimg + L.w_off;
        const int16_t *B = bimg + L.bias_off;
        const bool last = (li == M.numlayers - 1);
        const int rounds = L.nrows_pad >> 5;
        if (L.type == LAYER_LSTM) {
            const uint32_t *Wr = wimg + L.wrec_off;
            const int16_t *hh = ws->h + ho;
            if (ho & 3) { stage_h_row(y, hh, L.rows, L.k4rec, lane, 32); __syncwarp(); hh = y; }
            for (int r = 0; r < rounds; r += 4) {
                const int nr = min(4, rounds - r), r0 = r * 32 + lane;
                int32_t ax[4] = { 0, 0, 0, 0 }, ah[4] = { 0, 0, 0, 0 };
                dot_rows_n(nr, W, L.nrows_pad, L.k4, x, r0, ax);
                dot_rows_n(nr, Wr, L.nrows_pad, L.k4rec, hh, r0, ah);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int n = r0 + 32 * i;
                    if (i < nr && n < L.nrows) {
                        const int32_t pre = finish_gate(L, ax[i], ah[i], B[n]);
                        const int g = (n >= L.rows) + (n >= 2 * L.rows) + (n >= 3 * L.rows);
                        ws->gates[n] = (int16_t)((g == 1) ? tanh_q15(pre, tanh_lut) : sigmoid_q15(pre, tanh_lut));   /* lstm.c:65,78,91,104 */
                    }
                }
            }
            __syncwarp();
            const int H = L.rows;
            for (int u = lane; u < H; u += 32) {
                const int32_t gi = ws->gates[u], gj = ws->gates[H + u], gf = ws->gates[2 * H + u], go = ws->gates[3 * H + u];
                const int64_t t = ((int64_t)gi * (int64_t)gj + (int64_t)gf * (int64_t)ws->c[ho + u]) >> 15;   /* lstm.c:108-109 */
                const int32_t cn = sat32_dev(t);
                ws->c[ho + u] = cn;
                int32_t o = (tanh_q15(cn, tanh_lut) * go) >> 15;                                              /* lstm.c:111-115 */
                o = o > 32767 ? 32767 : (o < -32768 ? -32768 : o);
                y[u] = (int16_t)o;
                ws->h[ho + u] = (int16_t)o;                                                                   /* lstm.c:205-206 (all gates already used the old h) */
            }
            ho += H;
        } else {
            for (int r = 0; r < rounds; r += 4) {
                const int nr = min(4, rounds - r), r0 = r * 32 + lane;
                int32_t ax[4] = { 0, 0, 0, 0 };
                dot_rows_n(nr, W, L.nrows_pad, L.k4, x, r0, ax);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int n = r0 + 32 * i;
                    if (i < nr && n < L.nrows) {
                        const int32_t pre = finish_fc(L, ax[i], B[n]);
                        if (L.act == ACT_LINEAR) ws->logits[n] = pre;          /* linear_fix keeps int32 (activation.c:19-29) */
                        else y[n] = (int16_t)activate16(L.act, pre, tanh_lut);
                    }
                }
            }
        }
        __syncwarp();
        if (!last) {
            if (tap_act) for (int n = lane; n < L.rows; n += 32) tap_act[ao + n] = y[n];
            ao += L.rows;
        } else {
            const bool is32 = (L.type == LAYER_FC && L.act == ACT_LINEAR);     /* neural_nets.c:152-167 */
            if (!is32) { for (int n = lane; n < L.rows; n += 32) ws->logits[n] = y[n]; __syncwarp(); }
            if (tap_logits) for (int n = lane; n < L.rows; n += 32) tap_logits[n] = ws->logits[n];
        }
        x = y;
        pp ^= 1;
    }
}

/* net_forward by a group of GW warps that share one stream: the 32-row rounds of every layer are dealt
 * out to the warps in contiguous runs, the LSTM cell and the copies go over all threads of the group, and a named barrier
 * (`bar_id`, 32 GW threads) separates the phases. Same arithmetic, same order per row: bit-exact with net_forward. A stream
 * that one warp walks frame by frame is latency-bound; this shortens the chain per inference about threefold. */
template <int GW>
__device__ __forceinline__ void group_sync(int bar_id) { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(32 * GW) : "memory"); }

template <int GW, class WS>
__device__ __forceinline__ void net_forward_group(const DevModel &M, const uint32_t *__restrict__ wimg,
                                                  const int16_t *__restrict__ bimg, const int16_t *__restrict__ tanh_lut,
                                                  WS *ws, int wg, int lane, int bar_id)
{
    const int gt = wg * 32 + lane;
    const int16_t *x = ws->ctx;
    int pp = 0, ho = 0;
    for (int li = 0; li < M.numlayers; li++) {
        const DevLayer &L = M.layer[li];
        int16_t *y = ws->buf[pp];
        const uint32_t *W = wimg + L.w_off;
        const int16_t *B = bimg + L.bias_off;
        const bool last = (li == M.numlayers - 1);
        const int rounds = L.nrows_pad >> 5;
        const int per = (rounds + GW - 1) / GW, rs = wg * per, re = min(rounds, rs + per);      /* this warp's run of rounds */
        if (L.type == LAYER_LSTM) {
            const uint32_t *Wr = wimg + L.wrec_off;
            const int16_t *hh = ws->h + ho;
            if (ho & 3) { stage_h_row(y, hh, L.rows, L.k4rec, gt, 32 * GW); group_sync<GW>(bar_id); hh = y; }
            for (int r = rs; r < re; r += 4) {
                const int nr = min(4, re - r), r0 = r * 32 + lane;
                int32_t ax[4] = { 0, 0, 0, 0 }, ah[4] = { 0, 0, 0, 0 };
                dot_rows_n(nr, W, L.nrows_pad, L.k4, x, r0, ax);
                dot_rows_n(nr, Wr, L.nrows_pad, L.k4rec, hh, r0, ah);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int n = r0 + 32 * i;
                    if (i < nr && n < L.nrows) {
                        const int32_t pre = finish_gate(L, ax[i], ah[i], B[n]);
                        const int g = (n >= L.rows) + (n >= 2 * L.rows) + (n >= 3 * L.rows);
                        ws->gates[n] = (int16_t)((g == 1) ? tanh_q15(pre, tanh_lut) : sigmoid_q15(pre, tanh_lut));   /* lstm.c:65,78,91,104 */
                    }
                }
            }
            group_sync<GW>(bar_id);                                        /* every gate of the layer is in place; all read the old h */
            const int H = L.rows;
            for (int u = gt; u < H; u += 32 * GW) {
                const int32_t gi = ws->gates[u], gj = ws->gates[H + u], gf = ws->gates[2 * H + u], go = ws->gates[3 * H + u];
                const int64_t t = ((int64_t)gi * (int64_t)gj + (int64_t)gf * (int64_t)ws->c[ho + u]) >> 15;   /* lstm.c:108-109 */
                const int32_t cn = sat32_dev(t);
                ws->c[ho + u] = cn;
                int32_t o = (tanh_q15(cn, tanh_lut) * go) >> 15;                                              /* lstm.c:111-115 */
                o = o > 32767 ? 32767 : (o < -32768 ? -32768 : o);
                y[u] = (int16_t)o;
                ws->h[ho + u] = (int16_t)o;
            }
            ho += H;
        } else {
            for (int r = rs; r < re; r += 4) {
                const int nr = min(4, re - r), r0 = r * 32 + lane;
                int32_t ax[4] = { 0, 0, 0, 0 };
                dot_rows_n(nr, W, L.nrows_pad, L.k4, x, r0, ax);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int n = r0 + 32 * i;
                    if (i < nr && n < L.nrows) {
                        const int32_t pre = finish_fc(L, ax[i], B[n]);
                        if (L.act == ACT_LINEAR) ws->logits[n] = pre;          /* linear_fix keeps int32 (activation.c:19-29) */
                        else y[n] = (int16_t)activate16(L.act, pre, tanh_lut);
                    }
                }
            }
        }
        group_sync<GW>(bar_id);
        if (last && !(L.type == LAYER_FC && L.act == ACT_LINEAR)) {    /* neural_nets.c:152-167 */
            for (int n = gt; n < L.rows; n += 32 * GW) ws->logits[n] = y[n];
            group_sync<GW>(bar_id);
        }
        x = y;
        pp ^= 1;
    }
}

/* s2i_post_proc, nn_speech.c:146-189 (run by one lane; sc = NNSPClass scalars) */
__device__ __forceinline__ void post_s2i(int16_t *sc, const int32_t *est, int16_t th_count)
{
    sc[SC_TRIGGER] = 0;
    sc[SC_OUT0] = sc[SC_OUT0 + 1] = sc[SC_OUT0 + 2] = 0;
    const int ai = argmax_last_wins(est, 7);
    const int last = sc[SC_ARGMAX_LAST];
    if (last == 0 || last == ai) {
        if (ai != 0) {
            const int16_t cnt = (int16_t)(sc[SC_CNT0 + ai] + 1);
            sc[SC_CNT0 + ai] = cnt;
            if (cnt > th_count) {
                sc[SC_TRIGGER] = 1;
                sc[SC_OUT0] = (int16_t)ai;
                sc[SC_OUT0 + 1] = (int16_t)argmax_last_wins(est + 7, 17);
                sc[SC_OUT0 + 2] = (int16_t)argmax_last_wins(est + 24, 17);
            }
        }
    } else {
        for (int i = 0; i < 7; i++) sc[SC_CNT0 + i] = 0;
    }
    sc[SC_ARGMAX_LAST] = (int16_t)ai;
}

/* binary_post_proc, nn_speech.c:191-227 */
__device__ __forceinline__ void post_binary(int16_t *sc, const int32_t *logits, int16_t thresh_prob, int16_t th_count)
{
    const int32_t l0 = logits[0], l1 = logits[1];
    const int32_t mx = l0 > l1 ? l0 : l1;
    int32_t est[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int32_t val = (int32_t)((uint32_t)(i ? l1 : l0) - (uint32_t)mx);
        int64_t ref = ((int64_t)val * 0xB8AA) >> 15;
        est[i] = pwr2_q15(sat32_dev(ref));
    }
    const int32_t den = (int32_t)((uint32_t)est[0] + (uint32_t)est[1]);
    const int32_t thresh = 32768 - (int32_t)thresh_prob;
    const int32_t tmp = (int32_t)(((int64_t)thresh * (int64_t)den) >> 15);
    const int16_t cnt = (est[0] <= tmp) ? (int16_t)(sc[SC_CNT0] + 1) : (int16_t)0;
    sc[SC_CNT0] = cnt;
    sc[SC_TRIGGER] = (cnt >= th_count) ? 1 : 0;
}

/* NNSPClass_reset for the warp's scratch copy of a stream (nn_speech.c:57-72) */
template <class WS>
__device__ __forceinline__ void reset_stream_scratch(const DevModel &M, WS *ws, int lane)
{
    for (int i = lane; i < 200; i += 32) ws->ctx[i] = M.silence[i % 40];     /* feature_module.c:32-43: rows 0..4 only, row 5 stays */
    for (int i = lane; i < WS::WIDTH; i += 32) { ws->h[i] = 0; ws->c[i] = 0; }   /* neural_nets.c:27-42 */
    if (lane < SC_N) {
        /* counts_category[7] survives a reset in the reference (nn_speech.c:64-65 clears 7 of 8);
         * nothing ever writes it, so it is always 0 */
        ws->scal[lane] = (lane == SC_SLIDES) ? 1 : 0;
    }
}

}  // namespace nnsp
