/* nnsp_device.cuh -- device-side arithmetic shared by the nnsp-b200 kernels (sm_100a).
 * Every helper states the reference lines whose integer semantics it reproduces bit for bit. */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nnsp {

enum { LAYER_FC = 0, LAYER_LSTM = 1 };
enum { ACT_RELU6 = 0, ACT_TANH = 1, ACT_SIGMOID = 2, ACT_LINEAR = 3 };

/* Frames stream s advances in a call of T frames. nfr: the per-stream counts of a ragged cascade call
 * (nnsp_b200_cascade_exec_ragged), clamped to [0, T]; null for every other call, which advances every stream by T. */
__device__ __forceinline__ int stream_frames(const int32_t *nfr, long long s, int T)
{
    if (!nfr) return T;
    const int n = __ldg(nfr + s);
    return n < 0 ? 0 : (n > T ? T : n);
}

/* ---- Q15 products ------------------------------------------------------------------- */
/* (a*b) >> 15 with a 64-bit intermediate and floor: the ">>= 15" of complex.c:66-69. The
 * int32 saturation that follows in the reference cannot fire for int16 PCM input: with the
 * shipped window sum|fft_in| <= 8 175 452, so every FFT intermediate stays below 2^24
 * (DESIGN.md "Why the FFT clamps are elided"; tests/test_tables_and_format.py::test_window_bound_behind_the_elided_fft_clamps). */
__device__ __forceinline__ int32_t mul_q15(int32_t a, int32_t b)
{
    return (int32_t)(((int64_t)a * (int64_t)b) >> 15);
}
/* (ar*wr - ai*wi) >> 15 */
__device__ __forceinline__ int32_t msub_q15(int32_t ar, int32_t wr, int32_t ai, int32_t wi)
{
    return (int32_t)(((int64_t)ar * (int64_t)wr - (int64_t)ai * (int64_t)wi) >> 15);
}
__device__ __forceinline__ int32_t madd_q15(int32_t ar, int32_t wi, int32_t ai, int32_t wr)
{
    return (int32_t)(((int64_t)ar * (int64_t)wi + (int64_t)ai * (int64_t)wr) >> 15);
}
/* Three-input adds. The FMA-heavy pipe (IMAD at 2, IMAD.WIDE at 4 cycles per warp) is the busiest one in the front
 * end (ncu: sm__pipe_fmaheavy_cycles_active 71 %, ALU 51 %). A private-temporary add pair is fused by ptxas into ONE
 * IADD3 on the ALU pipe: fewer instructions, on the pipe that has room. (Forcing the remaining two-input adds onto the
 * ALU pipe with a run-time-zero third operand was measured and is slower: 0.508 vs 0.482 ms.) */
__device__ __forceinline__ int32_t add3(int32_t a, int32_t b, int32_t c)        /* a + b + c */
{
    int32_t r;
    asm("{\n\t.reg .s32 t;\n\tadd.s32 t, %1, %2;\n\tadd.s32 %0, t, %3;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ int32_t add2sub(int32_t a, int32_t b, int32_t c)     /* a + b - c */
{
    int32_t r;
    asm("{\n\t.reg .s32 t;\n\tadd.s32 t, %1, %2;\n\tsub.s32 %0, t, %3;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ int32_t sub2add(int32_t a, int32_t b, int32_t c)     /* a - b + c */
{
    int32_t r;
    asm("{\n\t.reg .s32 t;\n\tsub.s32 t, %1, %2;\n\tadd.s32 %0, t, %3;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ int32_t sub3(int32_t a, int32_t b, int32_t c)        /* a - b - c */
{
    int32_t r;
    asm("{\n\t.reg .s32 t;\n\tsub.s32 t, %1, %2;\n\tsub.s32 %0, t, %3;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

/* a * 0x7fff >> 15 == a + floor(-a / 2^15): the reference's Q15 "1.0" (twiddle_fft_dif.c:9) */
__device__ __forceinline__ int32_t mul_one_q15(int32_t a) { return a + ((-a) >> 15); }

__device__ __forceinline__ int32_t sat32_dev(int64_t v)
{
    v = v > 0x7fffffffLL ? 0x7fffffffLL : v;
    v = v < -0x80000000LL ? -0x80000000LL : v;
    return (int32_t)v;
}

/* ---- activations (activation.c) ------------------------------------------------------ */
/* tanh_fix, activation.c:31-69; lut = coeffs_tanh. x == INT32_MIN is undefined in the
 * reference (LUT index out of bounds); defined here as -0x7fff, same as the oracle. */
__device__ __forceinline__ int32_t tanh_q15(int32_t x, const int16_t *__restrict__ lut)
{
    const bool neg = x < 0;
    const int32_t xi = neg ? (int32_t)(0u - (uint32_t)x) : x;
    int32_t y;
    if (xi < 0 || xi >= (5 << 15)) y = 0x7fff;
    else {
        int32_t kx = (xi - 512) >> 10;
        kx = kx < 0 ? 0 : kx;
        const int32_t dx = xi - 512 - (kx << 10);
        const int32_t v = (int32_t)lut[kx << 1] + ((dx * (int32_t)lut[(kx << 1) + 1]) >> 15);
        y = v > 0 ? v : 0;
    }
    return neg ? -y : y;          /* fits int16 */
}
/* sigmoid_fix, activation.c:72-86 */
__device__ __forceinline__ int32_t sigmoid_q15(int32_t x, const int16_t *__restrict__ lut)
{
    return (tanh_q15(x >> 1, lut) >> 1) + 16384;
}
/* relu6_fix, activation.c:6-17 (Q15 in, Q12 out) */
__device__ __forceinline__ int32_t relu6_q12(int32_t x)
{
    int32_t v = x >> 3;
    v = v > (6 << 12) ? (6 << 12) : v;
    return v < 0 ? 0 : v;
}

/* ---- accumulator shifts (affine.c:565-591, affine_acc32b.c:566-592) ------------------- */
__device__ __forceinline__ int64_t shift64_dev(int64_t x, int sh)
{
    if (sh == 0) return x;
    if (sh < 0) return x >> (-sh);
    int64_t M = (int64_t)1 << (63 - sh);
    const int64_t m = -M;
    M -= 1;
    x = x < m ? m : (x > M ? M : x);
    return (int64_t)((uint64_t)x << sh);
}
__device__ __forceinline__ int32_t shift32_dev(int32_t x, int sh)
{
    if (sh == 0) return x;
    if (sh < 0) return x >> (-sh);
    int32_t M = (int32_t)(1u << (31 - sh));
    const int32_t m = (int32_t)(0u - (uint32_t)M);
    M -= 1;
    x = x < m ? m : (x > M ? M : x);
    return (int32_t)((uint32_t)x << sh);
}

/* ---- fixed-point log10 (fixlog10.c:9-61 with bit_frac_in = 15) ------------------------ */
__device__ __forceinline__ int32_t log10_q15(int32_t x, const int16_t *__restrict__ lut)
{
    x = (x == 0) ? 1 : x;
    /* norm_oneTwo scans bits 30..0: the MSB of a positive value; a negative x (impossible
     * here, mel energies are >= 0) would behave differently in the reference */
    const int msb = 31 - __clz(x & 0x7fffffff);
    const int sh = 15 - msb;                        /* y = x * 2^sh in [1,2) Q15 */
    const int32_t y = (sh >= 0) ? (int32_t)((uint32_t)x << sh) : (x >> (-sh));
    const int32_t kx = (y - 32768) >> 8, dx = (y - 32768) - (kx << 8);
    int32_t t = (int32_t)lut[kx << 1] + (((int32_t)lut[1 + (kx << 1)] * dx) >> 15);
    t = (int32_t)(((int64_t)t * 0x3796) >> 15);
    return t + 0x2688 * (-sh);
}

/* ---- post-processing (nn_speech.c) ---------------------------------------------------- */
/* ceiling + compute_pwr2, nn_speech.c:229-258 */
__device__ __forceinline__ int32_t pwr2_q15(int32_t in)
{
    int32_t ce = (int32_t)((uint32_t)(in >> 15) << 15);
    if (ce != in) ce = (int32_t)((uint32_t)ce + 32768u);
    in = (int32_t)((uint32_t)in - (uint32_t)ce);
    const int32_t shift = ce >> 15;
    if (shift <= -15) return 0;
    const int32_t t = (int32_t)(((uint32_t)in << 1) + 32768u);
    int32_t o = 0x1fd7 + ((int32_t)((uint32_t)t * 0x057au) >> 15);
    o = 0x5a82 + ((int32_t)((uint32_t)t * (uint32_t)o) >> 15);
    return (shift < 0) ? (o >> (-shift)) : (int32_t)((uint32_t)o << shift);
}
/* my_argmax, nn_speech.c:130-144: ">=" so ties resolve to the LAST index */
__device__ __forceinline__ int argmax_last_wins(const int32_t *v, int n)
{
    int im = 0;
    int32_t mx = v[0];
    for (int i = 1; i < n; i++)
        if (v[i] >= mx) { mx = v[i]; im = i; }
    return im;
}

/* (x - mean) * stdR >> (30 - q), int16 saturation: feature_module.c:34-37, 69-72 */
__device__ __forceinline__ int16_t standardise(int32_t v, int32_t mean, int32_t stdR, int rshift)
{
    int64_t t = ((int64_t)v - (int64_t)mean) * (int64_t)stdR;
    t >>= rshift;
    t = t > 32767 ? 32767 : (t < -32768 ? -32768 : t);
    return (int16_t)t;
}

}  // namespace nnsp
