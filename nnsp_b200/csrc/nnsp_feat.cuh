/* nnsp_feat.cuh -- the FeatureClass front end for one frame, computed by one half-warp.
 *
 * Reference path (per frame, per stream): FeatureClass_execute (feature_module.c:47-75) ->
 * stftModule_analyze (spectrogram_module.c:47-77) -> rfft/fft (fft.c:27-221, complex.c:14-72)
 * -> spec2pspec (spectrogram_module.c:33-45) -> melSpecProc (melSpecProc.c:6-27) ->
 * log10_vec (fixlog10.c:53-61).
 *
 * Mapping: 16 lanes own the 256 complex points of the packed real FFT, 16 points each, in
 * registers. Radix-4 DIF stages 0 and 1 touch points {L + 16a}; one padded 16x16 transpose
 * through shared memory; stages 2 and 3 touch points {16L + b}. The bit-reversed result is
 * scattered to shared memory, each lane then forms the real-FFT bins i and 256-i from the
 * pair (Z[i], Z[256-i]), squares them into the power spectrum, and finally 40 mel bands and
 * their log10 are produced (up to three bands per lane).
 * All arithmetic is integer and identical to the reference's; see nnsp_device.cuh for why the
 * reference's int32 clamps inside the FFT are unreachable and therefore not emitted. */
#pragma once
#include "nnsp_device.cuh"
#include "nnsp_engine.cuh"

namespace nnsp {

struct FeatSmemTables {            /* = the leading members of DevTables, same order */
    int4     mel_tap4[MEL_GROUPS];
    int2     win2[240];
    int2     tw0[4][3][16];
    int2     tw1[3][16];
    int2     tw2[4][3];
    int2     rtw[257];
    uint32_t mel_meta[40];
    int16_t  log_lut[256];
};

struct alignas(16) FrameScratch {  /* per half-warp */
    int2    x[272];                /* 256 complex points, one pad slot per 16; later the power spectrum
                                      (int32 bins 0..256 over the first 1040 bytes, read in groups of 4 bins) */
};

struct FeatDump {                  /* optional stage taps (global memory), all may be null */
    int32_t *fft_in, *spec, *pspec, *mel;
};

__device__ __forceinline__ void load_feat_tables(FeatSmemTables *dst, const DevTables *__restrict__ src,
                                                 int tid, int nthreads)
{
    /* DevTables starts with the same members in the same order: copy the common prefix word by word */
    const int *s = reinterpret_cast<const int *>(src);
    int *d = reinterpret_cast<int *>(dst);
    for (int i = tid; i < (int)(sizeof(FeatSmemTables) / 4); i += nthreads) d[i] = s[i];
}

#define NNSP_TW_RE(w) ((int32_t)(int16_t)((w) & 0xffff))
#define NNSP_TW_IM(w) ((int32_t)(w) >> 16)

/* radix-4 DIF butterfly on register slots A,C,B,D = x[i0], x[i0+q], x[i0+2q], x[i0+3q]
 * (fft.c:171-193 with M4_ of fft.c:12-15 written out), outputs times tw[0..3] (complex.c:54-72).
 * W0 is always the Q15 "one"; ALLONE marks the last stage where every twiddle is. */
template <bool ALLONE>
__device__ __forceinline__ void bfly4(int32_t &ar, int32_t &ai, int32_t &cr, int32_t &ci,
                                      int32_t &br, int32_t &bi, int32_t &dr, int32_t &di,
                                      int2 w1, int2 w2, int2 w3)
{
    /* 12 three-input adds instead of 16 two-input ones (wrapping int32 adds: any association gives the same bits) */
    const int32_t s1r = cr + dr, s1i = ci + di, d1r = cr - dr, d1i = ci - di;
    const int32_t o0r = add3(ar, br, s1r), o0i = add3(ai, bi, s1i);
    const int32_t o1r = add2sub(ar, br, s1r), o1i = add2sub(ai, bi, s1i);
    const int32_t o2r = sub2add(ar, br, d1i), o2i = sub3(ai, bi, d1r);
    const int32_t o3r = sub3(ar, br, d1i), o3i = sub2add(ai, bi, d1r);
    ar = mul_one_q15(o0r);
    ai = mul_one_q15(o0i);
    if (ALLONE) {
        cr = mul_one_q15(o1r); ci = mul_one_q15(o1i);
        br = mul_one_q15(o2r); bi = mul_one_q15(o2i);
        dr = mul_one_q15(o3r); di = mul_one_q15(o3i);
    } else {
        const int32_t w1r = w1.x, w1i = w1.y, w2r = w2.x, w2i = w2.y, w3r = w3.x, w3i = w3.y;
        cr = msub_q15(o1r, w1r, o1i, w1i); ci = madd_q15(o1r, w1i, o1i, w1r);
        br = msub_q15(o2r, w2r, o2i, w2i); bi = madd_q15(o2r, w2i, o2i, w2r);
        dr = msub_q15(o3r, w3r, o3i, w3i); di = madd_q15(o3r, w3i, o3i, w3r);
    }
}

/* Stage 2 of the 256-point FFT uses the twiddles of k = 0, 16, 32, 48 -- the same for every lane, so their special
 * shapes can be compiled in (fill_dev_tables verifies that the generated table has them; the values are floor-quantised,
 * twiddle_fft_dif.c:9):
 *   TW_ONE   (0x7fff, 0)        the Q15 "one": a + ((-a) >> 15)
 *   TW_NEGI  (0, -32768)        exactly -j: (re, im) -> (im, -re), no product at all
 *   TW_DIAG  (c, c)             re = ((a.re - a.im) c) >> 15, im = ((a.re + a.im) c) >> 15: one 64-bit product each
 *   TW_ADIAG (c, -(c + 1))      re = ((a.re + a.im) c + a.im) >> 15, im = ((a.im - a.re) c - a.re) >> 15
 *   TW_ANY   the general complex product (complex.c:54-72)
 * Every form is the reference's (ar wr - ai wi) >> 15, (ar wi + ai wr) >> 15 with the 64-bit sum rearranged exactly. */
enum { TW_ANY = 0, TW_ONE = 1, TW_NEGI = 2, TW_DIAG = 3, TW_ADIAG = 4 };
template <int KIND>
__device__ __forceinline__ void cmul_tw(int32_t or_, int32_t oi, int2 w, int32_t &re, int32_t &im)
{
    if (KIND == TW_ONE) { re = mul_one_q15(or_); im = mul_one_q15(oi); }
    else if (KIND == TW_NEGI) { re = oi; im = -or_; }
    else if (KIND == TW_DIAG) {
        re = (int32_t)(((int64_t)(or_ - oi) * (int64_t)w.x) >> 15);
        im = (int32_t)(((int64_t)(or_ + oi) * (int64_t)w.x) >> 15);
    } else if (KIND == TW_ADIAG) {
        re = (int32_t)(((int64_t)(or_ + oi) * (int64_t)w.x + (int64_t)oi) >> 15);
        im = (int32_t)(((int64_t)(oi - or_) * (int64_t)w.x - (int64_t)or_) >> 15);
    } else { re = msub_q15(or_, w.x, oi, w.y); im = madd_q15(or_, w.y, oi, w.x); }
}
/* bfly4 with the kinds of its three twiddles compiled in */
template <int K1, int K2, int K3>
__device__ __forceinline__ void bfly4_tw(int32_t &ar, int32_t &ai, int32_t &cr, int32_t &ci,
                                         int32_t &br, int32_t &bi, int32_t &dr, int32_t &di,
                                         int2 w1, int2 w2, int2 w3)
{
    const int32_t s1r = cr + dr, s1i = ci + di, d1r = cr - dr, d1i = ci - di;
    const int32_t o0r = add3(ar, br, s1r), o0i = add3(ai, bi, s1i);
    const int32_t o1r = add2sub(ar, br, s1r), o1i = add2sub(ai, bi, s1i);
    const int32_t o2r = sub2add(ar, br, d1i), o2i = sub3(ai, bi, d1r);
    const int32_t o3r = sub3(ar, br, d1i), o3i = sub2add(ai, bi, d1r);
    ar = mul_one_q15(o0r);
    ai = mul_one_q15(o0i);
    cmul_tw<K1>(o1r, o1i, w1, cr, ci);
    cmul_tw<K2>(o2r, o2i, w2, br, bi);
    cmul_tw<K3>(o3r, o3i, w3, dr, di);
}

__device__ __forceinline__ int xpad(int p) { return p + (p >> 4); }

/* One frame by the 16 lanes of a half-warp (L = lane & 15). `load_pair(a, p)` returns PCM samples
 * 2p and 2p+1 of the 480-sample analysis window packed in one word (p = L + 16a = 0..239; `a` is a
 * compile-time constant after unrolling, so callers can address with immediates).
 * Every lane of the WARP must call this together (full-warp __syncwarp inside). */
/* norm (optional, shared memory): mean[40], stdR[40], rshift of a model. When given, the standardised row
 * (feature_module.c:67-73) is written to out_feat as int16 instead of the log-mel row to out_logmel.
 * out_copy (optional, log-mel mode): a second place the log-mel row is written to. */
template <bool DUMP, typename LoadPair>
__device__ __forceinline__ void frame_logmel(const FeatSmemTables &tb, FrameScratch &fs, int L,
                                             LoadPair load_pair, int32_t *__restrict__ out_logmel,
                                             bool store, FeatDump dump, const int32_t *norm = nullptr,
                                             int16_t *__restrict__ out_feat = nullptr, int32_t *__restrict__ out_copy = nullptr)
{
    int32_t xr[16], xi[16];
    /* window, Q15 x Q15 >> 15 (spectrogram_module.c:62-66); zero padding 480..511 (:68-71) */
#pragma unroll
    for (int a = 0; a < 15; a++) {
        const int p = L + 16 * a;
        const uint32_t s = load_pair(a, p);
        const int2 w = tb.win2[p];
        xr[a] = (w.x * (int32_t)(int16_t)(s & 0xffff)) >> 15;
        xi[a] = (w.y * ((int32_t)s >> 16)) >> 15;
    }
    xr[15] = 0; xi[15] = 0;
    if (DUMP && dump.fft_in && store) {
#pragma unroll
        for (int a = 0; a < 16; a++) { dump.fft_in[2 * (L + 16 * a)] = xr[a]; dump.fft_in[2 * (L + 16 * a) + 1] = xi[a]; }
    }
    /* stage 0: Nf = 256, q = 64, butterflies m = L + 16a', twiddle index k = m (fft.c:162-200) */
#pragma unroll
    for (int a = 0; a < 4; a++) {
        bfly4<false>(xr[a], xi[a], xr[a + 4], xi[a + 4], xr[a + 8], xi[a + 8], xr[a + 12], xi[a + 12],
                     tb.tw0[a][0][L], tb.tw0[a][1][L], tb.tw0[a][2][L]);
    }
    /* stage 1: Nf = 64, q = 16, group g, m = L, k = 4L */
    {
        const int2 w1 = tb.tw1[0][L], w2 = tb.tw1[1][L], w3 = tb.tw1[2][L];
#pragma unroll
        for (int g = 0; g < 4; g++)
            bfly4<false>(xr[4 * g], xi[4 * g], xr[4 * g + 1], xi[4 * g + 1], xr[4 * g + 2], xi[4 * g + 2],
                         xr[4 * g + 3], xi[4 * g + 3], w1, w2, w3);
    }
    /* 16x16 transpose: point L + 16a -> lane a, slot L */
#pragma unroll
    for (int a = 0; a < 16; a++) fs.x[xpad(L + 16 * a)] = make_int2(xr[a], xi[a]);
    __syncwarp();
#pragma unroll
    for (int b = 0; b < 16; b++) { const int2 v = fs.x[xpad(16 * L + b)]; xr[b] = v.x; xi[b] = v.y; }
    __syncwarp();
    /* stage 2: Nf = 16, q = 4, group g = L, m = 0..3, k = 16m (same for every lane): twiddles tw^2k, tw^k, tw^3k of
     * k = 0 (all ones), 16 (-45 deg, general, general), 32 (-j, -45 deg, -135 deg), 48 (-135 deg, general, general) */
    bfly4_tw<TW_ONE, TW_ONE, TW_ONE>(xr[0], xi[0], xr[4], xi[4], xr[8], xi[8], xr[12], xi[12], tb.tw2[0][0], tb.tw2[0][1], tb.tw2[0][2]);
    bfly4_tw<TW_ADIAG, TW_ANY, TW_ANY>(xr[1], xi[1], xr[5], xi[5], xr[9], xi[9], xr[13], xi[13], tb.tw2[1][0], tb.tw2[1][1], tb.tw2[1][2]);
    bfly4_tw<TW_NEGI, TW_ADIAG, TW_DIAG>(xr[2], xi[2], xr[6], xi[6], xr[10], xi[10], xr[14], xi[14], tb.tw2[2][0], tb.tw2[2][1], tb.tw2[2][2]);
    bfly4_tw<TW_DIAG, TW_ANY, TW_ANY>(xr[3], xi[3], xr[7], xi[7], xr[11], xi[11], xr[15], xi[15], tb.tw2[3][0], tb.tw2[3][1], tb.tw2[3][2]);
    /* stage 3: Nf = 4, q = 1, k = 0: every twiddle is 0x7fff + 0j */
#pragma unroll
    for (int g = 0; g < 4; g++)
        bfly4<true>(xr[4 * g], xi[4 * g], xr[4 * g + 1], xi[4 * g + 1], xr[4 * g + 2], xi[4 * g + 2],
                    xr[4 * g + 3], xi[4 * g + 3], make_int2(0, 0), make_int2(0, 0), make_int2(0, 0));
    /* bit-reversed read-out (fft.c:217-220): Z[brev8(p)] = x[p]; store at index m = brev8(16L + b) */
#pragma unroll
    for (int b = 0; b < 16; b++) {
        const int m = (int)(__brev((unsigned)(16 * L + b)) >> 24);
        fs.x[m] = make_int2(xr[b], xi[b]);
    }
    __syncwarp();
    /* real-FFT split (fft.c:66-124) and power spectrum (spectrogram_module.c:33-45): each lane turns the pairs
     * (Z[i], Z[256-i]), i = L + 16j, into bins i and 256-i. Lane 0's pair (0, 0) would give bins 0 and 256, which no
     * mel band reads (melSpec_coeff.c: bins 1..255), so it takes the self-mirrored centre bin 128 in that turn
     * instead. The power spectrum is kept in registers until every lane has read its Z pairs, then it overwrites
     * the front of the same scratch (ps[] aliases x[]). */
    int32_t pa[8], pb[8];
    int32_t p0 = 0, p256 = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const bool centre = (j == 0 && L == 0);
        const int i = centre ? 128 : L + 16 * j;
        const int2 zi = fs.x[i], zr = fs.x[256 - i];
        const int2 w = tb.rtw[i], v = tb.rtw[256 - i];
        const int32_t er = (zi.x + zr.x) >> 1, ei = (zi.y - zr.y) >> 1;
        const int32_t orr = (zi.y + zr.y) >> 1, oi = (zr.x - zi.x) >> 1;
        const int32_t xr0 = er + msub_q15(orr, w.x, oi, w.y), xi0 = ei + madd_q15(orr, w.y, oi, w.x);
        pa[j] = (int32_t)(((int64_t)xr0 * xr0 + (int64_t)xi0 * xi0) >> 15);
        /* mirrored bin 256 - i from the same pair, roles of Z[i] and Z[256-i] swapped */
        const int32_t fi = (zr.y - zi.y) >> 1, pi = (zi.x - zr.x) >> 1;
        const int32_t xr1 = er + msub_q15(orr, v.x, pi, v.y), xi1 = fi + madd_q15(orr, v.y, pi, v.x);
        pb[j] = (int32_t)(((int64_t)xr1 * xr1 + (int64_t)xi1 * xi1) >> 15);
        if (DUMP && dump.spec && store) {
            dump.spec[2 * i] = xr0; dump.spec[2 * i + 1] = xi0;
            if (!centre) { dump.spec[2 * (256 - i)] = xr1; dump.spec[2 * (256 - i) + 1] = xi1; }
        }
    }
    if (DUMP && L == 0) {
        /* taps only: bin 0 from the pair (Z[0], Z[0]) and the Nyquist bin X[256] = Xe[0] - Xo[0] (fft.c:123-124) */
        const int2 z0 = fs.x[0], w = tb.rtw[0];
        const int32_t er = z0.x, orr = z0.y;
        const int32_t xr0 = er + msub_q15(orr, w.x, 0, w.y), xi0 = madd_q15(orr, w.y, 0, w.x);
        const int32_t re = z0.x - z0.y;
        p0 = (int32_t)(((int64_t)xr0 * xr0 + (int64_t)xi0 * xi0) >> 15);
        p256 = (int32_t)(((int64_t)re * re) >> 15);
        if (dump.spec && store) { dump.spec[0] = xr0; dump.spec[1] = xi0; dump.spec[512] = re; dump.spec[513] = 0; }
    }
    __syncwarp();
    int32_t *ps = reinterpret_cast<int32_t *>(fs.x);
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const bool centre = (j == 0 && L == 0);
        const int i = centre ? 128 : L + 16 * j;
        ps[i] = pa[j];
        if (!centre) ps[256 - i] = pb[j];
    }
    if (DUMP && L == 0) { ps[0] = p0; ps[256] = p256; }
    __syncwarp();
    if (DUMP && dump.pspec && store)
        for (int i = L; i < 257; i += 16) dump.pspec[i] = ps[i];
    /* mel filterbank (melSpecProc.c:6-27) + log10 (fixlog10.c:53-61). Bands are handed out widest first
     * (b = 39 - L - 16r) so that the lanes of a round have similar trip counts; taps and bins come in groups of 4
     * (one 128-bit load each), two independent 64-bit accumulators. The int64 sum is exact in any order. */
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const int b = 39 - L - 16 * r;
        if (b >= 0) {
            const uint32_t meta = tb.mel_meta[b];
            const int ng = (meta >> 8) & 0xff;
            const int4 *tap = &tb.mel_tap4[meta & 0xff];
            const int4 *bin = reinterpret_cast<const int4 *>(&ps[meta >> 16]);
            int64_t m0 = 0, m1 = 0;
            /* trip counts are bounded per round (MEL_MAXG, checked when the tables are built): fully unrolled and
             * predicated, so the loads of a round are issued together */
#pragma unroll
            for (int i = 0; i < (r == 0 ? MEL_MAXG0 : (r == 1 ? MEL_MAXG1 : MEL_MAXG2)); i++) {
                if (i < ng) {
                    const int4 w = tap[i], v = bin[i];
                    m0 += (int64_t)w.x * (int64_t)v.x; m1 += (int64_t)w.y * (int64_t)v.y;
                    m0 += (int64_t)w.z * (int64_t)v.z; m1 += (int64_t)w.w * (int64_t)v.w;
                }
            }
            const int32_t mel = sat32_dev((m0 + m1) >> 15);
            if (DUMP && dump.mel && store) dump.mel[b] = mel;
            if (store) {
                const int32_t lm = log10_q15(mel, tb.log_lut);
                if (norm) out_feat[b] = standardise(lm, norm[b], norm[40 + b], norm[80]);
                else {
                    out_logmel[b] = lm;
                    if (out_copy) out_copy[b] = lm;
                }
            }
        }
    }
    __syncwarp();
}

}  // namespace nnsp
