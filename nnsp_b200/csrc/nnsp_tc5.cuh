/* nnsp_tc5.cuh -- layer 0 of the batched network path on the 5th-generation tensor cores (tcgen05.mma kind::i8).
 *
 * What it computes (unchanged, bit for bit): the first fc layer of NeuralNetClass_exe (neural_nets.c:44-168 ->
 * fc_8x16, affine.c:409-490) with tanh_fix (activation.c:31-69) for every (stream, inference) row of one exec call:
 * 240 int16 inputs = the 6 x 40 context window of standardised feature rows ending at the inference frame
 * (feature_module.c:54-73), int8 weights, the exact 32-bit finish of MmaLayer.fast. Output: the activation byte planes
 * [tile][inference][hi|lo][16][pa] the scan kernel reads, exactly what seg_kernel<1> writes.
 *
 * Formulation (developed and measured in tools/tc5_gemm_bench.cu; profiles/r2_tc5_gemm_bench.txt):
 *   int16 x int8 = 256 (hi(x) . w) + (lo(x) . w): two tcgen05.mma kind::i8 chains, s8 x s8 into TMEM columns [0, NP) and
 *   u8 x s8 into [NP, 2 NP), both int32 and exact.
 *   A tile is 2 streams x 64 inference slots = the 128 rows (TMEM lanes) of one M = 128 instruction. Row (q, i) needs the
 *   rows 2 i .. 2 i + 5 of stream q's feature sequence. Those windows overlap, so instead of expanding them (6 x the bytes,
 *   and the expansion was what bound the first version) the sequence is stored ONCE as 16-byte entries, entry e of an
 *   array = 16 bytes of frame 2 e + parity, and an instruction's A descriptor starts (f >> 1) entries in: without swizzle
 *   the K-major operand is addressed as start + (row / 8) * SBO + (k chunk) * LBO + (row % 8) * 16 with SBO = 128, so row
 *   r simply reads entry r + (f >> 1). Five arrays per byte plane: (even frames, bytes 0..15), (even, 16..31), (odd, 0..15),
 *   (odd, 16..31) and the tails (bytes 32..39 of frame 2 e | of frame 2 e + 1). The second 16-byte chunk of a K = 32
 *   instruction is either the NEXT entry of the same array (LBO = 16: frames f and f + 2) or the same entry of the
 *   next array (LBO = the array stride): 15 chunks -> 8 instructions per plane, 16 per tile.
 *   Roles (one persistent CTA per SM, 13 warps): 8 finish warps (TMEM lane quarter x share of the 16-unit blocks; TMEM ->
 *   registers -> bias, shift, tanh -> the tile's byte planes assembled in shared memory -> coalesced 16-byte stores),
 *   4 conversion warps (TMA bulk copies of the raw int16 rows through a 4-deep ring -> byte planes in entry layout), 1 warp
 *   whose lane 0 issues the MMAs -- its own warp because the issue of a queued tcgen05.mma blocks, which would stall the
 *   conversion behind it. Three A buffers / TMEM stages in flight.
 * Eligibility (launch_split_layers): a range selection (the batched NNSPClass; the cascade's first round only under
 * NNSP_B200_TC5=2, through vseq_kernel), layer 0 = fc 240 -> rows <= 80 with tanh and the exact 32-bit finish, followed by
 * an LSTM, and at least 45 % of the tiles' inference slots in use (tc5_wanted, nnsp_split.cu). Taps do not change the
 * choice: with an activation tap, tc5_tap_kernel decodes the output planes into it right after this kernel.
 * NNSP_B200_TC5=0 keeps the mma.sync kernel, =2 takes this one whenever the layer qualifies. */
#pragma once

namespace nnsp {

constexpr int TC5_SLOTS = 64, TC5_STREAMS = 2;                               /* 128 rows = 2 streams x 64 inference slots */
constexpr int TC5_KC = TC5_SLOTS - 2;                                        /* usable slots: slot i reads entries i .. i + 2 of its stream's 64 */
constexpr int TC5_FRAMES = 2 * TC5_KC + 4;                                   /* feature rows a tile reads per stream: 128 */
constexpr int TC5_SPITCH = TC5_SLOTS * 16;                                   /* a stream's entries in one array */
constexpr int TC5_CH = TC5_STREAMS * TC5_SPITCH + 160;                       /* one array + the entries the last rows read past it (64 B); 2208 = 32 mod 128:
                                                                              * the even- and odd-frame lanes of a conversion store (arrays j, j + 2) take different banks */
constexpr int TC5_LUTC = 4;                                                  /* tanh table copies: lane l reads copy l % 4 (16 would remove every bank conflict; the room goes to the output staging) */
constexpr int TC5_PAMAX = 128;                                               /* widest plane pitch the output staging holds (2 pa = 16 lanes x 16 bytes) */
constexpr int TC5_PLANE = 5 * TC5_CH;
constexpr int TC5_STAGES = 3, TC5_RING = 4;
constexpr int TC5_NPMAX = 80;                                                /* 3 stages x 2 x NP TMEM columns <= 512 */
constexpr int TC5_FINISH_WARPS = 8, TC5_CONV_THREADS = 128;
constexpr int TC5_THREADS = TC5_FINISH_WARPS * 32 + TC5_CONV_THREADS + 32;
constexpr int TC5_GROUPS = TC5_FINISH_WARPS / 4;
constexpr int TC5_WBYTES = 8 * TC5_NPMAX * 32;

struct Tc5Smem {
    alignas(1024) uint8_t a[TC5_STAGES][2][TC5_PLANE];             /* [stage][hi|lo][array][stream][entry][16] */
    alignas(1024) uint8_t w[TC5_WBYTES];                           /* [instruction j][unit / 8][2 chunks][8][16] */
    alignas(128) int16_t raw[TC5_RING][TC5_STREAMS][TC5_FRAMES * 40 + 8];
    alignas(128) uint8_t outst[TC5_SLOTS * (4 * TC5_PAMAX + 16)];   /* finished tile: [slot][hi|lo][2 streams][pa] */
    int2 lut2[LUT2_N * TC5_LUTC];
    int32_t bias[TC5_NPMAX];
    alignas(8) uint64_t mma_done[TC5_STAGES], tmem_free[TC5_STAGES], a_full[TC5_STAGES], raw_full[TC5_RING];
    uint32_t tmem;
};

struct Tc5Args {
    const uint8_t *img;             /* tc5 image of the model: 8 x np x 32 weight bytes, then np int32 biases (pre-shifted) */
    const DevTables *tables;
    int np, rs;                     /* padded units (multiple of 16), right shift of the finish (-sh_out) */
    int s0, ns, tile0;              /* stream range and the plane tile of s0 */
    int T, first, n_inf, nchunks;   /* inference k is frame first + 2 k; chunks of TC5_KC inferences */
    int pa;
    long long tile_bytes;
    const int16_t *feat16;          /* [S][T][40] */
    const int16_t *ctx;             /* [S][240] */
    uint8_t *out_planes;
    /* cascade rounds (vseq != null): the selection is a device-side list (count, plane tile offset as in StreamSel), stream s
     * has its own first inference frame tstart[s], hence (Ts - tstart[s] + 1) / 2 inferences (Ts: its end frame, T unless
     * the call is ragged), and its window rows were
     * written by vseq_kernel: vseq[s][v] = row of frame tstart[s] - 5 + v, already standardised, context rows included */
    const int *list, *count, *tile_off, *tstart;
    const int16_t *vseq;
    int vf;                         /* rows per stream in vseq */
    const int32_t *nfr;             /* ragged cascade call: stream s ends at frame stream_frames(nfr, s, T) (null: at T) */
};
__device__ __forceinline__ int tc5_nsel(const Tc5Args &a) { return a.list ? *a.count : a.ns; }
__device__ __forceinline__ long long tc5_sid(const Tc5Args &a, int p) { return a.list ? a.list[p] : (long long)a.s0 + p; }
/* inferences of stream position p that fall into the chunk starting at inference k0 */
__device__ __forceinline__ int tc5_nk(const Tc5Args &a, int p, int nsel, int k0)
{
    if (p >= nsel) return 0;
    int ninf = a.n_inf;
    if (a.vseq) {
        const long long s = tc5_sid(a, p);
        const int ts = a.tstart[s], Ts = stream_frames(a.nfr, s, a.T);
        ninf = ts < Ts ? (Ts - ts + 1) >> 1 : 0;
    }
    return max(0, min(TC5_KC, ninf - k0));
}

__device__ __forceinline__ uint64_t tc5_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{   /* shared-memory matrix descriptor, no swizzle: address, leading / stride byte offsets in 16-byte units, version 1 */
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ uint32_t tc5_idesc(int n, bool a_signed)
{   /* kind::i8: D = s32, A = s8 / u8, B = s8, both K-major, N >> 3, M = 128 */
    return (2u << 4) | ((a_signed ? 1u : 0u) << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | (8u << 24);
}
__device__ __forceinline__ void tc5_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
                 :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
}
__device__ __forceinline__ void tc5_ld16(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc5_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}

__global__ void __launch_bounds__(TC5_THREADS, 1)
seg0_tc5_kernel(Tc5Args a)
{
    /* aligned by hand (the launch adds 1 KB): an alignment attribute here would apply to the dynamic shared memory of every
     * kernel of the translation unit and push the seg / scan kernels past the 227 KB limit */
    extern __shared__ __align__(128) unsigned char smem_tc5[];
    Tc5Smem &sm = *reinterpret_cast<Tc5Smem *>(smem_tc5 + ((1024u - (smem_u32(smem_tc5) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int np = a.np, T = a.T;
    const uint32_t st_cols = 2u * (uint32_t)np;                              /* TMEM columns of a stage: hi sums | lo sums */
    const int nsel = tc5_nsel(a);
    const int npairs = (nsel + 1) >> 1, nitems = npairs * a.nchunks;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&sm.tmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        for (int b = 0; b < TC5_STAGES; b++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&sm.mma_done[b])));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(&sm.tmem_free[b])), "r"((uint32_t)TC5_FINISH_WARPS));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&sm.a_full[b])));
        }
        for (int b = 0; b < TC5_RING; b++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&sm.raw_full[b])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 8 * np * 32 / 16; i += TC5_THREADS) reinterpret_cast<uint4 *>(sm.w)[i] = __ldg(reinterpret_cast<const uint4 *>(a.img) + i);
    for (int i = tid; i < np; i += TC5_THREADS) sm.bias[i] = reinterpret_cast<const int32_t *>(a.img + 8 * np * 32)[i];
    fill_lut2<TC5_LUTC>(sm.lut2, a.tables, tid, TC5_THREADS);
    for (int i = tid; i < (int)(sizeof(sm.outst) / 16); i += TC5_THREADS) reinterpret_cast<uint4 *>(sm.outst)[i] = make_uint4(0, 0, 0, 0);   /* columns np .. pa stay zero */
    /* entries no conversion writes (the slots past a short chunk, the pad behind the last stream) must hold defined bytes:
     * their rows are computed and dropped */
    for (int i = tid; i < (int)(sizeof(sm.a) / 16); i += TC5_THREADS) reinterpret_cast<uint4 *>(&sm.a[0][0][0])[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = sm.tmem;

    if (warp == TC5_FINISH_WARPS + TC5_CONV_THREADS / 32) {
        /* ---------------- MMA issue ---------------- */
        if (lane == 0) {
            const uint32_t idh = tc5_idesc(np, true), idl = tc5_idesc(np, false);
            int n = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, n++) {
                const int b = n % TC5_STAGES, use = n / TC5_STAGES;
                tc5_wait(&sm.a_full[b], (uint32_t)(use & 1));                                   /* the conversion of item n is in a[b] */
                if (use >= 1) tc5_wait(&sm.tmem_free[b], (uint32_t)((use - 1) & 1));            /* the finish has drained TMEM stage b */
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t ah = smem_u32(sm.a[b][0]), al = smem_u32(sm.a[b][1]), wb = smem_u32(sm.w), td = tmem + st_cols * b;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    /* j 0..3: frames f, f + 2 of array j (next entry: LBO = 16); 4, 5: bytes 0..15 | 16..31 of frame 4 + parity
                     * (next array); 6: tails of frames 0..3; 7: tails of frames 4, 5 | a chunk of zero weights */
                    const uint32_t arr = j < 4 ? j : (j < 6 ? 2 * (j - 4) : 4);
                    const uint32_t aoff = arr * TC5_CH + ((j == 4 || j == 5 || j == 7) ? 32 : 0);
                    const uint32_t lbo = (j == 4 || j == 5) ? TC5_CH : 16;
                    const uint64_t db = tc5_desc(wb + j * np * 32, 128, 256);
                    tc5_mma(td, tc5_desc(ah + aoff, lbo, 128), db, idh, j ? 1u : 0u);
                    tc5_mma(td + np, tc5_desc(al + aoff, lbo, 128), db, idl, j ? 1u : 0u);
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(&sm.mma_done[b])) : "memory");
            }
        }
    } else if (warp >= TC5_FINISH_WARPS) {
        /* ---------------- conversion: raw int16 rows (TMA ring) -> byte planes in entry layout ---------------- */
        const int ptid = tid - TC5_FINISH_WARPS * 32;
        /* rows v = 0 .. 2 nk + 3 of the item are frames f_lo + v; frames before the call are the carried context rows
         * (feature_module.c:54-57: row 6 + f of the stored window for f = -5 .. -1) */
        auto fetch = [&](int item, int rb) {
            const int chunk = item / npairs, pair = item - chunk * npairs;
            const int k0 = chunk * TC5_KC;
            const int f_lo = a.first - 5 + 2 * k0, nctx = (!a.vseq && f_lo < 0) ? -f_lo : 0;
            int nrow[TC5_STREAMS];
            uint32_t bytes = 0;
            for (int q = 0; q < TC5_STREAMS; q++) {
                const int nk = tc5_nk(a, 2 * pair + q, nsel, k0);
                nrow[q] = nk > 0 ? 2 * nk + 4 : 0;
                bytes += (uint32_t)(nrow[q] * 80);
            }
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&sm.raw_full[rb])), "r"(bytes) : "memory");
            for (int q = 0; q < TC5_STREAMS; q++) {
                if (!nrow[q]) continue;
                const long long s = tc5_sid(a, 2 * pair + q);
                if (nctx)
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 :: "r"(smem_u32(&sm.raw[rb][q][0])), "l"(a.ctx + s * 240 + (6 + f_lo) * 40), "r"((uint32_t)(nctx * 80)), "r"(smem_u32(&sm.raw_full[rb])) : "memory");
                const int16_t *src = a.vseq ? a.vseq + (s * a.vf + 2 * k0) * 40 : a.feat16 + (s * T + f_lo + nctx) * 40;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(smem_u32(&sm.raw[rb][q][nctx * 40])), "l"(src), "r"((uint32_t)((nrow[q] - nctx) * 80)), "r"(smem_u32(&sm.raw_full[rb])) : "memory");
            }
        };
        if (ptid == 0)
            for (int m = 0; m < TC5_RING - 1; m++)
                if ((int)blockIdx.x + m * (int)gridDim.x < nitems) fetch(blockIdx.x + m * gridDim.x, m);
        int n = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x, n++) {
            const int b = n % TC5_STAGES, use = n / TC5_STAGES, rb = n % TC5_RING;
            /* ring slot (n - 1) % RING was read by the conversion of item n - 1: every conversion thread is past that iteration's barrier */
            if (ptid == 0 && item + (TC5_RING - 1) * (int)gridDim.x < nitems) fetch(item + (TC5_RING - 1) * gridDim.x, (n + TC5_RING - 1) % TC5_RING);
            if (use >= 1) tc5_wait(&sm.mma_done[b], (uint32_t)((use - 1) & 1));                  /* the MMAs that read a[b] are complete */
            tc5_wait(&sm.raw_full[rb], (uint32_t)((n / TC5_RING) & 1));
            const int chunk = item / npairs, pair = item - chunk * npairs;
            const int nrow = 2 * max(tc5_nk(a, 2 * pair, nsel, chunk * TC5_KC), tc5_nk(a, 2 * pair + 1, nsel, chunk * TC5_KC)) + 4;   /* rows past a stream's own count are stale: their slots are dropped */
            for (int e = ptid; e < TC5_STREAMS * nrow; e += TC5_CONV_THREADS) {
                const int q = e / nrow, fr = e - q * nrow;
                const uint4 *src = reinterpret_cast<const uint4 *>(&sm.raw[rb][q][fr * 40]);
                const uint4 v0 = src[0], v1 = src[1], v2 = src[2], v3 = src[3], v4 = src[4];
                uint4 h0, l0, h1, l1;
                uint2 h2, l2;
                l0.x = __byte_perm(v0.x, v0.y, 0x6420); h0.x = __byte_perm(v0.x, v0.y, 0x7531);
                l0.y = __byte_perm(v0.z, v0.w, 0x6420); h0.y = __byte_perm(v0.z, v0.w, 0x7531);
                l0.z = __byte_perm(v1.x, v1.y, 0x6420); h0.z = __byte_perm(v1.x, v1.y, 0x7531);
                l0.w = __byte_perm(v1.z, v1.w, 0x6420); h0.w = __byte_perm(v1.z, v1.w, 0x7531);
                l1.x = __byte_perm(v2.x, v2.y, 0x6420); h1.x = __byte_perm(v2.x, v2.y, 0x7531);
                l1.y = __byte_perm(v2.z, v2.w, 0x6420); h1.y = __byte_perm(v2.z, v2.w, 0x7531);
                l1.z = __byte_perm(v3.x, v3.y, 0x6420); h1.z = __byte_perm(v3.x, v3.y, 0x7531);
                l1.w = __byte_perm(v3.z, v3.w, 0x6420); h1.w = __byte_perm(v3.z, v3.w, 0x7531);
                l2.x = __byte_perm(v4.x, v4.y, 0x6420); h2.x = __byte_perm(v4.x, v4.y, 0x7531);
                l2.y = __byte_perm(v4.z, v4.w, 0x6420); h2.y = __byte_perm(v4.z, v4.w, 0x7531);
                const int off = q * TC5_SPITCH + (fr >> 1) * 16, par = fr & 1;
                uint8_t *ph = sm.a[b][0] + off, *pl = sm.a[b][1] + off;
                *reinterpret_cast<uint4 *>(ph + 2 * par * TC5_CH) = h0; *reinterpret_cast<uint4 *>(ph + (2 * par + 1) * TC5_CH) = h1;
                *reinterpret_cast<uint2 *>(ph + 4 * TC5_CH + par * 8) = h2;
                *reinterpret_cast<uint4 *>(pl + 2 * par * TC5_CH) = l0; *reinterpret_cast<uint4 *>(pl + (2 * par + 1) * TC5_CH) = l1;
                *reinterpret_cast<uint2 *>(pl + 4 * TC5_CH + par * 8) = l2;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, %0;" :: "n"(TC5_CONV_THREADS) : "memory");
            if (ptid == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(&sm.a_full[b])) : "memory");
        }
    } else {
        /* ---------------- finish: TMEM lane r = 64 (stream of the pair) + inference slot; the warps of a lane quarter share the 16-unit blocks ---------------- */
        /* A thread's 16 bytes of a byte plane are 32 pa bytes away from its lane neighbour's: written straight from the
         * registers every 16-byte store was its own sector and the L1 store path (one sector per cycle) cost 120 of the
         * kernel's 266 us. So the tile is assembled in shared memory in the layout of the planes and copied out with lanes
         * along the 2 pa contiguous bytes that the two streams of a pair share per inference and byte plane (full sectors,
         * four per cycle). The four warps that own the same 32 slots (two streams x two block shares) synchronise among
         * themselves only: two 128-thread named barriers per tile. */
        const int grp = warp >> 2, set = warp & 1;                               /* set: slots 0..31 / 32..63 of both streams */
        const int r = (warp & 3) * 32 + lane, q = r >> 6, slot = r & (TC5_SLOTS - 1);
        const int nblk = np >> 4, pa = a.pa, rs = a.rs;
        const int2 *lutl = sm.lut2 + (lane & (TC5_LUTC - 1));
        const size_t XB = (size_t)32 * pa;
        const int spitch = 4 * pa + 16;                                          /* staging bytes of a slot: [hi|lo][2 streams][pa], + 16 to spread the banks */
        uint8_t *stg = sm.outst + (size_t)slot * spitch + q * pa;               /* this row's bytes of the high plane; low plane 2 pa on */
        const int ctid = (warp >> 1) * 32 + lane;                                /* 0..127 within the set: copy-out role */
        const int half = ctid >> 4, piece = ctid & 15, npc = pa >> 3;            /* 16 lanes per (slot, plane) run of 2 pa bytes = npc 16-byte pieces */
        int n = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x, n++) {
            const int b = n % TC5_STAGES, use = n / TC5_STAGES;
            const int chunk = item / npairs, pair = item - chunk * npairs;
            const int k0 = chunk * TC5_KC;
            const int nk0 = tc5_nk(a, 2 * pair, nsel, k0), nk1 = tc5_nk(a, 2 * pair + 1, nsel, k0), nk = max(nk0, nk1);
            const int nstr = min(TC5_STREAMS, nsel - 2 * pair);
            const bool live = slot < (q ? nk1 : nk0);
            tc5_wait(&sm.mma_done[b], (uint32_t)(use & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem + st_cols * b + ((uint32_t)((warp & 3) * 32) << 16);
            for (int j0 = 0; j0 < nblk; j0 += TC5_GROUPS) {                      /* blocks of 16 units: one 16-byte piece per byte plane */
                const int j = j0 + grp, c = j * 16;
                const bool have = j < nblk, last = j0 + TC5_GROUPS >= nblk;
                uint32_t hi[16], lo[16];
                if (have) {
                    tc5_ld16(taddr + c, hi);
                    tc5_ld16(taddr + np + c, lo);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                }
                if (last) {                                                      /* this warp's share of the stage is in registers: hand it back before the arithmetic */
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(&sm.tmem_free[b])) : "memory");
                }
                if (have && live) {
                    uint32_t oh[4] = { 0, 0, 0, 0 }, ol[4] = { 0, 0, 0, 0 };
#pragma unroll
                    for (int e = 0; e < 16; e++) {
                        const int32_t pre = (int32_t)((hi[e] << 8) + lo[e] + (uint32_t)sm.bias[c + e]) >> rs;
                        const uint32_t y = (uint32_t)tanh_q15v<TC5_LUTC>(pre, lutl);
                        oh[e >> 2] |= ((y >> 8) & 0xffu) << (8 * (e & 3));
                        ol[e >> 2] |= (y & 0xffu) << (8 * (e & 3));
                    }
                    *reinterpret_cast<uint4 *>(stg + c) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
                    *reinterpret_cast<uint4 *>(stg + 2 * pa + c) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
                }
            }
            asm volatile("bar.sync %0, 128;" :: "r"(2 + set) : "memory");        /* the set's 32 slots are assembled */
            {   /* copy out: the plane columns past the padded units leave as the zeros the staging buffer was cleared to */
                const size_t tile_abs = (size_t)a.tile0 + (a.list ? (size_t)*a.tile_off : 0) + (size_t)((2 * pair) >> 4);
                uint8_t *gbase = a.out_planes + tile_abs * (size_t)a.tile_bytes + (size_t)((2 * pair) & 15) * pa + (size_t)piece * 16;
                const int nrun = 2 * min(32, nk - 32 * set);                     /* (slot, plane) runs of this set; <= 0: nothing */
                if (piece * 16 < nstr * pa)
                    for (int run = half; run < nrun; run += 8) {
                        const int sl = 32 * set + (run >> 1), pl = run & 1;
                        const uint4 v = *reinterpret_cast<const uint4 *>(sm.outst + (size_t)sl * spitch + pl * 2 * pa + piece * 16);
                        *reinterpret_cast<uint4 *>(gbase + (size_t)(k0 + sl) * XB + (size_t)pl * 16 * pa) = v;
                    }
            }
            asm volatile("bar.sync %0, 128;" :: "r"(2 + set) : "memory");        /* ... and read: the next tile may overwrite them */
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512u) : "memory");
}

}   /* namespace nnsp */
