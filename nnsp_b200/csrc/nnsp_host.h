/* nnsp_host.h -- host-side internals shared by the engine translation units. */
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include "nnsp_b200.h"
#include "nnsp_engine.cuh"
#include "nnsp_model.h"
#include "nnsp_tables.h"

namespace nnsp {

extern std::atomic<long long> g_launches, g_tc5_launches;
extern std::atomic<long long> g_cascade_net_launches[3];   /* cascade_kernel<CsNarrow>, cascade_kernel<CsWide>, cascade_replay_kernel */
extern std::atomic<long long> g_scan_launches[6];          /* scan_kernel<4,4,1>, <4,4,0>, <8,2,2>, <9,2,3>, <9,2,0>, <16,1,0> */

#define NNSP_CUDA(expr)                                                                       \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            nnsp_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return NNSP_B200_ERR_CUDA;                                                        \
        }                                                                                     \
    } while (0)

#define NNSP_LAUNCH_CHECK()                                                                   \
    do {                                                                                      \
        ::nnsp::g_launches.fetch_add(1, std::memory_order_relaxed);                           \
        cudaError_t e__ = cudaGetLastError();                                                 \
        if (e__ != cudaSuccess) {                                                             \
            nnsp_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
            return NNSP_B200_ERR_CUDA;                                                        \
        }                                                                                     \
    } while (0)

/* device-resident copies of one model: descriptor + weight image + bias image */
struct DeviceModel {
    DevModel  h;              /* host copy of the descriptor */
    DevModel *d = nullptr;
    uint32_t *wimg = nullptr;
    int16_t  *bimg = nullptr;
};

int select_device(int device);                         /* cudaSetDevice + sm_100 check */
int get_device_tables(int device, const DevTables **out);
int upload_model(const nnsp_b200_model *m, DeviceModel *out);
void free_model(DeviceModel *dm);
int sm_count(int device);

/* kernel launchers (nnsp_engine.cu) */
struct FeatLaunch {
    const int16_t *pcm; long long stride;
    const int16_t *hist; int hist_frames;    /* [S][hist_frames*160], newest frames last */
    int s0, ns, T;
    int32_t *logmel;                          /* [S][T][40] */
    const int32_t *norm = nullptr;            /* device: mean[40], stdR[40], rshift -> write feat16 instead of logmel */
    int16_t *feat16 = nullptr;                /* [S][T][40] standardised rows (feature_module.c:67-73) */
    const int32_t *nfr = nullptr;             /* ragged cascade call: stream s has stream_frames(nfr, s, T) frames; the rows
                                                 of its later frames are neither computed nor written, their PCM not read */
};
int launch_feature(const DevTables *tb, const FeatLaunch &a, int device, cudaStream_t st);
/* hist <- newest hist_frames frames of (hist ++ src[0..T)); frames are words_per_frame 32-bit words. nfr (ragged
 * cascade call): stream s appends only its first stream_frames(nfr, s, T) frames, none when that is 0 */
int launch_hist_update(const void *src, long long stride_words, void *hist, int hist_frames, int words_per_frame,
                       int s0, int ns, int T, cudaStream_t st, const int32_t *nfr = nullptr);
/* the same, out of place (hist_in and hist_out distinct): lets the next call's front end start while kernels of this
 * call still read the old history */
int launch_hist_roll(const void *src, long long stride_words, const void *hist_in, void *hist_out, int hist_frames,
                     int words_per_frame, int s0, int ns, int T, cudaStream_t st, const int32_t *nfr = nullptr);


/* audio_frame_callback's conditioning (evb/src/main_nnsp.cc:58-65) of n_frames consecutive 160-sample frames, raw 32-bit
 * AUDADC words -> int16 PCM; both pointers 16-byte aligned */
int launch_ingest(const uint32_t *raw_dev, int16_t *pcm_dev, long long n_frames, int device, cudaStream_t st);

/* tensor-core (IMMA) network path, nnsp_mma.cu */
struct MmaModel;
struct MmaDeviceModel {
    MmaModel *h = nullptr;        /* host copy (heap) */
    MmaModel *d = nullptr;
    void     *frag = nullptr;     /* uint2 fragment image */
    int32_t  *bias32 = nullptr;
    uint8_t  *tc5 = nullptr;      /* layer 0 for the tcgen05 kernel (nnsp_tc5.cuh): 8 x tc5_np x 32 weight bytes + tc5_np biases; null when not eligible */
    int       tc5_np = 0;
    size_t    smem_base = 0, smem_warp = 0;
    int       off_bias = 0, off_lut = 0, off_model = 0, off_warps = 0;
};
/* NNSP_B200_ERR_UNSUPPORTED when the model does not fit the IMMA formulation (the dp2a kernel then runs) */
int upload_model_mma(const nnsp_b200_model *m, MmaDeviceModel *out);
void free_model_mma(MmaDeviceModel *mm);
struct NNLaunch {
    const DevTables *tables; StreamState st; const int32_t *logmel;
    int s0, ns, T; nnsp_b200_result *results; nnsp_b200_taps taps; int16_t thresh_prob, th_count;
    int raw_ctx = 0;              /* nnsp_b200_net_eval: the stored context is the network input as it stands */
};
int launch_nn_mma(const MmaDeviceModel &mm, const NNLaunch &a, int device, cudaStream_t st);

/* scan-split network path, nnsp_split.cu: fc runs for all (stream, inference) rows at once, the LSTM as a scan.
 * feat16: [S][T][40] standardised rows written by feat_kernel. first / n_inf: first inference frame (0 or 1) and number of inferences of this call (stride 2). planes0/1:
 * two buffers of split_plane_bytes(); dec: [S rounded up to 16][n_inf] int32. l.s0 must be a multiple of 16. */
/* one model over one selection of streams (the building block of launch_nn_split and of the cascade) */
struct SplitGroup {
    const DevTables *tables = nullptr;
    const int *list = nullptr, *count = nullptr, *tile_off = nullptr;   /* device-side selection, or ... */
    int s0 = 0, ns = 0;                                                 /* ... the range s0 .. s0+ns-1   */
    int tile0 = 0;                   /* first plane tile of the range / of the caller's plane region     */
    int max_streams = 0;             /* upper bound of the selection's size (sizes the grids)             */
    long long tile_bytes = 0;        /* plane bytes reserved per tile (0: n_inf * 32 * pa)               */
    int T = 0, first = 0, n_inf = 0;
    int mode = 1;                    /* 1: feat16 rows, 2: log-mel rows + look-back                       */
    const int16_t *feat16 = nullptr;
    const int32_t *logmel = nullptr, *lmhist = nullptr; int dmax = 0, dback = 0;
    const int16_t *ctx = nullptr;    /* [S][240] */
    int16_t *h = nullptr; int32_t *c = nullptr; int h_stride = 0;       /* LSTM state arrays [S][h_stride] */
    uint8_t *planes0 = nullptr, *planes1 = nullptr;
    int32_t *dec = nullptr; int dec_stride = 0;
    int16_t thresh_prob = 0;
    const int16_t *thr_prob = nullptr; int thr_stride = 0;   /* cascade: threshold of stream s = thr_prob[s * thr_stride] instead */
    nnsp_b200_taps taps{};
    /* cascade rounds (null in the batched path): per stream, the first inference frame of this round (inference k of
     * stream s is frame tstart[s] + 2k, it has (T - tstart[s] + 1) / 2 of them), the frame at which the live instance's
     * life in this call began (earlier frames of its window come from the stored context), the instance's age (frames
     * since its reset, capped at 2) at that frame, and the log-mel rows of the instance's first two frames, whose STFT
     * buffer is still partly zero (spectrogram_module.c:25-31) */
    const int *tstart = nullptr, *tb = nullptr, *age0 = nullptr;
    const int32_t *lmfix = nullptr;      /* [S][2][40] */
    /* cascade, first round: scratch for the streams' standardised window rows, [S][vseq_rows][40] (vseq_kernel); with it
     * layer 0 runs on the tcgen05 kernel. Null: seg_kernel<2> standardises while staging (later rounds, few streams) */
    int16_t *vseq = nullptr; int vseq_rows = 0;
    /* ragged cascade call (null otherwise): stream s ends at frame stream_frames(nfr, s, T), so a row of a round has
     * (Ts - tstart[s] + 1) / 2 inferences */
    const int32_t *nfr = nullptr;
};
int launch_split_layers(const MmaDeviceModel &mm, const SplitGroup &q, int device, cudaStream_t st);
int split_supported(const MmaDeviceModel &mm);
size_t split_plane_bytes(const MmaDeviceModel &mm, int n_streams, int n_inf);
int launch_nn_split(const MmaDeviceModel &mm, const NNLaunch &l, const int16_t *feat16, int first, int n_inf,
                    uint8_t *planes0, uint8_t *planes1, int32_t *dec, int cap_inf, int device, cudaStream_t st);

}  // namespace nnsp
