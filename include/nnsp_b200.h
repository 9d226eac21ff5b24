/*
 * nnsp_b200.h -- C ABI of libnnsp_b200.so: the ns-nnsp streaming-inference hot path
 * (FeatureClass -> NeuralNetClass -> NNSPClass post-processing, and the VAD->KWS->S2I
 * cascade of nnCntrlClass) batched over thousands of independent 16 kHz streams on one
 * NVIDIA B200 (sm_100a).
 *
 * Plain C types only. All device work runs in hand-written CUDA kernels; there is NO CPU
 * fallback: every entry point that computes returns NNSP_B200_ERR_CUDA when no usable
 * device is present.
 *
 * What each entry point replaces in the reference (AmbiqAI/nnsp, file:line):
 *   nnsp_b200_model_from_net ........ reading a linked model table, e.g. evb/src/def_nn1_vad.c:8-110
 *                                     (mean/stdR arrays + the `NeuralNetClass net_*` literal)
 *   nnsp_b200_model_from_table_text . compiling + linking a generated table file, python/c_code_table_converter.py:143-347
 *   nnsp_b200_batch_create .......... NNSPClass_init            ns-nnsp/src/nn_speech.c:23-55
 *                                     (+ FeatureClass_construct  ns-nnsp/src/feature_module.c:12-24)
 *   nnsp_b200_batch_reset ........... NNSPClass_reset           ns-nnsp/src/nn_speech.c:57-72
 *   nnsp_b200_batch_exec[_host] ..... NNSPClass_exec            ns-nnsp/src/nn_speech.c:74-127
 *                                     called n_frames times for each of n_streams instances
 *   nnsp_b200_cascade_create ........ nnCntrlClass_init         evb/src/nnCntrlClass.c:56-128
 *   nnsp_b200_cascade_reset ......... nnCntrlClass_reset        evb/src/nnCntrlClass.c:130-150
 *   nnsp_b200_cascade_exec[_host] ... nnCntrlClass_exec         evb/src/nnCntrlClass.c:152-272
 *   nnsp_b200_cascade_exec_*ragged* . the same, called a different number of times on each instance
 *   nnsp_b200_ingest_audadc ......... audio_frame_callback      evb/src/main_nnsp.cc:58-65 (mask + glitch fix)
 *   nnsp_b200_feature_stages ........ stftModule_analyze/spec2pspec/melSpecProc/log10_vec
 *                                     ns-nnsp/src/spectrogram_module.c:33-77, melSpecProc.c:6-27,
 *                                     fixlog10.c:53-61 (debug tap of every intermediate)
 * The nine legacy single-instance symbols themselves (NNSPClass_*, FeatureClass_*,
 * NeuralNetClass_*) are also exported, see include/nnsp_compat/nnsp_legacy_api.h.
 */
#ifndef NNSP_B200_H
#define NNSP_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define NNSP_B200_OK             0
#define NNSP_B200_ERR_ARG       (-1)   /* bad argument / malformed model            */
#define NNSP_B200_ERR_CUDA      (-2)   /* CUDA runtime failure or no device         */
#define NNSP_B200_ERR_NOMEM     (-3)
#define NNSP_B200_ERR_UNSUPPORTED (-4) /* model shape outside the engine's limits   */

#define NNSP_B200_FRAME          160   /* samples per hop  (ambiq_nnsp_const.h:5)   */
#define NNSP_B200_NMEL           40    /* mel bands        (ambiq_nnsp_const.h:6)   */
#define NNSP_B200_NCTX           6     /* context frames   (ambiq_nnsp_const.h:7)   */
#define NNSP_B200_MAX_LAYERS     10    /* neural_nets.h:18-30                       */
#define NNSP_B200_MAX_WIDTH      128   /* widest hidden layer / LSTM state the kernels support */
#define NNSP_B200_MAX_OUT        128   /* widest final layer                        */

/* post-processing flavour, keyed like NNSP_ID (nnsp_identification.h:3-9) */
#define NNSP_B200_ID_S2I         0
#define NNSP_B200_ID_VAD         1
#define NNSP_B200_ID_KWS         2

const char *nnsp_b200_version(void);
const char *nnsp_b200_strerror(int code);
/* text of the last error raised on the calling thread ("" if none) */
const char *nnsp_b200_last_error(void);
/* number of CUDA kernels launched by this library since load (all handles) */
long long nnsp_b200_kernel_launches(void);
/* how many of them were the tcgen05 (5th-generation tensor core) layer-0 kernel of the batched network path */
long long nnsp_b200_tc5_launches(void);
/* how many of them were the cascade's per-stream network kernels, by kind: 0 the sequential kernel in its narrow shape
 * (every layer at most 80 wide, LSTM state at most 80, at most 48 outputs), 1 the sequential kernel in its wide shape,
 * 2 the two-warps-per-stream replay kernel behind the stage-sorted rounds (-1 for any other kind). Launches, not work:
 * after the stage-sorted rounds the replay (kind 2, or kind 0 / 1 when the replay kernel is not used) is launched once
 * per call and returns at once when no stream is left for it. */
long long nnsp_b200_cascade_kernel_launches(int kind);
/* how many of them were the LSTM scan kernel of the split network path (batched NNSPClass, net_eval, the cascade's
 * stage-sorted rounds), by specialisation (unit groups NT, CTAs per SM, k-steps compiled in, 0 = read at run time), in
 * the order the dispatch tries them: 0 <4,4,1>, 1 <4,4,0>, 2 <8,2,2>, 3 <9,2,3>, 4 <9,2,0>, 5 <16,1,0> (-1 for any other
 * kind). Which one runs depends only on the LSTM layer's shape, so a test can tell which code path evaluated a model. */
long long nnsp_b200_scan_kernel_launches(int kind);

/* ------------------------------------------------------------------------------------ */
/* Models                                                                               */
/* ------------------------------------------------------------------------------------ */
typedef struct nnsp_b200_model nnsp_b200_model;

/* Read a live reference model table (`NeuralNetClass`, ARM 4-row weight interleave as
 * written by python/nnsp_pack/c_weight_man.py) plus its normalisation stats.
 * Accumulator width per layer is taken from layer_func[] (== &fc_8x16_acc32b etc.). */
int nnsp_b200_model_from_net(const void *neural_net_class, const int32_t *feature_mean,
                             const int32_t *feature_stdR, int nn_id, nnsp_b200_model **out);
/* The reference's on-disk model format: the generated C source `evb/src/def_nn{id}_{name}.c`
 * (python/c_code_table_converter.py:143-347; weight layout python/nnsp_pack/c_weight_man.py:5-124), parsed as
 * text -- no C compiler involved. nn_id < 0: inferred from the table name (s2i / vad / kws*). acc32: 1 selects
 * the `#ifdef DEF_ACC32BIT_OPT` branch (wrapping 32-bit accumulators), 0 the 64-bit one, -1 = 0.
 * model_to_table_text writes the same text back (call with buf = NULL to get the size). */
int nnsp_b200_model_from_table_text(const char *text, size_t nbytes, int nn_id, int acc32, nnsp_b200_model **out);
int nnsp_b200_model_to_table_text(const nnsp_b200_model *m, const char *nn_name, char *buf, size_t cap, size_t *nbytes);
/* Same model from / to the flat little-endian container described in DESIGN.md ("NNSPM1"). */
int nnsp_b200_model_from_blob(const void *blob, size_t nbytes, nnsp_b200_model **out);
int nnsp_b200_model_to_blob(const nnsp_b200_model *m, void *buf, size_t cap, size_t *nbytes);
/* Force accumulator semantics: 0 = 64-bit saturating (affine.c), 1 = wrapping 32-bit
 * (affine_acc32b.c, what -DDEF_ACC32BIT_OPT selects in def_nn*.c:68-84). */
int nnsp_b200_model_set_acc32(nnsp_b200_model *m, int acc32);
int nnsp_b200_model_info(const nnsp_b200_model *m, int *nn_id, int *numlayers,
                         int16_t size_layer[NNSP_B200_MAX_LAYERS + 1], int *acc32);
void nnsp_b200_model_free(nnsp_b200_model *m);

/* ------------------------------------------------------------------------------------ */
/* Per-stream-frame result record                                                       */
/* ------------------------------------------------------------------------------------ */
typedef struct {
    int16_t trigger;      /* return value of NNSPClass_exec for this frame (nn_speech.c:126) */
    int16_t outputs[3];   /* NNSPClass.outputs after this frame: intent, slot0, slot1        */
} nnsp_b200_result;       /* 8 bytes */

/* Optional debug taps (device pointers, any may be NULL). Index [s][t] = stream s, frame t
 * of the current exec call; rows are dense, stream-major. Frames on which the network did
 * not run (NNSPClass.slides == 0) get zero-filled act/logits rows.                      */
typedef struct {
    int32_t *logmel;      /* [S][T][40]  FeatureClass.feature after log10_vec            */
    int16_t *feat;        /* [S][T][40]  newest normFeatContext row                      */
    int16_t *act;         /* [S][T][act_stride] outputs of layers 0..L-2 back to back    */
    int32_t *logits;      /* [S][T][n_out]  final linear layer (Q15)                     */
    int16_t *hstate;      /* [S][T][h_stride] LSTM h after the frame (all LSTM layers)   */
    int32_t *cstate;      /* [S][T][h_stride] LSTM c after the frame                     */
    int16_t *post;        /* [S][T][16]: trigger, outputs[3], counts_category[8],
                                         argmax_last, slides(after), ran_nn, stage      */
} nnsp_b200_taps;

/* ------------------------------------------------------------------------------------ */
/* Batched NNSPClass: n_streams independent instances of one model                      */
/* ------------------------------------------------------------------------------------ */
typedef struct nnsp_b200_batch nnsp_b200_batch;

int nnsp_b200_batch_create(const nnsp_b200_model *m, int n_streams, int device,
                           int16_t thresh_prob, int16_t th_count_trigger,
                           nnsp_b200_batch **out);
int nnsp_b200_batch_reset(nnsp_b200_batch *b);
/* Advance every stream by n_frames hops.
 *   pcm      device pointer; sample i of frame t of stream s at pcm[s*stream_stride + t*160 + i]
 *   results  device pointer [n_streams][n_frames] (may be NULL)
 * Asynchronous: the call returns once the work is queued. On the default network path consecutive calls are
 * pipelined over two CUDA streams (front end of call N+1 while the network kernels of call N finish), so results
 * and state are complete only after nnsp_b200_batch_sync.
 * Ownership: `pcm_dev` and `results_dev` belong to the library from the call until nnsp_b200_batch_sync returns.
 * The engine's streams are non-blocking, so a refill through cudaMemcpy / nnsp_b200_memcpy_h2d (legacy stream) or
 * through a stream of the caller is NOT ordered against them. The one exception: work the caller enqueues on
 * nnsp_b200_batch_stream() AFTER the next exec call has been issued is ordered behind every reader of this call's
 * PCM (the feature and history kernels run on that stream); a serving loop that wants no sync therefore rotates
 * three PCM buffers and fills buffer k+1 on that stream.                                   */
int nnsp_b200_batch_exec(nnsp_b200_batch *b, const int16_t *pcm_dev, long long stream_stride,
                         int n_frames, nnsp_b200_result *results_dev,
                         const nnsp_b200_taps *taps);
/* Same with HOST buffers (pageable or pinned): H2D of the PCM, kernels, D2H of the results,
 * pipelined over stream slices; returns after the results are in `results`.             */
int nnsp_b200_batch_exec_host(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride,
                              int n_frames, nnsp_b200_result *results);
/* The same call without the wait at its end: it returns once the copies and kernels are queued and hands back a
 * ticket (1, 2, ...). `pcm` and `results` (pinned host memory, or the copies degrade to synchronous ones) belong
 * to the library until nnsp_b200_batch_wait_host(ticket) -- or any later ticket, or nnsp_b200_batch_sync --
 * returns. Calls complete in order; with two PCM/result buffer pairs a server keeps one call in flight while it
 * consumes the previous one, and the host link never idles between calls.                */
int nnsp_b200_batch_exec_host_async(nnsp_b200_batch *b, const int16_t *pcm, long long stream_stride,
                                    int n_frames, nnsp_b200_result *results, long long *ticket);
int nnsp_b200_batch_wait_host(nnsp_b200_batch *b, long long ticket);
int nnsp_b200_batch_sync(nnsp_b200_batch *b);
/* Device time (ms) spent in the kernels of the most recent exec call, per kernel:
 * [0] feature kernel, [1] network/post-processing kernel, [2] everything else.          */
int nnsp_b200_batch_last_kernel_ms(nnsp_b200_batch *b, float ms[3]);
int nnsp_b200_batch_dims(const nnsp_b200_batch *b, int *n_streams, int *act_stride,
                         int *h_stride, int *n_out);
/* Which network kernels run: 0 = automatic (3 when the model fits it, else 2, else 1), 1 = dp2a warp-per-stream
 * kernel, 2 = tensor-core IMMA kernel with the whole network inside the time loop, 3 = scan-split (fc layers
 * for all frames of the call at once, only the LSTM recurrence sequential; nnsp_split.cu). 2 and 3 return an
 * error when the model does not fit them. All three are bit-exact. */
int nnsp_b200_batch_set_nn_path(nnsp_b200_batch *b, int path);
/* the path the next call will take (1, 2 or 3): what `automatic` resolved to for this model */
int nnsp_b200_batch_get_nn_path(const nnsp_b200_batch *b);
/* CUDA stream the front end is launched on (cudaStream_t as void*), for callers that time it; the network
 * kernels of the default path run on a second, internal stream -- bracket timed regions with nnsp_b200_batch_sync. */
void *nnsp_b200_batch_stream(nnsp_b200_batch *b);
void nnsp_b200_batch_destroy(nnsp_b200_batch *b);

/* ------------------------------------------------------------------------------------ */
/* Batched nnCntrlClass: VAD -> KWS -> S2I gated cascade per stream                     */
/* ------------------------------------------------------------------------------------ */
typedef struct {
    int16_t thresh_prob_vad,  thresh_cnts_vad;                         /* ParamsNNCntrl.h:8-9   */
    int16_t frs_vbufBk_s2i,   thresh_timeout_s2i, thresh_prob_s2i, thresh_cnts_s2i; /* :12-15 */
    int16_t frs_vbufBk_kws,   thresh_timeout_kws, thresh_prob_kws, thresh_cnts_kws; /* :18-21 */
} nnsp_b200_cascade_params;   /* same fields, same order as ParamCntrlClass (nnCntrlClass.h:12-29) */

typedef struct {
    int8_t  stage_id;     /* NNSP id that executed this frame (seq[current_pos_seq] on entry) */
    int8_t  pos_after;    /* current_pos_seq on return                                     */
    int16_t detected;     /* NNSPClass_exec return value for the instance that ran         */
    int16_t outputs[3];   /* that instance's outputs[] right after exec (before any reset)  */
    uint16_t cnt_timeout; /* cnt_timeout_kws / _s2i on return (0 for VAD frames)            */
} nnsp_b200_cascade_result;   /* 12 bytes */

typedef struct nnsp_b200_cascade nnsp_b200_cascade;

void nnsp_b200_cascade_default_params(nnsp_b200_cascade_params *p);
/* models[id] indexed by NNSP id (0 s2i, 1 vad, 2 kws); seq = ids in cascade order,
 * e.g. {1,2,0} (evb/src/main_nnsp.cc:109). */
int nnsp_b200_cascade_create(const nnsp_b200_model *const models[3], const int *seq, int len_seq,
                             const nnsp_b200_cascade_params *params, int n_streams, int device,
                             nnsp_b200_cascade **out);
int nnsp_b200_cascade_reset(nnsp_b200_cascade *c);
/* Reset individual streams of a live handle, e.g. to hand a server slot to a new caller without touching the others.
 *   NNSP_B200_RESET_INSTANCE: nnCntrlClass_reset (nnCntrlClass.c:130-150) of that stream's controller, what
 *     nnsp_b200_cascade_reset does to every stream: PCM ring and log-mel history cleared, every instance reset, time-out
 *     counters zeroed; the stage position and context row 5 of every instance are kept (DESIGN.md section 2, quirks 2, 3).
 *   NNSP_B200_RESET_FRESH: nnCntrlClass_init + reset, the state nnsp_b200_cascade_create leaves.
 * `streams` is host memory, copied before the call returns. An id outside [0, n_streams), n < 0 or an unknown mode returns
 * NNSP_B200_ERR_ARG and records nothing; n == 0 does nothing. The call does not wait for the device: the listed streams
 * start the NEXT exec call of any kind (device, ragged, host, host-async, tapped) from the reset state. Calls issued
 * before it keep their results and the state they leave; a reset issued between two asynchronous host tickets affects
 * only the second. Resets compose in call order: a stream listed twice before a call is reset FRESH if either listing
 * was FRESH, and nnsp_b200_cascade_reset issued while resets are pending leaves what it would leave had they come first.
 * Per-stream parameters (nnsp_b200_cascade_set_stream_params) are configuration and survive both modes. A reset stream
 * given n_frames[s] == 0 in a ragged call stays in its reset state. A call with no pending reset launches and copies
 * exactly what it would without this function and never waits for the device. A call with some uploads the list and
 * resets those streams on the device before its kernels read them; before it reuses the list's staging buffer it waits
 * on the host until the device has run the list copies of the reset-carrying call before last, which are queued behind
 * the work issued before them on their stream (pipelined device calls: the chain two calls back; host calls: the same
 * slice of the previous ticket). A caller that resets before every call thus runs at most about two calls ahead of the
 * device. */
#define NNSP_B200_RESET_INSTANCE 0
#define NNSP_B200_RESET_FRESH    1
int nnsp_b200_cascade_reset_streams(nnsp_b200_cascade *c, const int32_t *streams, int n, int mode);
/* ParamCntrlClass belongs to a controller instance (nnCntrlClass.h:12-29), i.e. to a stream: params[i] becomes the
 * parameter set of stream first_stream + i (thresholds, counts, time-outs; the two look-back depths must equal the
 * handle's, they size its history buffers). Waits for the handle's work in flight; takes effect with the next call and
 * survives nnsp_b200_cascade_reset, like the reference's params pointer survives nnCntrlClass_reset. */
int nnsp_b200_cascade_set_stream_params(nnsp_b200_cascade *c, int first_stream, int n_streams,
                                        const nnsp_b200_cascade_params *params);
/* Asynchronous and pipelined like nnsp_b200_batch_exec: results, state and the PCM buffer of a call are settled
 * only after nnsp_b200_cascade_sync -- the kernels that handle the first frames after a stage change read the call's
 * PCM on an internal stream while the next call's front end already runs, so there is NO stream of the caller's on
 * which a refill of that buffer would be ordered. Rotate buffers and sync before reusing one. */
int nnsp_b200_cascade_exec(nnsp_b200_cascade *c, const int16_t *pcm_dev, long long stream_stride,
                           int n_frames, nnsp_b200_cascade_result *results_dev,
                           const nnsp_b200_taps *taps);
int nnsp_b200_cascade_exec_host(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride,
                                int n_frames, nnsp_b200_cascade_result *results);
/* asynchronous twin of the host-buffer call: see nnsp_b200_batch_exec_host_async */
int nnsp_b200_cascade_exec_host_async(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride,
                                      int n_frames, nnsp_b200_cascade_result *results, long long *ticket);
/* Ragged calls: stream s advances by n_frames[s] frames (0 <= n_frames[s] <= max_frames), exactly as if nnCntrlClass_exec
 * had been called n_frames[s] times on its instance -- a server passes what each stream has buffered, 0 for an idle slot.
 * PCM layout as nnsp_b200_cascade_exec with T = max_frames; no sample of a frame t >= n_frames[s] is used. Records
 * and tap rows of frames t >= n_frames[s] are written as "no frame": stage_id = -1 and every other field 0 (taps: zero
 * rows). A stream with n_frames[s] == 0 keeps its whole state (counters, time-outs, PCM and log-mel history).
 *   exec_ragged: n_frames_dev is a device array of n_streams counts, owned and pipelined like pcm_dev; values outside
 *     [0, max_frames] are clamped on the device. No sample of a frame t >= n_frames[s] is read. A call whose counts all
 *     equal max_frames is nnsp_b200_cascade_exec: same bytes, the same sequence of kernel launches.
 *   exec_host_ragged_async: n_frames is host memory (same lifetime rules as pcm); a value outside [0, max_frames] returns
 *     NNSP_B200_ERR_ARG before anything is queued. Follows nnsp_b200_cascade_set_host_format, slices and pipelines like
 *     nnsp_b200_cascade_exec_host_async and completes in ticket order (nnsp_b200_cascade_wait_host). Like the uniform
 *     call it copies every stream's max_frames frames (and conditions them, for AUDADC words); only the feature and
 *     history kernels read PCM, and they read none past a stream's count. */
int nnsp_b200_cascade_exec_ragged(nnsp_b200_cascade *c, const int16_t *pcm_dev, long long stream_stride, int max_frames,
                                  const int32_t *n_frames_dev, nnsp_b200_cascade_result *results_dev,
                                  const nnsp_b200_taps *taps);
int nnsp_b200_cascade_exec_host_ragged_async(nnsp_b200_cascade *c, const int16_t *pcm, long long stream_stride,
                                             int max_frames, const int32_t *n_frames, nnsp_b200_cascade_result *results,
                                             long long *ticket);
int nnsp_b200_cascade_wait_host(nnsp_b200_cascade *c, long long ticket);
int nnsp_b200_cascade_sync(nnsp_b200_cascade *c);
int nnsp_b200_cascade_last_kernel_ms(nnsp_b200_cascade *c, float ms[3]);
/* Device timeline of the last n <= 8 device-buffer calls, oldest first: ms[4 k + 0..3] = front end (feature kernel)
 * starts / done, controller-and-network chain starts / done, in ms after the oldest call's front end started (CUDA events
 * on the handle's own streams). Synchronises the handle. */
int nnsp_b200_cascade_timeline(nnsp_b200_cascade *c, float *ms, int *n_calls);
void *nnsp_b200_cascade_stream(nnsp_b200_cascade *c);
/* 0 = automatic, 1 = sequential warp-per-stream kernel only, 2 = stage-sorted pass (the scan-split network kernels
 * over the streams of each (model, phase) group) + replay of the frames after a stage change. Bit-exact either way;
 * calls that request debug taps always take 1. */
int nnsp_b200_cascade_set_path(nnsp_b200_cascade *c, int path);
void nnsp_b200_cascade_destroy(nnsp_b200_cascade *c);

/* ------------------------------------------------------------------------------------ */
/* Several GPUs of one box behind one handle                                            */
/* ------------------------------------------------------------------------------------ */
/* The streams are independent (no reference function looks at another instance: nn_speech.c:74-127,
 * evb/src/nnCntrlClass.c:152-272), so a group block-partitions them over `n_devices` devices -- member k owns streams
 * [S k / G, S (k + 1) / G) -- with one host thread per device and no inter-GPU traffic. A member is an ordinary
 * nnsp_b200_batch / nnsp_b200_cascade handle; `devices` may name a device more than once (two members, two threads).
 * exec_host takes HOST buffers laid out like the single-device calls: pcm[s * stream_stride + t * 160 + i], results
 * [n_streams][n_frames] records (nnsp_b200_result for a batch group, nnsp_b200_cascade_result for a cascade group).
 * The asynchronous form returns a ticket; buffers belong to the library until nnsp_b200_group_wait(ticket) (or a later
 * one) returns. Calls complete in order; with two buffer pairs every device keeps its host link busy across calls. */
typedef struct nnsp_b200_group nnsp_b200_group;
int nnsp_b200_group_create_batch(const nnsp_b200_model *m, int n_streams, const int *devices, int n_devices,
                                 int16_t thresh_prob, int16_t th_count_trigger, nnsp_b200_group **out);
int nnsp_b200_group_create_cascade(const nnsp_b200_model *const models[3], const int *seq, int len_seq,
                                   const nnsp_b200_cascade_params *params, int n_streams, const int *devices,
                                   int n_devices, nnsp_b200_group **out);
int nnsp_b200_group_size(const nnsp_b200_group *g);
int nnsp_b200_group_range(const nnsp_b200_group *g, int member, int *device, int *first_stream, int *n_streams);
int nnsp_b200_group_reset(nnsp_b200_group *g);
/* nnsp_b200_cascade_set_stream_params in the group's stream numbering (cascade groups); waits for the calls issued so far */
int nnsp_b200_group_set_stream_params(nnsp_b200_group *g, int first_stream, int n_streams, const nnsp_b200_cascade_params *params);
/* nnsp_b200_cascade_reset_streams in the group's stream numbering (cascade groups; a batch group returns
 * NNSP_B200_ERR_ARG). Checked and copied before it returns, queued in order with the group's calls in each member's
 * command queue: the listed streams start the next call issued after it from the reset state. Does not wait. */
int nnsp_b200_group_reset_streams(nnsp_b200_group *g, const int32_t *streams, int n, int mode);
int nnsp_b200_group_exec_host(nnsp_b200_group *g, const int16_t *pcm, long long stream_stride, int n_frames, void *results);
int nnsp_b200_group_exec_host_async(nnsp_b200_group *g, const int16_t *pcm, long long stream_stride, int n_frames,
                                    void *results, long long *ticket);
int nnsp_b200_group_wait(nnsp_b200_group *g, long long ticket);
void nnsp_b200_group_destroy(nnsp_b200_group *g);

/* ------------------------------------------------------------------------------------ */
/* Stage-by-stage tap of the feature front end (parity tool)                            */
/* ------------------------------------------------------------------------------------ */
/* For n windows of 480 int16 samples each (host pointers), computes on `device`:
 *   fft_in [n][512] int32   windowed, zero-padded frame      spectrogram_module.c:62-71
 *   spec   [n][514] int32   257 complex bins, re/im pairs    fft.c:27-126
 *   pspec  [n][257] int32   power spectrum                   spectrogram_module.c:33-45
 *   mel    [n][40]  int32   mel energies                     melSpecProc.c:6-27
 *   logmel [n][40]  int32   log10 Q15                        fixlog10.c:53-61
 * Any output pointer may be NULL. */
int nnsp_b200_feature_stages(int device, const int16_t *windows, int n, int32_t *fft_in,
                             int32_t *spec, int32_t *pspec, int32_t *mel, int32_t *logmel);

/* ------------------------------------------------------------------------------------ */
/* One network evaluation on explicit inputs (parity tool)                              */
/* ------------------------------------------------------------------------------------ */
/* NeuralNetClass_exe(net, input, output, -1) (ns-nnsp/src/neural_nets.c:44-168) for n independent evaluations on the
 * network kernels of `nn_path` (0 automatic, 1 dp2a, 2 IMMA in the time loop, 3 scan-split; see
 * nnsp_b200_batch_set_nn_path), no front end involved. Host pointers:
 *   x      [n][240] int16   the 6 x 40 context the network reads (normFeatContext)
 *   h0, c0 [n][h_stride]    LSTM state of all lstm layers back to back before the evaluation (NULL = zeros)
 *   act    [n][act_stride]  outputs of layers 0..L-2 back to back          (may be NULL)
 *   logits [n][n_out]       final layer (int32; int16 values when it is not linear, neural_nets.c:152-167)
 *   h1, c1 [n][h_stride]    LSTM state after the evaluation                (may be NULL)
 * act_stride / h_stride / n_out as reported by nnsp_b200_batch_dims. This is how adversarial inputs and states
 * (full-scale x, saturated c, wrap-around under ACC32BIT_OPT) reach every CUDA network path. */
int nnsp_b200_net_eval(const nnsp_b200_model *m, int device, int nn_path, int n, const int16_t *x,
                       const int16_t *h0, const int32_t *c0, int16_t *act, int32_t *logits,
                       int16_t *h1, int32_t *c1);

/* ------------------------------------------------------------------------------------ */
/* Ingest: the application's PCM conditioning in front of the path                      */
/* ------------------------------------------------------------------------------------ */
/* evb/src/main_nnsp.cc:58-65 (audio_frame_callback): raw AUDADC words -> int16 PCM, `raw & 0x0000FFF0`, and
 * sample 3 of each 160-sample frame := (sample 2 + sample 4) >> 1. raw_dev: n_frames*160 uint32 (device),
 * pcm_dev: n_frames*160 int16 (device), both 16-byte aligned; frames are consecutive in both, so any
 * [stream][frame] arrangement works. Asynchronous on `stream` (a handle's stream or NULL). */
int nnsp_b200_ingest_audadc(int device, const uint32_t *raw_dev, int16_t *pcm_dev, long long n_frames, void *stream);
/* The same conditioning chained in front of the HOST-buffer calls of a handle: with NNSP_B200_HOST_AUDADC the `pcm`
 * argument of *_exec_host / *_exec_host_async is read as `const uint32_t *` raw AUDADC words (same indexing,
 * stream_stride still in samples); they cross the link as they are and are conditioned on the device, slice by slice,
 * right before the feature kernel. Switching the format waits for the handle's work in flight. */
#define NNSP_B200_HOST_PCM16     0
#define NNSP_B200_HOST_AUDADC    1
int nnsp_b200_batch_set_host_format(nnsp_b200_batch *b, int format);
int nnsp_b200_cascade_set_host_format(nnsp_b200_cascade *c, int format);

/* ------------------------------------------------------------------------------------ */
/* Audio front door: RIFF/WAVE files -> the [stream][frame][160] PCM layout (host code)  */
/* ------------------------------------------------------------------------------------ */
/* Stands where the reference has the AUDADC interrupt (evb/src/main_nnsp.cc:46-74) and, off the device, the Python tools
 * reading python/test_wavs with soundfile (python/test_s2i.py etc.): 16 kHz, 16-bit integer PCM, any channel count (one
 * channel is picked), chunks in any order, WAVE_FORMAT_EXTENSIBLE accepted. Other rates are NNSP_B200_ERR_UNSUPPORTED
 * (the reference has no resampler). Frames past the end of a file are digital silence; frames_read tells how many held
 * file samples. load_streams fills stream s of a host buffer (pcm[s * stream_stride + t * 160 + i]) from paths[s]. */
int nnsp_b200_wav_info(const char *path, int *sample_rate, int *channels, int *bits, long long *n_samples);
int nnsp_b200_wav_read_frames(const char *path, int channel, long long first_frame, int n_frames, int16_t *pcm, int *frames_read);
int nnsp_b200_wav_load_streams(const char *const *paths, int n_streams, int channel, long long first_frame, int n_frames,
                               int16_t *pcm, long long stream_stride, int *frames_read);

/* Constant tables the engine generates at load time (host copies; see nnsp_tables.c).
 * name: "stft_win" int16[480], "fft_tw" int32[256], "rfft_tw" int32[256], "bitrev" int16[256],
 *       "mel" int16[534], "log_lut" int16[256], "tanh_lut" int16[384].
 * Returns element count or a negative error. */
int nnsp_b200_table(const char *name, const void **data, int *elem_bytes);

/* CUDA-event timing on a handle's stream (so callers can time exactly what the engine runs,
 * on the stream it runs on, without CUDA headers). stream = nnsp_b200_*_stream() or NULL. */
int nnsp_b200_event_create(int device, void **event);
int nnsp_b200_event_record(void *event, void *stream);
int nnsp_b200_event_elapsed_ms(void *start, void *stop, float *ms);   /* synchronises on `stop` */
int nnsp_b200_event_destroy(void *event);
/* Self-measured integer-pipe peaks of the device, in giga warp-lane instructions per second, from
 * register-resident dependent chains (8 per thread): gops[0] IMAD, gops[1] IMAD + ALU interleaved 1:1
 * (both pipes), gops[2] IMAD.WIDE, gops[3] IDP.2A. MEASURED_PEAKS.json has no integer figure, so the
 * int-ALU roofline of bench.py uses gops[1]. */
int nnsp_b200_int_peak(int device, double gops[4]);

/* Device utilities so that C callers need no CUDA headers. */
int nnsp_b200_device_count(void);
/* PCI bus id ("0000:1b:00.0") of CUDA device `device`: the key by which NVML / nvidia-smi name the same GPU whatever
 * CUDA_VISIBLE_DEVICES says */
int nnsp_b200_device_pci_bus_id(int device, char *buf, int len);
int nnsp_b200_dev_alloc(int device, size_t nbytes, void **ptr);
int nnsp_b200_dev_free(int device, void *ptr);
int nnsp_b200_host_alloc_pinned(size_t nbytes, void **ptr);
int nnsp_b200_host_free_pinned(void *ptr);
int nnsp_b200_memcpy_h2d(int device, void *dst, const void *src, size_t nbytes);
int nnsp_b200_memcpy_d2h(int device, void *dst, const void *src, size_t nbytes);
int nnsp_b200_memset(int device, void *dst, int value, size_t nbytes);

#ifdef __cplusplus
}
#endif
#endif /* NNSP_B200_H */
