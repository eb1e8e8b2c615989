/*
 * owwb200.h - C ABI of libowwb200.so: the B200 (sm_100a) replacement for the three
 * inference sessions on openWakeWord's streaming hot path, plus the device-resident
 * stream state that sits between them.
 *
 * What each entry point replaces in the reference (paths under /root/reference/):
 *   oww_melspectrogram   -> AudioFeatures.melspec_model_predict   openwakeword/utils.py:84-87,202
 *                           (melspectrogram.onnx; graph spec notebooks/converting_google_speech_embedding_model.ipynb:426-477)
 *   oww_embed_windows    -> AudioFeatures.embedding_model_predict openwakeword/utils.py:90-93,235,443
 *                           (embedding_model.onnx; graph spec same notebook :871-951)
 *   oww_head_predict     -> Model.model_prediction_function[name] openwakeword/model.py:137-138,158-159
 *                           (<head>.onnx; family openwakeword/train.py:56-83,144-165)
 *   oww_set_streams / oww_reset / oww_step / oww_step_host
 *                        -> AudioFeatures buffers + _streaming_features + the per-head window reads of
 *                           Model.predict                         openwakeword/utils.py:163-178,387-460; model.py:282-302
 *   oww_embed_clips      -> AudioFeatures.embed_clips             openwakeword/utils.py:358-385
 *   oww_predict_clips    -> Model.predict_clip over many clips (bulk_predict's inner loop)
 *                                                                 openwakeword/model.py:388-426; utils.py:467-539
 *   oww_get_features / oww_get_mel
 *                        -> AudioFeatures.get_features / .melspectrogram_buffer   openwakeword/utils.py:454-460,165
 *
 * Conventions: every function returns 0 (OWW_OK) or a negative code; oww_last_error() gives the
 * message of the last failure on that handle (or, with NULL, of the last failed oww_create).
 * No exceptions cross the boundary.  Pointers named d_* are CUDA device addresses on the handle's
 * device (e.g. torch.Tensor.data_ptr()); h_* are host addresses.  `stream` is a cudaStream_t
 * passed as void* (NULL = the legacy default stream); all device work of a call is enqueued on it
 * and the call does not synchronise unless stated.  The caller owns every buffer it passes; the
 * library owns weights, rings and scratch inside the handle.  A handle is single-producer: one
 * host thread at a time.
 */
#ifndef OWWB200_H
#define OWWB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OWW_OK            0
#define OWW_EINVAL      (-1)   /* bad argument / wrong call order            */
#define OWW_ECUDA       (-2)   /* a CUDA runtime call failed                 */
#define OWW_ENOMEM      (-3)   /* host or device allocation failed           */
#define OWW_EUNSUPPORTED (-4)  /* graph shape outside what the kernels cover */

#define OWW_SAMPLES_PER_CHUNK 1280   /* 80 ms @ 16 kHz                         */
#define OWW_MEL_BINS            32
#define OWW_WINDOW_ROWS         76   /* mel rows per embedding window          */
#define OWW_EMBEDDING_DIM       96
#define OWW_INIT_FEATURE_ROWS   41   /* rows AudioFeatures seeds the ring with */
#define OWW_MAX_HEAD_FRAMES    120   /* rows AudioFeatures keeps (utils.py:170): the widest head window */
#define OWW_MAX_HEAD_LAYERS      8

/* embedding-CNN execution modes */
#define OWW_CNN_FP32_WINDOW       0  /* CUDA-core fp32, full 76-row window per frame (reference-shaped)  */
#define OWW_CNN_TC_WINDOW         2  /* tcgen05 fp16-operand/fp32-accumulate implicit GEMM, full window  */
#define OWW_CNN_TC_INCREMENTAL    3  /* tcgen05, fused 20-layer kernel on the 8 new mel rows per stream
                                        (per-stream activation tails in HBM); first step after a reset and
                                        the stateless/batch calls use the full-window tcgen05 kernels      */

typedef struct oww_ctx oww_ctx;

typedef struct oww_config {
    int32_t device;        /* CUDA device ordinal                                               */
    int32_t max_chunks;    /* largest n_chunks a single oww_step may carry (>=1)                */
    int32_t cnn_mode;      /* OWW_CNN_*                                                         */
    int32_t window_batch;  /* windows per CNN sub-batch in the window modes (0 = default)       */
    int32_t reserved[4];   /* reserved[0] bit 0: 1 = keep mode 3's steady-state step as separate launches
                              (mel, CNN, append, heads) instead of the single fused step kernel;
                              bit 1: 1 = heads on CUDA cores (heads.cu) even in the tensor-core modes;
                              bit 2: 1 = tensor-core heads with plain fp16 operands (1 MMA term instead of the
                              fp32-grade 3-term hi/lo split);
                              bit 3: 1 = one tensor-core heads CTA per (128 streams, head) reading the fp32 rings
                              (heads_tc.cu) instead of one CTA per 128 streams for all heads that share a window,
                              fed from the fp16 mirror of the rings (heads_grp.cu);
                              bit 4: 1 = the incremental late (3,1) layers keep the window-mode tensor layout
                              (per-stream [tails | new rows] x (W+1): most accumulator rows of a tile are not outputs)
                              instead of the block-major layout of tc_conv_blk_kernel;
                              bit 5: 1 = no programmatic dependent launches inside the late chain.
                              reserved[1]: first conv layer that takes fp16 hi/lo split operands in the
                              tensor-core modes, 2..20 (0 = default 11; 20 = plain fp16 everywhere)           */
} oww_config;

typedef struct oww_head_desc {
    int32_t n_in;                              /* embedding frames read per prediction (model_inputs),
                                                  1..OWW_MAX_HEAD_FRAMES: no wider window exists in the reference,
                                                  and up to that every window fits the stream's feature ring      */
    int32_t n_layers;                          /* Linear layers (>=1, <= OWW_MAX_HEAD_LAYERS)          */
    int32_t dims[OWW_MAX_HEAD_LAYERS + 1];     /* dims[0] = n_in*96, dims[n_layers] = n_out            */
    int32_t layernorm;                         /* 1: LayerNorm(eps 1e-5) after every hidden Linear     */
    int32_t final_act;                         /* 0 none, 1 sigmoid, 2 softmax, 3 relu then softmax,
                                                  4 relu (train.py's multi-class Net before the softmax wrapper) */
} oww_head_desc;

/* ---- lifetime ---------------------------------------------------------------------------- */
int  oww_create(const oww_config* cfg, oww_ctx** out);
void oww_destroy(oww_ctx* ctx);
const char* oww_last_error(const oww_ctx* ctx);
const char* oww_version(void);

/* ---- weights (host pointers; copied) ------------------------------------------------------ */
/* window512: the 512-tap analysis window (periodic Hann(400) centred); mel_fb: [257][32] filterbank.
 * Either may be NULL to use the built-in constants computed in double precision.                */
int oww_load_mel(oww_ctx* ctx, const float* h_window512, const float* h_mel_fb);
/* blob layout: openwakeword_b200/weights.py:pack_embedding_blob (20 x {HWIO kernel, scale, bias}). */
int oww_load_embedding(oww_ctx* ctx, const float* h_blob, size_t n_floats);
/* blob layout: weights.py:pack_head_blob.  *head_id receives the index; score columns are
 * appended in head order (head 0's n_out columns first).                                        */
int oww_add_head(oww_ctx* ctx, const oww_head_desc* desc, const float* h_blob, size_t n_floats, int* head_id);
/* Conditional verifier pair (the released hey_jarvis graph, docs/models/hey_jarvis.md:9,38: "the second network ...
 * only predicting on audio frames that have a score > 0.5 from the first"): wherever the score of single-output head
 * `main_head` exceeds `threshold` it is replaced by the score of single-output head `verifier_head`, per chunk, before
 * the max over a multi-chunk call.  Both columns stay in d_scores (the verifier's holds its raw score).          */
int oww_add_gate(oww_ctx* ctx, int main_head, int verifier_head, float threshold);
int oww_n_heads(const oww_ctx* ctx);
int oww_n_outputs(const oww_ctx* ctx);          /* total score columns over all heads           */

/* ---- stateless graph calls (drop-in for the three ORT sessions) --------------------------- */
/* d_pcm [n_clips][n_samples] int16 -> d_mel [n_clips][T][32], T = (n_samples-512)/160+1.
 * The -80 dB clamp is per clip (the reference's CPU path runs the graph one clip per call).
 * affine != 0 applies AudioFeatures' x/10+2 (utils.py:180,206).                                 */
int oww_melspectrogram(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples,
                       float* d_mel, int affine, void* stream);
/* d_windows [n][76][32] float32 -> d_emb [n][96] */
int oww_embed_windows(oww_ctx* ctx, const float* d_windows, int n, float* d_emb, void* stream);
/* d_feats [n][n_in][96] -> d_out [n][n_out] */
int oww_head_predict(oww_ctx* ctx, int head_id, const float* d_feats, int n, float* d_out, void* stream);

/* ---- streaming state ----------------------------------------------------------------------- */
int oww_set_streams(oww_ctx* ctx, int n_streams);    /* (re)allocates rings; implies reset of all */
int oww_n_streams(const oww_ctx* ctx);
/* Reset streams to AudioFeatures.__init__/reset() state: empty PCM history, mel ring = ones(76,32),
 * feature ring = h_feature_init[n_rows][96] (NULL -> zeros(41,96); the reference fills it with
 * embeddings of unseeded noise, SURVEY.md F6 - pass the same rows to both sides for parity).
 * h_stream_ids NULL = all streams.  Synchronises.                                              */
int oww_reset(oww_ctx* ctx, const int32_t* h_stream_ids, int n, const float* h_feature_init, int n_rows);
/* Same, stream-ordered: no allocation, no synchronisation.  Enqueue it on the stream the steps run on (the one passed
 * to oww_step).  Streams that were reset re-prime from a full 76-row window at their next step (their first chunk
 * yields 5 mel rows, utils.py:393-398) on a side stream while every other stream keeps the incremental fused kernel. */
int oww_reset_async(oww_ctx* ctx, const int32_t* h_stream_ids, int n, const float* h_feature_init, int n_rows, void* stream);
/* One predict() worth of work for every stream: n_chunks*1280 new samples per stream.
 * d_pcm row b starts at d_pcm + b*pcm_stride (samples).  d_scores [n_streams][oww_n_outputs]:
 * per head the element-wise max over the n_chunks window positions (model.py:287-298).          */
int oww_step(oww_ctx* ctx, const int16_t* d_pcm, int64_t pcm_stride, int n_chunks,
             float* d_scores, void* stream);
/* Same, host buffers: H2D of the PCM and D2H of the scores through pinned staging inside the handle;
 * returns after the scores have landed in h_scores (= submit + collect).                          */
int oww_step_host(oww_ctx* ctx, const int16_t* h_pcm, int64_t pcm_stride, int n_chunks, float* h_scores);
/* Pipelined form for serving loops: submit copies the PCM to pinned memory, enqueues H2D (copy stream),
 * the step (compute stream, in submission order) and the D2H of the scores, and returns a ticket (0/1)
 * without waiting; at most two tickets may be in flight, so the H2D of step k+1 overlaps the kernels
 * of step k.  collect blocks until that step's scores are in h_scores.                          */
int oww_step_host_submit(oww_ctx* ctx, const int16_t* h_pcm, int64_t pcm_stride, int n_chunks, int* ticket);
int oww_step_host_collect(oww_ctx* ctx, int ticket, float* h_scores);
/* last n rows of one stream's feature ring, ending `back` rows before the newest -> h_out[n][96];
 * rows older than the ring holds come back as zeros.  Synchronises.                             */
int oww_get_features(oww_ctx* ctx, int stream_id, int n, int back, float* h_out);
int oww_get_mel(oww_ctx* ctx, int stream_id, int n_rows, float* h_out);   /* last n_rows<=76 mel rows */
/* rows written to the stream's mel / feature buffer since its last reset, initial rows included (76 ones / the
 * feature_init rows) - len(melspectrogram_buffer) / len(feature_buffer) of the reference before its 970 / 120 caps
 * (utils.py:400-401,449-450).  Either pointer may be NULL.  Synchronises.                                     */
int oww_get_counts(oww_ctx* ctx, int stream_id, int* mel_rows, int* feature_rows);

/* ---- batch paths --------------------------------------------------------------------------- */
/* d_pcm [n_clips][n_samples] -> d_emb [n_clips][W][96], W = (T-76)/8+1 (utils.py:322).           */
int oww_embed_clips(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples, float* d_emb, void* stream);
/* predict_clip for n_clips equal-length clips, each from a FRESH state seeded with h_feature_init
 * (SURVEY.md F9): pad_samples zeros each side, 1280-sample steps, steps = len(range(0, L-1280, 1280)).
 * d_scores [n_clips][steps][oww_n_outputs].  Raw head outputs (the first-5-zeroing of
 * model.py:330-333 is label bookkeeping done by the host wrapper).  Uses a private stream set.  */
int oww_predict_clips(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples, int pad_samples,
                      const float* h_feature_init, int n_rows, float* d_scores, void* stream);

/* ---- score metrics on the device (openwakeword/metrics.py:24-100) --------------------------------
 * d_scores holds n_series score sequences of n_frames float32 each, series i at d_scores + i*series_stride.
 * oww_metrics_false_positives: h_counts[i][j] = get_false_positives(series i, h_thresholds[j], grouping_window)
 * with the reference's grouping rule (restated in oracle/metrics.py); generate_roc_curve_fprs is this count at
 * np.linspace(0.01, 0.99, n_points) divided by the hours the series spans.
 * oww_metrics_count_ge: h_counts[j] = number of the n scores >= h_thresholds[j] (generate_roc_curve_tprs * len).
 * Comparisons are done in double, as NumPy does for float32 scores against np.float64 thresholds.  Both synchronise. */
int oww_metrics_false_positives(oww_ctx* ctx, const float* d_scores, int64_t series_stride, int n_series, int n_frames,
                                const double* h_thresholds, int n_thresholds, int grouping_window, int32_t* h_counts, void* stream);
int oww_metrics_count_ge(oww_ctx* ctx, const float* d_scores, int64_t n, const double* h_thresholds, int n_thresholds,
                         uint64_t* h_counts, void* stream);

/* ---- parity instrumentation --------------------------------------------------------------- */
/* Runs the embedding CNN on d_windows [n][76][32] (n <= window_batch) up to and including conv
 * layer `layer` (0..18) and its max-pool, and writes that activation as NHWC float32
 * [n][T][F][C] to d_out - used by the tests to localise a mismatch layer by layer.             */
int oww_debug_layer(oww_ctx* ctx, const float* d_windows, int n, int layer, float* d_out, void* stream);

/* Geometry plan of the fused incremental CNN kernel for groups of `group` streams, as raw int32
 * (struct IncPlan of csrc/oww_internal.h); returns the number of ints written (> 0) or an error.
 * Pure host computation (usable without a GPU): tests/test_inc_plan.py replays it in NumPy.          */
int oww_debug_inc_plan(oww_ctx* ctx, int group, int n_streams, int32_t* out, int max_ints);

/* cnn_mode 3 only, instrumentation: oww_debug_inc_clocks arms a clock buffer; the next step then records clock64()
 * stamps taken by CTA 0 on its first group; oww_debug_inc_clocks_read synchronises and returns 104 values:
 * [0..19] start of each layer phase, [20] end of layer 19, per layer l [21+l] cycles the MMA warp waited for weights,
 * [41+l] its MMA issue time, [61+l] phase start -> first accumulator ready, [81+l] phase start -> last tile stored,
 * [101] group start (before the fused frontend), [102] end of the fused heads phase (0 when the step was not fused). */
int oww_debug_inc_clocks(oww_ctx* ctx, int64_t* h_unused);
int oww_debug_inc_clocks_read(oww_ctx* ctx, int64_t* h_out104);
/* Instrumentation of the grouped heads kernel (heads_grp.cu): the first call arms the stamps, later calls synchronise and
 * return 8 clock64() values per head group (tile 0's CTA): start, producer done, last first-layer MMA issued,
 * first-layer accumulators complete, team 0 done, CTA end, 0, 0. */
int oww_debug_heads_clocks(oww_ctx* ctx, int64_t* h_out64);

/* ---- multi-GPU gather over peer memory (one process per GPU) ---------------------------------
 * The reference has no multi-device path; SURVEY.md section 8e defines the only exchange of the sharded hot path: the
 * per-step scores float32[B/G][n_labels] of every rank gathered on one rank.  Instead of a collective call after the
 * step, a rank moves its finished score block into the gathering rank's memory (a buffer opened with oww_peer_open)
 * with oww_peer_copy - one DMA over NVLink; d_scores of oww_step may also point into the mapping directly, at the
 * price of scattered 4-byte remote stores - then publishes a step counter with oww_peer_signal; the gathering rank
 * orders its consumer behind oww_peer_wait.  openwakeword_b200.distributed.PeerGather drives the protocol
 * (double-buffered slots, acknowledgement counters); validated on 2 x B200 by tests/test_gpu_multi.py.
 *   oww_peer_alloc  - cudaMalloc'd, zero-filled buffer on this handle's device + its 64-byte CUDA IPC handle
 *   oww_peer_open   - map another process's buffer (peer access is enabled lazily); oww_peer_close unmaps it
 *   oww_peer_signal - stream-ordered: after all earlier work of `stream`, *d_flag = value (system-scope release;
 *                     d_flag may be local or peer-mapped)
 *   oww_peer_wait   - stream-ordered: later work of `stream` starts once d_flags[i*stride] >= value for all i < n
 *                     (n <= 1024).  If that takes longer than timeout_s (<= 0: 10 s) the kernel gives up, the stream
 *                     goes on and oww_peer_status reports the timeout - a dead peer can neither hang the GPU nor
 *                     poison the CUDA context.                                                                    */
int oww_peer_alloc(oww_ctx* ctx, size_t bytes, void** d_ptr, unsigned char handle_out[64]);
int oww_peer_free(oww_ctx* ctx, void* d_ptr);
int oww_peer_open(oww_ctx* ctx, const unsigned char handle[64], void** d_ptr);
int oww_peer_close(oww_ctx* ctx, void* d_ptr);
/* stream-ordered block copy into (or out of) a peer mapping (4-byte words, a copy kernel with coalesced 16-byte stores:
 * full lines over NVLink instead of the step kernels' scattered 4-byte stores) - the way
 * openwakeword_b200.distributed moves a rank's [rows x columns] score block */
int oww_peer_copy(oww_ctx* ctx, void* d_dst, const void* d_src, size_t bytes, void* stream);
int oww_peer_signal(oww_ctx* ctx, uint64_t* d_flag, uint64_t value, void* stream);
int oww_peer_wait(oww_ctx* ctx, const uint64_t* d_flags, int n, int stride, uint64_t value, double timeout_s, void* stream);
/* a wait that ran into its timeout lets the stream continue and raises a flag on the handle: *timed_out = 1 (the flag is
 * cleared by the read).  Synchronises the device. */
int oww_peer_status(oww_ctx* ctx, int* timed_out);

/* ---- introspection ------------------------------------------------------------------------- */
uint64_t oww_launch_count(const oww_ctx* ctx);       /* kernels launched by this handle so far   */
/* n_slots > 0: every following oww_step / oww_step_host brackets its three stages (mel, embedding
 * CNN + ring append, heads) with CUDA events on the launching stream, step k in slot k % n_slots;
 * 0 disables.  oww_stage_ms synchronises on the recorded events and returns the per-step AVERAGE
 * {mel, cnn, heads} milliseconds over the steps recorded since enabling (at most n_slots).      */
int oww_enable_stage_timing(oww_ctx* ctx, int n_slots);
int oww_stage_ms(oww_ctx* ctx, float out_ms[3]);

#ifdef __cplusplus
}
#endif
#endif /* OWWB200_H */
