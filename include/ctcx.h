/* ctcx -- B200-native CTC "extended" beam-search decode (sm_100a): C-ABI boundary.
 *
 * This header is the drop-in boundary for ONE operator of prouast/ctc-beam-search-op: the TensorFlow
 * custom op `CTCExtBeamSearchDecoder`. Citations are relative to
 * tensorflow_ctc_ext_beam_search_decoder/cc/ in the reference:
 *   ops/ctc_ext_beam_search_decoder_ops.cc:9-24          the op signature (inputs, attrs, outputs)
 *   kernels/ctc_ext_beam_search_decoder_kernels.cc:20-95 CTCExtBeamSearchDecoderOp<T>::Compute
 *   kernels/...kernels.cc:97-160                         ValidateInputsGenerateOutputs
 *   kernels/...kernels.cc:163-257                        StoreAllDecodedSequences (sparse packing)
 *   util/ctc_ext_beam_search_decoder.h:229-261           TopPaths (its two InvalidArgument errors)
 *
 * Plain pointers and sizes only; no torch/TF types. Output sizes are data dependent, so a decode is
 * two calls: ctcx_decode_* runs the kernels and reports, per path, how many sparse entries there are;
 * the caller allocates and ctcx_pack_* fills the 6*top_paths int64 tensors and log_probability.
 * The library keeps no global state: everything lives in the caller's workspace, so calls on
 * different streams/workspaces may run concurrently (the reference's Compute is re-entrant too).
 *
 * There is NO CPU fallback: every entry point needs a CUDA device of compute capability 10.x.
 */
#ifndef CTCX_H_
#define CTCX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Return codes. 1-7 map 1:1 to the reference's Status errors (message text in ctcx_strerror). */
enum {
  CTCX_OK = 0,
  CTCX_ERR_INPUTS_NOT_3D = 1,       /* kernels.cc:111-113 "inputs is not a 3-Tensor" (host side) */
  CTCX_ERR_MAX_TIME_ZERO = 2,       /* kernels.cc:118-120 "max_time is 0" */
  CTCX_ERR_SEQ_LEN_NOT_VECTOR = 3,  /* kernels.cc:122-124 "sequence_length is not a vector" (host) */
  CTCX_ERR_SEQ_LEN_BATCH = 4,       /* kernels.cc:126-130 "len(sequence_length) != batch_size. ..." */
  CTCX_ERR_SEQ_LEN_RANGE = 5,       /* kernels.cc:134-138 "sequence_length(b) <= max_time" */
  CTCX_ERR_TOO_MANY_PATHS = 6,      /* decoder.h:237-239 "requested more paths than the beam width." */
  CTCX_ERR_TOO_FEW_LEAVES = 7,      /* decoder.h:240-243 "Less leaves in the beam search than requested." */
  CTCX_ERR_BAD_ARGUMENT = 8,        /* not validated by the reference (UB there): blank_index outside
                                       [0,C), negative sequence_length, beam_width/top_paths < 1 */
  CTCX_ERR_UNSUPPORTED = 9,         /* shape outside what this build supports (see ctcx_limits) */
  CTCX_ERR_WORKSPACE = 10,          /* workspace too small / NULL / not 256-byte aligned */
  CTCX_ERR_CUDA = 11                /* a CUDA runtime call failed; ctcx_last_cuda_error() has it */
};

/* Human-readable text of a return code; for 1-7 the reference's own message (for
 * CTCX_ERR_SEQ_LEN_RANGE with the offending batch index of this thread's last decode filled in). */
const char* ctcx_strerror(int code);

/* Batch index of this thread's last CTCX_ERR_SEQ_LEN_RANGE (kernels.cc:134-138 reports it in the
 * message); a caller that decodes a shard [b0, b1) of a batch adds b0 before reporting. */
int ctcx_error_batch_index(void);

/* Last CUDA error string seen by this thread ("" if none). */
const char* ctcx_last_cuda_error(void);

/* Library build info: returns the sm arch the kernels were built for (100), fills limits. */
typedef struct {
  int max_beam_width;  /* largest supported beam_width */
  int max_classes;     /* largest supported num_classes */
  int max_top_paths;   /* bounded by beam_width anyway */
} ctcx_limits;
int ctcx_get_limits(ctcx_limits* out);

/* Bytes of device workspace needed by ctcx_decode_f32 for this shape (0 on invalid shape). */
size_t ctcx_workspace_bytes(int max_time, int batch, int num_classes, int beam_width, int top_paths);

/* Per-path sparse sizes produced by a decode (host memory, caller-allocated, top_paths entries each). */
typedef struct {
  int64_t* n_decoded;     /* [P] total decoded entries over the batch   (rows of decoded_indices[p]) */
  int64_t* max_decoded;   /* [P] longest decoded sequence               (decoded_shape[p][1])        */
  int64_t* n_alignment;   /* [P] total alignment entries over the batch (rows of alignment_indices[p]) */
  int64_t* max_alignment; /* [P] longest alignment                      (alignment_shape[p][1])      */
} ctcx_sizes;

/* Decode: replaces Compute's validation + batch/time loops + TopPaths (kernels.cc:20-90).
 *   logits_dev   [max_time, batch, num_classes] float32, time-major, raw logits, DEVICE memory
 *   seq_len_dev  [batch] int32, DEVICE memory
 *   attrs        as ops.cc:12-16 (merge_repeated / blank_index / blank_label defaults are the host's job)
 *   workspace    DEVICE memory of at least ctcx_workspace_bytes(...) bytes, 256-byte aligned; it holds
 *                the decode result until ctcx_pack_f32 has run
 *   stream       cudaStream_t (as void*), may be NULL for the default stream
 *   sizes        host output, see ctcx_sizes. NULL = DEFERRED: the decode is only enqueued, nothing is
 *                synchronised and only argument errors are returned; ctcx_finish() later brings the
 *                sizes, the flags and the reference's run-time errors. Every ctcx_decode_* entry on
 *                device or page-locked inputs accepts it.
 *   flags_out    optional host int32: bit0 = some utterance hit the documented rounding anomaly
 * Synchronises `stream` once (sizes must reach the host). */
int ctcx_decode_f32(const float* logits_dev, int max_time, int batch, int num_classes,
                    const int32_t* seq_len_dev, int beam_width, int top_paths, int merge_repeated,
                    int blank_index, int blank_label, void* workspace, size_t workspace_bytes,
                    void* stream, ctcx_sizes* sizes, int32_t* flags_out);

/* Element types of a logits tensor. The reference registers float and double (kernels.cc:269-275);
 * half and bfloat16 are what an acoustic model's projection emits -- they are read by the kernels as
 * they are (widened exactly to float32 in registers), so the result equals the reference op run on
 * the widened values. */
enum { CTCX_F32 = 0, CTCX_F16 = 1, CTCX_BF16 = 2, CTCX_F64 = 3 };

/* Decode a VIEW: logits_dev points at element (t = 0, b = 0, c = 0) of a [max_time, batch, num_classes]
 * view whose frames are `time_stride` ELEMENTS apart (0 = batch * num_classes, i.e. contiguous) -- e.g.
 * the batch shard inputs[:, b0:b1, :] of a wider time-major tensor (pointer = &inputs[0, b0, 0], stride
 * = total_batch * num_classes) is decoded in place, without a repack. Utterances are independent
 * (kernels.cc:67-89), so a shard's result is the corresponding slice of the whole batch's. dtype is
 * one of CTCX_F32 / F16 / BF16 / F64 (F64: pack with ctcx_pack_f64). Everything else as
 * ctcx_decode_f32. */
int ctcx_decode_view(const void* logits_dev, int dtype, int64_t time_stride, int max_time, int batch,
                     int num_classes, const int32_t* seq_len_dev, int beam_width, int top_paths,
                     int merge_repeated, int blank_index, int blank_label, void* workspace,
                     size_t workspace_bytes, void* stream, ctcx_sizes* sizes, int32_t* flags_out);

/* Decode HOST logits, with the host->device copy off the critical path. logits_host is a
 * [max_time, batch, num_classes] view in host memory (frames host_time_stride elements apart, 0 =
 * contiguous; pinned memory copies asynchronously, pageable memory works too), seq_len_host [batch]
 * int32 in host memory. The logits are copied into staging_dev (device memory, at least
 * ctcx_hostin_staging_bytes(...) bytes) in time slabs on `copy_stream` while, for the char-CTC shapes
 * (num_classes <= 32), the beam kernel on `stream` already consumes the frames that have landed; for
 * wide vocabularies (the wide fast path) the decode follows the copy slab by slab in stream order; other
 * shapes, and pageable sources, start after the copy. copy_stream must be a different stream from `stream`. The decode result
 * is left in the workspace exactly as by ctcx_decode_f32 (follow with ctcx_pack_f32 / _f64).
 * Synchronises `stream` once. */
size_t ctcx_hostin_staging_bytes(int dtype, int max_time, int batch, int num_classes);
int ctcx_decode_hostin(const void* logits_host, int dtype, int64_t host_time_stride, int max_time,
                       int batch, int num_classes, const int32_t* seq_len_host, int beam_width,
                       int top_paths, int merge_repeated, int blank_index, int blank_label,
                       void* staging_dev, size_t staging_bytes, void* workspace, size_t workspace_bytes,
                       void* stream, void* copy_stream, ctcx_sizes* sizes, int32_t* flags_out);

/* Pack: replaces StoreAllDecodedSequences (kernels.cc:163-257) and the log-prob copy (:87-89).
 * All pointers are DEVICE memory; arrays of `top_paths` device pointers are HOST arrays.
 *   decoded_indices[p]   int64 [n_decoded[p], 2]   rows [b, position], row-major over b then position
 *   decoded_values[p]    int64 [n_decoded[p]]
 *   decoded_shape[p]     int64 [2] = [batch, max_decoded[p]]
 *   alignment_*          likewise
 *   log_probability      float32 [batch, top_paths]
 * Does not synchronise: the pack kernel is only enqueued on `stream` (the part of the workspace it
 * reads is laid out by max_time, batch and top_paths alone). A workspace decoded as float64 must be
 * packed with ctcx_pack_f64. */
int ctcx_pack_f32(const void* workspace, int max_time, int batch, int top_paths,
                  int64_t* const* decoded_indices, int64_t* const* decoded_values,
                  int64_t* const* decoded_shape, int64_t* const* alignment_indices,
                  int64_t* const* alignment_values, int64_t* const* alignment_shape,
                  float* log_probability, void* stream);

/* Compact pack for a host that does not know the sizes yet (a deferred decode): ALL outputs go into one
 * int64 DEVICE buffer of packed_elems elements -- per path p: decoded_indices [n_decoded[p], 2],
 * decoded_values [n_decoded[p]], decoded_shape [2], alignment_indices [n_alignment[p], 2],
 * alignment_values [n_alignment[p]], alignment_shape [2]; after the last path log_probability [batch,
 * top_paths] (real_bytes = 4: float32, two per slot, or 8: float64) -- laid out ON THE DEVICE from the
 * sizes the decode left in the workspace. A sufficient size is top_paths * (6 * A + 4) + batch *
 * top_paths slots, A = sum of the (clamped) sequence lengths <= batch * max_time. Only enqueues; a
 * buffer that turns out too small writes nothing and makes ctcx_finish return CTCX_ERR_WORKSPACE. */
int ctcx_pack_compact(void* workspace, int max_time, int batch, int top_paths, int real_bytes,
                      int64_t* packed_dev, size_t packed_elems, void* stream);

/* Completes a deferred decode (sizes == NULL above): one device->host copy of the sizes and status
 * words, one synchronisation of `stream`, then the reference's checks exactly as the synchronous entry
 * would have returned them. */
int ctcx_finish(const void* workspace, int max_time, int batch, int top_paths, void* stream,
                ctcx_sizes* sizes, int32_t* flags_out);

/* ctcx_finish in two halves, for callers that keep SEVERAL decodes in flight on one stream (ctcx_finish
 * would wait for all of them): ctcx_result_copy_async enqueues the copy of the sizes / status block
 * (ctcx_result_bytes(top_paths) bytes) into result_host -- page-locked memory, or the call blocks --
 * right behind the decode; the caller records an event of its own there, waits for it when it wants
 * the result, and ctcx_result_parse (host only) turns the block into sizes, flags and the return code. */
size_t ctcx_result_bytes(int top_paths);
int ctcx_result_copy_async(const void* workspace, int max_time, int batch, int top_paths, void* result_host,
                           size_t result_bytes, void* stream);
int ctcx_result_parse(const void* result_host, int max_time, int batch, int top_paths, ctcx_sizes* sizes,
                      int32_t* flags_out);

/* Host-buffer entry point: what a TensorFlow CPU OpKernel::Compute (the reference's only
 * registration, kernels.cc:269-275) would call with its host tensors. Copies the inputs to the
 * device, decodes, and returns one malloc'd host block per output group which the caller copies into
 * its framework-allocated tensors and releases with ctcx_free_host. Layout of the result:
 *   for p in [0,P): dec_indices[p] (n_decoded[p]*2 int64), dec_values[p], dec_shape[p] (2),
 *                   ali_indices[p], ali_values[p], ali_shape[p]; then log_probability.
 * device = CUDA device ordinal. */
typedef struct {
  int top_paths;
  int64_t* n_decoded;       /* [P] */
  int64_t* n_alignment;     /* [P] */
  int64_t** decoded_indices;   /* [P] -> [n_decoded[p]*2] */
  int64_t** decoded_values;    /* [P] -> [n_decoded[p]]   */
  int64_t** decoded_shape;     /* [P] -> [2]              */
  int64_t** alignment_indices; /* [P] -> [n_alignment[p]*2] */
  int64_t** alignment_values;  /* [P] -> [n_alignment[p]] */
  int64_t** alignment_shape;   /* [P] -> [2]              */
  float* log_probability;      /* [batch*top_paths]; NULL after ctcx_decode_host_f64 */
  int32_t flags;
  double* log_probability_f64; /* [batch*top_paths]; NULL after ctcx_decode_host_f32 */
} ctcx_host_result;

int ctcx_decode_host_f32(const float* logits_host, int max_time, int batch, int num_classes,
                         const int32_t* seq_len_host, int beam_width, int top_paths,
                         int merge_repeated, int blank_index, int blank_label, int device,
                         ctcx_host_result** result);
/* T = double registration (kernels.cc:275): float64 host logits, log_probability_f64 in the result. */
int ctcx_decode_host_f64(const double* logits_host, int max_time, int batch, int num_classes,
                         const int32_t* seq_len_host, int beam_width, int top_paths,
                         int merge_repeated, int blank_index, int blank_label, int device,
                         ctcx_host_result** result);
void ctcx_free_host(ctcx_host_result* result);

/* Half-precision logits: logits_dev is [max_time, batch, num_classes] IEEE half (dtype 0) or bfloat16
 * (dtype 1) in DEVICE memory. The kernels read them directly and widen them exactly to float32 in
 * registers, i.e. the result equals the reference op run on the widened values. scratch_dev is
 * IGNORED (the first version of this entry upcast into it; the argument stays for ABI stability and
 * may be NULL). Everything else as ctcx_decode_f32. */
int ctcx_decode_half(const void* logits_dev, int dtype, float* scratch_dev, int max_time, int batch,
                     int num_classes, const int32_t* seq_len_dev, int beam_width, int top_paths,
                     int merge_repeated, int blank_index, int blank_label, void* workspace,
                     size_t workspace_bytes, void* stream, ctcx_sizes* sizes, int32_t* flags_out);

/* T = double (the reference registers the op for float and double, kernels.cc:269-275, and its own
 * test feeds float64): logits_dev is [max_time, batch, num_classes] float64 in DEVICE memory; scores
 * are computed in float64 exactly as the reference does (LogSumExp still through the float
 * functions, util/ctc_loss_util.h:39-40); ctcx_pack_f64 writes log_probability as float64 [batch,
 * top_paths]. Same workspace size, same error codes. A workspace decoded with one dtype must be
 * packed with the same one. */
int ctcx_decode_f64(const double* logits_dev, int max_time, int batch, int num_classes,
                    const int32_t* seq_len_dev, int beam_width, int top_paths, int merge_repeated,
                    int blank_index, int blank_label, void* workspace, size_t workspace_bytes,
                    void* stream, ctcx_sizes* sizes, int32_t* flags_out);
int ctcx_pack_f64(const void* workspace, int max_time, int batch, int top_paths,
                  int64_t* const* decoded_indices, int64_t* const* decoded_values,
                  int64_t* const* decoded_shape, int64_t* const* alignment_indices,
                  int64_t* const* alignment_values, int64_t* const* alignment_shape,
                  double* log_probability, void* stream);

/* Scorer extension point. The reference's decoder takes a BaseBeamScorer (util/ctc_beam_scorer.h:
 * 31-65; call sites decoder.h:103,114,171,176,182) whose GetStateExpansionScore(state, s) is applied
 * whenever a beam entry is extended by a label; the op itself only ever passes the default scorer
 * (kernels.cc:260-265), i.e. s unchanged. This entry point plugs a table-driven scorer in:
 *   expansion_scores_dev  [num_classes + 1, num_classes] float32, DEVICE memory, every entry <= 0
 *                         (log-probabilities; CTCX_ERR_BAD_ARGUMENT otherwise): row = label of the
 *                         entry being extended + 1 (row 0: the empty prefix), column = the new label;
 *                         GetStateExpansionScore(state, s) = s + entry  -- e.g. a label-bigram LM with
 *                         its weight folded in, or a constant insertion penalty.
 * NULL gives ctcx_decode_f32. With a table the generic beam kernel is used (the fast kernels'
 * candidate search assumes scores monotone in the frame's log-probs). A constant table reproduces
 * the reference compiled with a stateless scorer subclass bit for bit (tests/test_oracle.py). */
int ctcx_decode_scorer_f32(const float* logits_dev, int max_time, int batch, int num_classes,
                           const int32_t* seq_len_dev, int beam_width, int top_paths,
                           int merge_repeated, int blank_index, int blank_label,
                           const float* expansion_scores_dev, void* workspace, size_t workspace_bytes,
                           void* stream, ctcx_sizes* sizes, int32_t* flags_out);

/* ---- Streaming: the reference decoder's Step / TopPaths / Reset
 * (util/ctc_ext_beam_search_decoder.h:39-53) for all utterances of a batch at once. The beam state
 * lives in the workspace between calls, so logits can be fed in chunks of frames as they arrive:
 *   ctcx_stream_reset(...)                       Reset():    decoder.h:212-227
 *   ctcx_stream_step_f32(..., chunk, lens ...)   Step() x lens[b] frames: decoder.h:67-210
 *   ctcx_stream_top_paths(...) + ctcx_pack_f32   TopPaths(): decoder.h:229-261 (does not disturb the state)
 * Feeding the same frames in any chunking gives bit-identical results to one one-shot decode of the
 * same score type (ctcx_decode_view / ctcx_decode_f64 / ctcx_decode_scorer_f32 with the same table).
 * max_time_total bounds the frames per utterance over the whole stream (feeding more is reported by
 * ctcx_stream_top_paths as CTCX_ERR_SEQ_LEN_RANGE). The shape arguments must be the same in every
 * call on one workspace. None of the step calls synchronises. The un-suffixed entries are the float32
 * stream of the _v entries (same workspace size). ---- */
size_t ctcx_stream_workspace_bytes(int max_time_total, int batch, int num_classes, int beam_width,
                                   int top_paths);
int ctcx_stream_reset(void* workspace, size_t workspace_bytes, int max_time_total, int batch,
                      int num_classes, int beam_width, int top_paths, void* stream);
/* logits_dev [chunk_time, batch, num_classes] float32 DEVICE; chunk_len_dev [batch] int32 DEVICE =
 * number of leading frames of this chunk to consume per utterance (0 .. chunk_time). */
int ctcx_stream_step_f32(void* workspace, int max_time_total, int batch, int num_classes,
                         int beam_width, int top_paths, const float* logits_dev, int chunk_time,
                         const int32_t* chunk_len_dev, int blank_index, void* stream);
/* A stream with score_dtype scores: CTCX_F32 (float32 / float16 / bfloat16 chunks) or CTCX_F64 (float64
 * chunks, double scores; pack with ctcx_pack_f64). workspace_bytes 0 = bad arguments. */
size_t ctcx_stream_workspace_bytes_v(int score_dtype, int max_time_total, int batch, int num_classes,
                                     int beam_width, int top_paths);
int ctcx_stream_reset_v(void* workspace, size_t workspace_bytes, int score_dtype, int max_time_total,
                        int batch, int num_classes, int beam_width, int top_paths, void* stream);
/* One Step() of a chunk of element type `dtype` (CTCX_F32 / F16 / BF16 step a float32 stream, CTCX_F64 a
 * float64 one), row (t, b) at element t * time_stride + b * num_classes (0 = batch * num_classes: a batch
 * shard [:, b0:b1, :] of a wider tensor is stepped in place). expansion_scores_dev: the scorer table of
 * ctcx_decode_scorer_f32 (float32 streams; NULL = the default scorer); with float16 / bfloat16 chunks it
 * returns CTCX_ERR_UNSUPPORTED wherever ctcx_decode_scorer_f32 would not take them (widen the chunk).
 * Errors: CTCX_ERR_WORKSPACE when workspace_bytes is short of the chunk's score type; unknown dtype or a
 * stride shorter than a frame: CTCX_ERR_BAD_ARGUMENT. A table entry > 0, or float32 and float64 steps
 * since the last reset, make the next ctcx_stream_top_paths return CTCX_ERR_BAD_ARGUMENT. */
int ctcx_stream_step_v(void* workspace, size_t workspace_bytes, int max_time_total, int batch,
                       int num_classes, int beam_width, int top_paths, const void* logits_dev, int dtype,
                       int64_t time_stride, int chunk_time, const int32_t* chunk_len_dev, int blank_index,
                       const float* expansion_scores_dev, void* stream);
/* Leaves the dense result in the workspace and reports the sparse sizes; follow with
 * ctcx_pack_f32(workspace, max_time_total, batch, top_paths, ...) (ctcx_pack_f64 for a float64
 * stream). Synchronises `stream` once. */
int ctcx_stream_top_paths(void* workspace, int max_time_total, int batch, int num_classes,
                          int beam_width, int top_paths, int merge_repeated, int blank_label,
                          void* stream, ctcx_sizes* sizes, int32_t* flags_out);

/* ---- Per-utterance lifecycle of a stream: each of the `batch` positions (slots) of a stream can start
 * and finish on its own. slot_mask_dev is a DEVICE int32 [batch]; non-zero selects the slot. Both
 * entries only enqueue device work with no host staging of the mask, so the mask may be built or kept on
 * the device, and ctcx_stream_reset_slots can be captured in a CUDA graph. A NULL mask is
 * CTCX_ERR_BAD_ARGUMENT; the other argument checks are those of ctcx_stream_reset_v /
 * ctcx_stream_top_paths, plus top_paths > beam_width (CTCX_ERR_TOO_MANY_PATHS), all before any CUDA call.
 *
 * ctcx_stream_reset_slots: Reset() (decoder.h:212-227) of the selected slots; the others keep their
 * beams untouched. The workspace must have been reset once with ctcx_stream_reset_v(score_dtype, ...).
 * A reset slot has consumed zero frames, so its max_time_total budget starts again (max_time_total
 * bounds the longest utterance, not the frames that pass through a slot); its anomaly, overflow and
 * too-few-leaves flags and its record of float32 / float64 steps are cleared; TopPaths of the slot before
 * any step returns the root (one leaf, log-probability 0, empty sequences; "Less leaves" for
 * top_paths > 1). The stream-wide mark of a scorer table with a positive entry is NOT cleared: only
 * ctcx_stream_reset_v clears it. */
int ctcx_stream_reset_slots(void* workspace, size_t workspace_bytes, int score_dtype, int max_time_total,
                            int batch, int num_classes, int beam_width, int top_paths,
                            const int32_t* slot_mask_dev, void* stream);
/* ctcx_stream_top_paths_slots: TopPaths() (decoder.h:229-261) of the selected slots; does not disturb
 * any state. The result has the workspace layout of ctcx_stream_top_paths for the whole batch: selected
 * slots are traced as there, unselected ones contribute no decoded or alignment entries (lengths 0) and
 * their log_probability rows are unspecified; dense_shape[p][1] is the maximum over the selected slots.
 * The run-time checks cover the selected slots only: a slot fed more than max_time_total frames
 * (CTCX_ERR_SEQ_LEN_RANGE, ctcx_error_batch_index() = the slot), too few leaves, mixed score types and
 * the rounding-anomaly flag, so a finished slot can be read beside an over-fed or freshly reset one.
 * sizes != NULL: synchronises `stream` once; follow with ctcx_pack_f32 / ctcx_pack_f64(workspace,
 * max_time_total, batch, ...). sizes == NULL: deferred, only enqueues; complete it exactly like a deferred
 * decode (ctcx_pack_compact + ctcx_finish, or ctcx_result_copy_async + ctcx_result_parse).
 * Ordering, in both forms: the pack (ctcx_pack_f32 / _f64 / _compact) must be enqueued before the next
 * ctcx_stream_step_*, ctcx_stream_reset* or ctcx_stream_top_paths* on the workspace, because it reads
 * log_probability from the final beam, which every step and reset rewrites; ctcx_finish or
 * ctcx_result_copy_async must come before the next ctcx_stream_top_paths*, which rewrites the sizes and
 * status words. Steps and resets enqueued after the pack leave the result alone: it reflects the frames
 * consumed by the steps enqueued before this call, even when it is read later. */
int ctcx_stream_top_paths_slots(void* workspace, int max_time_total, int batch, int num_classes,
                                int beam_width, int top_paths, int merge_repeated, int blank_label,
                                const int32_t* slot_mask_dev, void* stream, ctcx_sizes* sizes,
                                int32_t* flags_out);

/* ---- Measurement and test hooks (not part of the operator's contract) ---- */

/* Dense per-(b,p) rows as left in the workspace by a decode (device pointers into the workspace;
 * stride max_time per row). Any output pointer may be NULL. Synchronises the device (it validates
 * the workspace header). */
int ctcx_workspace_views(const void* workspace, int max_time, int batch, int top_paths,
                         const int32_t** dec_len, const int32_t** dec, const int32_t** ali_len,
                         const int32_t** ali, const float** logp);

/* Per-kernel device times of the calling thread's last decode, from CUDA events recorded on the
 * launching stream (bench.py's roofline line): out_ms[5] = {pre-pass, beam kernel, trace-back,
 * scan + flags, whole decode}. */
void ctcx_profile_enable(int on);
void ctcx_profile_get(float* out_ms);

/* Device buffer [batch, 24] int64 receiving per-phase clock64 cycles of the fast beam kernels (thread
 * 0 of every CTA, summed over frames; a separately compiled timing build of the kernel is launched
 * while it is set) for the calling thread's decodes; NULL switches it off. tools/phase_cycles.py.
 * The _n form takes rows of `slots` >= 24 entries; the narrow kernel fills its revisit-wipe event
 * counters 24-26 (at-risk members listed, contested members, fixed-point rounds) where they fit. */
void ctcx_debug_set_cycles_buffer(long long* dev_buf);
void ctcx_debug_set_cycles_buffer_n(long long* dev_buf, int slots);

/* 0 = dispatch by shape (default); 1 = route every decode of the process to the generic beam kernel,
 * the independently written second implementation the parity tests compare with the fast kernels. */
void ctcx_debug_set_beam_impl(int impl);

/* y = f(x) element-wise with the exact device math (bit-identical to glibc 2.39, DESIGN.md section 6):
 * f32 op 0 expf (x <= 0), 1 log1pf (0 <= x <= 1), 2 logf (x >= 1), 3 LogSumExp(x, 0), 4 LogSumExp(0, x);
 * f64 op 0 exp, 1 log, 2 LogSumExp(x, 0). */
int ctcx_debug_math_f32(int op, const float* x_dev, float* y_dev, int n, void* stream);
int ctcx_debug_math_f64(int op, const double* x_dev, double* y_dev, int n, void* stream);

/* The softmax-normaliser pre-pass of a decode, run alone on the T*B rows of a [T, B, C] tensor of
 * element type `in_dtype` (CTCX_F32 ... ; time stride `tstride` elements, 0 = B*C) through the same
 * pre-pass function a decode calls. off_dev[T*B] (double for CTCX_F64, float otherwise) receives max + log(sum exp).
 * route 0: the generic path's normaliser (half inputs are upcast to float32 first).
 * route 1: the wide path's fused pre-pass (32 < C <= 2048, shapes the wide kernel takes, not CTCX_F64):
 *   also srt_pl_dev / srt_cls_dev[T*B, *ks_out] receive per row the first min(C-1, 2*beam_width+3)
 *   non-blank classes by (log-prob desc, class asc), then (-inf, 0xffff) padding.
 * Returns CTCX_ERR_UNSUPPORTED for a shape the route does not serve. Asynchronous on `stream`. */
int ctcx_debug_prepass(int route, const void* logits_dev, int in_dtype, int T, int B, int C, long long tstride,
                       int blank_index, int beam_width, void* off_dev, float* srt_pl_dev, uint16_t* srt_cls_dev,
                       int* ks_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTCX_H_ */
