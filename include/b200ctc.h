/*
 * b200ctc.h -- C ABI of the B200-native CTC loss-and-gradient engine.
 *
 * This is the drop-in boundary for the CTC path of
 * carolinebear/pytorch_end2end_speech_recognition.  The reference reaches its
 * CTC arithmetic through the un-vendored warp-ctc binding
 * (tools/install_warpctc_pytorch.sh:7-18):
 *
 *   models/pytorch_v3/ctc/ctc.py:35,39-45   warpctc_pytorch.gpu_ctc(acts, grads,
 *                                           labels, label_lens, act_lens,
 *                                           minibatch_size, costs)
 *   models/pytorch_v3/ctc/ctc.py:30-52      _CTC.forward (costs.sum(), ctx.grads)
 *   models/pytorch_v3/ctc/decoders/greedy_decoder.py:19-47   GreedyDecoder.__call__
 *
 * warp-ctc's own C interface has the two-call shape
 * get_workspace_size(...) / compute_ctc_loss(...) [recollection -- the source is
 * not under /root/reference]; the entry points below keep that shape so that
 * the reference-side binding is a one-to-one replacement (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; no exceptions cross this boundary; every function
 *     returns a b200ctc_status_t (0 == success).
 *   - the caller owns every buffer, including the device workspace (the
 *     PyTorch binding takes it from the caching allocator: no cudaMalloc per
 *     call).  The library keeps no global mutable state; the only state is the
 *     handle, which owns a small ring of pinned host staging buffers.  Calls on
 *     one handle must be serialised by the caller; different handles are
 *     independent (two CTC calls per step with different shapes --
 *     models/pytorch_v3/ctc/hierarchical_ctc.py:323-330 -- may share a handle
 *     because they are issued from one thread in order).
 *   - all device work is enqueued on `stream` (a cudaStream_t passed as
 *     void*); nothing synchronises the host unless stated.
 *   - there is NO CPU fallback: if no CUDA device is usable the calls fail
 *     with B200CTC_STATUS_EXECUTION_FAILED.
 */
#ifndef B200CTC_H_
#define B200CTC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200CTC_VERSION 200 /* 0.2.0 */

#if defined(__GNUC__)
#define B200CTC_API __attribute__((visibility("default")))
#else
#define B200CTC_API
#endif

typedef enum {
  B200CTC_STATUS_SUCCESS = 0,
  B200CTC_STATUS_INVALID_VALUE = 1,     /* bad argument: shape, length, label range, null pointer */
  B200CTC_STATUS_EXECUTION_FAILED = 2,  /* CUDA runtime / launch error */
  B200CTC_STATUS_UNSUPPORTED = 3,       /* size outside what the kernels handle */
  B200CTC_STATUS_WORKSPACE_TOO_SMALL = 4
} b200ctc_status_t;

typedef struct b200ctc_handle b200ctc_handle;

/* Element type of the logits (and of the gradient) of b200ctc_loss_and_grad_dev_typed, and of the input of
   b200ctc_greedy_decode_typed, b200ctc_beam_search_typed and b200ctc_softmax_temperature_typed. */
typedef enum {
  B200CTC_FLOAT32 = 0,
  B200CTC_BFLOAT16 = 1,
  B200CTC_FLOAT16 = 2
} b200ctc_dtype_t;

/*
 * Arithmetic of the reference's loss call site fused into the kernels (SURVEY 8(f) ranks 1-2), for
 * b200ctc_loss_and_grad_dev.  With z = logit_scale * acts and y = softmax(z):
 *
 *   loss_sum  = loss_scale * sum_b [ (1 - label_smoothing) * cost_b
 *                                    + (label_smoothing / V) * sum_{t < act_lens[b]} sum_k -log y[t,b,k] ]
 *   grads     = grad_scale * [ y - (1 - label_smoothing) * occupancy - label_smoothing / V ]     (t < act_lens[b])
 *
 * i.e. grads = grad_scale * d(loss_sum / loss_scale) / dz.  The reference computes exactly this with separate
 * tensor passes: `logits /= logits_temperature` (models/pytorch_v3/ctc/ctc.py:306-307: logit_scale =
 * 1/temperature), `/ len(xs)` (ctc.py:323: loss_scale = 1/B), and the label-smoothing cross entropy with a
 * uniform distribution, a second log_softmax and a python loop over the mini-batch (ctc.py:329-337,
 * models/pytorch_v3/criterion.py:51-80).  For the gradient with respect to the UNSCALED logits of a loss
 * scaled by loss_scale pass grad_scale = loss_scale * logit_scale.
 * A NULL options pointer means {1, 0, 1, 1}: results are bit-identical to b200ctc_loss_and_grad.
 */
typedef struct {
  float logit_scale;      /* > 0 */
  float label_smoothing;  /* in [0, 1) */
  float loss_scale;
  float grad_scale;
} b200ctc_options;

/* Replaces warp-ctc's get_warpctc_version(). */
B200CTC_API int b200ctc_version(void);

/* Replaces warp-ctc's ctcGetStatusString(). */
B200CTC_API const char* b200ctc_status_string(int status);

/* Handle life cycle.  `device` is the CUDA device ordinal the handle is used with. */
B200CTC_API int b200ctc_create(b200ctc_handle** handle, int device);
B200CTC_API int b200ctc_destroy(b200ctc_handle* handle);

/*
 * Replaces warp-ctc's get_workspace_size(label_lengths, input_lengths,
 * alphabet_size, minibatch, options, &bytes).
 * label_lens/act_lens: HOST int32 [B].  T: padded number of frames of acts.
 */
B200CTC_API int b200ctc_get_workspace_size(const int* label_lens, const int* act_lens,
                               int T, int V, int B, size_t* bytes);

/*
 * Workspace bound from the shape alone (no length arrays): enough for any lengths with
 * label_lens[b] <= max_label_len and act_lens[b] <= T.  This is the size the device-resident call
 * b200ctc_loss_and_grad_dev needs; it is also valid for b200ctc_loss_and_grad.
 */
B200CTC_API int b200ctc_get_workspace_bound(int T, int V, int B, int max_label_len, size_t* bytes);

/*
 * Replaces warp-ctc's compute_ctc_loss(activations, gradients, flat_labels,
 * label_lengths, input_lengths, alphabet_size, minibatch, costs, workspace,
 * options) as called by pytorch_binding's gpu_ctc
 * (reference call site: models/pytorch_v3/ctc/ctc.py:35,39-45).
 *
 *   acts        DEVICE fp32 unnormalised logits, logical shape [T,B,V]; element
 *               (t,b,v) lives at acts[t*acts_stride_t + b*acts_stride_b + v]
 *               (strides in elements).  A [B,T,V] batch-major tensor viewed as
 *               transpose(0,1) is accepted as is, which removes the
 *               acts.contiguous() copy of ctc.py:34.
 *   grads       DEVICE fp32 [T,B,V] contiguous, or NULL for cost only.  Fully
 *               overwritten: rows t >= act_lens[b] are set to zero (the
 *               reference wrapper pre-zeros them, ctc.py:36), so the caller
 *               need not clear it.
 *   flat_labels HOST int32 [sum(label_lens)], values in [0,V) and != blank.
 *   label_lens  HOST int32 [B];  act_lens HOST int32 [B], 0 <= act_lens[b] <= T.
 *   blank       blank symbol index (the reference uses 0, ctc.py:267-269).
 *   costs       DEVICE fp32 [B]: -log p(labels_b | acts_b) per utterance.  An
 *               utterance with no valid alignment (L_b + repeats_b > T_b) gets
 *               +inf and an all-zero gradient.
 *   loss_sum    DEVICE fp32 [1] or NULL: sum_b costs[b] (ctc.py:50), fixed
 *               summation order.
 *   workspace   DEVICE, >= b200ctc_get_workspace_size bytes, 256-byte aligned.
 *
 * Limits: T * B rows, B * V * 4 < 2^31; label sequences of any length the fp64 safe lattice can hold in
 * shared memory (about 4000 labels); longer ones return B200CTC_STATUS_UNSUPPORTED.
 * A call whose lengths and labels equal those of the previous call on the same handle and stream reuses
 * that call's plan (no planning, no host-to-device copy of the tables).
 */
B200CTC_API int b200ctc_loss_and_grad(b200ctc_handle* handle,
                          const float* acts, int64_t acts_stride_t, int64_t acts_stride_b,
                          float* grads,
                          const int* flat_labels, const int* label_lens, const int* act_lens,
                          int T, int V, int B, int blank,
                          float* costs, float* loss_sum,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same evaluation with DEVICE-resident labels and lengths: the rewritten call site of
 * models/pytorch_v3/ctc/ctc.py:294-326 (SURVEY 8(f) rank 1) keeps ys / x_lens / y_lens on the GPU, so
 * nothing crosses PCIe and the host does no per-utterance work.  The call is kernel launches only
 * (plan -> softmax rows -> lattice) and may be captured into a CUDA graph.
 *
 *   labels         DEVICE int32, utterance b's labels at labels[b*label_stride .. + label_lens[b])
 *                  (a padded [B, Lmax] tensor with label_stride = Lmax, or a flat vector with equal strides)
 *   label_lens     DEVICE int32 [B], 0 <= label_lens[b] <= max_label_len
 *   act_lens       DEVICE int32 [B], 0 <= act_lens[b] <= T
 *   max_label_len  host-side bound on label_lens (sizes shared memory and the workspace regions)
 *   opts           fused call-site arithmetic (b200ctc_options above) or NULL
 *   costs          DEVICE fp32 [B]: the plain CTC cost -log p(labels_b | z_b), whatever the options
 *   ls_costs       DEVICE fp32 [B] or NULL: sum_{t<act_lens[b]} sum_k -log y[t,b,k] (written when label_smoothing > 0)
 *   workspace      DEVICE, >= b200ctc_get_workspace_bound(T, V, B, max_label_len) bytes
 *
 * Inputs cannot be validated on the host: an utterance with a length out of range or a label outside
 * [0,V) or equal to blank gets cost NaN and an all-zero gradient (b200ctc_get_last_fallbacks counts[2]).
 * B <= 65536.
 */
B200CTC_API int b200ctc_loss_and_grad_dev(b200ctc_handle* handle,
                              const float* acts, int64_t acts_stride_t, int64_t acts_stride_b,
                              float* grads,
                              const int* labels, int label_stride, const int* label_lens, const int* act_lens,
                              int T, int V, int B, int max_label_len, int blank,
                              const b200ctc_options* opts,
                              float* costs, float* loss_sum, float* ls_costs,
                              void* workspace, size_t workspace_bytes, void* stream);

/*
 * b200ctc_loss_and_grad_dev for logits of element type `acts_dtype` (b200ctc_dtype_t); `grads` has the same element
 * type.  A bfloat16 / float16 logit is widened to fp32 when it is loaded, and everything after that is the fp32
 * evaluation of b200ctc_loss_and_grad_dev.  The gradient rows are formed in fp32 in a staging region of the
 * workspace and rounded once, to nearest even, into `grads`; rows t >= act_lens[b] and rows of rejected or
 * infeasible utterances are exact zeros.  costs, loss_sum and ls_costs stay fp32.  With B200CTC_FLOAT32 this is
 * exactly b200ctc_loss_and_grad_dev.
 *   workspace   DEVICE, >= b200ctc_get_workspace_bound_typed(T, V, B, max_label_len, acts_dtype, grads != NULL) bytes
 */
B200CTC_API int b200ctc_loss_and_grad_dev_typed(b200ctc_handle* handle, const void* acts, int64_t acts_stride_t, int64_t acts_stride_b, int acts_dtype, void* grads, const int* labels, int label_stride, const int* label_lens, const int* act_lens, int T, int V, int B, int max_label_len, int blank, const b200ctc_options* opts, float* costs, float* loss_sum, float* ls_costs, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Workspace of b200ctc_loss_and_grad_dev_typed.  For B200CTC_FLOAT32, or without a gradient (need_grad == 0), it
 * equals b200ctc_get_workspace_bound; a bfloat16 / float16 call with a gradient adds the fp32 [T,B,V] staging region
 * (4 * T * B * V bytes, rounded up to 256).
 */
B200CTC_API int b200ctc_get_workspace_bound_typed(int T, int V, int B, int max_label_len, int dtype, int need_grad, size_t* bytes);

/*
 * Backward of a loss on bfloat16 / float16 logits: out[t,b,v] = grads[t,b,v] * scale[s], multiplied in fp32 and rounded
 * once, to nearest even, to `dtype`; s = 0 when n_scale == 1 (one grad_output for the whole loss), s = b when
 * n_scale == B (one per utterance).
 *   grads, out  DEVICE [T,B,V] contiguous, of type dtype (B200CTC_BFLOAT16 or B200CTC_FLOAT16); may be the same buffer
 *   scale       DEVICE fp32 [n_scale]
 * One kernel launch on `stream`.
 */
B200CTC_API int b200ctc_scale_grads(const void* grads, void* out, int dtype, int T, int B, int V, const float* scale, int n_scale, void* stream);

/*
 * Batched best-path decoder; replaces the numpy loops of
 * models/pytorch_v3/ctc/decoders/greedy_decoder.py:32-45 (per-frame argmax with
 * first-index tie break, collapse repeats, then drop blanks).
 *
 *   logits      DEVICE fp32, logical [B,T,V]; element (b,t,v) at
 *               logits[b*stride_b + t*stride_t + v].
 *   lens        DEVICE int32 [B] (x_lens); values outside [0, T] are clamped to that range.
 *   out_tokens  DEVICE int32 [B,T]: hypothesis of utterance b in
 *               out_tokens[b*T .. b*T+out_lens[b]); the rest of the row is -1.
 *   out_lens    DEVICE int32 [B].
 */
B200CTC_API int b200ctc_greedy_decode(const float* logits, int64_t stride_b, int64_t stride_t,
                          const int* lens, int T, int V, int B, int blank,
                          int* out_tokens, int* out_lens, void* stream);

/*
 * b200ctc_greedy_decode for logits of element type `dtype` (b200ctc_dtype_t); the other parameters are the same and the
 * outputs stay int32.  A bfloat16 / float16 call gives, bit for bit, what the fp32 call gives on the logits widened to
 * fp32 (widening is exact and monotone: the same arg-max, ties and NaN included), and reads half the bytes.  With
 * B200CTC_FLOAT32 this is exactly b200ctc_greedy_decode.  An unknown dtype returns B200CTC_STATUS_INVALID_VALUE.
 */
B200CTC_API int b200ctc_greedy_decode_typed(const void* logits, int dtype, int64_t stride_b, int64_t stride_t,
                          const int* lens, int T, int V, int B, int blank,
                          int* out_tokens, int* out_lens, void* stream);

/*
 * Batched CTC prefix beam search without a language model; replaces the python loops of
 * models/pytorch_v3/ctc/decoders/beam_search_decoder.py:33-124 (called with beam_width 10 for every published
 * error rate and with beam_width 2 by every reference test).  One CTA per utterance; scores are accumulated in
 * float64 with numpy's logaddexp formula on the float32 log-probabilities; the surviving prefixes and their
 * order (ties included) are the reference's.
 *
 *   log_probs   DEVICE fp32 log-probabilities (log_softmax output, ctc.py:439-441), element (b,t,v) at
 *               log_probs[b*stride_b + t*stride_t + v]
 *   lens        DEVICE int32 [B]; clamped to [0, T]
 *   beam_width  1..64
 *   out_tokens  DEVICE int32 [B,T]: the best hypothesis of utterance b in out_tokens[b*T .. b*T+out_lens[b]), then -1
 *   out_lens    DEVICE int32 [B];  out_scores  DEVICE fp32 [B] or NULL: log p of the best prefix
 *   workspace   DEVICE, >= b200ctc_beam_search_workspace(B, T, V, beam_width) bytes
 */
B200CTC_API int b200ctc_beam_search_workspace(int B, int T, int V, int beam_width, size_t* bytes);
B200CTC_API int b200ctc_beam_search(const float* log_probs, int64_t stride_b, int64_t stride_t,
                        const int* lens, int T, int V, int B, int blank, int beam_width,
                        int* out_tokens, int* out_lens, float* out_scores,
                        void* workspace, size_t workspace_bytes, void* stream);
/*
 * b200ctc_beam_search for log-probabilities of element type `dtype` (b200ctc_dtype_t); the other parameters and the
 * workspace size are the same, tokens and lengths stay int32 and scores fp32.  The arithmetic is float64 on the
 * widened values, so a bfloat16 / float16 call gives, bit for bit, the tokens, lengths and scores of the fp32 call on
 * the log-probabilities widened to fp32.  With B200CTC_FLOAT32 this is exactly b200ctc_beam_search.  An unknown dtype
 * returns B200CTC_STATUS_INVALID_VALUE.
 */
B200CTC_API int b200ctc_beam_search_typed(const void* log_probs, int dtype, int64_t stride_b, int64_t stride_t,
                        const int* lens, int T, int V, int B, int blank, int beam_width,
                        int* out_tokens, int* out_lens, float* out_scores,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * Batched edit distance with error counts; replaces the python loops of compute_wer
 * (utils/evaluation/edit_distance.py:53-126), which the metric code calls once per utterance
 * (examples/timit/s5/exp/metrics/phone.py:93-101 and its twins).
 *
 *   refs / hyps   DEVICE int32 token ids, pair b at refs[b*ref_stride ..+ref_lens[b]) / hyps[b*hyp_stride ..+hyp_lens[b])
 *   ref_lens / hyp_lens  DEVICE int32 [B]; values outside [0, max_ref] / [0, max_hyp] are clamped
 *   out4          DEVICE int32 [B,4]: distance, substitutions, insertions, deletions, with the backtrace
 *                 preference of the reference (:99-117): match, insertion, substitution, deletion.
 *   workspace     DEVICE, >= b200ctc_edit_distance_workspace(B, max_ref, max_hyp) bytes
 * max_ref <= 17000 (three anti-diagonals of the matrix live in shared memory).  The reference indexes its
 * matrix with -1 at the borders and raises for some inputs (its callers swallow the exception and skip the
 * utterance); here the first row / column always backtrace as insertions / deletions.
 */
B200CTC_API int b200ctc_edit_distance_workspace(int B, int max_ref, int max_hyp, size_t* bytes);
B200CTC_API int b200ctc_edit_distance(const int* refs, int ref_stride, const int* ref_lens,
                          const int* hyps, int hyp_stride, const int* hyp_lens,
                          int B, int max_ref, int max_hyp, int* out4,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * probs[b,t,:] = softmax(logits[b,t,:] / temperature): the tensor work of CTC.posteriors
 * (models/pytorch_v3/ctc/ctc.py:455-502) in one pass.  logits: DEVICE fp32, element (b,t,v) at
 * logits[b*stride_b + t*stride_t + v]; probs: DEVICE fp32 [B,T,V] contiguous.
 */
B200CTC_API int b200ctc_softmax_temperature(const float* logits, int64_t stride_b, int64_t stride_t,
                                int T, int V, int B, float temperature, float* probs, void* stream);
/*
 * b200ctc_softmax_temperature for logits of element type `dtype` (b200ctc_dtype_t); `probs` stays fp32 [B,T,V] for
 * every type.  A bfloat16 / float16 call gives, bit for bit, the probabilities of the fp32 call on the logits widened
 * to fp32 (same element-to-lane assignment and summation order).  With B200CTC_FLOAT32 this is exactly
 * b200ctc_softmax_temperature.  An unknown dtype returns B200CTC_STATUS_INVALID_VALUE.
 */
B200CTC_API int b200ctc_softmax_temperature_typed(const void* logits, int dtype, int64_t stride_b, int64_t stride_t,
                                int T, int V, int B, float temperature, float* probs, void* stream);

/*
 * Measurement hooks (no counterpart in the reference; used by bench.py for the roofline line).
 * With profiling enabled every b200ctc_loss_and_grad call on this handle brackets each of its
 * kernels with CUDA events on `stream`; b200ctc_get_last_kernel_ms waits for the last call and
 * returns the device time of {softmax rows, lattice, gradient completion} in milliseconds.  The third
 * slot holds the occupancy pass of large vocabularies and, for bfloat16 / float16 logits, the pass
 * that rounds the fp32 staged gradient into the caller's buffer.
 */
B200CTC_API int b200ctc_set_profiling(b200ctc_handle* handle, int enable);
B200CTC_API int b200ctc_get_last_kernel_ms(b200ctc_handle* handle, float* ms3);
/*
 * Diagnostics: number of utterances of the LAST call on this handle that were evaluated by the
 * fp64 safe lattice instead of the block-exponent fast lattice (counts[0]: flagged by the softmax
 * pass for extreme probabilities, counts[1]: the fast lattice lost range and was redone), and
 * counts[2]: utterances of a device-resident call with invalid lengths or labels.
 * Synchronises `stream`; the workspace of that call must still be alive.
 */
B200CTC_API int b200ctc_get_last_fallbacks(b200ctc_handle* handle, int* counts3, void* stream);
/* Plan cache of b200ctc_loss_and_grad: calls that reused the previous call's plan / calls that planned. */
B200CTC_API int b200ctc_get_plan_cache_stats(b200ctc_handle* handle, long long* hits, long long* misses);

#ifdef __cplusplus
}
#endif
#endif /* B200CTC_H_ */
