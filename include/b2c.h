/* b2c — C ABI of the B200-native KD hot path of VeeraKarthick609/ImageCaptioner.
 *
 * The reference is pure Python/PyTorch and has no FFI of its own; what this library replaces are the
 * bodies of the reference's Python entry points on the hot path (citations are into /root/reference):
 *
 *   b2c_decoder_forward   <- LSTMDecoder.forward                    src/student_model.py:205-256
 *                            (attention_mechanism :173-203, nn.LSTM step :244, output_projection :247)
 *   b2c_decoder_prepare / b2c_decoder_forward_prepared <- the same forward split at the point where the image features are first read
 *   b2c_decoder_set_initial_state <- the optional `hidden=(h0, c0)` argument of LSTMDecoder.forward   src/student_model.py:205,219-222
 *   b2c_decoder_forward_eval <- validate_student_model's forward + loss + argmax without a logits tensor   src/train_student_kd.py:29-86
 *   b2c_decoder_backward  <- autograd of the above (loss.backward(), src/train_student_kd.py:288)
 *   b2c_greedy_decode     <- CaptioningStudent.caption_image loop   src/student_model.py:339-381 (batched)
 *   b2c_attention_step    <- LSTMDecoder.attention_mechanism          src/student_model.py:173-203 (stand-alone accessor)
 *   b2c_refinement_forward/backward <- AttentionRefinement.forward (+ autograd)   src/student_model.py:72-118
 *   b2c_refinement_forward_dual <- the same, also emitting the output in the compute type for the decoder that follows (:313-320)
 *   b2c_projector_forward/backward  <- FeatureProjector.forward (+ autograd)      src/distillation_utils.py:203-252
 *   b2c_count_valid       <- CrossEntropyLoss(ignore_index=0) normaliser  src/distillation_utils.py:22
 *   b2c_kd_token_loss     <- token_level_distillation :30-54 + CE term :154 (+ their gradient)
 *   b2c_kd_token_loss_pitched / b2c_decoder_backward_pitched <- the same two calls with the logits gradient at a padded row pitch
 *   *_steps               <- the training calls for a batch of fewer steps than shape->T (data_loader.py pads each batch to its own
 *                            longest caption): a device step count, so one CUDA graph serves every caption length
 *   b2c_kd_token_eval     <- validate_student_model: loss without gradients + logits.argmax(-1)   src/train_student_kd.py:29-86
 *   b2c_bleu1             <- compute_bleu_score (per sample, on the device)                       src/distillation_utils.py:398-409
 *   b2c_aux_loss          <- encoder_feature_distillation :56-94 + decoder_hidden_state_distillation :96-136
 *   b2c_loss_finalize     <- the alpha/beta/gamma weighting and loss_dict  :184-198
 *   b2c_scale_inplace     <- the scalar grad_output of loss.backward() (GradScaler / accumulation, train_student_kd.py:285-288)
 *   b2c_optimizer_step    <- scaler.unscale_ + clip_grad_norm_ (x2) + AdamW.step + scaler.update   src/train_student_kd.py:230-236,290-303
 *   b2c_set_gemm_cta_limit <- (no reference counterpart) CTA budget for calls a host overlaps with the decoder's recurrences
 *   b2c_gemm              <- test hook for the tcgen05 / SIMT contraction tiles used inside the decoder
 *
 * Conventions
 *   - Plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host.
 *   - The caller (PyTorch) owns every buffer; the library allocates nothing per call and keeps no pointer.
 *   - All work is enqueued on `stream` (a cudaStream_t passed as void*); calls are asynchronous.
 *   - Return 0 on success, a negative B2C_E* code otherwise; message via b2c_last_error() (thread local).
 *   - `dtype` selects the precision mode: B2C_F32 (parity mode: fp32 storage + FFMA contractions) or
 *     B2C_BF16 (throughput mode: bf16 storage, tcgen05 contractions, fp32 accumulation and cell state).
 *   - `teacher_dtype` (the *_teacher entry points) is the element type of the teacher's outputs: B2C_F32, B2C_BF16 or B2C_F16, as
 *     a teacher run under autocast or a half-precision cache of its outputs leaves them.  The kernels widen half-precision values
 *     to fp32 exactly as they load them, so the results are bit-identical to those for the same values given as fp32.
 *     Each entry point without the suffix is its _teacher form with teacher_dtype = B2C_F32.
 *   - Time-major layouts like the reference: captions/targets (T,B) int64, logits (T,B,V).
 *   - There is no CPU fallback.
 */
#ifndef B2C_H_
#define B2C_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2C_ABI_VERSION 5
#define B2C_MAX_LAYERS 4

enum { B2C_OK = 0, B2C_EINVAL = -1, B2C_EARCH = -2, B2C_ECUDA = -3, B2C_ENOMEM = -4 };
enum { B2C_F32 = 0, B2C_BF16 = 1, B2C_F16 = 2 };      /* B2C_F16: a teacher_dtype only, never a compute dtype */
enum { B2C_WS_TRAIN = 0, B2C_WS_DECODE = 1, B2C_WS_ATTN = 2, B2C_WS_REFINE = 3, B2C_WS_PROJ = 4 };

/* B batch (per GPU), T decode steps, S image tokens (49), E embed, H hidden, L LSTM layers, V vocab. */
typedef struct B2CShape { int32_t B, T, S, E, H, L, V; } B2CShape;

/* fp32 master parameters of LSTMDecoder in the reference's own layouts (src/student_model.py:125-165);
 * field <-> state_dict key:  embedding = decoder.embedding.weight (V,E); attn_w/attn_b = decoder.attention
 * (E,H+E)/(E) [hidden columns first]; comb_w/comb_b = decoder.attention_combine (E,2E)/(E) [embedding
 * columns first]; w_ih[k] (4H,in_k), w_hh[k] (4H,H), b_ih[k], b_hh[k] (4H) = decoder.lstm.*_l{k}, gate order
 * i,f,g,o; out0_* = decoder.output_projection.0 (E,H); out3_* = decoder.output_projection.3 (V,E). */
typedef struct B2CParams {
  const float* embedding;
  const float* attn_w;  const float* attn_b;
  const float* comb_w;  const float* comb_b;
  const float* w_ih[B2C_MAX_LAYERS]; const float* w_hh[B2C_MAX_LAYERS];
  const float* b_ih[B2C_MAX_LAYERS]; const float* b_hh[B2C_MAX_LAYERS];
  const float* out0_w;  const float* out0_b;
  const float* out3_w;  const float* out3_b;
} B2CParams;

/* fp32 gradients, same layouts; every buffer is overwritten (not accumulated into). */
typedef struct B2CGrads {
  float* embedding;
  float* attn_w;  float* attn_b;
  float* comb_w;  float* comb_b;
  float* w_ih[B2C_MAX_LAYERS]; float* w_hh[B2C_MAX_LAYERS];
  float* b_ih[B2C_MAX_LAYERS]; float* b_hh[B2C_MAX_LAYERS];
  float* out0_w;  float* out0_b;
  float* out3_w;  float* out3_b;
} B2CGrads;

/* Dropout of the reference's training mode (decoder p in output_projection and between LSTM layers,
 * src/student_model.py:142-156).  p == 0 disables it (eval mode / parity runs).  The keep mask is a
 * counter-based hash of (seed, site, element index): backward regenerates it, nothing is stored.
 * seed_dev (may be NULL): a device counter that is mixed into the seed by the kernels at run time, so a captured CUDA graph
 * (whose kernel arguments, `seed` included, are frozen at capture) draws a fresh mask on every replay: the caller bumps the
 * counter once per step, before the forward (b2c_bump_counter), and passes the same pointer to forward and backward. */
typedef struct B2CDropout { float p; uint64_t seed; const uint64_t* seed_dev; } B2CDropout;
/* *counter += 1 (device, on `stream`): the per-step dropout counter of B2CDropout.seed_dev. */
int b2c_bump_counter(uint64_t* counter, void* stream);

int b2c_abi_version(void);
const char* b2c_last_error(void);
/* Number of kernels this library has launched so far in this process (bench.py reports the per-step delta). */
uint64_t b2c_launch_count(void);

/* Bytes of caller-provided workspace for mode B2C_WS_TRAIN (forward saves + backward scratch) or
 * B2C_WS_DECODE (greedy decode; shape->T = max_len).  0 on invalid shape. */
size_t b2c_workspace_bytes(const B2CShape* shape, int dtype, int mode);

/* LSTMDecoder.forward with hidden=None.  feats (B,S,E) [dtype]; captions (T,B) int64;
 * out: logits (T,B,V) [dtype], hidden_top (T,B,H) [dtype] (top-layer h_t), attn_w (T,B,S) fp32.
 * The workspace keeps what backward needs and must be passed unchanged to b2c_decoder_backward. */
int b2c_decoder_forward(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                        void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                        int dtype, const B2CDropout* dropout, void* stream);

/* Validation forward WITHOUT materialising the logits (validate_student_model, src/train_student_kd.py:29-86; SURVEY.md section 8f
 * row 4): the teacher-forced decoder forward in eval mode whose vocabulary-head contraction reduces every accumulator tile, in its
 * epilogue, to per-row partials of the token-KD term, the CE term and the argmax against the teacher logits it streams alongside
 * (online-softmax form); a second small kernel merges the partials.  Outputs as b2c_kd_token_eval: row_kl (T*B), row_ce (T*B, 0 on
 * PAD rows), argmax_out (T*B, may be NULL) = student_logits.argmax(-1); hidden_top / attn_w as b2c_decoder_forward.  bf16 mode only.
 * The (T,B,V) logits are never written: 102 MB less written and 102 MB less read at BASELINE configs[1] sizes. */
int b2c_decoder_forward_eval(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                             const float* teacher_logits, const int64_t* targets, float temperature,
                             void* hidden_top, float* attn_w, float* row_kl, float* row_ce, int32_t* argmax_out,
                             void* workspace, size_t ws_bytes, int dtype, void* stream);
/* b2c_decoder_forward_eval on teacher logits of element type teacher_dtype: the epilogue streams them in that type. */
int b2c_decoder_forward_eval_teacher(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                     const void* teacher_logits, int teacher_dtype, const int64_t* targets, float temperature,
                                     void* hidden_top, float* attn_w, float* row_kl, float* row_ce, int32_t* argmax_out,
                                     void* workspace, size_t ws_bytes, int dtype, void* stream);

/* The part of b2c_decoder_forward that does not read the image features: operand packing (compute-type copies of the weights,
 * attention_combine folded into layer 0), the embedding rows of `captions`, the time-batched embedding half of layer 0's
 * gates and the zero initial state, all written into `workspace` (mode B2C_WS_TRAIN).  It may be enqueued on a different
 * stream while the features are still being produced (e.g. under AttentionRefinement); b2c_decoder_forward_prepared then
 * does the rest.  The caller orders the two calls (event / stream wait); shape, params, captions, workspace and dtype must be
 * identical in both.  b2c_decoder_forward == b2c_decoder_prepare + b2c_decoder_forward_prepared on one stream. */
int b2c_decoder_prepare(const B2CShape* shape, const B2CParams* params, const int64_t* captions, void* workspace, size_t ws_bytes,
                        int dtype, void* stream);
int b2c_decoder_forward_prepared(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                        void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                        int dtype, const B2CDropout* dropout, void* stream);

/* LSTMDecoder.forward(image_features, captions, hidden) with a caller-supplied initial state (reference src/student_model.py:205,
 * :219-222: `hidden` replaces init_hidden's zeros and seeds nn.LSTM at :243).  h0, c0: (L,B,H) fp32 on the device.  Call it between
 * b2c_decoder_prepare (which writes the zero state) and b2c_decoder_forward_prepared, on the same stream as the latter; the backward
 * then differentiates through the non-zero state (no gradient with respect to h0 / c0 is returned). */
int b2c_decoder_set_initial_state(const B2CShape* shape, const float* h0, const float* c0, void* workspace, size_t ws_bytes,
                                  int dtype, void* stream);

/* Backward of b2c_decoder_forward.  dlogits (T,B,V) [dtype]; dhidden_top (T,B,H) [dtype] or NULL;
 * hidden_top / attn_w are the forward outputs.  out: grads (fp32, all fields), dfeats (B,S,E) fp32. */
int b2c_decoder_backward(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                         const void* hidden_top, const float* attn_w, const void* dlogits, const void* dhidden_top,
                         const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                         int dtype, const B2CDropout* dropout, int flags, void* stream);

/* b2c_decoder_backward with the logits gradient at row pitch ld_dlogits >= V (elements): row r of dlogits starts at
 * dlogits + r * ld_dlogits, and only its first V columns are read.  The caller owns the buffer.  In bf16 mode a pitch with
 * ld_dlogits % 8 == 0 and a 16-byte-aligned dlogits lets the vocabulary head's data-gradient and weight-gradient contractions
 * run on tensor cores for any V (TMA needs 16-byte row pitches); with ld_dlogits == V this is b2c_decoder_backward. */
int b2c_decoder_backward_pitched(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                 const void* hidden_top, const float* attn_w, const void* dlogits, int64_t ld_dlogits, const void* dhidden_top,
                                 const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                                 int dtype, const B2CDropout* dropout, int flags, void* stream);

/* ---- Variable-length batches.  The *_steps entry points take `steps`, a device int32 scalar with 1 <= *steps <= shape->T (NULL
 * means shape->T): the buffers keep their shape->T-step layout, and the call computes what the plain call computes for a batch of
 * the first *steps steps.  The value is read by the kernels when they run, so a CUDA graph captured once at a capacity T replays
 * for any length up to it.  It must be written before the call on `stream` and not change until the call's work is complete.
 *   - forward: the rows of steps >= *steps of logits are unspecified, those of hidden_top and attn_w are zeros;
 *   - backward: the rows of steps >= *steps of dlogits and dhidden_top must be zeros (b2c_kd_token_loss_steps and b2c_aux_loss_steps
 *     write them so); the gradients are those of the *steps-step batch;
 *   - the recurrences launch their per-step kernels for all shape->T steps, and the ones past *steps return at once; the
 *     whole-sequence recurrence kernels (B2C_PERSISTENT, B2C_CLUSTER), sub-batch streams (B2C_SUB_BATCHES) and weight-gradient
 *     chunks under the reverse loop (B2C_WGRAD_CHUNKS) are not used. */
int b2c_decoder_forward_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                              void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                              int dtype, const B2CDropout* dropout, const int32_t* steps, void* stream);
int b2c_decoder_forward_prepared_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                       void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                                       int dtype, const B2CDropout* dropout, const int32_t* steps, void* stream);
/* b2c_decoder_backward_pitched with a step count (ld_dlogits == V: contiguous dlogits). */
int b2c_decoder_backward_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                               const void* hidden_top, const float* attn_w, const void* dlogits, int64_t ld_dlogits, const void* dhidden_top,
                               const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                               int dtype, const B2CDropout* dropout, int flags, const int32_t* steps, void* stream);

/* b2c_decoder_backward contracts every weight gradient on an internal (per-device) side stream next to the chain that produces
 * dfeats, and by default makes `stream` wait for that branch before it returns ("all work is enqueued on stream").  A caller that
 * does not read parameter gradients until later (an optimizer step after the rest of the backward) passes
 * flags = B2C_BWD_DEFER_JOIN so that whatever it enqueues next (the refinement backward) overlaps the weight-gradient
 * contractions, and calls b2c_join_side_work(stream) before the gradients are read.  The choice is per call: there is no
 * process-wide state besides the per-device stream / event set. */
#define B2C_BWD_DEFER_JOIN 1
int b2c_join_side_work(void* stream);

/* Background hint for the CALLING THREAD's subsequent b2c calls: their tensor-core contractions use at most `max_ctas` CTAs
 * (0 = no limit, the default).  The GEMM kernels are persistent -- a CTA keeps its SM until the kernel ends -- so a caller that
 * overlaps one b2c call on a side stream with a latency-bound one on another stream (e.g. b2c_projector_backward next to the reverse
 * recurrence of b2c_decoder_backward) wraps the background call in b2c_set_gemm_cta_limit(20) ... b2c_set_gemm_cta_limit(0). */
int b2c_set_gemm_cta_limit(int32_t max_ctas);

/* Batched greedy decode: every sample starts at start_id and steps shape->T (= max_len) times with its own
 * argmax fed back on the device (no host sync per token).  out: tokens (T,B) int64; lengths (B) int32 =
 * number of tokens emitted before the first end_id (T if none) == len(caption_image(...)). */
int b2c_greedy_decode(const B2CShape* shape, const B2CParams* params, const void* feats, int64_t start_id, int64_t end_id,
                      int64_t* tokens, int32_t* lengths, void* workspace, size_t ws_bytes, int dtype, void* stream);

/* One stand-alone attention step: hidden (B,H), feats (B,S,E) [dtype] -> context (B,E) [dtype], weights (B,S) fp32.
 * Only shape->{B,S,E,H} are read; workspace size from b2c_workspace_bytes(shape, dtype, B2C_WS_ATTN). */
int b2c_attention_step(const B2CShape* shape, const float* attn_w, const float* attn_b, const void* hidden, const void* feats,
                       void* context, float* weights, void* workspace, size_t ws_bytes, int dtype, void* stream);

/* ---- AttentionRefinement: x1 = LN1(x + MHA(x)), out = LN2(x1 + FFN(x1)); nn.MultiheadAttention(batch_first) packing:
 * in_w (3E,E) / in_b (3E) = in_proj_{weight,bias}, out_w (E,E) / out_b = out_proj; ffn0 (2E,E), ffn3 (E,2E); n1 / n2 = LayerNorm
 * weight, bias.  Workspace: b2c_workspace_bytes with shape {B, S, E, H = heads}, mode B2C_WS_REFINE. */
typedef struct B2CRefineParams {
  const float *in_w, *in_b, *out_w, *out_b, *ffn0_w, *ffn0_b, *ffn3_w, *ffn3_b, *n1_w, *n1_b, *n2_w, *n2_b;
} B2CRefineParams;
typedef struct B2CRefineGrads {
  float *in_w, *in_b, *out_w, *out_b, *ffn0_w, *ffn0_b, *ffn3_w, *ffn3_b, *n1_w, *n1_b, *n2_w, *n2_b;
} B2CRefineGrads;
/* x (B,S,E) fp32 -> out (B,S,E) fp32 in both modes: the residual stream (x, LN1's output, out) is carried in fp32 like torch.autocast
 * does (LayerNorm runs in fp32 there); `dtype` selects the type of the contraction operands and of the branch activations.
 * dropout->p is the reference's 0.1 in training (attention probabilities and FFN), 0 in eval. */
int b2c_refinement_forward(const B2CShape* shape, const B2CRefineParams* params, const float* x, float* out,
                           void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);
/* The same forward that ALSO leaves the output in the compute type (`out_compute`, (B,S,E) of `dtype`, may be NULL): the decoder
 * consumes the refined features in the compute type (TMA operands), and taking them from the final LayerNorm saves the separate
 * fp32 -> bf16 pass over the features that would otherwise sit between the two calls on the critical path. */
int b2c_refinement_forward_dual(const B2CShape* shape, const B2CRefineParams* params, const float* x, float* out, void* out_compute,
                                void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);
/* x = the forward's input, dout (B,S,E) fp32 -> grads (fp32, overwritten), dx (B,S,E) fp32. */
int b2c_refinement_backward(const B2CShape* shape, const B2CRefineParams* params, const float* x, const float* dout, const B2CRefineGrads* grads,
                            float* dx, void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);

/* ---- FeatureProjector: LN(Drop(ReLU(x W^T + b))) on the channel axis, then AdaptiveAvgPool1d over tokens St -> So.
 * w (Es,Et), b (Es), ln_w / ln_b (Es); all four NULL = identity channel projection (Et == Es): pooling only.
 * Workspace: shape {B, S = St, E = Et, H = Es, T = So}, mode B2C_WS_PROJ. */
typedef struct B2CProjParams { const float *w, *b, *ln_w, *ln_b; } B2CProjParams;
typedef struct B2CProjGrads { float *w, *b, *ln_w, *ln_b; } B2CProjGrads;
/* x (B,St,Et) fp32 (teacher features, no gradient) -> out (B,So,Es) fp32 */
int b2c_projector_forward(const B2CShape* shape, const B2CProjParams* params, const float* x, float* out,
                          void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);
/* b2c_projector_forward on teacher features x of element type teacher_dtype (in either compute mode).  The backward is unchanged:
 * it reads the compute-type copy of x the forward keeps in the workspace. */
int b2c_projector_forward_teacher(const B2CShape* shape, const B2CProjParams* params, const void* x, int teacher_dtype, float* out,
                                  void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);
/* dout (B,So,Es) fp32 -> grads (fp32, overwritten) */
int b2c_projector_backward(const B2CShape* shape, const B2CProjParams* params, const float* dout, const B2CProjGrads* grads,
                           void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream);

/* n_valid_out[0] = #{ i < n : 0 < targets[i] < V }   (int32 on the device). */
int b2c_count_valid(const int64_t* targets, int64_t n, int32_t V, int32_t* n_valid_out, void* stream);

/* Streaming token pass over N = T*B rows of V logits: one read of student logits [dtype] and teacher logits
 * (fp32), one write of dlogits [dtype]:
 *   row_kl[r] = KL(softmax(z_r/Temp) || softmax(y_r/Temp)),  row_ce[r] = logsumexp(y_r) - y_r[tgt] (0 on PAD rows)
 *   dlogits   = alpha*Temp/N * (pS - pT) + w_ce*ce_mult/n_valid * [tgt != 0] * (softmax(y) - onehot(tgt))
 * n_valid points at the (global, under data parallelism) non-PAD count on the device; ce_mult = world size. */
int b2c_kd_token_loss(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                      int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                      const int32_t* n_valid, void* dlogits, float* row_kl, float* row_ce, int dtype, void* stream);

/* b2c_kd_token_loss writing dlogits at row pitch ld_dlogits >= V (elements); the student and teacher logits keep pitch V.  The caller
 * owns dlogits, (N, ld_dlogits) elements.  In bf16 mode with ld_dlogits % 8 == 0, ld_dlogits >= roundup(V, 8) and a 16-byte-aligned
 * dlogits (any V <= 16384, any alignment of the logits) the rows are streamed by the TMA-pipelined pass and written with 16-byte
 * stores; columns V .. roundup(V, 8) - 1 of every row are written as exact zeros, columns beyond that are not written.  Any other
 * pitched call (fp32 mode, or a pitch that misses those conditions) returns B2C_EINVAL unless ld_dlogits == V, which is
 * b2c_kd_token_loss. */
int b2c_kd_token_loss_pitched(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                              int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                              const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype, void* stream);

/* b2c_kd_token_loss_pitched with a step count over N = T * rows_per_step rows (rows_per_step = B): the n = *steps * rows_per_step
 * first rows are computed with the KD scale alpha*Temp/n; the rows past them are never used (a few bytes of row n may be fetched with
 * the last row's enclosing 16-byte range), and get row_kl = row_ce = 0 and a dlogits row of zeros (padding columns included).
 * The caller keeps the targets of those rows PAD (0), so n_valid (b2c_count_valid over all N rows) is that of the n rows. */
int b2c_kd_token_loss_steps(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                            int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                            const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype,
                            const int32_t* steps, int64_t rows_per_step, void* stream);

/* The token pass on teacher logits of element type teacher_dtype: the arguments of b2c_kd_token_loss_steps, where steps == NULL is a
 * batch of all N rows and ld_dlogits == V a contiguous dlogits, so this covers b2c_kd_token_loss, _pitched and _steps. */
int b2c_kd_token_loss_teacher(const void* student_logits, const void* teacher_logits, int teacher_dtype, const int64_t* targets,
                              int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                              const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype,
                              const int32_t* steps, int64_t rows_per_step, void* stream);

/* Evaluation form of the token pass (validate_student_model, src/train_student_kd.py:29-86): the same per-row KL and CE partials,
 * NO gradient, plus (argmax_out != NULL) the teacher-forced prediction argmax_v student_logits[r, v] of every row (lowest index on
 * ties, like torch.argmax) from the same read of the logits -- `student_logits.argmax(dim=-1)` (:74) without a second pass. */
int b2c_kd_token_eval(const void* student_logits, const float* teacher_logits, const int64_t* targets, int64_t N, int32_t V,
                      float temperature, const int32_t* n_valid, float* row_kl, float* row_ce, int32_t* argmax_out, int dtype, void* stream);

/* b2c_kd_token_eval on teacher logits of element type teacher_dtype. */
int b2c_kd_token_eval_teacher(const void* student_logits, const void* teacher_logits, int teacher_dtype, const int64_t* targets, int64_t N,
                              int32_t V, float temperature, const int32_t* n_valid, float* row_kl, float* row_ce, int32_t* argmax_out,
                              int dtype, void* stream);

/* compute_bleu_score (src/distillation_utils.py:398-409) for every sample of a batch on the device: predicted (T,B) int32,
 * targets (T,B) int64 -> bleu_out (B) = |set(pred) & set(target)| / |set(target)| over token ids outside {PAD=0, START=1, END=2}
 * (0 when the target set is empty).  Token ids stand for the words (vocab.itos is one-to-one). */
int b2c_bleu1(const int32_t* predicted, const int64_t* targets, int32_t T, int32_t B, float* bleu_out, void* stream);

/* Fused feature-KD + hidden-KD reduction and gradients.
 *   feats_s (B,Ss,E) [feat_dtype] or NULL, feats_t (B,St,E) fp32 (the projected teacher features).  feat_dtype may be B2C_F32 in
 *   bf16 mode: the student's UN-refined encoder features reach the loss in fp32 (src/student_model.py:301-312), and the pooled
 *   term takes a softmax over token sums of E of them, where bf16 rounding of the inputs costs ~3 % in the pooling weights;
 *   hid_s (T,B,H) [dtype] or NULL, hid_t (Th,B,H) fp32, Th <= T steps are compared (list truncation).
 *   out: dfeats_s, dfeats_t (fp32, scaled by beta; may be NULL), dhid_s (T,B,H) [dtype] scaled by gamma (may be NULL),
 *   feat_part (B*2) and hid_part (Th*B*2) fp32 partials consumed by b2c_loss_finalize. */
int b2c_aux_loss(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                 const void* hid_s, const float* hid_t, int32_t T, int32_t Th, int32_t H,
                 float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                 float* feat_part, float* hid_part, int dtype, int feat_dtype, void* stream);

/* b2c_aux_loss with a step count: hidden KD over the first min(Th, *steps) steps (the steps past them are not read, get zero
 * partials and a zero dhid_s, and the mean over steps divides by min(Th, *steps)); feature KD is unchanged. */
int b2c_aux_loss_steps(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                       const void* hid_s, const float* hid_t, int32_t T, int32_t Th, int32_t H,
                       float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                       float* feat_part, float* hid_part, int dtype, int feat_dtype, const int32_t* steps, void* stream);

/* b2c_aux_loss_steps (steps may be NULL: all steps) with teacher hidden states hid_t of element type hid_t_dtype.  feats_t stays
 * fp32: it is the projector's output, and dfeats_t flows back into the projector. */
int b2c_aux_loss_teacher(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                         const void* hid_s, const void* hid_t, int hid_t_dtype, int32_t T, int32_t Th, int32_t H,
                         float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                         float* feat_part, float* hid_part, int dtype, int feat_dtype, const int32_t* steps, void* stream);

/* out5 = { total, ce, token_kd, feature_kd, hidden_kd } (device, fp32); fixed-order fp64 reduction. */
int b2c_loss_finalize(const float* row_kl, const float* row_ce, int64_t N, const int32_t* n_valid, float ce_mult,
                      const float* feat_part, int32_t B, int32_t E, const float* hid_part, int32_t Th, int32_t H,
                      float temperature, float alpha, float beta, float gamma, float w_ce, float* out5, void* stream);
/* b2c_loss_finalize with a step count: token KD divided by *steps * B rows, hidden KD by min(Th, *steps) steps. */
int b2c_loss_finalize_steps(const float* row_kl, const float* row_ce, int64_t N, const int32_t* n_valid, float ce_mult,
                            const float* feat_part, int32_t B, int32_t E, const float* hid_part, int32_t Th, int32_t H,
                            float temperature, float alpha, float beta, float gamma, float w_ce, float* out5, const int32_t* steps,
                            void* stream);

/* p[i] *= *scale for i < n  (scale is a device fp32 scalar: autograd's grad_output). */
int b2c_scale_inplace(void* p, int64_t n, int dtype, const float* scale, void* stream);

/* ---- optimizer side of the step on flat fp32 buffers (every trainable parameter, its gradient and both Adam moments laid
 * out in the same order in four equally long arrays).
 * A segment is a run of parameters that share a learning rate, a weight decay and a clip group: the reference builds
 * AdamW with three LR groups (encoder 0.1*lr, decoder lr, refinement + projectors lr; weight_decay 0.01;
 * src/train_student_kd.py:230-234) and clips student_model.parameters() and each projector's parameters separately with
 * max_norm 1.0 (:293-297), i.e. two clip groups.  Segments must start on a multiple of 4 elements. */
#define B2C_OPT_MAX_SEG 8
#define B2C_OPT_MAX_CLIP 4
#define B2C_OPT_SCRATCH_BYTES 16384      /* device scratch; zero-filled ONCE by the caller before the first call */
#define B2C_OPT_NSTATS (B2C_OPT_MAX_CLIP + 2)
typedef struct {
  int64_t begin, end;      /* [begin, end) in elements; begin % 4 == 0 */
  int32_t lr_index;        /* which entry of the device array lr[] */
  int32_t clip_group;      /* 0 .. B2C_OPT_MAX_CLIP-1: gradients of one group share one global L2 norm; -1: never clipped */
  float weight_decay;      /* decoupled (AdamW): p *= 1 - lr * weight_decay */
} B2COptSegment;
typedef struct {
  double beta1, beta2, eps; /* torch.optim.AdamW defaults 0.9, 0.999, 1e-8 (doubles, as in torch: 1 - beta is formed in fp64) */
  float max_norm;          /* clip_grad_norm_ threshold per clip group; <= 0 disables clipping */
  float grad_scale;        /* every gradient is multiplied by this first (1/world after a SUM all-reduce; 1 otherwise) */
  float growth_factor, backoff_factor;   /* torch.amp.GradScaler defaults 2.0, 0.5 */
  int32_t growth_interval;               /* default 2000; only read when loss_scale != NULL */
} B2COptHyper;

/* One optimizer step, two kernel launches, no host synchronisation:
 *   g' = grad * grad_scale / *loss_scale (data-parallel average + unscale_);  if any g' is non-finite the parameters, the moments and *step are left untouched
 *   (scaler.step skips) and *loss_scale is multiplied by backoff_factor;  otherwise each clip group is scaled by
 *   min(1, max_norm / (||g'||_2 + 1e-6)) and AdamW is applied with bias correction for step *step + 1, *step is
 *   incremented, and *loss_scale grows by growth_factor after growth_interval consecutive clean steps (scaler.update).
 * lr (device, one float per LR group) is read by the kernel, so a scheduler can change it between CUDA-graph replays.
 * loss_scale / growth_tracker may be NULL (no loss scaling: bf16 autocast).  grad is not modified.
 * stats (device, B2C_OPT_NSTATS floats, may not be NULL): [g] = unscaled pre-clip norm of clip group g,
 * [B2C_OPT_MAX_CLIP] = 1 if the step was skipped, [B2C_OPT_MAX_CLIP+1] = the loss scale that was applied. */
int b2c_optimizer_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                       const B2COptSegment* segments_host, int32_t n_segments, const B2COptHyper* hyper_host,
                       const float* lr, int32_t n_lr, int32_t* step, float* loss_scale, int32_t* growth_tracker,
                       float* stats, void* scratch, void* stream);

/* Debug aid: with B2C_RECUR_TRACE=1 in the environment the persistent forward-recurrence kernel stamps clock64() at its phase
 * boundaries (per CTA, per time step, 8 stamps); this copies the last launch's stamps to the host (synchronises the device). */
int b2c_debug_recur_trace(uint64_t* out_host, int64_t n, int32_t* grid_out, int32_t* steps_out);

/* C[m,n] = act(alpha * sum_k A(m,k) B(n,k) + bias[n]) + beta*C[m,n];  a_mn/b_mn = 1 when the operand is stored
 * MN-major (A[k*lda+m]) instead of K-major (A[m*lda+k]).  dtype = operand type; c_dtype = output type.
 * impl: 0 = the mode's default (tcgen05 for bf16 when TMA can describe the operands, FFMA otherwise), 1 = force FFMA tiles. */
int b2c_gemm(int32_t M, int32_t N, int32_t K, float alpha, const void* A, int64_t lda, int a_mn,
             const void* B, int64_t ldb, int b_mn, float beta, void* C, int64_t ldc, const float* bias, int relu,
             int dtype, int c_dtype, int impl, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2C_H_ */
