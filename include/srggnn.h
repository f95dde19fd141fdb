/*
 * srggnn.h -- C ABI of libsrggnn.so: the B200 (sm_100a) implementation of the GGNN role-graph stage of
 * vFones/situation-recognition.  The reference has no FFI layer (its boundary is the Python class API of
 * model.py), so every entry point below cites the reference code it replaces.  The Python host side
 * (situation_recognition_b200/) binds these with ctypes; INTEGRATION.md shows the stub a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - all tensor pointers are DEVICE pointers owned by the caller (torch `tensor.data_ptr()`), row-major;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = OK, non-zero = error; srg_last_error() returns a thread-local message;
 *   - no exceptions cross the ABI; a handle is bound to one device and is not thread-safe;
 *   - there is NO CPU fallback: on a machine without an sm_100a GPU every compute call fails.
 */
#ifndef SRGGNN_H_
#define SRGGNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct srg_handle srg_handle;

enum { SRG_DT_F32 = 1, SRG_DT_BF16 = 2 };
/* arithmetic of the tensor-core contractions:
 *   SRG_PREC_BF16 : bf16 operands, fp32 accumulate (training / throughput mode)
 *   SRG_PREC_FP32 : every operand split into three bf16 parts x = hi + mid + lo, a product expanded into the six terms
 *                   of weight >= 2^-16 (hi*hi + hi*mid + mid*hi + hi*lo + lo*hi + mid*mid), fp32 accumulate --
 *                   fp32-parity mode, forward only */
enum { SRG_PREC_BF16 = 0, SRG_PREC_FP32 = 1 };
/* GGSNN.forward(..., verb=True|False), model.py:59-77 */
enum { SRG_MODE_NOUN = 0, SRG_MODE_VERB = 1 };

const char* srg_last_error(void);
int srg_version(void);

/* FCGGNN.__init__ (model.py:90-111): D = hidden size (2048), R = encoder.get_max_role_count() (6), T = 4 (model.py:60),
 * n_verbs/n_roles/n_labels = encoder.get_num_{verbs,roles,labels}().  srg_set_cta_group selects 1 or 2 CTAs per
 * tcgen05.mma (default 2: M=256 x N=256 tiles on a CTA pair; 1 = 128 x 128 tiles, kept for tests). */
int srg_create(srg_handle** out, int device, int D, int R, int T, int n_verbs, int n_roles, int n_labels);
int srg_destroy(srg_handle* h);
int srg_set_cta_group(srg_handle* h, int cta_group);

/* Row layout of the role-graph paths (srg_nouns_forward / srg_nouns_backward).  on = 1 (default): only the REAL role
 * nodes of an image (n = encoder.get_role_count(verb) of its R slots) are materialised as rows, plus ONE shared pad row
 * per call: pad nodes start at the zero padding_idx embedding and only see themselves (model.py:95-97,
 * imsitu_encoder.py:223-225), so all pad nodes of a batch follow one trajectory that depends on the weights only.  The
 * row count is a function of the verb ids, which for the predicted-verb path exist only on the device: it stays there
 * (the kernels read it), so a step has no host synchronisation.  Logits still come out for all B*R slots.
 * on = 0: R rows per image, as the reference lays them out (A/B measurements). */
int srg_set_compact_rows(srg_handle* h, int on);

/* imsitu_encoder.roles_to_verb_tensor_list (imsitu_encoder.py:71-89) and get_role_count (158-159) as flat host tables:
 * verb2roles[v*R + r] (pad value = n_roles), role_count[v]. */
int srg_set_tables(srg_handle* h, const int32_t* verb2roles, const int32_t* role_count);

/* imsitu_encoder.get_role_ids_batch (imsitu_encoder.py:172-180) + get_adj_matrix_noself (209-229), bit-exact:
 * role_idx[b,r] = verb2roles[verb[b], r];  mask[b,i,j] = (i<n && j<n && i!=j) || (i>=n && i==j), n = role_count[verb[b]].
 * Either output may be NULL.  Returns an error flag in *bad_verb (device int, nullable) if a verb id is out of range. */
int srg_gather_mask(srg_handle* h, const int64_t* verb, int B, int64_t* role_idx, float* mask, int* bad_verb,
                    void* stream);

/* The role-graph forward calls clamp a verb id outside [0, n_verbs) to 0 (the reference raises an IndexError,
 * imsitu_encoder.py:172-180) and raise a device flag.  srg_check_verbs synchronises `stream`, returns an error if the
 * flag was raised since the last check, and clears it.  Debugging aid: it costs a host synchronisation. */
int srg_check_verbs(srg_handle* h, void* stream);

/* The 7 shared GGSNN linears + both classifiers (model.py:47-56,105-111); fp32, nn.Linear layout [out, in]. */
typedef struct srg_params {
  const float *W_p, *b_p;
  const float *W_z, *b_Wz, *U_z, *b_Uz;
  const float *W_r, *b_Wr, *U_r, *b_Ur;
  const float *W_h, *b_Wh, *U_h, *b_Uh;
  const float *Wc_verb, *bc_verb;   /* verb_classifier.1 : [n_verbs, D]  */
  const float *Wc_noun, *bc_noun;   /* nouns_classifier.1: [n_labels, D] */
} srg_params;

/* Gradient accumulators (fp32, same shapes as srg_params; kernels ACCUMULATE into them, caller zeroes). */
typedef struct srg_grads {
  float *W_p, *b_p;
  float *W_z, *b_Wz, *U_z, *b_Uz;
  float *W_r, *b_Wr, *U_r, *b_Ur;
  float *W_h, *b_Wh, *U_h, *b_Uh;
  float *Wc_verb, *bc_verb;
  float *Wc_noun, *bc_noun;
  float *role_emb;   /* [n_roles+1, D] (padding row never touched) */
  float *verb_emb;   /* [n_verbs, D] */
} srg_grads;

/* Convert/pack the fp32 parameters into the bf16 tensor-core operand layout held by the handle.
 * Must be called after every optimizer step (weights changed) and before the forward calls. */
int srg_pack_weights(srg_handle* h, const srg_params* p, int precision, void* stream);

/* Bytes of caller-provided workspace needed by one forward(+backward) pass over the graph nodes of B images
 * (B*R node slots + the shared pad row for SRG_MODE_NOUN -- sized for the worst case of R real roles per image --
 * B nodes for SRG_MODE_VERB). */
size_t srg_workspace_bytes(srg_handle* h, int mode, int B, int precision, int save_for_backward);

/* predict_nouns minus the backbone (model.py:117-155):
 *   role gather + mask (117,147) -> node = relu(feat * role_emb[role_idx] * verb_emb[verb]) (124-144)
 *   -> GGSNN(node, mask) (151) -> Dropout + Linear (152) -> logits[B*R, ldl] (first n_labels columns valid).
 * feat: fp32 [B, D]; verb: int64 [B].
 * Dropout (model.py:110, training mode only; drop_p = 0 or both sources NULL = identity):
 *   keep      : explicit uint8 keep-mask [B*R, D] (parity tests), or NULL;
 *   drop_seed : device int64 scalar; with keep == NULL the keep decisions are Bernoulli(1 - drop_p) draws of a
 *               counter-based Philox4x32-10 generator keyed by (*drop_seed, drop_stream, slot row, column), regenerated
 *               identically by the matching backward call -- no mask is stored or read.  drop_stream separates the
 *               paths of one step that share a seed (FCGGNN uses 0 = verb, 1 = predicted-verb nouns, 2 = gt-verb nouns).
 * The role ids / row layout stay inside the workspace; srg_gather_mask returns ids and mask when a caller wants them. */
int srg_nouns_forward(srg_handle* h, const float* feat, const int64_t* verb, int B, const float* role_emb,
                      const float* verb_emb, const uint8_t* keep, float drop_p, const int64_t* drop_seed,
                      int64_t drop_stream, float* logits, int64_t ldl, int precision, int save_for_backward,
                      void* workspace, size_t workspace_bytes, void* stream);

/* predict_verb minus the backbone (model.py:160-168): node = relu(feat) -> GGSNN(verb=True) -> Dropout + Linear.
 * keep: uint8 [B, D]; dropout arguments as above. */
int srg_verb_forward(srg_handle* h, const float* feat, int B, const uint8_t* keep, float drop_p,
                     const int64_t* drop_seed, int64_t drop_stream, float* logits, int64_t ldl, int precision,
                     int save_for_backward, void* workspace, size_t workspace_bytes, void* stream);

/* Row-wise top-k + log-softmax: for each of `rows` rows of logits [rows, ldl], the k largest of the first n columns in
 * descending order (ties go to the lower column, as torch.argmax and a stable descending sort) and their log-softmax
 * over those n columns (fp32, accurate expf / logf).  Columns >= n are never read, so padding may hold anything;
 * -inf entries are allowed.  1 <= k <= 16, k <= n <= ldl.  idx int64 [rows, k], logp fp32 [rows, k]. */
int srg_topk_logsoftmax(const float* logits, int64_t ldl, int rows, int n, int k, int64_t* idx, float* logp,
                        void* stream);

/* Top-k situation decode (a situation = a verb + one label per role of that verb).
 * srg_situation_nouns runs the role graphs of the B*k (image, verb) pairs verbs[b*k + j] (int64 [B, k]) in eval mode
 * (no dropout): it is srg_nouns_forward on B*k graphs whose node init reads feat[b] (fp32 [B, D]; the features are
 * not copied k times), followed by a decode.  Per candidate:
 *   labels     int64 [B, k, R]: top-1 label of every role slot, -1 on the pad slots (r >= role_count[verb]);
 *   label_logp fp32  [B, k, R]: its log-softmax over the n_labels labels, 0 on the pad slots;
 *   score      fp32  [B, k]   : (verb_logp ? verb_logp[b*k + j] : 0) + the sum of the real slots' label_logp.
 * verb_logp (nullable) fp32 [B, k].  Out-of-range verb ids are clamped and flagged as in srg_nouns_forward
 * (srg_check_verbs).  1 <= k <= min(16, n_verbs); both precisions.
 * Workspace (srg_situation_workspace_bytes, enough at any 16-byte aligned address): the forward buffers of B*k role
 * graphs plus their noun logits
 * [B*k*R, n_labels padded to 256] fp32.  At D = 2048, R = 6, 2001 labels, B = 6144, k = 5 that is about 7.5 GB in bf16
 * (184 k slot rows of state, operand copies and logits; estimated from the buffer list, not measured); the fp32-parity
 * mode needs more for its split operands. */
size_t srg_situation_workspace_bytes(srg_handle* h, int B, int k, int precision);
int srg_situation_nouns(srg_handle* h, const float* feat, const int64_t* verbs, int B, int k, const float* role_emb,
                        const float* verb_emb, const float* verb_logp, int64_t* labels, float* label_logp,
                        float* score, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* N-best situation decode: the n highest-scoring situations of each image b over its kv candidate verbs
 * verbs[b*kv + j] (int64 [B, kv]).  A situation is a candidate j < kv plus one label per real role slot of its verb;
 * its score is (verb_logp ? verb_logp[b*kv + j] : 0) + l_0 + l_1 + ..., summed in fp32 in slot order (as
 * srg_situation_nouns sums it, so the 1-best score is bit-identical to that call's best candidate), where l_r is the
 * label's log-softmax over the n_labels labels.  Order: score descending, then lower j, then the per-slot label ranks
 * compared lexicographically from slot 0.  A situation with a label of rank >= n in some slot has n situations before
 * it (replace that label by a better-ranked one), so only the top n labels of each slot are searched.
 *   out_verbs     int64 [B, n]   : the verb of each entry (out-of-range ids clamped and flagged as in srg_nouns_forward)
 *   out_verb_logp fp32  [B, n]   : its verb_logp (nullable; written when verb_logp is given)
 *   labels        int64 [B, n, R]: -1 on the pad slots;  label_logp fp32 [B, n, R]: l_r, 0 on the pad slots
 *   score         fp32  [B, n]
 *   exact         uint8 [B]      : (nullable) 1 when the list is the n-best over ALL verbs, certified by
 *                                  score[b, n-1] >= verb_bound[b]; verb_bound fp32 [B] (nullable) is the log-prob of
 *                                  the best verb outside the beam.  Every l_r <= 0, and adding a non-positive number
 *                                  never increases an fp32 sum, so no situation of an outside verb scores above it.
 *                                  NULL verb_bound: no verb is outside the beam and every exact[b] is 1.
 * If kv < n and no candidate verb has a role, fewer than n situations exist; the entries past them hold verb -1,
 * score -inf, labels -1 and label log-probs 0.  The partial sums are pruned to n per slot, so two situations whose
 * scores lie within one fp32 rounding of each other may come out in the other order than an exhaustive enumeration
 * would give.  Deterministic: repeated calls are bit-identical.
 * 1 <= kv <= min(16, n_verbs), 1 <= n <= min(16, n_labels); both precisions.  Workspace
 * (srg_situation_nbest_workspace_bytes, enough at any 16-byte aligned address): srg_situation_workspace_bytes(B, kv)
 * plus the per-slot lists [B*kv*R, n] int64 + fp32 (35 MB at B = 6144, kv = 5, R = 6, n = 16). */
size_t srg_situation_nbest_workspace_bytes(srg_handle* h, int B, int kv, int n, int precision);
int srg_situation_nbest(srg_handle* h, const float* feat, const int64_t* verbs, int B, int kv, const float* role_emb,
                        const float* verb_emb, const float* verb_logp, const float* verb_bound, int n,
                        int64_t* out_verbs, float* out_verb_logp, int64_t* labels, float* label_logp, float* score,
                        uint8_t* exact, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* The keep-mask the Philox path applies for (*drop_seed, drop_stream, drop_p) on a [rows, D] slot matrix, written as
 * uint8 0/1 (tests: lets the oracle replay exactly the dropout a training step used). */
int srg_dropout_mask(const int64_t* drop_seed, int64_t drop_stream, float drop_p, int64_t rows, int D, uint8_t* keep,
                     void* stream);

/* GGSNN.forward (model.py:59-86) on caller-provided node states: hidden fp32 [rows, D] is updated in place.
 * mask: fp32 [B, R, R] (SRG_MODE_NOUN, rows = B*R) or NULL (SRG_MODE_VERB, rows = B). */
int srg_ggnn_forward(srg_handle* h, int mode, float* hidden, const float* mask, int B, int precision,
                     int save_for_backward, void* workspace, size_t workspace_bytes, void* stream);

/* autograd backward of srg_ggnn_forward(..., save_for_backward = 1): `workspace`, `mask` and B must be that call's.
 * dhidden_out: fp32 [rows, D] = dL/d(the updated states), only read.  dhidden_in (nullable): fp32 [rows, D], receives
 * dL/d(the states passed in).  dmask (nullable, SRG_MODE_NOUN only): fp32 [B, R, R], receives dL/dmask (overwritten;
 * deterministic).  The 14 GGSNN gradients accumulate into `g` (its classifier and embedding fields are ignored); the
 * deferred chain rule (srg_set_deferred_chain) applies as in srg_*_backward.  bf16-packed weights only. */
int srg_ggnn_backward(srg_handle* h, int mode, const float* dhidden_out, const float* mask, float* dmask,
                      float* dhidden_in, int B, const srg_grads* g, void* workspace, size_t workspace_bytes,
                      void* stream);

/* FCGGNN.nouns_loss (model.py:189-201): sum over the 3 annotations of CrossEntropy(ignore_index = n_labels), each a
 * mean over its non-ignored targets.  counts: device fp32 [3] = number of non-ignored targets per annotation over the
 * GLOBAL batch (srg_count_targets, all-reduced by the caller when the batch is sharded).  loss: device fp32 scalar,
 * accumulated (+=).  dlogits: fp32 [B*R, ldl] or NULL; receives grad_scale * dLoss/dlogits (padding columns = 0). */
int srg_count_targets(srg_handle* h, const int64_t* gt_nouns, int B, float* counts, void* stream);
int srg_nouns_loss(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                   const float* counts, float* loss, float* dlogits, float grad_scale, const float* stats,
                   void* stream);

/* FCGGNN.verb_loss (model.py:182-187): CrossEntropy(pred_verb[B, n_verbs], gt_verb[B]); the mean is taken over the
 * GLOBAL batch: inv_batch = 1/B_global, or -- when batch_total (device fp32 scalar, nullable) is given -- 1 / *batch_total,
 * which lets a sharded caller all-reduce its local batch sizes on the stream without a host synchronisation (shards
 * of unequal size: the tail batch of an epoch). */
int srg_verb_loss(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B, float inv_batch,
                  const float* batch_total, float* loss, float* dlogits, float grad_scale, const float* stats,
                  void* stream);

/* Backward of the two losses as its own pass: grad_scale * (*grad_out) * dLoss/dlogits, where grad_out is the DEVICE
 * scalar autograd hands to the loss node (nullable = 1).  With these, the forward calls can be given dlogits = NULL (they
 * then only read the target logits when `stats` is available) and no separate scaling pass over the [rows, ldl]
 * gradient is needed.  The gradient goes to ONE of two places:
 *   dlogits      : fp32 [rows, ldl] (a caller that wants the gradient as a tensor), or
 *   dlogits_bf16 : the zero-padded bf16 [rows, padded classes] operand the classifier's backward GEMMs read, i.e. the
 *                  address `workspace + srg_workspace_dlogits_offset(...)` of the forward call that produced the logits
 *                  (accumulate = 1: added to what is there, for a second loss on the same logits).  The fp32 gradient
 *                  is then never written or re-read; srg_nouns_backward / srg_verb_backward are told with
 *                  dlogits_in_workspace = 1. */
int srg_nouns_loss_backward(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                            const float* counts, const float* grad_out, float grad_scale, float* dlogits,
                            void* dlogits_bf16, int accumulate, const float* stats, void* stream);
int srg_verb_loss_backward(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B,
                           float inv_batch, const float* batch_total, const float* grad_out, float grad_scale,
                           float* dlogits, void* dlogits_bf16, int accumulate, const float* stats, void* stream);
size_t srg_workspace_dlogits_offset(srg_handle* h, int mode, int B, const void* workspace);

/* Class weights, label smoothing and the reduction of the two losses: torch.nn.functional.cross_entropy(weight,
 * label_smoothing, reduction), exactly.  For logits z over C classes, target y, class weights w (NULL = all 1),
 * W = sum_c w_c and smoothing eps in [0, 1], the loss of one target is
 *   l = (1 - eps) w_y (lse - z_y) + (eps / C) sum_c w_c (lse - z_c),   0 for an ignored target (nouns: y = n_labels),
 * and dl/dz_c = (1 - eps) w_y (p_c - [c == y]) + (eps / C) (W p_c - w_c).  Reductions:
 *   SRG_REDUCTION_MEAN : sum l / (sum of w_y over the non-ignored targets): the nouns per annotation, summed over the 3
 *                        (counts = srg_count_targets_weighted), the verbs over the batch (batch_total =
 *                        srg_verb_weight_total, or inv_batch when there are no class weights).  A zero denominator
 *                        contributes 0, not NaN as torch gives.
 *   SRG_REDUCTION_SUM  : sum l (counts, inv_batch and batch_total are not read);
 *   SRG_REDUCTION_NONE : l per target into per_target_loss (fp32, laid out like the targets: [B] verbs, [B, 3, R] nouns;
 *                        0 on ignored targets); `loss` may be NULL.  The backward calls take d(loss)/dl per target in
 *                        grad_per_target (same layout), times grad_scale and *grad_out when given.
 * per_target_loss under MEAN / SUM (nullable): receives each target's term of the scalar, and *loss += their sum in a
 * fixed order (one more launch), so that repeated calls give bit-identical losses; NULL: per-CTA atomics, as the
 * default options.  Only the forward calls write it.  class_weight: device fp32 [n_classes] (n_verbs or n_labels).
 * A NULL srg_loss_opts, or one whose fields all hold their defaults (no weight, eps = 0, MEAN, no per-target pointers),
 * runs exactly the default-option kernels.  Bad options (eps outside [0, 1], an unknown reduction, NONE without
 * per_target_loss in a forward call or without grad_per_target in a call that writes a gradient) return an error and
 * launch nothing. */
enum { SRG_REDUCTION_MEAN = 0, SRG_REDUCTION_SUM = 1, SRG_REDUCTION_NONE = 2 };
typedef struct srg_loss_opts {
  const float* class_weight;
  float label_smoothing;
  int reduction;
  float* per_target_loss;
  const float* grad_per_target;
} srg_loss_opts;

/* Weighted denominators of the MEAN reduction, summed by one CTA in a fixed order (no atomics, so an eager step and a
 * replayed CUDA graph get bit-identical values).  counts: device fp32 [3] = sum of class_weight[y] over the
 * non-ignored targets of each annotation (overwritten; class_weight NULL = srg_count_targets).  total: device fp32
 * scalar = sum of class_weight[y] over the B verbs (overwritten).  All-reduce both over the ranks of a sharded batch. */
int srg_count_targets_weighted(srg_handle* h, const int64_t* gt_nouns, int B, const float* class_weight, float* counts,
                               void* stream);
int srg_verb_weight_total(srg_handle* h, const int64_t* gt_verb, int B, const float* class_weight, float* total,
                          void* stream);

/* srg_nouns_loss / srg_verb_loss / srg_*_loss_backward with options (opts nullable = those calls). */
int srg_nouns_loss_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                      const float* counts, float* loss, float* dlogits, float grad_scale, const float* stats,
                      const srg_loss_opts* opts, void* stream);
int srg_verb_loss_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B, float inv_batch,
                     const float* batch_total, float* loss, float* dlogits, float grad_scale, const float* stats,
                     const srg_loss_opts* opts, void* stream);
int srg_nouns_loss_backward_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                               const float* counts, const float* grad_out, float grad_scale, float* dlogits,
                               void* dlogits_bf16, int accumulate, const float* stats, const srg_loss_opts* opts,
                               void* stream);
int srg_verb_loss_backward_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B,
                              float inv_batch, const float* batch_total, const float* grad_out, float grad_scale,
                              float* dlogits, void* dlogits_bf16, int accumulate, const float* stats,
                              const srg_loss_opts* opts, void* stream);

/* `stats` (nullable) of the two loss calls: the per-column-tile (row max, row sum-exp) pairs the classifier GEMM of the
 * matching forward call left in its workspace, at this byte offset; with them the loss reads each logits row once
 * instead of three times.  They are only valid for the logits that forward call produced. */
size_t srg_workspace_stats_offset(srg_handle* h, int mode, int B, int precision, int save_for_backward,
                                  const void* workspace);

/* autograd backward of srg_nouns_forward / srg_verb_forward (sr.py:76-79).  `workspace` must be the one used by the
 * matching forward call with save_for_backward = 1, and the dropout arguments must be that call's (the seed scalar
 * must still hold the same value).  The gradient of the logits: dlogits fp32 [rows, ldl] (nullable), and / or
 * dlogits_in_workspace = 1 when srg_*_loss_backward already wrote it into the workspace as bf16 (both: their sum).
 * Gradients accumulate into `g`. */
int srg_nouns_backward(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, const float* feat,
                       const int64_t* verb, int B, const float* role_emb, const float* verb_emb, const uint8_t* keep,
                       float drop_p, const int64_t* drop_seed, int64_t drop_stream, const srg_grads* g, void* workspace,
                       size_t workspace_bytes, void* stream);
int srg_verb_backward(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, int B,
                      const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                      const srg_grads* g, void* workspace, size_t workspace_bytes, void* stream);

/* srg_nouns_backward / srg_verb_backward plus the gradient w.r.t. the backbone features `feat` of the forward call:
 * dfeat (nullable) fp32 [B, D] is OVERWRITTEN (not accumulated), like dhidden_in of srg_ggnn_backward.
 *   nouns (model.py:124-144): node[b,r] = relu(feat[b] * role_emb[role(b,r)] * verb_emb[verb[b]]), so
 *          dfeat[b] = sum over the real roles r of [node[b,r] > 0] * dL/dnode[b,r] * role_emb[role(b,r)] * verb_emb[verb[b]]
 *          (pad slots contribute nothing); the embedding gradients in `g` are computed in the same pass when both
 *          g->role_emb and g->verb_emb are set, and the pass is skipped when neither they nor dfeat are;
 *   verb  (model.py:160): node = relu(feat), so dfeat = [node > 0] * dL/dnode.
 * The mask [node > 0] is taken from the bf16 copy of the initial state (relu'(0) = 0, as torch).  No atomics: dfeat is
 * deterministic.  With dfeat = NULL these are srg_nouns_backward / srg_verb_backward, launch for launch. */
int srg_nouns_backward_feat(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace,
                            const float* feat, const int64_t* verb, int B, const float* role_emb, const float* verb_emb,
                            const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                            const srg_grads* g, float* dfeat, void* workspace, size_t workspace_bytes, void* stream);
int srg_verb_backward_feat(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, int B,
                           const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                           const srg_grads* g, float* dfeat, void* workspace, size_t workspace_bytes, void* stream);

/* Deferred chain rule.  The verb node and the role graph share one GGNN (model.py:28-35, 226), so one training step
 * (sr.py:63-79) calls both backward functions with the same weights.  Their gradients w.r.t. the message-side weights
 * W_p, b_p, W_z, W_r, W_h go through the same chain rule (d/dP_x -> dW_x, dW_p, db_p; P_x = W_x W_p), which is linear
 * in d/dP_x: with on = 1 the backward calls only accumulate d/dP_x and the bias column sums into buffers owned by the
 * handle (safe from two streams at once), and srg_chain_finalize applies the chain rule ONCE, adds the result into `g`
 * and clears the accumulators.  Until srg_chain_finalize has run on a stream ordered after every backward call, the
 * five message-side gradients in `g` are incomplete.  on = 0 (default): every backward call is self-contained. */
int srg_set_deferred_chain(srg_handle* h, int on, void* stream);
int srg_chain_finalize(srg_handle* h, const srg_grads* g, void* stream);

/* sr.py:80-83 on flat fp32 buffers of all trainable tensors (one launch instead of ~40 small ones):
 * torch.nn.utils.clip_grad_norm_(params, max_norm) -- grads are scaled in place by min(1, max_norm / (||g||_2 + 1e-6)) --
 * followed by torch.optim.Adamax(lr, betas = (beta1, beta2), eps).  scratch: device fp32 [2] = {||g||^2 of this step,
 * number of steps taken so far (incremented by the call)}; n must be a multiple of 4. */
int srg_clip_adamax(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                    float beta2, float eps, float max_norm, float* scratch, void* stream);

/* The two halves of srg_clip_adamax for a data-parallel caller that SHARDS the flat buffers over its ranks (each rank
 * updates 1/N of the parameters after a reduce-scatter of the gradients, then the parameters are all-gathered):
 * srg_sumsq writes sum x^2 of the local gradient shard to *out (device fp32), the caller all-reduces that scalar, and
 * srg_adamax_step clips with the global *norm_sq and applies Adamax to the shard (step: device fp32 counter, incremented). */
int srg_sumsq(const float* x, int64_t n, float* out, void* stream);
int srg_adamax_step(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                    float beta2, float eps, float max_norm, const float* norm_sq, float* step, void* stream);

/* Raw tensor-core GEMM (tests / micro-benchmarks):  C[M,N] = alpha * A[M,K] * B[N,K]^T + bias[N]
 * a_mn / b_mn = 1: the operand is stored transposed (A as [K,M], B as [K,N]).  c_dtype: SRG_DT_F32 | SRG_DT_BF16.
 * reduce = 1 (fp32 only): C += ... with k_splits-way split-K. */
int srg_gemm_bf16(const void* A, int64_t lda, int a_mn, const void* B, int64_t ldb, int b_mn, void* C, int64_t ldc,
                  int c_dtype, int M, int N, int K, const float* bias, float alpha, int cta_group, int k_splits,
                  int reduce, void* stream);

/* Accounting used by bench.py: number of kernels this library has launched so far, and an optional CUDA-event
 * bracket around every tensor-core GEMM launch, accumulated per kernel kind (kind = 4*epilogue + 2*a_mn + b_mn). */
long long srg_launch_count(void);
int srg_profile_begin(void);
int srg_profile_end(int max_kinds, double* ms, double* flops, long long* launches);
const char* srg_profile_kind_name(int kind);

#ifdef __cplusplus
}
#endif
#endif /* SRGGNN_H_ */
