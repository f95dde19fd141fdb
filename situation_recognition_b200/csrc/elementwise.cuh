// HBM-bound kernels of the GGNN role-graph stage: index gather / mask build, node initialisation, neighbour
// aggregation, weight packing, dropout, cross-entropy, and the elementwise pieces of the backward pass.
// All of them are launched on grids sized in multiples of the SM count with 16-byte vector accesses.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <cuda_bf16.h>

namespace srg {

typedef __nv_bfloat16 bf16;

// Compact row layout of a role-graph path, built on the device by launch_prep_rows (all pointers are device pointers):
//   cnt[b]  = number of real roles n_b of image b's verb            off[b] = first row of image b (off[B] = sum L_b)
//   meta[0] = rows incl. the ONE shared pad row (the GEMMs' M)      meta[1] = index of the shared pad row
//   meta[2] = meta[0] rounded up to 256: the rows the GEMM tiles touch; every one of them holds finite values
// compact = 1: image b owns L_b = n_b rows (pad nodes are not materialised: they all follow the shared pad row's
// trajectory); compact = 0: L_b = R rows per image as the reference lays them out (kept for A/B measurements).
// All members null: the path has a static dense row layout (verb node path, srg_ggnn_forward).
struct RowMap {
  const int* cnt = nullptr;
  const int* off = nullptr;
  const int* meta = nullptr;
  int compact = 0;
};

// Dropout in front of a classifier: explicit uint8 keep-mask [rows, D] (tests), or Philox keyed by (*seed, stream, row,
// column); neither: identity.  thresh = (1 - p) * 65536, scale = 1 / (1 - p).
struct DropSpec {
  const uint8_t* keep = nullptr;
  const long long* seed = nullptr;
  long long stream = 0;
  uint32_t thresh = 65536;
  float scale = 1.f;
};

int launch_gather_mask(const int32_t* verb2roles, const int32_t* role_count, int n_verbs, int R, const int64_t* verb,
                       int B, int64_t* role_idx, float* mask, int* bad, cudaStream_t s);

// cnt / off / meta of `rm` from the verb ids (imsitu_encoder.py:158-159 per image + an exclusive scan); one block
int launch_prep_rows(const int32_t* role_count, int n_verbs, int R, const int64_t* verb, int B, int compact, RowMap rm,
                     int* bad, cudaStream_t s);
// node[row(b,r), :] = relu(feat[b / feat_rep,:] * role_emb[verb2roles[verb[b], r], :] * verb_emb[verb[b], :])
// (model.py:124-144) for the rows `rm` materialises; the self-loop rows are set to 0.  feat_rep > 1: consecutive groups
// of feat_rep graphs share one feature row (the k candidate verbs of an image, srg_situation_nouns)
int launch_node_init_noun(const float* feat, const float* role_emb, const float* verb_emb, const int64_t* verb,
                          const int32_t* verb2roles, int n_verbs, int B, int R, int D, RowMap rm, int feat_rep,
                          float* h32, bf16* hb_hi, bf16* hb_mid, bf16* hb_lo, cudaStream_t s);
// the same aggregation as launch_aggregate on the rows of `rm`, from the role counts instead of a [B,R,R] mask
int launch_aggregate_rows(const float* h32, RowMap rm, int B, int R, int D, bf16* a_hi, bf16* a_mid, bf16* a_lo,
                          cudaStream_t s);
// ada = e + aggregate^T(da) on the rows of `rm` (rm.cnt == nullptr: B dense rows, identity aggregation)
int launch_aggregate_t_rows(const bf16* da, const bf16* e, RowMap rm, int B, int R, int D, bf16* ada, cudaStream_t s);
// backward of launch_aggregate on B*R dense rows with the caller's fp32 mask [B,R,R] (any values):
// ada[b,j] = e[b,j] + sum_i mask[b,i,j] da[b,i]; with dmask (nullable): dmask[b,i,j] += sum_d da[b,i,d] h[b,j,d], where
// h is the state operand that entered the step.  dmask is deterministic (no atomics); without it h is not read.
int launch_aggregate_t(const bf16* da, const bf16* e, const float* mask, const bf16* h, int B, int R, int D,
                       bf16* ada, float* dmask, cudaStream_t s);
// x[row] = dropout(h32[row of slot `row` under rm]) for all `rows` node slots -> bf16 hi (+ mid, lo)
int launch_classifier_input(const float* h32, RowMap rm, int R, int64_t rows, int D, DropSpec ds, bf16* x_hi,
                            bf16* x_mid, bf16* x_lo, cudaStream_t s);
// GRU-gate derivatives of the LAST propagation step, fused into launch_classifier_input_bwd for the rows it writes
// (z == nullptr: off): dpre_z = g (hc - h) z (1 - z), dpre_h = g z (1 - hc^2), dh_acc = g (1 - z) with g = dL/dh'
struct GruPre {
  const bf16* z = nullptr;
  const bf16* hc = nullptr;
  const bf16* h = nullptr;
  bf16* dpre_z = nullptr;
  bf16* dpre_h = nullptr;
  int64_t ld_out = 0;
  float* dh_acc = nullptr;
};
// dh[row under rm] = dropout'(dx[slot]) with all pad slots summed into the shared pad row; with `gp` the real rows get
// their gate derivatives instead of dh (launch_gru_bwd_pre_ld then only has to run on the self-loop rows)
int launch_classifier_input_bwd(const float* dx, RowMap rm, int B, int R, int D, DropSpec ds, float* dh, GruPre gp,
                                cudaStream_t s);
// out[rows, D] uint8 = the keep decisions `ds` makes (tests: feeds the oracle the mask the Philox path used)
int launch_dropout_mask(DropSpec ds, int64_t rows, int D, uint8_t* out, cudaStream_t s);
// node = relu(feat)  (model.py:160)
int launch_node_init_verb(const float* feat, int B, int D, float* h32, bf16* hb_hi, bf16* hb_mid, bf16* hb_lo,
                          cudaStream_t s);
// fp32 -> bf16 hi (+ mid, lo residual parts when non-null)
int launch_split_cast(const float* x, int64_t n, bf16* hi, bf16* mid, bf16* lo, cudaStream_t s);

// a[b,i,:] = sum_j mask[b,i,j] * h[b,j,:]    (model.py:67-75 with the projection hoisted out of the sum)
int launch_aggregate(const float* h32, const float* mask, int B, int R, int D, bf16* a_hi, bf16* a_mid, bf16* a_lo,
                     cudaStream_t s);

// dst[r, col_off + c] = bf16 part `part` (0 hi, 1 mid, 2 lo) of src[r, c] (r < rows), 0 for rows <= r < rows_pad;
// many such jobs in one launch (all with `cols` columns)
struct PackJob {
  const float* src;
  bf16* dst;
  int64_t ld_dst;
  int64_t col_off;
  int rows, rows_pad, part;
};
constexpr int kMaxPackJobs = 48;
int launch_pack_weight_multi(const PackJob* jobs, int n_jobs, int cols, cudaStream_t s);
// dst[i] = a[i] (+ b[i]) for i < n, 0 for n <= i < n_pad
int launch_pack_bias(const float* a, const float* b, int n, int n_pad, float* dst, cudaStream_t s);

int launch_count_targets(const int64_t* gt, int B, int R, int ignore_index, float* counts, cudaStream_t s);
// out[a] = sum of cw[gt[t]] over the targets t of annotation a = (t / R) % n_ann with gt[t] != ignore_index
// (targets outside [0, n_classes) count 0), n targets in all; overwritten.  One CTA in a fixed order, no atomics:
// repeated calls are bit-identical.  n_ann <= 3.
int launch_weighted_count(const int64_t* gt, int64_t n, int R, int n_ann, int ignore_index, const float* cw,
                          int n_classes, float* out, cudaStream_t s);

// Options of the cross-entropy kernels (srg_loss_opts).  With none of them given the kernels run the default-option
// instantiation, launch for launch.
enum { kCeMean = 0, kCeSum = 1, kCeNone = 2 };
struct CeOpts {
  const float* cw;          // class weights [n_classes] or null (all 1)
  float eps;                // label smoothing in [0, 1]
  int reduction;            // kCeMean / kCeSum / kCeNone
  float* per_target;        // forward: kCeNone: the loss of every target; mean / sum: its term of the scalar, which
                            // is then their sum in a fixed order
  const float* gpt;         // kCeNone gradient: d(loss)/d(per-target loss), laid out like the targets
};
inline bool ce_opts_active(const CeOpts* o) {
  return o != nullptr && (o->cw != nullptr || o->eps > 0.f || o->reduction != kCeMean || o->per_target != nullptr);
}

// one warp per logits row; loss and dlogits are both optional; the gradient is scaled by grad_scale and, when
// gscale_dev is not null, by that device scalar as well
// dlb (nullable, instead of dlogits): the gradient as the zero-padded bf16 [rows, n_pad] operand of the classifier's
// backward GEMMs; accumulate: added to what dlb already holds
// opt (nullable): class weights, label smoothing and the reduction; the option arithmetic is only compiled into the
// instantiation that ce_opts_active(opt) selects.  Mean: counts[a] / *batch_total are the weighted denominators.
int launch_nouns_ce(const float* logits, int64_t ldl, int n_labels, const int64_t* gt, int B, int R,
                    const float* counts, float* loss, float* dlogits, float grad_scale, const float* gscale_dev,
                    const float* stats, int stats_tiles, bf16* dlb, int n_pad, int accumulate, const CeOpts* opt,
                    cudaStream_t s);
int launch_verb_ce(const float* logits, int64_t ldl, int n_verbs, const int64_t* gt, int B, float inv_batch,
                   float* loss, float* dlogits, float grad_scale, const float* gscale_dev, const float* stats,
                   int stats_tiles, const float* batch_total, bf16* dlb, int n_pad, int accumulate, const CeOpts* opt,
                   cudaStream_t s);
// Per row of x [rows, ldl]: the k largest of the first n columns in descending order (ties: lower column first, as
// torch.argmax) and their log-softmax over those n columns.  Columns >= n are never read.  1 <= k <= 16, k <= n.
// idx int64 [rows, k], logp fp32 [rows, k].
int launch_row_topk_logsoftmax(const float* x, int64_t ldl, int rows, int n, int k, int64_t* idx, float* logp,
                               cudaStream_t s);
// Decode of the situation candidates u < n_cand (verb[u]): slots r >= role_count[verb[u]] get label -1 and log-prob 0;
// score[u] = (verb_logp ? verb_logp[u] : 0) + sum of the real slots' label log-probs.  labels / label_logp [n_cand, R]
// hold the per-slot top-1 on entry and are finished in place.
int launch_situation_finish(const int64_t* verb, const int32_t* role_count, int n_verbs, int R, int n_cand,
                            const float* verb_logp, int64_t* labels, float* label_logp, float* score, cudaStream_t s);
// N-best decode of image b < B from its kv candidates verbs[b*kv + j] (one CTA per image, one warp per candidate):
// the n best (score desc, then lower j, then the per-slot label ranks lexicographically) of the situations built from
// the per-slot top-n lists slot_idx / slot_logp [B*kv*R, n].  score = (verb_logp ? verb_logp : 0) + l_0 + l_1 + ...
// in fp32, slot order.  out_verbs [B,n], out_verb_logp [B,n] (written when both it and verb_logp are given), labels /
// label_logp [B,n,R] (-1 / 0 on pad slots), score [B,n]; exact [B] (nullable) = no verb_bound or score[b,n-1] >=
// verb_bound[b].  1 <= kv, n <= 16, R <= 8.
int launch_situation_nbest(const int64_t* verbs, const int32_t* role_count, int n_verbs, int R, int B, int kv, int n,
                           const float* verb_logp, const float* verb_bound, const int64_t* slot_idx,
                           const float* slot_logp, int64_t* out_verbs, float* out_verb_logp, int64_t* labels,
                           float* label_logp, float* score, uint8_t* exact, cudaStream_t s);
// fp32 [rows, ld] (first n_valid columns) -> bf16 [rows, n_pad], zero padded
int launch_cast_pad(const float* src, int64_t ld, int rows, int n_valid, int n_pad, bf16* dst, int accumulate,
                    cudaStream_t s);

// out1[c] (+= scale1 * colsum) , out2[c] (+= scale2 * colsum); X bf16 [rows, ld], first n_cols columns
int launch_colsum(const bf16* X, int64_t ld, int rows, int n_cols, float* out1, float scale1, float* out2,
                  float scale2, cudaStream_t s);
// node-init backward of the role graph, model.py:124-144, from dh0 = dL/dnode and the bf16 copy h0b of the node's
// initial state (relu'(0) = 0): the embedding gradients (accumulated; both pointers null: skipped) and / or
// dfeat fp32 [B, D] = sum over the image's rows of [node > 0] dh0 * role_emb * verb_emb (overwritten; nullable)
int launch_node_init_bwd(const float* dh0, const bf16* h0b, const float* feat, const float* role_emb,
                         const float* verb_emb, const int64_t* verb, const int32_t* verb2roles, int n_verbs,
                         int n_roles, int B, int R, int D, RowMap rm, float* d_role_emb, float* d_verb_emb,
                         float* dfeat, cudaStream_t s);
// node-init backward of the verb node, model.py:160: dfeat [B, D] = h0b > 0 ? dh0 : 0 (overwritten)
int launch_node_init_verb_bwd(const float* dh0, const bf16* h0b, int B, int D, float* dfeat, cudaStream_t s);

// up to 4 column sums in one launch: out1/out2 += scale * colsum, out3 += scale3 * colsum
struct ColsumJob {
  const bf16* X;
  float* out1;
  float* out2;
  float scale;
  float* out3;
  float scale3;
};
// rows: nseg segments of `rows` rows (rows_dev, nullable: device count of valid rows per segment), segment s at row
// s * seg_stride of X
int launch_colsum_multi(const ColsumJob* jobs, int n_jobs, int64_t ld, int rows, const int* rows_dev, int nseg,
                        int64_t seg_stride, int n_cols, cudaStream_t s);


// clip_grad_norm_(max_norm) + Adamax on flat fp32 buffers (sr.py:80-83).  scratch: device fp32 [2] = {sum g^2, step}.
// the two halves of launch_clip_adamax, for a caller that shards the flat buffers over ranks and all-reduces the
// squared norm in between: out = sum x^2 (device scalar, overwritten); then clip with the given *norm_sq + Adamax + ++*step
int launch_sumsq(const float* x, int64_t n, float* out, cudaStream_t s);
int launch_adamax_step(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                       float beta2, float eps, float max_norm, const float* norm_sq, float* step, cudaStream_t s);
int launch_clip_adamax(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                       float beta2, float eps, float max_norm, float* norm_sq, float* step, cudaStream_t s);

// GRU backward prologue writing into column blocks of a wider matrix (leading dimension ld_out elements)
// rows [row0, rows): rows_dev / row0_dev (nullable) are device-resident overrides (`rows` then only sizes the grid)
int launch_gru_bwd_pre_ld(const float* dh, const bf16* z, const bf16* hc, const bf16* h, int rows, const int* rows_dev,
                          const int* row0_dev, int D, bf16* dpre_z, bf16* dpre_h, int64_t ld_out, float* dh_acc,
                          cudaStream_t s);
// y[o] = sum_k W[o,k] x[k]                       (fp32, W row-major [rows, cols])
int launch_matvec(const float* W, const float* x, int rows, int cols, float* y, cudaStream_t s);
// y[k] += sum_x sum_o W_x[o,k] s[x*rows + o]    (three [rows, cols] matrices in one launch; null W_x skipped)
int launch_matvec_t_acc3(const float* const W[3], const float* sv, int rows, int cols, float* y, cudaStream_t s);
// dW_x[o,k] += s[x*rows + o] * b[k]              (three matrices in one launch; null dW_x skipped);
// atomic = the destination may be accumulated into from another stream at the same time
int launch_outer_acc3(const float* sv, const float* b, int rows, int cols, float* const dW[3], bool atomic,
                      cudaStream_t s);
// dst[i] = a[i] + b[i] + scale * c[i]   (b, c nullable; zero beyond n up to n_pad)
int launch_pack_bias3(const float* a, const float* b, const float* c, float scale, int n, int n_pad, float* dst,
                      cudaStream_t s);

}  // namespace srg
