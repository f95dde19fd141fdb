// C-ABI of the GGNN role-graph stage (include/srggnn.h): handle, weight packing, forward and backward
// orchestration.  Every contraction is one launch of the tcgen05 kernel in gemm.cuh; everything HBM-bound
// is in kernels_elementwise.cu.
#include <new>
#include <vector>
#include "elementwise.cuh"
#include "host.cuh"
#include "../../include/srggnn.h"

using namespace srg;

namespace srg {
int query_device(DeviceInfo* d);
}

namespace {
constexpr int kMaxT = 8;
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
}  // namespace

struct srg_handle {
  int device = 0, D = 0, R = 0, T = 0, V = 0, n_roles = 0, L = 0;
  int Vpad = 0, Lpad = 0;
  int cg = 2;
  int compact = 1;      // role-node rows: 1 = real rows + ONE shared pad row (default), 0 = R rows per image
  DeviceInfo dev;
  int32_t* d_verb2roles = nullptr;
  int32_t* d_role_count = nullptr;
  bool tables_set = false;
  int* d_bad = nullptr;
  // ---- packed tensor-core operands (rebuilt by srg_pack_weights)
  // The neighbour projection is folded into the gate weights:  (a W_p^T + c b_p) W_x^T = a (W_x W_p)^T + c W_x b_p,
  // so the message GEMM disappears and the gates read the aggregated state `a` directly.  P_x = W_x W_p.
  int packed_prec = -1;
  int alloc_split = 0;  // K replication factor the forward buffers were allocated for (1 or 6)
  srg_params params;    // fp32 masters seen by the last srg_pack_weights (needed by the backward chain rule)
  bf16 *Wzr = nullptr;  // [2D, 2D*s]  rows z|r, K blocks [P_x | U_x]
  bf16 *Wh = nullptr;   // [D,  2D*s]  [P_h | U_h]
  bf16 *Wcn = nullptr, *Wcv = nullptr;
  bf16 *Wm_hi = nullptr, *Wm_mid = nullptr, *Wm_lo = nullptr;  // [3D, D] = [W_h; W_z; W_r] as bf16 hi + mid + lo parts
  bf16 *Wp6 = nullptr;                                         // [6D, D] = W_p parts [hi; mid; hi; lo; hi; mid]
  bf16 *P_hi = nullptr, *P_mid = nullptr, *P_lo = nullptr;     // [3D, D] = [P_h; P_z; P_r]
  bf16 *U_stack = nullptr, *Uh = nullptr;   // [2D, D] = [U_z; U_r], [D, D]
  float *wb = nullptr;                      // [3D] = [W_h b_p; W_z b_p; W_r b_p]
  float *bzr[2] = {nullptr, nullptr};       // [2D] per mode (noun, verb): b_Wx + b_Ux + c W_x b_p
  float *bh[2] = {nullptr, nullptr};        // [D]  per mode
  float *bcn = nullptr, *bcv = nullptr;
  // ---- deferred chain rule (srg_set_deferred_chain): d/dP_x and bias column sums of ALL paths of one training step
  bool defer_chain = false;
  float* acc_GP = nullptr;   // [3D, D] fp32
  bf16* acc_GPb = nullptr;   // [3D, D] bf16 operand copy
  float* acc_s = nullptr;    // [3D]
};

namespace {

// ------------------------------------------------------------------------------------------------ workspace
struct StepBufs {
  bf16 *a_hi = nullptr, *a_mid = nullptr, *a_lo = nullptr, *rh_hi = nullptr, *rh_mid = nullptr, *rh_lo = nullptr;
  bf16 *r = nullptr, *hc = nullptr;
  void* z = nullptr;
};

struct PathBufs {
  int M = 0;       // rows the state buffers are allocated (and the tensor maps built) for
  int Mfull = 0;   // node slots B*R (role graph) or B (verb node): the rows of the classifier GEMM and of the logits
  RowMap rm;       // role-graph paths: device-resident compact row layout (the GEMMs read their M from rm.meta)
  float* h32 = nullptr;
  bf16* hb_hi[kMaxT + 1] = {};
  bf16* hb_mid[kMaxT + 1] = {};
  bf16* hb_lo[kMaxT + 1] = {};
  StepBufs st[kMaxT];
  bf16 *xd_hi = nullptr, *xd_mid = nullptr, *xd_lo = nullptr;
  float* stats = nullptr;
  // backward
  float *dh = nullptr, *dh_acc = nullptr, *dx = nullptr;
  bf16* dpre_all = nullptr;  // [T*M, 3D]: per step t (row offset t*M) the column blocks [dpre_h | dpre_z | dpre_r]
  bf16 *da = nullptr, *ada = nullptr, *e = nullptr, *dlb = nullptr;
  float* G_P = nullptr;   // [3D, D] fp32: d/dP_x accumulated over the steps of this path
  bf16* G_Pb = nullptr;   // bf16 copy for the chain-rule GEMMs
  float* s_all = nullptr; // [3D]: c * colsum(dpre_x), for the W_x b_p bias term
  size_t bytes = 0;
};

struct Bump {
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* b) : base(static_cast<uint8_t*>(b)) {
    // absolute 1024-byte alignment (the size query reserves the worst-case slack for it)
    if (base) off = (1024 - (reinterpret_cast<uintptr_t>(base) & 1023)) & 1023;
  }
  template <typename T>
  T* take(size_t n) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += (n * sizeof(T) + 1023) & ~static_cast<size_t>(1023);
    return p;
  }
};

inline bool base_is_null(const void* ws) { return ws == nullptr; }

// Lay the buffers of one path out in `ws` (ws == nullptr: only compute the size).
// rowmap: the path uses the device-resident row layout (srg_nouns_*): B*R node slots + the shared pad row, rounded up to
// whole 256-row tiles, is the upper bound of its rows; otherwise the rows are the dense B*R / B rows of the caller.
PathBufs carve(const srg_handle* h, int mode, int B, int prec, int save, void* ws, bool rowmap) {
  PathBufs pb;
  const int D = h->D, T = h->T;
  const int Mfull = (mode == SRG_MODE_NOUN) ? B * h->R : B;
  const int M = rowmap ? round_up(Mfull + 1, 256) : Mfull;
  const size_t MD = static_cast<size_t>(M) * D;
  const size_t MfD = static_cast<size_t>(Mfull) * D;
  const bool f32 = (prec == SRG_PREC_FP32);
  const int npad = (mode == SRG_MODE_NOUN) ? h->Lpad : h->Vpad;
  Bump bump(ws);
  pb.M = M;
  pb.Mfull = Mfull;
  if (rowmap) {
    pb.rm.cnt = bump.take<int>(B);
    pb.rm.off = bump.take<int>(static_cast<size_t>(B) + 1);
    pb.rm.meta = bump.take<int>(4);
    pb.rm.compact = h->compact;
  }
  pb.h32 = bump.take<float>(MD);
  // operand copies of the state, one per step boundary: ONE contiguous [(T+1)*M, D] array in training mode (the
  // weight-gradient GEMMs read steps 0..T-1 as a single K = T*M operand), two ping-pong blocks otherwise
  const int n_hb = save ? T + 1 : 2;
  bf16* hb_all = bump.take<bf16>(static_cast<size_t>(n_hb) * MD);
  bf16* hb_mid_all = f32 ? bump.take<bf16>(static_cast<size_t>(n_hb) * MD) : nullptr;
  bf16* hb_lo_all = f32 ? bump.take<bf16>(static_cast<size_t>(n_hb) * MD) : nullptr;
  for (int t = 0; t <= T; ++t) {
    const size_t off = static_cast<size_t>(save ? t : (t & 1)) * MD;
    pb.hb_hi[t] = hb_all ? hb_all + off : nullptr;
    pb.hb_mid[t] = hb_mid_all ? hb_mid_all + off : nullptr;
    pb.hb_lo[t] = hb_lo_all ? hb_lo_all + off : nullptr;
  }
  // per-step buffers; in training mode each kind is ONE contiguous [T*M, D] array (step t at row offset t*M), so the
  // weight-gradient GEMMs can contract over all T steps in a single launch (K = T*M)
  const int n_st = save ? T : 1;
  const size_t n_all = static_cast<size_t>(n_st) * MD;
  bf16* a_all = (mode == SRG_MODE_NOUN) ? bump.take<bf16>(n_all) : nullptr;
  bf16* a_mid_all = (mode == SRG_MODE_NOUN && f32) ? bump.take<bf16>(n_all) : nullptr;
  bf16* a_lo_all = (mode == SRG_MODE_NOUN && f32) ? bump.take<bf16>(n_all) : nullptr;
  bf16* rh_all = bump.take<bf16>(n_all);
  bf16* rh_mid_all = f32 ? bump.take<bf16>(n_all) : nullptr;
  bf16* rh_lo_all = f32 ? bump.take<bf16>(n_all) : nullptr;
  uint8_t* z_all = f32 ? reinterpret_cast<uint8_t*>(bump.take<float>(n_all)) : reinterpret_cast<uint8_t*>(bump.take<bf16>(n_all));
  bf16* r_all = save ? bump.take<bf16>(n_all) : nullptr;
  bf16* hc_all = save ? bump.take<bf16>(n_all) : nullptr;
  for (int t = 0; t < T; ++t) {
    const size_t off = (save ? static_cast<size_t>(t) : 0) * MD;
    StepBufs& st = pb.st[t];
    st.a_hi = a_all ? a_all + off : nullptr;
    st.a_mid = a_mid_all ? a_mid_all + off : nullptr;
    st.a_lo = a_lo_all ? a_lo_all + off : nullptr;
    st.rh_hi = rh_all + off;
    st.rh_mid = rh_mid_all ? rh_mid_all + off : nullptr;
    st.rh_lo = rh_lo_all ? rh_lo_all + off : nullptr;
    st.z = (base_is_null(ws)) ? nullptr : static_cast<void*>(z_all + off * (f32 ? 4 : 2));
    st.r = r_all ? r_all + off : nullptr;
    st.hc = hc_all ? hc_all + off : nullptr;
  }
  // classifier side: one row per node slot
  pb.xd_hi = bump.take<bf16>(MfD);
  pb.xd_mid = f32 ? bump.take<bf16>(MfD) : nullptr;
  pb.xd_lo = f32 ? bump.take<bf16>(MfD) : nullptr;
  pb.stats = bump.take<float>(static_cast<size_t>(Mfull) * (npad / 128) * 2);
  if (save) {
    pb.dh = bump.take<float>(MD);
    pb.dh_acc = bump.take<float>(MD);
    pb.dx = bump.take<float>(MfD);
    pb.dpre_all = bump.take<bf16>(static_cast<size_t>(T) * 3 * MD);
    pb.da = bump.take<bf16>(MD);
    pb.ada = bump.take<bf16>(MD);
    pb.e = bump.take<bf16>(MD);
    pb.dlb = bump.take<bf16>(static_cast<size_t>(Mfull) * npad);
    pb.G_P = bump.take<float>(static_cast<size_t>(3) * D * D);
    pb.G_Pb = bump.take<bf16>(static_cast<size_t>(3) * D * D);
    pb.s_all = bump.take<float>(static_cast<size_t>(3) * D);
  }
  pb.bytes = bump.off + 1024;
  return pb;
}

int check_ws(const srg_handle* h, int mode, int B, int prec, int save, void* ws, size_t ws_bytes, PathBufs* out,
             bool rowmap) {
  SRG_CHECK(h != nullptr, "null handle");
  SRG_CHECK(B > 0, "batch must be positive (got %d)", B);
  SRG_CHECK(prec == SRG_PREC_BF16 || prec == SRG_PREC_FP32, "bad precision %d", prec);
  SRG_CHECK(!(save && prec != SRG_PREC_BF16), "save_for_backward requires SRG_PREC_BF16 (the fp32 mode is forward-only)");
  SRG_CHECK(ws != nullptr, "null workspace");
  SRG_CHECK((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "workspace must be 16-byte aligned");
  *out = carve(h, mode, B, prec, save, ws, rowmap);
  const size_t need = carve(h, mode, B, prec, save, nullptr, rowmap).bytes;
  if (need > ws_bytes)
    return set_error(SRG_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, ws_bytes);
  return SRG_OK;
}

// ------------------------------------------------------------------------------------------------ GEMM helpers
GemmProblem base_problem(const srg_handle* h, int M, int N) {
  GemmProblem p;
  p.cg = h->cg;
  p.M = M;
  p.N = N;
  return p;
}

// a GEMM over the node rows of a path: M is the allocated upper bound, the kernel reads the actual row count
GemmProblem path_problem(const srg_handle* h, const PathBufs& pb, int N) {
  GemmProblem p = base_problem(h, pb.M, N);
  p.m_dev = pb.rm.meta;   // meta[0]; nullptr = static rows
  return p;
}

void add_seg_ld(GemmProblem& p, const bf16* a, int64_t rows, int64_t cols, int64_t ld, int k_off, int k_len) {
  GemmSeg& s = p.seg[p.nseg++];
  s.a = mat(a, rows, cols, ld, DT_BF16);
  s.k_off = k_off;
  s.k_len = k_len;
}
void add_seg(GemmProblem& p, const bf16* a, int64_t rows, int64_t cols, int k_off, int k_len) {
  add_seg_ld(p, a, rows, cols, cols, k_off, k_len);
}

// fp32-parity arithmetic: every operand is x = hi + mid + lo (three bf16 parts, 24 significant bits) and a product is
// expanded into the six terms of weight >= 2^-16:  hi*hi + hi*mid + mid*hi + hi*lo + lo*hi + mid*mid.
// K block b of the packed weights holds part kPartB[b]; the activation segments carry part kPartA[b].
constexpr int kSplitTerms = 6;
constexpr int kPartA[kSplitTerms] = {0, 0, 1, 0, 2, 1};
constexpr int kPartB[kSplitTerms] = {0, 1, 0, 2, 0, 1};

struct Split3 {
  const bf16* part[3];
};

// A = [x0 | x1 | ...] (each [M, D]), replicated per split term in fp32 mode
void add_split_segs(GemmProblem& p, int M, int D, bool f32, const Split3* x, int n) {
  const int terms = f32 ? kSplitTerms : 1;
  for (int b = 0; b < terms; ++b)
    for (int i = 0; i < n; ++i) add_seg(p, x[i].part[kPartA[b]], M, D, 0, D);
  if (f32) p.corr_seg_begin = n;   // term 0 (hi*hi) -> main accumulator, terms 1..5 -> correction accumulator
}

int wgrad_splits(const srg_handle* h, int out_rows, int out_cols, int K) {
  const int bn = (h->cg == 2) ? 256 : 128;
  const int tiles = ((out_rows + 128 * h->cg - 1) / (128 * h->cg)) * (out_cols / bn);
  const int clusters = h->dev.num_sms / h->cg;
  int s = (clusters * 7 + tiles - 1) / tiles;  // ~7 waves
  const int kb = (K + kBlockK - 1) / kBlockK;
  if (s > kb) s = kb;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  return s;
}

// dW[out, in] += dY^T[out, K] * X[K, in]   (both operands MN-major, split-K, TMA reduce-add).
// dY is a column block (out_rows columns, leading dimension dy_ld) of a wider matrix.  K runs over `nseg` row segments
// of `seg_rows` rows each, segment t starting at row t * seg_stride of BOTH operands (the T propagation steps of a
// path); k_dev (nullable) = device-resident number of valid rows per segment (seg_rows is then its upper bound).
int wgrad(const srg_handle* h, const bf16* dY, int64_t dy_ld, int out_rows, const bf16* X, int in_cols, int nseg,
          int seg_rows, int64_t seg_stride, const int* k_dev, float* dW, cudaStream_t s) {
  if (dW == nullptr) return SRG_OK;
  const int64_t phys_rows = static_cast<int64_t>(nseg - 1) * seg_stride + seg_rows;
  GemmProblem p = base_problem(h, out_rows, in_cols);
  p.a_mn = true;
  p.b_mn = true;
  p.epi = EPI_STORE_F32;
  p.flags = FLAG_REDUCE;
  if (nseg > 1 && seg_stride == seg_rows && k_dev == nullptr) {   // dense: one long K
    nseg = 1;
    seg_rows = static_cast<int>(phys_rows);
  }
  SRG_CHECK(nseg >= 1 && nseg <= kMaxSeg, "wgrad: bad segment count %d", nseg);
  p.nseg = nseg;
  for (int t = 0; t < nseg; ++t) {
    p.seg[t].a = mat(dY, phys_rows, out_rows, dy_ld, DT_BF16);
    p.seg[t].k_off = static_cast<int>(t * seg_stride);
    p.seg[t].k_len = seg_rows;
  }
  if (nseg > 1 || k_dev != nullptr) p.flags |= FLAG_BK_A;
  p.k_dev = k_dev;
  p.b = mat(X, phys_rows, in_cols, in_cols, DT_BF16);
  p.io[0] = mat(dW, out_rows, in_cols, in_cols, DT_F32);
  // expected K for the split heuristic: the compact layout keeps ~0.6 of the slots (imSitu: 3.55 of 6 roles)
  const int64_t k_expect = static_cast<int64_t>(nseg) * seg_rows * ((k_dev != nullptr && h->compact) ? 3 : 5) / 5;
  p.k_splits = wgrad_splits(h, out_rows, in_cols, static_cast<int>(k_expect));
  return run_gemm(p, h->dev, s);
}

// ------------------------------------------------------------------------------------------------ forward
// mask: caller-provided [B,R,R] adjacency (srg_ggnn_forward on dense rows); nullptr on a role-graph path with a row map
// (the aggregation then follows from the role counts) and on the verb node path.
int ggnn_steps(srg_handle* h, int mode, PathBufs& pb, float* h32, const float* mask, int B, int prec, int save,
               cudaStream_t s) {
  const int D = h->D, T = h->T, M = pb.M;
  const bool f32 = (prec == SRG_PREC_FP32);
  const int kmul = f32 ? kSplitTerms : 1;
  const int mi = (mode == SRG_MODE_NOUN) ? 0 : 1;
  for (int t = 0; t < T; ++t) {
    StepBufs& st = pb.st[t];
    // aggregated neighbour state a[b,i] = sum_j mask[b,i,j] h[b,j]  (model.py:67-75); verb mode: a = h (62-64)
    const Split3 hcur = {{pb.hb_hi[t], pb.hb_mid[t], pb.hb_lo[t]}};
    Split3 a = hcur;
    if (mode == SRG_MODE_NOUN) {
      if (pb.rm.meta != nullptr) SRG_TRY(launch_aggregate_rows(h32, pb.rm, B, h->R, D, st.a_hi, st.a_mid, st.a_lo, s));
      else SRG_TRY(launch_aggregate(h32, mask, B, h->R, D, st.a_hi, st.a_mid, st.a_lo, s));
      a = Split3{{st.a_hi, st.a_mid, st.a_lo}};
    }
    const Split3 rh = {{st.rh_hi, st.rh_mid, st.rh_lo}};
    {  // gates: [z | r] = sigmoid([a | h] [P_z U_z ; P_r U_r]^T + b'), rh = r * h      (model.py:74,80-81)
      GemmProblem p = path_problem(h, pb, 2 * D);
      const Split3 ops[2] = {a, hcur};
      add_split_segs(p, M, D, f32, ops, 2);
      p.b = mat(h->Wzr, 2 * D, static_cast<int64_t>(2 * D) * kmul, static_cast<int64_t>(2 * D) * kmul, DT_BF16);
      p.epi = EPI_ZR;
      p.f32 = f32;
      p.bias = h->bzr[mi];
      p.n_split = D;
      p.flags = (f32 ? FLAG_LO : 0) | (save ? FLAG_STASH : 0);
      p.io[0] = mat(st.z, M, D, D, f32 ? DT_F32 : DT_BF16);
      p.io[1] = mat(h32, M, D, D, DT_F32);
      p.io[2] = mat(st.rh_hi, M, D, D, DT_BF16);
      if (f32) {
        p.io[3] = mat(st.rh_mid, M, D, D, DT_BF16);
        p.io[5] = mat(st.rh_lo, M, D, D, DT_BF16);
      }
      if (save) p.io[4] = mat(st.r, M, D, D, DT_BF16);
      SRG_TRY(run_gemm(p, h->dev, s));
    }
    {  // candidate + update: h' = h + z * (tanh([a | rh] [P_h U_h]^T + b') - h)      (model.py:82-84)
      GemmProblem p = path_problem(h, pb, D);
      const Split3 ops[2] = {a, rh};
      add_split_segs(p, M, D, f32, ops, 2);
      p.b = mat(h->Wh, D, static_cast<int64_t>(2 * D) * kmul, static_cast<int64_t>(2 * D) * kmul, DT_BF16);
      p.epi = EPI_H;
      p.f32 = f32;
      p.bias = h->bh[mi];
      p.flags = save ? FLAG_STASH : 0;
      p.io[0] = mat(h32, M, D, D, DT_F32);
      p.io[1] = mat(st.z, M, D, D, f32 ? DT_F32 : DT_BF16);
      p.io[2] = mat(pb.hb_hi[t + 1], M, D, D, DT_BF16);
      if (f32) {
        p.io[3] = mat(pb.hb_mid[t + 1], M, D, D, DT_BF16);
        p.io[5] = mat(pb.hb_lo[t + 1], M, D, D, DT_BF16);
      }
      if (save) p.io[4] = mat(st.hc, M, D, D, DT_BF16);
      SRG_TRY(run_gemm(p, h->dev, s));
    }
  }
  return SRG_OK;
}

// Dropout in front of a classifier (model.py:106,110): explicit keep-mask, or Philox keyed by the device seed, or none.
int make_drop(const uint8_t* keep, float drop_p, const int64_t* seed, int64_t stream_id, DropSpec* ds) {
  SRG_CHECK(drop_p >= 0.f && drop_p < 1.f, "dropout probability %f out of range", drop_p);
  *ds = DropSpec();
  if (drop_p > 0.f && (keep != nullptr || seed != nullptr)) {
    ds->keep = keep;
    ds->seed = (keep == nullptr) ? reinterpret_cast<const long long*>(seed) : nullptr;
    ds->stream = stream_id;
    ds->thresh = static_cast<uint32_t>((1.0 - static_cast<double>(drop_p)) * 65536.0 + 0.5);
    ds->scale = 1.0f / (1.0f - drop_p);
  }
  return SRG_OK;
}

int classifier_forward(srg_handle* h, int mode, PathBufs& pb, const float* h32, const DropSpec& ds, float* logits,
                       int64_t ldl, int prec, cudaStream_t s) {
  const int D = h->D, M = pb.Mfull;
  const bool f32 = (prec == SRG_PREC_FP32);
  const int kmul = f32 ? kSplitTerms : 1;
  const int ncls = (mode == SRG_MODE_NOUN) ? h->L : h->V;
  const int npad = (mode == SRG_MODE_NOUN) ? h->Lpad : h->Vpad;
  SRG_CHECK(ldl >= ncls && (ldl % 4) == 0, "logits leading dimension %lld must be >= %d and a multiple of 4",
            (long long)ldl, ncls);
  // The classifier runs on every node slot: a dense [Mfull, D] operand is gathered from the (compact) state rows with
  // the dropout applied per slot.  Dense rows without dropout (verb node in eval mode) read the state operand directly.
  Split3 x = {{pb.hb_hi[h->T], pb.hb_mid[h->T], pb.hb_lo[h->T]}};
  const bool use_drop = (ds.keep != nullptr || ds.seed != nullptr);
  if (use_drop || pb.rm.meta != nullptr) {
    SRG_TRY(launch_classifier_input(h32, pb.rm, h->R, M, D, ds, pb.xd_hi, pb.xd_mid, pb.xd_lo, s));
    x = Split3{{pb.xd_hi, pb.xd_mid, pb.xd_lo}};
  }
  GemmProblem p = base_problem(h, M, npad);
  add_split_segs(p, M, D, f32, &x, 1);
  const bf16* W = (mode == SRG_MODE_NOUN) ? h->Wcn : h->Wcv;
  p.b = mat(W, npad, static_cast<int64_t>(D) * kmul, static_cast<int64_t>(D) * kmul, DT_BF16);
  p.epi = EPI_LOGITS;
  p.f32 = f32;
  p.bias = (mode == SRG_MODE_NOUN) ? h->bcn : h->bcv;
  p.n_valid = ncls;
  p.stats = pb.stats;
  p.io[0] = mat(logits, M, ldl < npad ? ldl : npad, ldl, DT_F32);
  return run_gemm(p, h->dev, s);
}

// ------------------------------------------------------------------------------------------------ chain rule
// Through P_x = W_x W_p and b'_x = b_Wx + b_Ux + c W_x b_p  (x = h, z, r):
//   dW_x += dP_x W_p^T + s_x (x) b_p,   dW_p += sum_x W_x^T dP_x,   db_p += sum_x W_x^T s_x,   s_x = c colsum(dpre_x).
// shared_dst: another stream may be accumulating into the same gradients (per-path mode on two streams).
int chain_rule(srg_handle* h, const float* G_P, bf16* G_Pb, const float* s_all, const srg_grads* g, bool shared_dst,
               cudaStream_t s) {
  const int D = h->D;
  SRG_TRY(launch_split_cast(G_P, static_cast<int64_t>(3) * D * D, G_Pb, nullptr, nullptr, s));
  float* gW[3] = {g->W_h, g->W_z, g->W_r};
  const float* W32[3] = {h->params.W_h, h->params.W_z, h->params.W_r};
  for (int x3 = 0; x3 < 3; ++x3) {
    if (gW[x3] == nullptr) continue;
    GemmProblem p = base_problem(h, D, D);
    add_seg(p, G_Pb + static_cast<size_t>(x3) * D * D, D, D, 0, D);
    p.b = mat(h->Wp6, D, D, D, DT_BF16);  // first block of Wp6 = bf16(W_p), K-major [k, i]
    p.epi = EPI_STORE_F32;
    p.flags = FLAG_REDUCE;
    p.io[0] = mat(gW[x3], D, D, D, DT_F32);
    SRG_TRY(run_gemm(p, h->dev, s));
  }
  SRG_TRY(launch_outer_acc3(s_all, h->params.b_p, D, D, gW, shared_dst, s));
  if (g->b_p != nullptr) SRG_TRY(launch_matvec_t_acc3(W32, s_all, D, D, g->b_p, s));
  if (g->W_p != nullptr) {  // dW_p += [W_h; W_z; W_r]^T [dP_h; dP_z; dP_r]
    GemmProblem p = base_problem(h, D, D);
    p.a_mn = true;
    p.b_mn = true;
    p.nseg = 1;
    p.seg[0].a = mat(h->Wm_hi, 3 * D, D, D, DT_BF16);
    p.seg[0].k_off = 0;
    p.seg[0].k_len = 3 * D;
    p.b = mat(G_Pb, 3 * D, D, D, DT_BF16);
    p.epi = EPI_STORE_F32;
    p.flags = FLAG_REDUCE;
    p.io[0] = mat(g->W_p, D, D, D, DT_F32);
    p.k_splits = wgrad_splits(h, D, D, 3 * D);
    SRG_TRY(run_gemm(p, h->dev, s));
  }
  return SRG_OK;
}

// ------------------------------------------------------------------------------------------------ backward
// d/dP_x and the bias column sums of one backward call: per call (cleared here), or (deferred chain rule) shared by all
// paths of the step
int chain_acc(srg_handle* h, PathBufs& pb, float** G_P, float** s_all, cudaStream_t s) {
  const int D = h->D;
  *G_P = h->defer_chain ? h->acc_GP : pb.G_P;
  *s_all = h->defer_chain ? h->acc_s : pb.s_all;
  if (!h->defer_chain) {
    SRG_CUDA(cudaMemsetAsync(*G_P, 0, sizeof(float) * 3 * D * D, s));
    SRG_CUDA(cudaMemsetAsync(*s_all, 0, sizeof(float) * 3 * D, s));
  }
  return SRG_OK;
}

// The GGNN steps of a backward pass, on the stash of a save_for_backward forward: the gate derivatives of the last step
// from dh_T = dL/dh_T fp32 [M, D] (read only; nullptr: the caller already wrote them), steps t = T-1..0, the weight
// gradients, and the chain rule (or, deferred, only the accumulation into G_P / s_all).  mask: the [B,R,R] mask of
// srg_ggnn_forward on dense rows, whose aggregation backward also yields dL/dmask when dmask is given (the caller clears
// it); nullptr on a row-mapped role graph and on the verb node.  Leaves dL/d(initial states) in pb.dh.
int ggnn_backward(srg_handle* h, int mode, PathBufs& pb, int B, const float* dh_T, const float* mask, float* dmask,
                  float* G_P, float* s_all, const srg_grads* g, cudaStream_t s) {
  const int D = h->D, T = h->T, M = pb.M, R = h->R;
  const int64_t ld3 = 3 * static_cast<int64_t>(D);
  const float cmul = (mode == SRG_MODE_NOUN) ? static_cast<float>(R) : 1.f;  // how often b_p enters a message
  const bool mapped = (pb.rm.meta != nullptr);            // role-graph path on the device-resident row layout
  const int* m_dev = mapped ? pb.rm.meta : nullptr;          // rows incl. the shared pad row

  // dL/dh' of the last step comes from the caller; from there on the GRU-gate derivatives of step t-1 are fused into
  // the epilogue of the GEMM that completes dL/dh of step t (EPI_DH).
  // dpre_of(t) = [dpre_h | dpre_z | dpre_r] of step t as column blocks of one [M, 3D] matrix.
  float* dh_acc = pb.dh_acc;
  auto dpre_of = [&](int t) { return pb.dpre_all + static_cast<size_t>(t) * M * ld3; };
  if (dh_T != nullptr)
    SRG_TRY(launch_gru_bwd_pre_ld(dh_T, static_cast<const bf16*>(pb.st[T - 1].z), pb.st[T - 1].hc, pb.hb_hi[T - 1], M,
                                  nullptr, nullptr, D, dpre_of(T - 1) + D, dpre_of(T - 1), ld3, dh_acc, s));
  for (int t = T - 1; t >= 0; --t) {
    StepBufs& st = pb.st[t];
    bf16* dp = dpre_of(t);
    bf16* dpre_r = dp + 2 * D;   // column blocks of dp: [dpre_h | dpre_z | dpre_r]
    {  // d(r*h) = dpre_h U_h ; fused: dpre_r = drh*h*r*(1-r), e = drh*r (this path's share of dL/dh)
      GemmProblem p = path_problem(h, pb, D);
      add_seg_ld(p, dp, M, ld3, ld3, 0, D);
      p.b_mn = true;
      p.b = mat(h->Uh, D, D, D, DT_BF16);
      p.epi = EPI_DRH;
      p.io[0] = mat(pb.hb_hi[t], M, D, D, DT_BF16);
      p.io[1] = mat(st.r, M, D, D, DT_BF16);
      p.io[2] = mat(dpre_r, M, D, ld3, DT_BF16);
      p.io[3] = mat(pb.e, M, D, D, DT_BF16);
      SRG_TRY(run_gemm(p, h->dev, s));
    }
    {  // da = [dpre_h | dpre_z | dpre_r] [P_h ; P_z ; P_r]   (gradient w.r.t. the aggregated state)
      GemmProblem p = path_problem(h, pb, D);
      add_seg_ld(p, dp, M, ld3, ld3, 0, 3 * D);
      p.b_mn = true;
      p.b = mat(h->P_hi, 3 * D, D, D, DT_BF16);
      p.epi = EPI_STORE_BF16;
      p.io[0] = mat(pb.da, M, D, D, DT_BF16);
      SRG_TRY(run_gemm(p, h->dev, s));
    }
    // back through the aggregation, plus the r*h share:  ada[j] = e[j] + sum_i mask[i,j] da[i]
    // (verb node: the aggregation is the identity)
    if (mask != nullptr) SRG_TRY(launch_aggregate_t(pb.da, pb.e, mask, pb.hb_hi[t], B, R, D, pb.ada, dmask, s));
    else SRG_TRY(launch_aggregate_t_rows(pb.da, pb.e, pb.rm, mapped ? B : M, R, D, pb.ada, s));
    const bf16* ada = pb.ada;
    {  // dL/dh_t = dh_acc + ada + [dpre_z | dpre_r] [U_z ; U_r], then the gate derivatives of step t-1
      GemmProblem p = path_problem(h, pb, D);
      add_seg_ld(p, dp, M, ld3, ld3, D, 2 * D);
      p.b_mn = true;
      p.b = mat(h->U_stack, 2 * D, D, D, DT_BF16);
      p.epi = EPI_DH;
      p.flags = FLAG_ADD;
      p.io[0] = mat(dh_acc, M, D, D, DT_F32);
      p.io[6] = mat(ada, M, D, D, DT_BF16);
      if (t > 0) {
        bf16* dn = dpre_of(t - 1);
        p.flags |= FLAG_NEXT;
        p.io[1] = mat(pb.st[t - 1].z, M, D, D, DT_BF16);
        p.io[2] = mat(pb.st[t - 1].hc, M, D, D, DT_BF16);
        p.io[3] = mat(pb.hb_hi[t - 1], M, D, D, DT_BF16);
        p.io[4] = mat(dn + D, M, D, ld3, DT_BF16);  // dpre_z of step t-1
        p.io[5] = mat(dn, M, D, ld3, DT_BF16);      // dpre_h of step t-1
      }
      SRG_TRY(run_gemm(p, h->dev, s));
    }
  }
  // ---- weight gradients: one GEMM per weight group, contracting over all T steps at once.  Step t occupies rows
  // [t*M, t*M + rows) of every stash array; on the device-resident layout `rows` is read by the kernel and the rows
  // between it and the next k-block boundary hold dpre = 0 (their dL/dh is 0 from k_zero_self_rows on).
  {
    bf16* dp = pb.dpre_all;
    const bf16* a_all = (mode == SRG_MODE_NOUN) ? pb.st[0].a_hi : pb.hb_hi[0];   // step t at row offset t*M
    SRG_TRY(wgrad(h, dp, ld3, 3 * D, a_all, D, T, M, M, m_dev, G_P, s));                 // dP_h, dP_z, dP_r in one GEMM
    SRG_TRY(wgrad(h, dp + D, ld3, D, pb.hb_hi[0], D, T, M, M, m_dev, g->U_z, s));
    SRG_TRY(wgrad(h, dp + 2 * D, ld3, D, pb.hb_hi[0], D, T, M, M, m_dev, g->U_r, s));
    SRG_TRY(wgrad(h, dp, ld3, D, pb.st[0].rh_hi, D, T, M, M, m_dev, g->U_h, s));
    ColsumJob jobs[3] = {{dp, g->b_Wh, g->b_Uh, 1.f, s_all, cmul},
                         {dp + D, g->b_Wz, g->b_Uz, 1.f, s_all + D, cmul},
                         {dp + 2 * D, g->b_Wr, g->b_Ur, 1.f, s_all + 2 * D, cmul}};
    if (mapped) SRG_TRY(launch_colsum_multi(jobs, 3, ld3, M, m_dev, T, M, D, s));
    else SRG_TRY(launch_colsum_multi(jobs, 3, ld3, T * M, nullptr, 1, 0, D, s));
  }
  pb.dh = dh_acc;  // gradient w.r.t. the initial node states

  if (h->defer_chain) return SRG_OK;   // srg_chain_finalize applies the chain rule once for all paths
  return chain_rule(h, G_P, pb.G_Pb, s_all, g, /*shared_dst=*/true, s);
}

// dlogits (nullable) fp32 [Mfull, ldl]; dlb_ready: the bf16 gradient operand pb.dlb already holds a gradient written by
// the loss kernels (srg_*_loss_backward with dlogits_bf16); both given: their sum.
int path_backward(srg_handle* h, int mode, PathBufs& pb, const float* dlogits, int64_t ldl, int dlb_ready, int B,
                  const DropSpec& ds, const srg_grads* g, cudaStream_t s) {
  const int D = h->D, T = h->T, Mf = pb.Mfull, R = h->R;
  const int ncls = (mode == SRG_MODE_NOUN) ? h->L : h->V;
  const int npad = (mode == SRG_MODE_NOUN) ? h->Lpad : h->Vpad;
  const bf16* Wc = (mode == SRG_MODE_NOUN) ? h->Wcn : h->Wcv;
  float* gWc = (mode == SRG_MODE_NOUN) ? g->Wc_noun : g->Wc_verb;
  float* gbc = (mode == SRG_MODE_NOUN) ? g->bc_noun : g->bc_verb;
  const int64_t ld3 = 3 * static_cast<int64_t>(D);
  const bool use_drop = (ds.keep != nullptr || ds.seed != nullptr);
  const bool mapped = (pb.rm.meta != nullptr);            // role-graph path on the device-resident row layout
  const bool gathered = use_drop || mapped;               // the classifier read pb.xd_hi (see classifier_forward)
  const bf16* x = gathered ? pb.xd_hi : pb.hb_hi[T];
  const int* rows_dev = mapped ? pb.rm.meta + 2 : nullptr;   // rows the tiles touch (multiple of 256)

  float *G_P = nullptr, *s_all = nullptr;
  SRG_TRY(chain_acc(h, pb, &G_P, &s_all, s));

  // ---- classifier (model.py:105-111,152,168): one row per node slot
  SRG_CHECK(dlogits != nullptr || dlb_ready, "backward: no gradient of the logits was given");
  if (dlogits != nullptr) SRG_TRY(launch_cast_pad(dlogits, ldl, Mf, ncls, npad, pb.dlb, dlb_ready ? 1 : 0, s));
  SRG_TRY(launch_colsum(pb.dlb, npad, Mf, ncls, gbc, 1.f, nullptr, 0.f, s));
  SRG_TRY(wgrad(h, pb.dlb, npad, ncls, x, D, 1, Mf, Mf, nullptr, gWc, s));
  {
    GemmProblem p = base_problem(h, Mf, D);
    add_seg(p, pb.dlb, Mf, npad, 0, npad);
    p.b_mn = true;
    p.b = mat(Wc, npad, D, D, DT_BF16);
    p.epi = EPI_STORE_F32;
    p.io[0] = mat(gathered ? pb.dx : pb.dh, Mf, D, D, DT_F32);
    SRG_TRY(run_gemm(p, h->dev, s));
  }
  if (gathered) {
    // back through the dropout and the slot -> state-row gather, with the gate derivatives of the last step applied in
    // the same pass for every row that has exactly one slot; the pad slots of all images add up in the shared pad row,
    // whose derivatives (and the zero rows up to the tile boundary) follow in a launch over those few rows
    bf16* dp = pb.dpre_all + static_cast<size_t>(T - 1) * pb.M * ld3;
    GruPre gp;
    gp.z = static_cast<const bf16*>(pb.st[T - 1].z);
    gp.hc = pb.st[T - 1].hc;
    gp.h = pb.hb_hi[T - 1];
    gp.dpre_z = dp + D;
    gp.dpre_h = dp;
    gp.ld_out = ld3;
    gp.dh_acc = pb.dh_acc;
    SRG_TRY(launch_classifier_input_bwd(pb.dx, pb.rm, (mode == SRG_MODE_NOUN) ? B : Mf, (mode == SRG_MODE_NOUN) ? R : 1,
                                        D, ds, pb.dh, gp, s));
    if (mapped)
      SRG_TRY(launch_gru_bwd_pre_ld(pb.dh, gp.z, gp.hc, gp.h, 256, rows_dev, pb.rm.meta + 1, D, gp.dpre_z, gp.dpre_h,
                                    ld3, pb.dh_acc, s));
  }
  return ggnn_backward(h, mode, pb, B, gathered ? nullptr : pb.dh, nullptr, nullptr, G_P, s_all, g, s);
}

int ensure_pack_buffers(srg_handle* h, int split) {
  const size_t D = h->D;
  auto re = [&](bf16** p, size_t n) -> int {
    if (*p) cudaFree(*p);
    *p = nullptr;
    SRG_CUDA(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(bf16)));
    return SRG_OK;
  };
  auto f32buf = [&](float** p, size_t n) -> int {
    SRG_CUDA(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(float)));
    return SRG_OK;
  };
  if (!h->Wm_hi) {
    SRG_TRY(re(&h->Wm_hi, 3 * D * D));
    SRG_TRY(re(&h->Wm_mid, 3 * D * D));
    SRG_TRY(re(&h->Wm_lo, 3 * D * D));
    SRG_TRY(re(&h->Wp6, 6 * D * D));
    SRG_TRY(re(&h->P_hi, 3 * D * D));
    SRG_TRY(re(&h->P_mid, 3 * D * D));
    SRG_TRY(re(&h->P_lo, 3 * D * D));
    SRG_TRY(re(&h->U_stack, 2 * D * D));
    SRG_TRY(re(&h->Uh, D * D));
    SRG_TRY(f32buf(&h->wb, 3 * D));
    for (int i = 0; i < 2; ++i) {
      SRG_TRY(f32buf(&h->bzr[i], 2 * D));
      SRG_TRY(f32buf(&h->bh[i], D));
    }
    SRG_TRY(f32buf(&h->bcn, h->Lpad));
    SRG_TRY(f32buf(&h->bcv, h->Vpad));
  }
  if (h->alloc_split >= split) return SRG_OK;
  SRG_TRY(re(&h->Wzr, 2 * D * 2 * D * split));
  SRG_TRY(re(&h->Wh, D * 2 * D * split));
  SRG_TRY(re(&h->Wcn, static_cast<size_t>(h->Lpad) * D * split));
  SRG_TRY(re(&h->Wcv, static_cast<size_t>(h->Vpad) * D * split));
  h->alloc_split = split;
  return SRG_OK;
}

// dst[rows 0..D, col_off .. col_off+D] (leading dimension ld) <- src[D, D]
int copy_block(bf16* dst, int64_t ld, int64_t row_off, int64_t col_off, const bf16* src, int D, cudaStream_t s) {
  SRG_CUDA(cudaMemcpy2DAsync(dst + row_off * ld + col_off, ld * sizeof(bf16), src, D * sizeof(bf16), D * sizeof(bf16), D,
                             cudaMemcpyDeviceToDevice, s));
  return SRG_OK;
}

}  // namespace

// ================================================================================================== C ABI
extern "C" {

int srg_version(void) { return 100; }

int srg_create(srg_handle** out, int device, int D, int R, int T, int n_verbs, int n_roles, int n_labels) {
  SRG_CHECK(out != nullptr, "srg_create: null output pointer");
  SRG_CHECK(D > 0 && D % 256 == 0, "hidden size D=%d must be a positive multiple of 256", D);
  SRG_CHECK(R >= 1 && R <= 8, "max role count R=%d must be in [1, 8]", R);
  SRG_CHECK(T >= 1 && T <= kMaxT, "propagation steps T=%d must be in [1, %d]", T, kMaxT);
  SRG_CHECK(n_verbs > 0 && n_roles > 0 && n_labels > 0, "vocabulary sizes must be positive");
  SRG_CUDA(cudaSetDevice(device));
  srg_handle* h = new (std::nothrow) srg_handle();
  SRG_CHECK(h != nullptr, "out of host memory");
  h->device = device;
  h->D = D; h->R = R; h->T = T; h->V = n_verbs; h->n_roles = n_roles; h->L = n_labels;
  h->Vpad = round_up(n_verbs, 256);
  h->Lpad = round_up(n_labels, 256);
  int rc = query_device(&h->dev);
  if (rc != SRG_OK) { delete h; return rc; }
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&h->d_verb2roles), sizeof(int32_t) * n_verbs * R);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&h->d_role_count), sizeof(int32_t) * n_verbs);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&h->d_bad), sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(h->d_bad, 0, sizeof(int));
  if (e != cudaSuccess) {
    delete h;
    return set_error(SRG_ERR_CUDA, "srg_create: cudaMalloc failed: %s", cudaGetErrorString(e));
  }
  *out = h;
  return SRG_OK;
}

int srg_destroy(srg_handle* h) {
  if (!h) return SRG_OK;
  DeviceGuard guard_(h->device);
  void* ptrs[] = {h->d_verb2roles, h->d_role_count, h->d_bad, h->Wzr, h->Wh, h->Wcn, h->Wcv, h->Wm_hi, h->Wm_mid, h->Wm_lo, h->Wp6,
                  h->P_hi, h->P_mid, h->P_lo, h->U_stack, h->Uh, h->wb, h->bzr[0], h->bzr[1], h->bh[0], h->bh[1], h->bcn, h->bcv,
                  h->acc_GP, h->acc_GPb, h->acc_s};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  delete h;
  return SRG_OK;
}

int srg_set_cta_group(srg_handle* h, int cta_group) {
  SRG_CHECK(h != nullptr, "null handle");
  SRG_CHECK(cta_group == 1 || cta_group == 2, "cta_group must be 1 or 2");
  h->cg = cta_group;
  return SRG_OK;
}

int srg_set_compact_rows(srg_handle* h, int on) {
  SRG_CHECK(h != nullptr, "null handle");
  h->compact = (on != 0);
  return SRG_OK;
}

int srg_set_tables(srg_handle* h, const int32_t* verb2roles, const int32_t* role_count) {
  SRG_CHECK(h != nullptr, "srg_set_tables: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h && verb2roles && role_count, "srg_set_tables: null argument");
  for (int v = 0; v < h->V; ++v) {
    SRG_CHECK(role_count[v] >= 0 && role_count[v] <= h->R, "role_count[%d]=%d outside [0,%d]", v, role_count[v], h->R);
    for (int r = 0; r < h->R; ++r) {
      const int id = verb2roles[v * h->R + r];
      SRG_CHECK(id >= 0 && id <= h->n_roles, "verb2roles[%d,%d]=%d outside [0,%d]", v, r, id, h->n_roles);
    }
  }
  SRG_CUDA(cudaMemcpy(h->d_verb2roles, verb2roles, sizeof(int32_t) * h->V * h->R, cudaMemcpyHostToDevice));
  SRG_CUDA(cudaMemcpy(h->d_role_count, role_count, sizeof(int32_t) * h->V, cudaMemcpyHostToDevice));
  h->tables_set = true;
  return SRG_OK;
}

int srg_gather_mask(srg_handle* h, const int64_t* verb, int B, int64_t* role_idx, float* mask, int* bad_verb,
                    void* stream) {
  SRG_CHECK(h != nullptr, "srg_gather_mask: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h != nullptr && h->tables_set, "srg_gather_mask: call srg_set_tables first");
  SRG_CHECK(B >= 0, "negative batch");
  if (B == 0) return SRG_OK;
  SRG_CHECK(verb != nullptr, "null verb pointer");
  return launch_gather_mask(h->d_verb2roles, h->d_role_count, h->V, h->R, verb, B, role_idx, mask, bad_verb,
                            static_cast<cudaStream_t>(stream));
}

int srg_check_verbs(srg_handle* h, void* stream) {
  SRG_CHECK(h != nullptr, "srg_check_verbs: null handle");
  DeviceGuard guard_(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int bad = 0;
  SRG_CUDA(cudaMemcpyAsync(&bad, h->d_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  SRG_CUDA(cudaMemsetAsync(h->d_bad, 0, sizeof(int), s));
  SRG_CUDA(cudaStreamSynchronize(s));
  if (bad) return set_error(SRG_ERR_ARG, "a verb id outside [0, %d) was passed to srg_nouns_forward (it was computed as verb 0)", h->V);
  return SRG_OK;
}

int srg_pack_weights(srg_handle* h, const srg_params* p, int precision, void* stream) {
  SRG_CHECK(h != nullptr, "srg_pack_weights: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h && p, "srg_pack_weights: null argument");
  SRG_CHECK(precision == SRG_PREC_BF16 || precision == SRG_PREC_FP32, "bad precision %d", precision);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int D = h->D;
  const int split = (precision == SRG_PREC_FP32) ? kSplitTerms : 1;
  SRG_TRY(ensure_pack_buffers(h, split));
  h->params = *p;
  const size_t DD = static_cast<size_t>(D) * D;

  // All fp32 -> bf16 conversions of this call are queued as jobs and run as two launches (before / after the P GEMM).
  std::vector<PackJob> jobs;
  auto queue = [&](const float* src, int rows, int rows_pad, bf16* dst, int64_t ld, int64_t col_off, int part) {
    PackJob j;
    j.src = src; j.dst = dst; j.ld_dst = ld; j.col_off = col_off; j.rows = rows; j.rows_pad = rows_pad; j.part = part;
    jobs.push_back(j);
  };
  const bool f32 = (precision == SRG_PREC_FP32);

  // (1) bf16 parts (hi, mid, lo) of the message-side weights, stacked [W_h; W_z; W_r], and of W_p in block order kPartB.
  //     The training mode only needs the hi parts.
  const float* Wm32[3] = {p->W_h, p->W_z, p->W_r};
  bf16* Wm_part[3] = {h->Wm_hi, h->Wm_mid, h->Wm_lo};
  const int p_terms = f32 ? kSplitTerms : 1;
  for (int x = 0; x < 3; ++x)
    for (int part = 0; part < (f32 ? 3 : 1); ++part) queue(Wm32[x], D, D, Wm_part[part] + x * DD, D, 0, part);
  for (int b = 0; b < p_terms; ++b) queue(p->W_p, D, D, h->Wp6 + b * DD, D, 0, kPartB[b]);
  SRG_TRY(launch_pack_weight_multi(jobs.data(), static_cast<int>(jobs.size()), D, s));
  jobs.clear();

  // (2) P = [W_h; W_z; W_r] W_p.  Training mode: one bf16 x bf16 product with fp32 accumulation (the same operand
  //     rounding the unfused formulation has); fp32-parity mode: all six split terms, written as bf16 hi + mid + lo.
  {
    GemmProblem g = base_problem(h, 3 * D, D);
    for (int b = 0; b < p_terms; ++b) add_seg(g, Wm_part[kPartA[b]], 3 * D, D, 0, D);
    if (f32) g.corr_seg_begin = 1;
    g.b_mn = true;                                   // B[n = i, k] = W_p[k, i]: W_p as stored, K along rows
    g.b = mat(h->Wp6, static_cast<int64_t>(p_terms) * D, D, D, DT_BF16);
    g.epi = EPI_STORE_BF16;
    g.f32 = f32;                                     // instantiation with the 3-way split output
    g.flags = f32 ? FLAG_LO : 0;
    g.io[0] = mat(h->P_hi, 3 * D, D, D, DT_BF16);
    if (f32) {
      g.io[1] = mat(h->P_mid, 3 * D, D, D, DT_BF16);
      g.io[2] = mat(h->P_lo, 3 * D, D, D, DT_BF16);
    }
    SRG_TRY(run_gemm(g, h->dev, s));
  }

  // (3) forward operands: K blocks [P_x | U_x], one block per split term (part kPartB[b]) in fp32 mode
  const int64_t ld1 = static_cast<int64_t>(D) * split, ld2 = static_cast<int64_t>(2 * D) * split;
  const bf16* P_part[3] = {h->P_hi, h->P_mid, h->P_lo};
  auto pack_u = [&](const float* src, int rows, int rows_pad, bf16* dst, int64_t ld, int64_t row_off, int block_cols,
                    int col_in_block) {
    bf16* d = dst + row_off * ld;
    for (int b = 0; b < split; ++b)
      queue(src, rows, rows_pad, d, ld, static_cast<int64_t>(b) * block_cols + col_in_block, kPartB[b]);
  };
  auto pack_p = [&](int x, bf16* dst, int64_t row_off) -> int {  // x: 0 = h, 1 = z, 2 = r
    for (int b = 0; b < split; ++b)
      SRG_TRY(copy_block(dst, ld2, row_off, static_cast<int64_t>(b) * 2 * D, P_part[kPartB[b]] + x * DD, D, s));
    return SRG_OK;
  };
  SRG_TRY(pack_p(1, h->Wzr, 0));
  pack_u(p->U_z, D, D, h->Wzr, ld2, 0, 2 * D, D);
  SRG_TRY(pack_p(2, h->Wzr, D));
  pack_u(p->U_r, D, D, h->Wzr, ld2, D, 2 * D, D);
  SRG_TRY(pack_p(0, h->Wh, 0));
  pack_u(p->U_h, D, D, h->Wh, ld2, 0, 2 * D, D);
  pack_u(p->Wc_noun, h->L, h->Lpad, h->Wcn, ld1, 0, D, 0);
  pack_u(p->Wc_verb, h->V, h->Vpad, h->Wcv, ld1, 0, D, 0);
  if (!f32) {  // backward operands (MN-major B = stacks along K)
    queue(p->U_z, D, D, h->U_stack, D, 0, 0);
    queue(p->U_r, D, D, h->U_stack + DD, D, 0, 0);
    queue(p->U_h, D, D, h->Uh, D, 0, 0);
  }
  SRG_TRY(launch_pack_weight_multi(jobs.data(), static_cast<int>(jobs.size()), D, s));

  // (4) biases: b'_x(mode) = b_Wx + b_Ux + c W_x b_p, c = R for the noun graph (model.py:73-75: the projection bias is
  //     added for all R neighbours before the sum), c = 1 for the verb node (model.py:62-64)
  for (int x = 0; x < 3; ++x) SRG_TRY(launch_matvec(Wm32[x], p->b_p, D, D, h->wb + x * D, s));
  for (int mi = 0; mi < 2; ++mi) {
    const float c = (mi == 0) ? static_cast<float>(h->R) : 1.f;
    SRG_TRY(launch_pack_bias3(p->b_Wz, p->b_Uz, h->wb + D, c, D, D, h->bzr[mi], s));
    SRG_TRY(launch_pack_bias3(p->b_Wr, p->b_Ur, h->wb + 2 * D, c, D, D, h->bzr[mi] + D, s));
    SRG_TRY(launch_pack_bias3(p->b_Wh, p->b_Uh, h->wb, c, D, D, h->bh[mi], s));
  }
  SRG_TRY(launch_pack_bias(p->bc_noun, nullptr, h->L, h->Lpad, h->bcn, s));
  SRG_TRY(launch_pack_bias(p->bc_verb, nullptr, h->V, h->Vpad, h->bcv, s));
  h->packed_prec = precision;
  return SRG_OK;
}

size_t srg_workspace_stats_offset(srg_handle* h, int mode, int B, int precision, int save_for_backward,
                                  const void* workspace) {
  if (!h || B <= 0 || !workspace) return 0;
  // carve() only does pointer arithmetic; the offset depends on the alignment of the actual workspace address
  PathBufs pb = carve(h, mode, B, precision, save_for_backward, const_cast<void*>(workspace), mode == SRG_MODE_NOUN);
  return static_cast<size_t>(reinterpret_cast<const uint8_t*>(pb.stats) - static_cast<const uint8_t*>(workspace));
}

size_t srg_workspace_dlogits_offset(srg_handle* h, int mode, int B, const void* workspace) {
  if (!h || B <= 0 || !workspace) return 0;
  PathBufs pb = carve(h, mode, B, SRG_PREC_BF16, 1, const_cast<void*>(workspace), mode == SRG_MODE_NOUN);
  return static_cast<size_t>(reinterpret_cast<const uint8_t*>(pb.dlb) - static_cast<const uint8_t*>(workspace));
}

size_t srg_workspace_bytes(srg_handle* h, int mode, int B, int precision, int save_for_backward) {
  if (!h || B <= 0) return 0;
  // role-graph paths: the row-mapped layout of srg_nouns_* is the larger one (srg_ggnn_forward uses dense rows)
  return carve(h, mode, B, precision, save_for_backward, nullptr, mode == SRG_MODE_NOUN).bytes;
}

}  // extern "C"

namespace {
// predict_nouns minus the backbone on the B role graphs of `verb` (B = images x candidates): role graph b reads feature
// row b / feat_rep.  Shared by srg_nouns_forward (feat_rep = 1) and srg_situation_nouns (feat_rep = k).
int nouns_forward_body(srg_handle* h, PathBufs& pb, const float* feat, int feat_rep, const int64_t* verb, int B,
                       const float* role_emb, const float* verb_emb, const DropSpec& ds, float* logits, int64_t ldl,
                       int precision, int save_for_backward, cudaStream_t s) {
  // role counts -> compact row layout (device-resident: the predicted verbs never visit the host)
  SRG_TRY(launch_prep_rows(h->d_role_count, h->V, h->R, verb, B, h->compact, pb.rm, h->d_bad, s));
  SRG_TRY(launch_node_init_noun(feat, role_emb, verb_emb, verb, h->d_verb2roles, h->V, B, h->R, h->D, pb.rm, feat_rep,
                                pb.h32, pb.hb_hi[0], pb.hb_mid[0], pb.hb_lo[0], s));
  SRG_TRY(ggnn_steps(h, SRG_MODE_NOUN, pb, pb.h32, nullptr, B, precision, save_for_backward, s));
  return classifier_forward(h, SRG_MODE_NOUN, pb, pb.h32, ds, logits, ldl, precision, s);
}

// srg_situation_nouns' workspace: the role-graph buffers of B*k graphs (carve), then the noun logits [B*k*R, Lpad].
// Returns the bytes a workspace at ANY 16-byte aligned address needs: carve's size of the buffers alone (used + 1024
// bytes of slack for the 1024-byte alignment of the first buffer) plus the logits.  With ws != nullptr, *pb / *logits
// receive the layout in `ws`: carve starts at the alignment pad a <= 1023 and ends at ws + a + used (1024-aligned), where
// the logits begin; they end at a + used + logit_bytes < the returned size.
size_t situation_layout(const srg_handle* h, int B, int k, int prec, void* ws, PathBufs* pb, float** logits) {
  const int n = B * k;
  const size_t logit_bytes = static_cast<size_t>(n) * h->R * h->Lpad * sizeof(float);
  if (ws != nullptr) {
    const PathBufs p = carve(h, SRG_MODE_NOUN, n, prec, 0, ws, true);   // p.bytes = a + used + 1024
    if (pb) *pb = p;
    if (logits) *logits = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + p.bytes - 1024);
  }
  return carve(h, SRG_MODE_NOUN, n, prec, 0, nullptr, true).bytes + logit_bytes;
}

// srg_situation_nbest's workspace: situation_layout(B, kv), then the per-slot top-n lists [B*kv*R, n] as int64 label
// ids and fp32 log-probs.  The logits end 1024-aligned (their rows are Lpad = 256 m floats), so the lists are aligned
// too, and they end within situation_layout's 1024 bytes of alignment slack plus their own size.
size_t nbest_layout(const srg_handle* h, int B, int kv, int nb, int prec, void* ws, PathBufs* pb, float** logits,
                    int64_t** slot_idx, float** slot_logp) {
  const size_t slots = static_cast<size_t>(B) * kv * h->R * nb;
  if (ws != nullptr) {
    float* nl = nullptr;
    situation_layout(h, B, kv, prec, ws, pb, &nl);
    *logits = nl;
    *slot_idx = reinterpret_cast<int64_t*>(nl + static_cast<size_t>(B) * kv * h->R * h->Lpad);
    *slot_logp = reinterpret_cast<float*>(*slot_idx + slots);
  }
  return situation_layout(h, B, kv, prec, nullptr, nullptr, nullptr) + slots * (sizeof(int64_t) + sizeof(float));
}
}  // namespace

extern "C" {

int srg_nouns_forward(srg_handle* h, const float* feat, const int64_t* verb, int B, const float* role_emb,
                      const float* verb_emb, const uint8_t* keep, float drop_p, const int64_t* drop_seed,
                      int64_t drop_stream, float* logits, int64_t ldl, int precision, int save_for_backward,
                      void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_nouns_forward: null handle");
  DeviceGuard guard_(h->device);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_NOUN, B, precision, save_for_backward, workspace, workspace_bytes, &pb, true));
  SRG_CHECK(h->tables_set, "srg_nouns_forward: call srg_set_tables first");
  SRG_CHECK(h->packed_prec == precision, "srg_nouns_forward: weights are not packed for precision %d", precision);
  SRG_CHECK(feat && verb && role_emb && verb_emb && logits, "srg_nouns_forward: null argument");
  DropSpec ds;
  SRG_TRY(make_drop(keep, drop_p, drop_seed, drop_stream, &ds));
  return nouns_forward_body(h, pb, feat, 1, verb, B, role_emb, verb_emb, ds, logits, ldl, precision, save_for_backward,
                            static_cast<cudaStream_t>(stream));
}

int srg_topk_logsoftmax(const float* logits, int64_t ldl, int rows, int n, int k, int64_t* idx, float* logp,
                        void* stream) {
  SRG_CHECK(rows >= 0, "srg_topk_logsoftmax: negative row count %d", rows);
  SRG_CHECK(rows == 0 || (logits && idx && logp), "srg_topk_logsoftmax: null argument");
  return launch_row_topk_logsoftmax(logits, ldl, rows, n, k, idx, logp, static_cast<cudaStream_t>(stream));
}

size_t srg_situation_workspace_bytes(srg_handle* h, int B, int k, int precision) {
  if (!h || B <= 0 || k < 1 || k > 16) return 0;
  return situation_layout(h, B, k, precision, nullptr, nullptr, nullptr);
}

int srg_situation_nouns(srg_handle* h, const float* feat, const int64_t* verbs, int B, int k, const float* role_emb,
                        const float* verb_emb, const float* verb_logp, int64_t* labels, float* label_logp,
                        float* score, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_situation_nouns: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(k >= 1 && k <= 16 && k <= h->V, "srg_situation_nouns: k=%d must be in [1, min(16, n_verbs=%d)]", k, h->V);
  SRG_CHECK(B > 0 && static_cast<int64_t>(B) * k * h->R <= (1 << 30), "srg_situation_nouns: bad batch %d", B);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_NOUN, B * k, precision, 0, workspace, workspace_bytes, &pb, true));
  float* nl = nullptr;
  const size_t need = situation_layout(h, B, k, precision, workspace, &pb, &nl);
  if (need > workspace_bytes)
    return set_error(SRG_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  SRG_CHECK(h->tables_set, "srg_situation_nouns: call srg_set_tables first");
  SRG_CHECK(h->packed_prec == precision, "srg_situation_nouns: weights are not packed for precision %d", precision);
  SRG_CHECK(feat && verbs && role_emb && verb_emb && labels && label_logp && score, "srg_situation_nouns: null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int n = B * k;
  SRG_TRY(nouns_forward_body(h, pb, feat, k, verbs, n, role_emb, verb_emb, DropSpec(), nl, h->Lpad, precision, 0, s));
  SRG_TRY(launch_row_topk_logsoftmax(nl, h->Lpad, n * h->R, h->L, 1, labels, label_logp, s));
  return launch_situation_finish(verbs, h->d_role_count, h->V, h->R, n, verb_logp, labels, label_logp, score, s);
}

size_t srg_situation_nbest_workspace_bytes(srg_handle* h, int B, int kv, int n, int precision) {
  if (!h || B <= 0 || kv < 1 || kv > 16 || n < 1 || n > 16) return 0;
  return nbest_layout(h, B, kv, n, precision, nullptr, nullptr, nullptr, nullptr, nullptr);
}

int srg_situation_nbest(srg_handle* h, const float* feat, const int64_t* verbs, int B, int kv, const float* role_emb,
                        const float* verb_emb, const float* verb_logp, const float* verb_bound, int n,
                        int64_t* out_verbs, float* out_verb_logp, int64_t* labels, float* label_logp, float* score,
                        uint8_t* exact, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_situation_nbest: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(kv >= 1 && kv <= 16 && kv <= h->V, "srg_situation_nbest: kv=%d must be in [1, min(16, n_verbs=%d)]", kv,
            h->V);
  SRG_CHECK(n >= 1 && n <= 16 && n <= h->L, "srg_situation_nbest: n=%d must be in [1, min(16, n_labels=%d)]", n, h->L);
  SRG_CHECK(B > 0 && static_cast<int64_t>(B) * kv * h->R <= (1 << 30), "srg_situation_nbest: bad batch %d", B);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_NOUN, B * kv, precision, 0, workspace, workspace_bytes, &pb, true));
  float* nl = nullptr;
  int64_t* slot_idx = nullptr;
  float* slot_logp = nullptr;
  const size_t need = nbest_layout(h, B, kv, n, precision, workspace, &pb, &nl, &slot_idx, &slot_logp);
  if (need > workspace_bytes)
    return set_error(SRG_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  SRG_CHECK(h->tables_set, "srg_situation_nbest: call srg_set_tables first");
  SRG_CHECK(h->packed_prec == precision, "srg_situation_nbest: weights are not packed for precision %d", precision);
  SRG_CHECK(feat && verbs && role_emb && verb_emb && out_verbs && labels && label_logp && score,
            "srg_situation_nbest: null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int nc = B * kv;
  SRG_TRY(nouns_forward_body(h, pb, feat, kv, verbs, nc, role_emb, verb_emb, DropSpec(), nl, h->Lpad, precision, 0, s));
  SRG_TRY(launch_row_topk_logsoftmax(nl, h->Lpad, nc * h->R, h->L, n, slot_idx, slot_logp, s));
  return launch_situation_nbest(verbs, h->d_role_count, h->V, h->R, B, kv, n, verb_logp, verb_bound, slot_idx, slot_logp,
                                out_verbs, out_verb_logp, labels, label_logp, score, exact, s);
}

int srg_verb_forward(srg_handle* h, const float* feat, int B, const uint8_t* keep, float drop_p,
                     const int64_t* drop_seed, int64_t drop_stream, float* logits, int64_t ldl, int precision,
                     int save_for_backward, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_verb_forward: null handle");
  DeviceGuard guard_(h->device);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_VERB, B, precision, save_for_backward, workspace, workspace_bytes, &pb, false));
  SRG_CHECK(h->packed_prec == precision, "srg_verb_forward: weights are not packed for precision %d", precision);
  SRG_CHECK(feat && logits, "srg_verb_forward: null argument");
  DropSpec ds;
  SRG_TRY(make_drop(keep, drop_p, drop_seed, drop_stream, &ds));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SRG_TRY(launch_node_init_verb(feat, B, h->D, pb.h32, pb.hb_hi[0], pb.hb_mid[0], pb.hb_lo[0], s));
  SRG_TRY(ggnn_steps(h, SRG_MODE_VERB, pb, pb.h32, nullptr, B, precision, save_for_backward, s));
  return classifier_forward(h, SRG_MODE_VERB, pb, pb.h32, ds, logits, ldl, precision, s);
}

int srg_ggnn_forward(srg_handle* h, int mode, float* hidden, const float* mask, int B, int precision,
                     int save_for_backward, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_ggnn_forward: null handle");
  DeviceGuard guard_(h->device);
  PathBufs pb;
  SRG_CHECK(mode == SRG_MODE_NOUN || mode == SRG_MODE_VERB, "bad mode %d", mode);
  SRG_TRY(check_ws(h, mode, B, precision, save_for_backward, workspace, workspace_bytes, &pb, false));
  SRG_CHECK(h->packed_prec == precision, "srg_ggnn_forward: weights are not packed for precision %d", precision);
  SRG_CHECK(hidden != nullptr, "null hidden state");
  SRG_CHECK(mode == SRG_MODE_VERB || mask != nullptr, "noun mode needs a mask");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SRG_TRY(launch_split_cast(hidden, static_cast<int64_t>(pb.M) * h->D, pb.hb_hi[0], pb.hb_mid[0], pb.hb_lo[0], s));
  return ggnn_steps(h, mode, pb, hidden, mask, B, precision, save_for_backward, s);
}

int srg_dropout_mask(const int64_t* drop_seed, int64_t drop_stream, float drop_p, int64_t rows, int D, uint8_t* keep,
                     void* stream) {
  SRG_CHECK(drop_seed != nullptr && keep != nullptr, "srg_dropout_mask: null argument");
  SRG_CHECK(rows >= 0 && D > 0 && D % 8 == 0, "srg_dropout_mask: bad shape");
  DropSpec ds;
  SRG_TRY(make_drop(nullptr, drop_p, drop_seed, drop_stream, &ds));
  if (ds.seed == nullptr) {   // p == 0: everything is kept
    SRG_CUDA(cudaMemsetAsync(keep, 1, static_cast<size_t>(rows) * D, static_cast<cudaStream_t>(stream)));
    return SRG_OK;
  }
  return launch_dropout_mask(ds, rows, D, keep, static_cast<cudaStream_t>(stream));
}

int srg_count_targets(srg_handle* h, const int64_t* gt_nouns, int B, float* counts, void* stream) {
  SRG_CHECK(h != nullptr, "srg_count_targets: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h && gt_nouns && counts, "srg_count_targets: null argument");
  return launch_count_targets(gt_nouns, B, h->R, h->L, counts, static_cast<cudaStream_t>(stream));
}

int srg_count_targets_weighted(srg_handle* h, const int64_t* gt_nouns, int B, const float* class_weight, float* counts,
                               void* stream) {
  SRG_CHECK(h != nullptr, "srg_count_targets_weighted: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(gt_nouns && counts, "srg_count_targets_weighted: null argument");
  SRG_CHECK(B >= 0, "srg_count_targets_weighted: B = %d", B);
  return launch_weighted_count(gt_nouns, static_cast<int64_t>(B) * 3 * h->R, h->R, 3, h->L, class_weight, h->L,
                               counts, static_cast<cudaStream_t>(stream));
}

int srg_verb_weight_total(srg_handle* h, const int64_t* gt_verb, int B, const float* class_weight, float* total,
                          void* stream) {
  SRG_CHECK(h != nullptr, "srg_verb_weight_total: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(gt_verb && total, "srg_verb_weight_total: null argument");
  SRG_CHECK(B >= 0, "srg_verb_weight_total: B = %d", B);
  return launch_weighted_count(gt_verb, B, 1, 1, -100, class_weight, h->V, total, static_cast<cudaStream_t>(stream));
}

// srg_loss_opts -> CeOpts, refusing what the kernels cannot honour.  NULL = the default options.  fwd: the call writes
// a loss (and, for "none", needs per_target_loss); grad: it writes a gradient (for "none", needs grad_per_target).
static int loss_opts(const char* fn, const srg_loss_opts* o, bool fwd, bool grad, CeOpts* out) {
  *out = CeOpts{};
  if (o == nullptr) return SRG_OK;
  SRG_CHECK(o->label_smoothing >= 0.f && o->label_smoothing <= 1.f, "%s: label_smoothing %g outside [0, 1]", fn,
            static_cast<double>(o->label_smoothing));
  SRG_CHECK(o->reduction == SRG_REDUCTION_MEAN || o->reduction == SRG_REDUCTION_SUM ||
            o->reduction == SRG_REDUCTION_NONE, "%s: unknown reduction %d", fn, o->reduction);
  if (o->reduction == SRG_REDUCTION_NONE) {
    SRG_CHECK(!fwd || o->per_target_loss != nullptr, "%s: reduction 'none' needs per_target_loss", fn);
    SRG_CHECK(!grad || o->grad_per_target != nullptr, "%s: reduction 'none' needs grad_per_target", fn);
  }
  out->cw = o->class_weight;
  out->eps = o->label_smoothing;
  out->reduction = o->reduction;
  out->per_target = fwd ? o->per_target_loss : nullptr;
  out->gpt = grad ? o->grad_per_target : nullptr;
  return SRG_OK;
}

static bool mean_reduction(const srg_loss_opts* o) { return o == nullptr || o->reduction == SRG_REDUCTION_MEAN; }

int srg_nouns_loss_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                      const float* counts, float* loss, float* dlogits, float grad_scale, const float* stats,
                      const srg_loss_opts* opts, void* stream) {
  CeOpts o;
  SRG_TRY(loss_opts("srg_nouns_loss", opts, true, dlogits != nullptr, &o));
  SRG_CHECK(h != nullptr, "srg_nouns_loss: null handle");
  DeviceGuard guard_(h->device);
  const bool none = !mean_reduction(opts) && opts->reduction == SRG_REDUCTION_NONE;
  SRG_CHECK(logits && gt_nouns && (counts || !mean_reduction(opts)) && (loss || none), "srg_nouns_loss: null argument");
  SRG_CHECK(ldl >= h->L, "srg_nouns_loss: ldl %lld < n_labels %d", (long long)ldl, h->L);
  return launch_nouns_ce(logits, ldl, h->L, gt_nouns, B, h->R, counts, loss, dlogits, grad_scale, nullptr, stats,
                         h->Lpad / ((h->cg == 2) ? 256 : 128), nullptr, 0, 0, &o, static_cast<cudaStream_t>(stream));
}

int srg_nouns_loss(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                   const float* counts, float* loss, float* dlogits, float grad_scale, const float* stats,
                   void* stream) {
  return srg_nouns_loss_ex(h, logits, ldl, gt_nouns, B, counts, loss, dlogits, grad_scale, stats, nullptr, stream);
}

int srg_nouns_loss_backward_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                               const float* counts, const float* grad_out, float grad_scale, float* dlogits,
                               void* dlogits_bf16, int accumulate, const float* stats, const srg_loss_opts* opts,
                               void* stream) {
  CeOpts o;
  SRG_TRY(loss_opts("srg_nouns_loss_backward", opts, false, true, &o));
  SRG_CHECK(h != nullptr, "srg_nouns_loss_backward: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(logits && gt_nouns && (counts || !mean_reduction(opts)) && (dlogits || dlogits_bf16),
            "srg_nouns_loss_backward: null argument");
  SRG_CHECK(ldl >= h->L, "srg_nouns_loss_backward: ldl %lld < n_labels %d", (long long)ldl, h->L);
  return launch_nouns_ce(logits, ldl, h->L, gt_nouns, B, h->R, counts, nullptr, dlogits, grad_scale, grad_out, stats,
                         h->Lpad / ((h->cg == 2) ? 256 : 128), static_cast<bf16*>(dlogits_bf16), h->Lpad, accumulate,
                         &o, static_cast<cudaStream_t>(stream));
}

int srg_nouns_loss_backward(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_nouns, int B,
                            const float* counts, const float* grad_out, float grad_scale, float* dlogits,
                            void* dlogits_bf16, int accumulate, const float* stats, void* stream) {
  return srg_nouns_loss_backward_ex(h, logits, ldl, gt_nouns, B, counts, grad_out, grad_scale, dlogits, dlogits_bf16,
                                    accumulate, stats, nullptr, stream);
}

int srg_verb_loss_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B, float inv_batch,
                     const float* batch_total, float* loss, float* dlogits, float grad_scale, const float* stats,
                     const srg_loss_opts* opts, void* stream) {
  CeOpts o;
  SRG_TRY(loss_opts("srg_verb_loss", opts, true, dlogits != nullptr, &o));
  SRG_CHECK(h != nullptr, "srg_verb_loss: null handle");
  DeviceGuard guard_(h->device);
  const bool none = !mean_reduction(opts) && opts->reduction == SRG_REDUCTION_NONE;
  SRG_CHECK(logits && gt_verb && (loss || none), "srg_verb_loss: null argument");
  SRG_CHECK(ldl >= h->V, "srg_verb_loss: ldl %lld < n_verbs %d", (long long)ldl, h->V);
  return launch_verb_ce(logits, ldl, h->V, gt_verb, B, inv_batch, loss, dlogits, grad_scale, nullptr, stats,
                        h->Vpad / ((h->cg == 2) ? 256 : 128), batch_total, nullptr, 0, 0, &o,
                        static_cast<cudaStream_t>(stream));
}

int srg_verb_loss(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B, float inv_batch,
                  const float* batch_total, float* loss, float* dlogits, float grad_scale, const float* stats,
                  void* stream) {
  return srg_verb_loss_ex(h, logits, ldl, gt_verb, B, inv_batch, batch_total, loss, dlogits, grad_scale, stats,
                          nullptr, stream);
}

int srg_verb_loss_backward_ex(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B,
                              float inv_batch, const float* batch_total, const float* grad_out, float grad_scale,
                              float* dlogits, void* dlogits_bf16, int accumulate, const float* stats,
                              const srg_loss_opts* opts, void* stream) {
  CeOpts o;
  SRG_TRY(loss_opts("srg_verb_loss_backward", opts, false, true, &o));
  SRG_CHECK(h != nullptr, "srg_verb_loss_backward: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(logits && gt_verb && (dlogits || dlogits_bf16), "srg_verb_loss_backward: null argument");
  SRG_CHECK(ldl >= h->V, "srg_verb_loss_backward: ldl %lld < n_verbs %d", (long long)ldl, h->V);
  return launch_verb_ce(logits, ldl, h->V, gt_verb, B, inv_batch, nullptr, dlogits, grad_scale, grad_out, stats,
                        h->Vpad / ((h->cg == 2) ? 256 : 128), batch_total, static_cast<bf16*>(dlogits_bf16), h->Vpad,
                        accumulate, &o, static_cast<cudaStream_t>(stream));
}

int srg_verb_loss_backward(srg_handle* h, const float* logits, int64_t ldl, const int64_t* gt_verb, int B,
                           float inv_batch, const float* batch_total, const float* grad_out, float grad_scale,
                           float* dlogits, void* dlogits_bf16, int accumulate, const float* stats, void* stream) {
  return srg_verb_loss_backward_ex(h, logits, ldl, gt_verb, B, inv_batch, batch_total, grad_out, grad_scale, dlogits,
                                   dlogits_bf16, accumulate, stats, nullptr, stream);
}

int srg_clip_adamax(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                    float beta2, float eps, float max_norm, float* scratch, void* stream) {
  SRG_CHECK(params && grads && exp_avg && exp_inf && scratch, "srg_clip_adamax: null argument");
  return launch_clip_adamax(params, grads, exp_avg, exp_inf, n, lr, beta1, beta2, eps, max_norm, scratch, scratch + 1,
                            static_cast<cudaStream_t>(stream));
}

int srg_sumsq(const float* x, int64_t n, float* out, void* stream) {
  SRG_CHECK(x && out, "srg_sumsq: null argument");
  return launch_sumsq(x, n, out, static_cast<cudaStream_t>(stream));
}

int srg_adamax_step(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                    float beta2, float eps, float max_norm, const float* norm_sq, float* step, void* stream) {
  SRG_CHECK(params && grads && exp_avg && exp_inf && norm_sq && step, "srg_adamax_step: null argument");
  return launch_adamax_step(params, grads, exp_avg, exp_inf, n, lr, beta1, beta2, eps, max_norm, norm_sq, step,
                            static_cast<cudaStream_t>(stream));
}

int srg_set_deferred_chain(srg_handle* h, int on, void* stream) {
  SRG_CHECK(h != nullptr, "srg_set_deferred_chain: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h != nullptr, "null handle");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t D = h->D;
  if (on && h->acc_GP == nullptr) {
    SRG_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->acc_GP), 3 * D * D * sizeof(float)));
    SRG_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->acc_GPb), 3 * D * D * sizeof(bf16)));
    SRG_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->acc_s), 3 * D * sizeof(float)));
  }
  if (on) {
    SRG_CUDA(cudaMemsetAsync(h->acc_GP, 0, 3 * D * D * sizeof(float), s));
    SRG_CUDA(cudaMemsetAsync(h->acc_s, 0, 3 * D * sizeof(float), s));
  }
  h->defer_chain = (on != 0);
  return SRG_OK;
}

int srg_chain_finalize(srg_handle* h, const srg_grads* g, void* stream) {
  SRG_CHECK(h != nullptr, "srg_chain_finalize: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(h != nullptr && g != nullptr, "srg_chain_finalize: null argument");
  SRG_CHECK(h->defer_chain && h->acc_GP != nullptr, "srg_chain_finalize: call srg_set_deferred_chain(h, 1) first");
  SRG_CHECK(h->packed_prec == SRG_PREC_BF16, "srg_chain_finalize needs bf16-packed weights");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t D = h->D;
  SRG_TRY(chain_rule(h, h->acc_GP, h->acc_GPb, h->acc_s, g, /*shared_dst=*/false, s));
  SRG_CUDA(cudaMemsetAsync(h->acc_GP, 0, 3 * D * D * sizeof(float), s));
  SRG_CUDA(cudaMemsetAsync(h->acc_s, 0, 3 * D * sizeof(float), s));
  return SRG_OK;
}

int srg_nouns_backward_feat(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace,
                            const float* feat, const int64_t* verb, int B, const float* role_emb, const float* verb_emb,
                            const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                            const srg_grads* g, float* dfeat, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_nouns_backward: null handle");
  DeviceGuard guard_(h->device);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_NOUN, B, SRG_PREC_BF16, 1, workspace, workspace_bytes, &pb, true));
  SRG_CHECK(h->packed_prec == SRG_PREC_BF16, "backward needs bf16-packed weights");
  SRG_CHECK((dlogits || dlogits_in_workspace) && feat && verb && role_emb && verb_emb && g,
            "srg_nouns_backward: null argument");
  SRG_CHECK(dlogits == nullptr || ldl >= h->L, "srg_nouns_backward: ldl %lld < n_labels %d", (long long)ldl, h->L);
  DropSpec ds;
  SRG_TRY(make_drop(keep, drop_p, drop_seed, drop_stream, &ds));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SRG_TRY(path_backward(h, SRG_MODE_NOUN, pb, dlogits, ldl, dlogits_in_workspace, B, ds, g, s));
  const bool emb = (g->role_emb != nullptr && g->verb_emb != nullptr);
  return launch_node_init_bwd(pb.dh, pb.hb_hi[0], feat, role_emb, verb_emb, verb, h->d_verb2roles, h->V, h->n_roles, B,
                              h->R, h->D, pb.rm, emb ? g->role_emb : nullptr, emb ? g->verb_emb : nullptr, dfeat, s);
}

int srg_nouns_backward(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, const float* feat,
                       const int64_t* verb, int B, const float* role_emb, const float* verb_emb, const uint8_t* keep,
                       float drop_p, const int64_t* drop_seed, int64_t drop_stream, const srg_grads* g, void* workspace,
                       size_t workspace_bytes, void* stream) {
  return srg_nouns_backward_feat(h, dlogits, ldl, dlogits_in_workspace, feat, verb, B, role_emb, verb_emb, keep, drop_p,
                                 drop_seed, drop_stream, g, nullptr, workspace, workspace_bytes, stream);
}

int srg_verb_backward_feat(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, int B,
                           const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                           const srg_grads* g, float* dfeat, void* workspace, size_t workspace_bytes, void* stream) {
  SRG_CHECK(h != nullptr, "srg_verb_backward: null handle");
  DeviceGuard guard_(h->device);
  PathBufs pb;
  SRG_TRY(check_ws(h, SRG_MODE_VERB, B, SRG_PREC_BF16, 1, workspace, workspace_bytes, &pb, false));
  SRG_CHECK(h->packed_prec == SRG_PREC_BF16, "backward needs bf16-packed weights");
  SRG_CHECK((dlogits || dlogits_in_workspace) && g, "srg_verb_backward: null argument");
  SRG_CHECK(dlogits == nullptr || ldl >= h->V, "srg_verb_backward: ldl %lld < n_verbs %d", (long long)ldl, h->V);
  DropSpec ds;
  SRG_TRY(make_drop(keep, drop_p, drop_seed, drop_stream, &ds));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SRG_TRY(path_backward(h, SRG_MODE_VERB, pb, dlogits, ldl, dlogits_in_workspace, B, ds, g, s));
  if (dfeat != nullptr) SRG_TRY(launch_node_init_verb_bwd(pb.dh, pb.hb_hi[0], B, h->D, dfeat, s));
  return SRG_OK;
}

int srg_verb_backward(srg_handle* h, const float* dlogits, int64_t ldl, int dlogits_in_workspace, int B,
                      const uint8_t* keep, float drop_p, const int64_t* drop_seed, int64_t drop_stream,
                      const srg_grads* g, void* workspace, size_t workspace_bytes, void* stream) {
  return srg_verb_backward_feat(h, dlogits, ldl, dlogits_in_workspace, B, keep, drop_p, drop_seed, drop_stream, g,
                                nullptr, workspace, workspace_bytes, stream);
}

int srg_ggnn_backward(srg_handle* h, int mode, const float* dhidden_out, const float* mask, float* dmask,
                      float* dhidden_in, int B, const srg_grads* g, void* workspace, size_t workspace_bytes,
                      void* stream) {
  SRG_CHECK(h != nullptr, "srg_ggnn_backward: null handle");
  DeviceGuard guard_(h->device);
  SRG_CHECK(mode == SRG_MODE_NOUN || mode == SRG_MODE_VERB, "bad mode %d", mode);
  PathBufs pb;
  SRG_TRY(check_ws(h, mode, B, SRG_PREC_BF16, 1, workspace, workspace_bytes, &pb, false));
  SRG_CHECK(h->packed_prec == SRG_PREC_BF16, "backward needs bf16-packed weights");
  SRG_CHECK(dhidden_out != nullptr && g != nullptr, "srg_ggnn_backward: null argument");
  SRG_CHECK(mode == SRG_MODE_VERB || mask != nullptr, "noun mode needs a mask");
  SRG_CHECK(mode == SRG_MODE_NOUN || dmask == nullptr, "the verb node has no mask: dmask must be NULL");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float *G_P = nullptr, *s_all = nullptr;
  SRG_TRY(chain_acc(h, pb, &G_P, &s_all, s));
  if (dmask != nullptr)
    SRG_CUDA(cudaMemsetAsync(dmask, 0, sizeof(float) * static_cast<size_t>(B) * h->R * h->R, s));
  SRG_TRY(ggnn_backward(h, mode, pb, B, dhidden_out, (mode == SRG_MODE_NOUN) ? mask : nullptr, dmask, G_P, s_all, g, s));
  if (dhidden_in != nullptr)
    SRG_CUDA(cudaMemcpyAsync(dhidden_in, pb.dh, sizeof(float) * static_cast<size_t>(pb.M) * h->D,
                             cudaMemcpyDeviceToDevice, s));
  return SRG_OK;
}

#ifdef SRG_EPI_TIMING
/* debug builds only (tools/epi_timing.py): copy out and optionally clear the epilogue clock counters [8 kinds][8] */
int srg_debug_epi_timing(unsigned long long* out, int reset) {
  SRG_CUDA(cudaDeviceSynchronize());
  SRG_CHECK(srg::g_epi_t_dev != nullptr, "no GEMM has been launched yet");
  SRG_CUDA(cudaMemcpy(out, srg::g_epi_t_dev, sizeof(unsigned long long) * 64, cudaMemcpyDeviceToHost));
  if (reset) SRG_CUDA(cudaMemset(srg::g_epi_t_dev, 0, sizeof(unsigned long long) * 64));
  return SRG_OK;
}
#endif

}  // extern "C"
