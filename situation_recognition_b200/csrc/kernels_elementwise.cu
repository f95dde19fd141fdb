// HBM-bound kernels of the GGNN role-graph stage (see elementwise.cuh).
#include "elementwise.cuh"
#include "host.cuh"

namespace srg {

namespace {

constexpr int kMaxR = 8;
constexpr int kThreads = 256;

inline int grid_for(int64_t work, int threads = kThreads, int max_blocks = 148 * 16) {
  int64_t b = (work + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return static_cast<int>(b);
}

__device__ __forceinline__ uint2 pack4_bf16(float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&lo);
  r.y = *reinterpret_cast<uint32_t*>(&hi);
  return r;
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// bf16 operand parts of 4 values: hi = bf16(v); when `parts` carries the residual pointers also
// mid = bf16(v - hi) and lo = bf16(v - hi - mid)  (fp32-parity mode: x = hi + mid + lo to 24 bits)
struct Parts {
  bf16* mid;
  bf16* lo;
};
__device__ __forceinline__ void store4_split(bf16* hi, Parts parts, int64_t idx, float4 v) {
  *reinterpret_cast<uint2*>(hi + idx) = pack4_bf16(v.x, v.y, v.z, v.w);
  if (parts.mid != nullptr) {
    const float4 r1 = make_float4(v.x - bf16_round(v.x), v.y - bf16_round(v.y), v.z - bf16_round(v.z),
                                  v.w - bf16_round(v.w));
    *reinterpret_cast<uint2*>(parts.mid + idx) = pack4_bf16(r1.x, r1.y, r1.z, r1.w);
    *reinterpret_cast<uint2*>(parts.lo + idx) = pack4_bf16(r1.x - bf16_round(r1.x), r1.y - bf16_round(r1.y),
                                                           r1.z - bf16_round(r1.z), r1.w - bf16_round(r1.w));
  }
}

// ------------------------------------------------------------------------------------------------ K1
__global__ void k_gather_mask(const int32_t* __restrict__ verb2roles, const int32_t* __restrict__ role_count,
                              int n_verbs, int R, const int64_t* __restrict__ verb, int B,
                              int64_t* __restrict__ role_idx, float* __restrict__ mask, int* __restrict__ bad) {
  const int64_t total = static_cast<int64_t>(B) * R * R;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(t / (R * R));
    const int ij = static_cast<int>(t % (R * R));
    const int i = ij / R, j = ij % R;
    int64_t v = verb[b];
    const bool ok = (v >= 0 && v < n_verbs);
    if (!ok) {
      if (bad != nullptr) *bad = 1;
      v = 0;
    }
    const int n = role_count[v];
    if (mask != nullptr) {
      const bool on = (i < n && j < n && i != j) || (i >= n && i == j);
      mask[t] = on ? 1.0f : 0.0f;
    }
    if (role_idx != nullptr && i == 0) role_idx[static_cast<int64_t>(b) * R + j] = verb2roles[v * R + j];
  }
}

// ------------------------------------------------------------------------------------------------ node init
__global__ void k_node_init_verb(const float* __restrict__ feat, int64_t n4, float* __restrict__ h32,
                                 bf16* __restrict__ hb_hi, Parts hb_lo) {
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n4;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 f = *reinterpret_cast<const float4*>(feat + t * 4);
    f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); f.z = fmaxf(f.z, 0.f); f.w = fmaxf(f.w, 0.f);
    *reinterpret_cast<float4*>(h32 + t * 4) = f;
    store4_split(hb_hi, hb_lo, t * 4, f);
  }
}

__global__ void k_split_cast(const float* __restrict__ x, int64_t n4, bf16* __restrict__ hi, Parts lo) {
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n4;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 f = *reinterpret_cast<const float4*>(x + t * 4);
    store4_split(hi, lo, t * 4, f);
  }
}

// ------------------------------------------------------------------------------------------------ aggregation
__global__ void k_aggregate(const float* __restrict__ h32, const float* __restrict__ mask, int B, int R, int D,
                            bf16* __restrict__ a_hi, Parts a_lo) {
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(B) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(t / D4);
    const int d = static_cast<int>(t % D4) * 4;
    float4 h[kMaxR];
#pragma unroll
    for (int j = 0; j < kMaxR; ++j)
      if (j < R) h[j] = *reinterpret_cast<const float4*>(h32 + (static_cast<int64_t>(b) * R + j) * D + d);
    const float* mb = mask + static_cast<int64_t>(b) * R * R;
#pragma unroll
    for (int i = 0; i < kMaxR; ++i) {
      if (i < R) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < kMaxR; ++j) {
          if (j < R) {
            const float m = __ldg(mb + i * R + j);
            a.x = fmaf(m, h[j].x, a.x); a.y = fmaf(m, h[j].y, a.y);
            a.z = fmaf(m, h[j].z, a.z); a.w = fmaf(m, h[j].w, a.w);
          }
        }
        store4_split(a_hi, a_lo, (static_cast<int64_t>(b) * R + i) * D + d, a);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ compact role-node rows
// Row layout of a role-graph path (RowMap, elementwise.cuh).  Image b owns rows [off[b], off[b] + L_b), L_b = its number
// of real roles n_b (compact) or R (one row per slot); ONE shared pad row follows at meta[1] = sum L_b.  Pad nodes start
// at 0 and only see themselves (model.py:95-97, imsitu_encoder.py:223-225), so every pad node of a batch follows the same
// trajectory, which only depends on the weights: it is computed once.  Rows [meta[1], meta[2]) -- the shared pad row and
// the rest of its 256-row GEMM tile -- are "self-loop rows": zero initial state, aggregate = own state.
__global__ void __launch_bounds__(1024)
k_prep_rows(const int32_t* __restrict__ role_count, int n_verbs, int R, const int64_t* __restrict__ verb, int B,
            int compact, int* __restrict__ cnt, int* __restrict__ off, int* __restrict__ meta, int* __restrict__ bad) {
  __shared__ int s_part[1024];
  const int tid = threadIdx.x;
  const int per = (B + 1023) / 1024;
  const int b0 = min(B, tid * per), b1 = min(B, b0 + per);
  int sum = 0;
  for (int b = b0; b < b1; ++b) {
    int64_t v = verb[b];
    if (v < 0 || v >= n_verbs) {
      if (bad != nullptr) *bad = 1;
      v = 0;
    }
    const int n = role_count[v];
    cnt[b] = n;
    sum += compact ? n : R;
  }
  s_part[tid] = sum;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {   // inclusive scan of the per-thread partial sums
    const int v = (tid >= o) ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int run = s_part[tid] - sum;
  for (int b = b0; b < b1; ++b) {
    off[b] = run;
    run += compact ? cnt[b] : R;
  }
  if (tid == 1023) {
    const int n_real = s_part[1023];
    off[B] = n_real;
    meta[0] = n_real + 1;                        // rows, shared pad row included (the GEMMs' M)
    meta[1] = n_real;                            // index of the shared pad row
    meta[2] = (n_real + 1 + 255) / 256 * 256;    // rows the GEMM tiles touch (all of them hold finite values)
    meta[3] = 0;
  }
}

constexpr int kSelfRows = 256;   // upper bound of meta[2] - meta[1]

__device__ __forceinline__ void store8_split(bf16* hi, Parts parts, int64_t idx, float4 a, float4 b) {
  store4_split(hi, parts, idx, a);
  store4_split(hi, parts, idx + 4, b);
}

__global__ void k_node_init_noun(const float* __restrict__ feat, const float* __restrict__ role_emb,
                                 const float* __restrict__ verb_emb, const int64_t* __restrict__ verb,
                                 const int32_t* __restrict__ verb2roles, int n_verbs, int B, int R, int D, RowMap rm,
                                 int feat_rep, float* __restrict__ h32, bf16* __restrict__ hb_hi, Parts hb_lo) {
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(B + kSelfRows) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int u = static_cast<int>(t / D4);
    const int d = static_cast<int>(t % D4) * 4;
    if (u >= B) {   // self-loop rows start at exactly 0 (nn.Embedding padding_idx row)
      const int row = rm.meta[1] + (u - B);
      if (row < rm.meta[2]) {
        const int64_t off = static_cast<int64_t>(row) * D + d;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(h32 + off) = z;
        store4_split(hb_hi, hb_lo, off, z);
      }
      continue;
    }
    const int b = u;
    int64_t v = verb[b];
    if (v < 0 || v >= n_verbs) v = 0;
    const float4 f = *reinterpret_cast<const float4*>(feat + static_cast<int64_t>(b / feat_rep) * D + d);
    const float4 ve = *reinterpret_cast<const float4*>(verb_emb + v * D + d);
    const int L = rm.compact ? rm.cnt[b] : R;
    const int base = rm.off[b];
    for (int r = 0; r < L; ++r) {
      const int idx = verb2roles[v * R + r];
      const float4 re = *reinterpret_cast<const float4*>(role_emb + static_cast<int64_t>(idx) * D + d);
      float4 o;
      // same association as the reference: (img_features * role_embd) * verb_embed_expand
      o.x = fmaxf((f.x * re.x) * ve.x, 0.f);
      o.y = fmaxf((f.y * re.y) * ve.y, 0.f);
      o.z = fmaxf((f.z * re.z) * ve.z, 0.f);
      o.w = fmaxf((f.w * re.w) * ve.w, 0.f);
      const int64_t off = (static_cast<int64_t>(base) + r) * D + d;
      *reinterpret_cast<float4*>(h32 + off) = o;
      store4_split(hb_hi, hb_lo, off, o);
    }
  }
}

// a[i] = sum_{j < n, j != i} h[j] for the real nodes of an image (the closed form of the [R,R] mask of
// imsitu_encoder.py:209-229 applied as in model.py:67-75, summed in the same order); a = h on pad / self-loop rows.
__global__ void k_aggregate_rows(const float* __restrict__ h32, RowMap rm, int B, int R, int D, bf16* __restrict__ a_hi,
                                 Parts a_lo) {
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(B + kSelfRows) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int u = static_cast<int>(t / D4);
    const int d = static_cast<int>(t % D4) * 4;
    if (u >= B) {
      const int row = rm.meta[1] + (u - B);
      if (row < rm.meta[2]) {
        const int64_t off = static_cast<int64_t>(row) * D + d;
        store4_split(a_hi, a_lo, off, *reinterpret_cast<const float4*>(h32 + off));
      }
      continue;
    }
    const int n = rm.cnt[u];
    const int L = rm.compact ? n : R;
    const int64_t base = static_cast<int64_t>(rm.off[u]) * D + d;
    float4 h[kMaxR];
#pragma unroll
    for (int j = 0; j < kMaxR; ++j)
      if (j < L) h[j] = *reinterpret_cast<const float4*>(h32 + base + static_cast<int64_t>(j) * D);
#pragma unroll
    for (int i = 0; i < kMaxR; ++i) {
      if (i < L) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) {
#pragma unroll
          for (int j = 0; j < kMaxR; ++j) {
            if (j < n && j != i) {
              a.x += h[j].x; a.y += h[j].y; a.z += h[j].z; a.w += h[j].w;
            }
          }
        } else {
          a = h[i];
        }
        store4_split(a_hi, a_lo, base + static_cast<int64_t>(i) * D, a);
      }
    }
  }
}

// ---- dropout: explicit keep-mask (tests) or counter-based Philox4x32-10 keyed by (seed, path stream, row, column / 8),
// so the forward and the backward pass regenerate the same Bernoulli(1 - p) keep decisions without storing a mask
// (model.py:106,110: nn.Dropout(0.5) in front of both classifiers).  One Philox block = 8 x 16 random bits = the keep
// decisions of 8 consecutive columns: keep_i = (u16_i < (1 - p) * 65536).
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// bit i of the result = keep column (8 * col8 + i) of `row`
__device__ __forceinline__ uint32_t keep_bits8(const DropSpec& ds, int64_t row, int col8, int64_t ld_keep) {
  if (ds.keep != nullptr) {
    const uint2 k = *reinterpret_cast<const uint2*>(ds.keep + row * ld_keep + static_cast<int64_t>(col8) * 8);
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      m |= (((k.x >> (8 * i)) & 0xFFu) ? 1u : 0u) << i;
      m |= (((k.y >> (8 * i)) & 0xFFu) ? 1u : 0u) << (4 + i);
    }
    return m;
  }
  if (ds.seed == nullptr) return 0xFFu;
  const unsigned long long seed = static_cast<unsigned long long>(*ds.seed);
  const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(row), static_cast<uint32_t>(col8),
                                           static_cast<uint32_t>(ds.stream), static_cast<uint32_t>(row >> 32)),
                                make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m |= ((w[i] & 0xFFFFu) < ds.thresh ? 1u : 0u) << (2 * i);
    m |= ((w[i] >> 16) < ds.thresh ? 1u : 0u) << (2 * i + 1);
  }
  return m;
}

__global__ void k_dropout_mask(DropSpec ds, int64_t rows, int D, uint8_t* __restrict__ out) {
  const int D8 = D / 8;
  const int64_t total = rows * D8;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = t / D8;
    const int c8 = static_cast<int>(t % D8);
    const uint32_t m = keep_bits8(ds, row, c8, D);
    uint2 o;
    o.x = (m & 1u) | ((m >> 1 & 1u) << 8) | ((m >> 2 & 1u) << 16) | ((m >> 3 & 1u) << 24);
    o.y = (m >> 4 & 1u) | ((m >> 5 & 1u) << 8) | ((m >> 6 & 1u) << 16) | ((m >> 7 & 1u) << 24);
    *reinterpret_cast<uint2*>(out + row * D + static_cast<int64_t>(c8) * 8) = o;
  }
}

// Classifier input: x[row, :] = dropout(h[src(row), :]) as bf16 operand parts, for ALL B*R node slots (the dropout mask
// differs per slot, so the classifier runs on every slot even though the pad slots share one state row).
// rm.cnt == nullptr: src(row) = row (verb node path).
__global__ void k_classifier_input(const float* __restrict__ h32, RowMap rm, int R, int64_t rows, int D, DropSpec ds,
                                   bf16* __restrict__ x_hi, Parts x_lo) {
  const int D8 = D / 8;
  const int64_t total = rows * D8;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = t / D8;
    const int c8 = static_cast<int>(t % D8);
    int64_t src = row;
    if (rm.cnt != nullptr) {
      const int b = static_cast<int>(row / R), r = static_cast<int>(row % R);
      const int L = rm.compact ? rm.cnt[b] : R;
      src = (r < L) ? rm.off[b] + r : rm.meta[1];
    }
    const float* hp = h32 + src * D + c8 * 8;
    float4 a = *reinterpret_cast<const float4*>(hp), b4 = *reinterpret_cast<const float4*>(hp + 4);
    const uint32_t m = keep_bits8(ds, row, c8, D);
    const float sc = ds.scale;
    a.x = (m & 1u) ? a.x * sc : 0.f;
    a.y = (m & 2u) ? a.y * sc : 0.f;
    a.z = (m & 4u) ? a.z * sc : 0.f;
    a.w = (m & 8u) ? a.w * sc : 0.f;
    b4.x = (m & 16u) ? b4.x * sc : 0.f;
    b4.y = (m & 32u) ? b4.y * sc : 0.f;
    b4.z = (m & 64u) ? b4.z * sc : 0.f;
    b4.w = (m & 128u) ? b4.w * sc : 0.f;
    store8_split(x_hi, x_lo, row * D + c8 * 8, a, b4);
  }
}

__global__ void k_zero_self_rows(float* __restrict__ x, RowMap rm, int D) {
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(kSelfRows) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int row = rm.meta[1] + static_cast<int>(t / D4);
    if (row < rm.meta[2])
      *reinterpret_cast<float4*>(x + static_cast<int64_t>(row) * D + static_cast<int>(t % D4) * 4) =
          make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// Backward of k_classifier_input: dh[dst(row), :] = dx[row, :] * keep * scale; the rows of all pad slots are SUMMED into
// the shared pad row (the backward pass of one state row feeding many classifier rows), which k_zero_self_rows cleared.
// grid = (column chunks, image slabs); rm.cnt == nullptr: one row per "image", R = 1 (verb node path).
__global__ void k_classifier_input_bwd(const float* __restrict__ dx, RowMap rm, int B, int R, int D, DropSpec ds,
                                       float* __restrict__ dh, GruPre gp) {
  const int D8 = D / 8;
  const int c8 = blockIdx.x * blockDim.x + threadIdx.x;
  if (c8 >= D8) return;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  bool any_pad = false;
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const int L = (rm.cnt != nullptr) ? (rm.compact ? rm.cnt[b] : R) : R;
    const int64_t base = (rm.off != nullptr) ? rm.off[b] : static_cast<int64_t>(b) * R;
    for (int r = 0; r < R; ++r) {
      const int64_t row = static_cast<int64_t>(b) * R + r;
      const float* xp = dx + row * D + c8 * 8;
      const float4 a = *reinterpret_cast<const float4*>(xp), b4 = *reinterpret_cast<const float4*>(xp + 4);
      const uint32_t m = keep_bits8(ds, row, c8, D);
      const float sc = ds.scale;
      float v[8] = {a.x, a.y, a.z, a.w, b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = ((m >> i) & 1u) ? v[i] * sc : 0.f;
      if (r < L && gp.z != nullptr) {
        // v = dL/dh' of the last propagation step on this state row: its GRU-gate derivatives right here, so dL/dh'
        // is never written (k_gru_bwd_pre_ld only runs on the few self-loop rows, whose dL/dh' is a sum over slots)
        const int64_t o = (base + r) * D + c8 * 8;
        const uint4 zz = *reinterpret_cast<const uint4*>(gp.z + o), cc = *reinterpret_cast<const uint4*>(gp.hc + o),
                    hh = *reinterpret_cast<const uint4*>(gp.h + o);
        const uint32_t zw[4] = {zz.x, zz.y, zz.z, zz.w}, cw[4] = {cc.x, cc.y, cc.z, cc.w}, hw[4] = {hh.x, hh.y, hh.z, hh.w};
        float dz[8], dc[8], da[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float zv = (i & 1) ? bf16_hi_f(zw[i >> 1]) : bf16_lo_f(zw[i >> 1]);
          const float cv = (i & 1) ? bf16_hi_f(cw[i >> 1]) : bf16_lo_f(cw[i >> 1]);
          const float hv = (i & 1) ? bf16_hi_f(hw[i >> 1]) : bf16_lo_f(hw[i >> 1]);
          dz[i] = v[i] * (cv - hv) * zv * (1.f - zv);
          dc[i] = v[i] * zv * (1.f - cv * cv);
          da[i] = v[i] * (1.f - zv);
        }
        const int64_t oo = (base + r) * gp.ld_out + c8 * 8;
        uint4 pz, ph;
        const uint2 z0 = pack4_bf16(dz[0], dz[1], dz[2], dz[3]), z1 = pack4_bf16(dz[4], dz[5], dz[6], dz[7]);
        const uint2 c0 = pack4_bf16(dc[0], dc[1], dc[2], dc[3]), c1 = pack4_bf16(dc[4], dc[5], dc[6], dc[7]);
        pz.x = z0.x; pz.y = z0.y; pz.z = z1.x; pz.w = z1.y;
        ph.x = c0.x; ph.y = c0.y; ph.z = c1.x; ph.w = c1.y;
        *reinterpret_cast<uint4*>(gp.dpre_z + oo) = pz;
        *reinterpret_cast<uint4*>(gp.dpre_h + oo) = ph;
        *reinterpret_cast<float4*>(gp.dh_acc + o) = make_float4(da[0], da[1], da[2], da[3]);
        *reinterpret_cast<float4*>(gp.dh_acc + o + 4) = make_float4(da[4], da[5], da[6], da[7]);
      } else if (r < L) {
        float* dp = dh + (base + r) * D + c8 * 8;
        *reinterpret_cast<float4*>(dp) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(dp + 4) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
        any_pad = true;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += v[i];
      }
    }
  }
  if (any_pad) {
    float* dp = dh + static_cast<int64_t>(rm.meta[1]) * D + c8 * 8;
    atomicAdd(reinterpret_cast<float4*>(dp), make_float4(acc[0], acc[1], acc[2], acc[3]));
    atomicAdd(reinterpret_cast<float4*>(dp + 4), make_float4(acc[4], acc[5], acc[6], acc[7]));
  }
}

// ------------------------------------------------------------------------------------------------ packing
struct PackJobs {
  PackJob j[kMaxPackJobs];
};
// grid = (blocks per job, jobs)
__global__ void k_pack_weight_multi(PackJobs jobs, int cols) {
  const PackJob job = jobs.j[blockIdx.y];
  const int c4 = cols / 4;
  const int64_t total = static_cast<int64_t>(job.rows_pad) * c4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(t / c4);
    const int c = static_cast<int>(t % c4) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < job.rows) v = *reinterpret_cast<const float4*>(job.src + static_cast<int64_t>(r) * cols + c);
    for (int k = 0; k < job.part; ++k) {
      v.x -= bf16_round(v.x); v.y -= bf16_round(v.y); v.z -= bf16_round(v.z); v.w -= bf16_round(v.w);
    }
    *reinterpret_cast<uint2*>(job.dst + static_cast<int64_t>(r) * job.ld_dst + job.col_off + c) =
        pack4_bf16(v.x, v.y, v.z, v.w);
  }
}

__global__ void k_pack_bias(const float* __restrict__ a, const float* __restrict__ b, int n, int n_pad,
                            float* __restrict__ dst) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < n) v = a[i] + (b != nullptr ? b[i] : 0.f);
    dst[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ cross-entropy
__global__ void k_count_targets(const int64_t* __restrict__ gt, int B, int R, int ignore_index,
                                float* __restrict__ counts) {
  __shared__ int sc[3];
  if (threadIdx.x < 3) sc[threadIdx.x] = 0;
  __syncthreads();
  int local[3] = {0, 0, 0};
  const int64_t total = static_cast<int64_t>(B) * 3 * R;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int a = static_cast<int>((t / R) % 3);
    if (gt[t] != ignore_index) local[a]++;
  }
  for (int a = 0; a < 3; ++a)
    if (local[a]) atomicAdd(&sc[a], local[a]);
  __syncthreads();
  if (threadIdx.x < 3 && sc[threadIdx.x]) atomicAdd(&counts[threadIdx.x], static_cast<float>(sc[threadIdx.x]));
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per row.  NT = number of targets per row (3 for nouns, 1 for verbs).
//   loss += sum_a w_a * (lse - logit[t_a]);   dlogits[c] = gs * (sum_a w_a * (p_c - [c == t_a]))
template <int NT>
__global__ void k_cross_entropy(const float* __restrict__ logits, int64_t ldl, int n_classes, int rows,
                                const int64_t* __restrict__ gt, int R, int ignore_index,
                                const float* __restrict__ counts, float inv_fixed, float* __restrict__ loss,
                                float* __restrict__ dlogits, float grad_scale, const float* __restrict__ gscale_dev,
                                const float2* __restrict__ stats, int stats_tiles,
                                const float* __restrict__ total_dev, bf16* __restrict__ dlb, int64_t ld_b, int n_pad,
                                int accumulate) {
  // dlb (nullable): the gradient goes out as the zero-padded bf16 [rows, n_pad] operand of the classifier's backward
  // GEMMs instead of (not in addition to) the fp32 dlogits -- the fp32 gradient is then never written or re-read
  // (accumulate: add to what dlb holds, for a second loss on the same logits)
  __shared__ float s_loss[kThreads / 32];
  // total_dev: device scalar holding the GLOBAL number of rows the mean is taken over (all-reduced by the caller when
  // the batch is sharded unevenly); overrides inv_fixed
  if (total_dev != nullptr) inv_fixed = 1.0f / fmaxf(__ldg(total_dev), 1.0f);
  // gscale_dev: device scalar multiplied into the gradient (the incoming d(loss) of the autograd backward pass)
  if (gscale_dev != nullptr) grad_scale *= __ldg(gscale_dev);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warps_per_block = blockDim.x >> 5;
  float my_loss = 0.f;
  for (int row = blockIdx.x * warps_per_block + wib; row < rows; row += gridDim.x * warps_per_block) {
    const float* lr = logits + static_cast<int64_t>(row) * ldl;
    int64_t tgt[NT];
    float w[NT];
    float wsum = 0.f;
#pragma unroll
    for (int a = 0; a < NT; ++a) {
      if (NT == 3) {
        const int b = row / R, r = row % R;
        tgt[a] = gt[(static_cast<int64_t>(b) * 3 + a) * R + r];
        w[a] = (tgt[a] != ignore_index) ? 1.0f / counts[a] : 0.f;
      } else {
        tgt[a] = gt[row];
        w[a] = inv_fixed;
      }
      wsum += w[a];
    }
    if (wsum == 0.f && dlogits == nullptr && dlb == nullptr) continue;  // fully ignored row contributes nothing
    float mx = -INFINITY, se = 0.f;
    if (stats != nullptr) {
      // the classifier GEMM already reduced every 128/256-column tile of this row to (max, sum exp(x - max)):
      // combine the per-tile pairs instead of reading the logits row two more times
      float2 st = make_float2(-INFINITY, 0.f);
      if (lane < stats_tiles) st = stats[static_cast<int64_t>(row) * stats_tiles + lane];
      mx = warp_max(st.x);
      se = warp_sum(st.y > 0.f ? st.y * __expf(st.x - mx) : 0.f);
    } else {
      for (int c = lane; c < n_classes; c += 32) mx = fmaxf(mx, lr[c]);
      mx = warp_max(mx);
      for (int c = lane; c < n_classes; c += 32) se += __expf(lr[c] - mx);
      se = warp_sum(se);
    }
    const float lse = mx + __logf(se);
    if (lane == 0) {
#pragma unroll
      for (int a = 0; a < NT; ++a)
        if (w[a] != 0.f) my_loss += w[a] * (lse - lr[tgt[a]]);
    }
    if (dlb != nullptr) {
      bf16* br = dlb + static_cast<int64_t>(row) * ld_b;
      const float inv_se = 1.0f / se;
      const float ws = wsum * grad_scale;
      // n_pad is a multiple of 128 here (the classifier pads to 256 columns); logits rows are 16-byte aligned
      for (int c = lane * 4; c < n_pad; c += 128) {
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (c < n_classes && wsum != 0.f) {
          float x[4];
          if (c + 4 <= ldl && ((reinterpret_cast<uintptr_t>(lr) & 15) == 0) && (ldl & 3) == 0) {
            const float4 v = *reinterpret_cast<const float4*>(lr + c);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) x[k] = (c + k < n_classes) ? lr[c + k] : 0.f;
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (c + k < n_classes) {
              float v = ws * __expf(x[k] - mx) * inv_se;
#pragma unroll
              for (int a = 0; a < NT; ++a)
                if (w[a] != 0.f && tgt[a] == c + k) v -= w[a] * grad_scale;
              g[k] = v;
            }
          }
        }
        uint2* dst = reinterpret_cast<uint2*>(br + c);
        if (accumulate) {
          const uint2 old = *dst;
          g[0] += bf16_lo_f(old.x); g[1] += bf16_hi_f(old.x); g[2] += bf16_lo_f(old.y); g[3] += bf16_hi_f(old.y);
        }
        *dst = pack4_bf16(g[0], g[1], g[2], g[3]);
      }
    } else if (dlogits != nullptr) {
      float* dr = dlogits + static_cast<int64_t>(row) * ldl;
      const float inv_se = 1.0f / se;
      const float ws = wsum * grad_scale;
      if ((ldl & 3) == 0 && ((reinterpret_cast<uintptr_t>(lr) | reinterpret_cast<uintptr_t>(dr)) & 15) == 0) {
        // four columns per lane and access; consecutive iterations are independent, so several loads are in flight
#pragma unroll 4
        for (int c = lane * 4; c < ldl; c += 128) {
          const float4 x = *reinterpret_cast<const float4*>(lr + c);
          float g[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float v = 0.f;
            if (c + k < n_classes && wsum != 0.f) {
              v = ws * __expf(g[k] - mx) * inv_se;
#pragma unroll
              for (int a = 0; a < NT; ++a)
                if (w[a] != 0.f && tgt[a] == c + k) v -= w[a] * grad_scale;
            }
            g[k] = v;
          }
          *reinterpret_cast<float4*>(dr + c) = make_float4(g[0], g[1], g[2], g[3]);
        }
      } else {
        for (int c = lane; c < ldl; c += 32) {
          float g = 0.f;
          if (c < n_classes && wsum != 0.f) {
            g = ws * __expf(lr[c] - mx) * inv_se;
#pragma unroll
            for (int a = 0; a < NT; ++a)
              if (w[a] != 0.f && tgt[a] == c) g -= w[a] * grad_scale;
          }
          dr[c] = g;
        }
      }
    }
  }
  if (lane == 0) s_loss[wib] = my_loss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < warps_per_block; ++i) t += s_loss[i];
    if (t != 0.f && loss != nullptr) atomicAdd(loss, t);
  }
}

__global__ void k_cast_pad(const float* __restrict__ src, int64_t ld, int rows, int n_valid, int n_pad,
                           bf16* __restrict__ dst, int accumulate) {
  // eight columns per thread: two 16-byte loads, one 16-byte store (n_pad is a multiple of 8; ld a multiple of 4)
  const int c8 = n_pad / 8;
  const int64_t total = static_cast<int64_t>(rows) * c8;
  const bool vec = (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(t / c8);
    const int c = static_cast<int>(t % c8) * 8;
    const float* s = src + static_cast<int64_t>(r) * ld;
    float v[8];
    if (vec && c + 8 <= ld) {
      const float4 x = *reinterpret_cast<const float4*>(s + c), y = *reinterpret_cast<const float4*>(s + c + 4);
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = (c + k < n_valid) ? s[c + k] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (c + k >= n_valid) v[k] = 0.f;
    uint4* dp = reinterpret_cast<uint4*>(dst + static_cast<int64_t>(r) * n_pad + c);
    if (accumulate) {   // on top of a gradient a loss kernel already wrote there as bf16
      const uint4 old = *dp;
      v[0] += bf16_lo_f(old.x); v[1] += bf16_hi_f(old.x); v[2] += bf16_lo_f(old.y); v[3] += bf16_hi_f(old.y);
      v[4] += bf16_lo_f(old.z); v[5] += bf16_hi_f(old.z); v[6] += bf16_lo_f(old.w); v[7] += bf16_hi_f(old.w);
    }
    uint4 o;
    const uint2 lo = pack4_bf16(v[0], v[1], v[2], v[3]), hi = pack4_bf16(v[4], v[5], v[6], v[7]);
    o.x = lo.x; o.y = lo.y; o.z = hi.x; o.w = hi.y;
    *dp = o;
  }
}

// ------------------------------------------------------------------------------------------------ GRU backward
// column sums of a bf16 matrix; block = 8 warps x 64 columns, grid = (col chunks, row slabs)
__global__ void k_colsum(const bf16* __restrict__ X, int64_t ld, int rows, int n_cols, float* __restrict__ out1,
                         float scale1, float* __restrict__ out2, float scale2) {
  __shared__ float2 red[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + lane * 2;
  const int rows_per = (rows + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * rows_per, r1 = min(rows, r0 + rows_per);
  float2 acc = make_float2(0.f, 0.f);
  if (c < n_cols) {
    for (int r = r0 + w; r < r1; r += 8) {
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(X + static_cast<int64_t>(r) * ld + c);
      const float2 f = __bfloat1622float2(v);
      acc.x += f.x;
      acc.y += f.y;
    }
  }
  red[w][lane] = acc;
  __syncthreads();
  if (w == 0 && c < n_cols) {
    float2 t = red[0][lane];
#pragma unroll
    for (int i = 1; i < 8; ++i) {
      t.x += red[i][lane].x;
      t.y += red[i][lane].y;
    }
    if (out1 != nullptr) {
      atomicAdd(out1 + c, t.x * scale1);
      if (c + 1 < n_cols) atomicAdd(out1 + c + 1, t.y * scale1);
    }
    if (out2 != nullptr) {
      atomicAdd(out2 + c, t.x * scale2);
      if (c + 1 < n_cols) atomicAdd(out2 + c + 1, t.y * scale2);
    }
  }
}

// One thread per (image, 4 columns) walks the image's real role rows.  kEmb: the embedding gradients (atomics: ~190
// role rows receive the gradients of all node rows); kFeat: dfeat[b] = sum_r [node > 0] dh0 * role_emb * verb_emb, one
// register accumulator and a plain store (this thread owns the output element: deterministic, no atomics).
template <bool kEmb, bool kFeat>
__global__ void k_node_init_bwd(const float* __restrict__ dh0, const bf16* __restrict__ h0b,
                                const float* __restrict__ feat, const float* __restrict__ role_emb,
                                const float* __restrict__ verb_emb, const int64_t* __restrict__ verb,
                                const int32_t* __restrict__ verb2roles, int n_verbs, int n_roles, int B, int R,
                                int D, RowMap rm, float* __restrict__ d_role_emb, float* __restrict__ d_verb_emb,
                                float* __restrict__ dfeat) {
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(B) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(t / D4);
    const int d = static_cast<int>(t % D4) * 4;
    int64_t v = verb[b];
    if (v < 0 || v >= n_verbs) v = 0;   // same clamp as the forward kernels (which also raise the bad-verb flag)
    float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kEmb) f = *reinterpret_cast<const float4*>(feat + static_cast<int64_t>(b) * D + d);
    const float4 ve = *reinterpret_cast<const float4*>(verb_emb + v * D + d);
    float4 accv = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 accf = make_float4(0.f, 0.f, 0.f, 0.f);
    const int n = rm.cnt[b];
    const int64_t base = rm.off[b];
    for (int r = 0; r < n; ++r) {
      const int idx = verb2roles[v * R + r];
      if (idx == n_roles) continue;  // padding_idx row: never receives a gradient, contributes 0 to verb_emb
      const int64_t off = (base + r) * D + d;
      float4 g = *reinterpret_cast<const float4*>(dh0 + off);
      const uint2 hb = *reinterpret_cast<const uint2*>(h0b + off);
      g.x = (bf16_lo_f(hb.x) > 0.f) ? g.x : 0.f;
      g.y = (bf16_hi_f(hb.x) > 0.f) ? g.y : 0.f;
      g.z = (bf16_lo_f(hb.y) > 0.f) ? g.z : 0.f;
      g.w = (bf16_hi_f(hb.y) > 0.f) ? g.w : 0.f;
      const float4 re = *reinterpret_cast<const float4*>(role_emb + static_cast<int64_t>(idx) * D + d);
      if (kEmb) {
        // one 16-byte reduction per thread instead of four
        atomicAdd(reinterpret_cast<float4*>(d_role_emb + static_cast<int64_t>(idx) * D + d),
                  make_float4(g.x * f.x * ve.x, g.y * f.y * ve.y, g.z * f.z * ve.z, g.w * f.w * ve.w));
        accv.x = fmaf(g.x * f.x, re.x, accv.x);
        accv.y = fmaf(g.y * f.y, re.y, accv.y);
        accv.z = fmaf(g.z * f.z, re.z, accv.z);
        accv.w = fmaf(g.w * f.w, re.w, accv.w);
      }
      if (kFeat) {
        accf.x = fmaf(g.x * re.x, ve.x, accf.x);
        accf.y = fmaf(g.y * re.y, ve.y, accf.y);
        accf.z = fmaf(g.z * re.z, ve.z, accf.z);
        accf.w = fmaf(g.w * re.w, ve.w, accf.w);
      }
    }
    if (kEmb) atomicAdd(reinterpret_cast<float4*>(d_verb_emb + v * D + d), accv);
    if (kFeat) *reinterpret_cast<float4*>(dfeat + static_cast<int64_t>(b) * D + d) = accf;
  }
}

// verb node: node = relu(feat), so dfeat = dh0 where the initial state (its bf16 copy) is > 0, else 0
__global__ void k_node_init_verb_bwd(const float* __restrict__ dh0, const bf16* __restrict__ h0b, int64_t n4,
                                     float* __restrict__ dfeat) {
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n4;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 g = *reinterpret_cast<const float4*>(dh0 + t * 4);
    const uint2 hb = *reinterpret_cast<const uint2*>(h0b + t * 4);
    g.x = (bf16_lo_f(hb.x) > 0.f) ? g.x : 0.f;
    g.y = (bf16_hi_f(hb.x) > 0.f) ? g.y : 0.f;
    g.z = (bf16_lo_f(hb.y) > 0.f) ? g.z : 0.f;
    g.w = (bf16_hi_f(hb.y) > 0.f) ? g.w : 0.f;
    *reinterpret_cast<float4*>(dfeat + t * 4) = g;
  }
}

// ada[j] = e[j] + sum_{i < n, i != j} da[i] on the real nodes of an image (the aggregation is symmetric, so its backward
// pass is the same closed form), ada = e + da on pad / self-loop rows.  rm.cnt == nullptr: every one of the B rows is a
// self-loop row (verb node path: the aggregation is the identity).  bf16 in / bf16 out, 8 columns per thread.
__global__ void __launch_bounds__(kThreads, 4)
k_aggregate_t_rows(const bf16* __restrict__ da, const bf16* __restrict__ e, RowMap rm, int B, int R, int D,
                   bf16* __restrict__ ada) {
  const int D8 = D / 8;
  const bool rows_only = (rm.cnt == nullptr);
  const int64_t total = static_cast<int64_t>(rows_only ? B : B + kSelfRows) * D8;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int u = static_cast<int>(t / D8);
    const int d = static_cast<int>(t % D8) * 8;
    int n = 0, L = 1;
    int64_t base;
    if (rows_only) {
      base = static_cast<int64_t>(u) * D + d;
    } else if (u >= B) {
      const int row = rm.meta[1] + (u - B);
      if (row >= rm.meta[2]) continue;
      base = static_cast<int64_t>(row) * D + d;
    } else {
      n = rm.cnt[u];
      L = rm.compact ? n : R;
      base = static_cast<int64_t>(rm.off[u]) * D + d;
    }
    // the input rows stay packed as bf16 pairs and are widened where they are used (register pressure)
    uint4 g[kMaxR];
#pragma unroll
    for (int i = 0; i < kMaxR; ++i)
      if (i < L) g[i] = *reinterpret_cast<const uint4*>(da + base + static_cast<int64_t>(i) * D);
#pragma unroll
    for (int j = 0; j < kMaxR; ++j) {
      if (j < L) {
        const uint4 ad = *reinterpret_cast<const uint4*>(e + base + static_cast<int64_t>(j) * D);
        float a[8] = {bf16_lo_f(ad.x), bf16_hi_f(ad.x), bf16_lo_f(ad.y), bf16_hi_f(ad.y),
                      bf16_lo_f(ad.z), bf16_hi_f(ad.z), bf16_lo_f(ad.w), bf16_hi_f(ad.w)};
#pragma unroll
        for (int i = 0; i < kMaxR; ++i) {
          const bool on = (j < n) ? (i < n && i != j) : (i == j);
          if (i < L && on) {
            a[0] += bf16_lo_f(g[i].x); a[1] += bf16_hi_f(g[i].x);
            a[2] += bf16_lo_f(g[i].y); a[3] += bf16_hi_f(g[i].y);
            a[4] += bf16_lo_f(g[i].z); a[5] += bf16_hi_f(g[i].z);
            a[6] += bf16_lo_f(g[i].w); a[7] += bf16_hi_f(g[i].w);
          }
        }
        uint4 o;
        const uint2 lo = pack4_bf16(a[0], a[1], a[2], a[3]), hi = pack4_bf16(a[4], a[5], a[6], a[7]);
        o.x = lo.x; o.y = lo.y; o.z = hi.x; o.w = hi.y;
        *reinterpret_cast<uint4*>(ada + base + static_cast<int64_t>(j) * D) = o;
      }
    }
  }
}

// One 8-column chunk of the backward of k_aggregate for image rows [base, base + R*D) (see k_aggregate_t):
// ada[j] = e[j] + sum_i mb[i,j] da[i]; kGrad: acc[i*kMaxR + j] += the chunk's share of da[i] . h[j].
template <bool kGrad>
__device__ __forceinline__ void aggregate_t_chunk(const bf16* __restrict__ da, const bf16* __restrict__ e,
                                                  const float* __restrict__ mb, const bf16* __restrict__ h,
                                                  int64_t base, int R, int D, bf16* __restrict__ ada, float* acc) {
  uint4 g[kMaxR];
#pragma unroll
  for (int i = 0; i < kMaxR; ++i)
    if (i < R) g[i] = *reinterpret_cast<const uint4*>(da + base + static_cast<int64_t>(i) * D);
#pragma unroll
  for (int j = 0; j < kMaxR; ++j) {
    if (j < R) {
      const uint4 ad = *reinterpret_cast<const uint4*>(e + base + static_cast<int64_t>(j) * D);
      float a[8] = {bf16_lo_f(ad.x), bf16_hi_f(ad.x), bf16_lo_f(ad.y), bf16_hi_f(ad.y),
                    bf16_lo_f(ad.z), bf16_hi_f(ad.z), bf16_lo_f(ad.w), bf16_hi_f(ad.w)};
#pragma unroll
      for (int i = 0; i < kMaxR; ++i) {
        if (i < R) {
          const float m = __ldg(mb + i * R + j);
          a[0] = fmaf(m, bf16_lo_f(g[i].x), a[0]); a[1] = fmaf(m, bf16_hi_f(g[i].x), a[1]);
          a[2] = fmaf(m, bf16_lo_f(g[i].y), a[2]); a[3] = fmaf(m, bf16_hi_f(g[i].y), a[3]);
          a[4] = fmaf(m, bf16_lo_f(g[i].z), a[4]); a[5] = fmaf(m, bf16_hi_f(g[i].z), a[5]);
          a[6] = fmaf(m, bf16_lo_f(g[i].w), a[6]); a[7] = fmaf(m, bf16_hi_f(g[i].w), a[7]);
        }
      }
      uint4 o;
      const uint2 lo = pack4_bf16(a[0], a[1], a[2], a[3]), hi = pack4_bf16(a[4], a[5], a[6], a[7]);
      o.x = lo.x; o.y = lo.y; o.z = hi.x; o.w = hi.y;
      *reinterpret_cast<uint4*>(ada + base + static_cast<int64_t>(j) * D) = o;
      if constexpr (kGrad) {
        const uint4 hv = *reinterpret_cast<const uint4*>(h + base + static_cast<int64_t>(j) * D);
        const float hf[8] = {bf16_lo_f(hv.x), bf16_hi_f(hv.x), bf16_lo_f(hv.y), bf16_hi_f(hv.y),
                             bf16_lo_f(hv.z), bf16_hi_f(hv.z), bf16_lo_f(hv.w), bf16_hi_f(hv.w)};
#pragma unroll
        for (int i = 0; i < kMaxR; ++i) {
          if (i < R) {
            float s = acc[i * kMaxR + j];
            s = fmaf(bf16_lo_f(g[i].x), hf[0], s); s = fmaf(bf16_hi_f(g[i].x), hf[1], s);
            s = fmaf(bf16_lo_f(g[i].y), hf[2], s); s = fmaf(bf16_hi_f(g[i].y), hf[3], s);
            s = fmaf(bf16_lo_f(g[i].z), hf[4], s); s = fmaf(bf16_hi_f(g[i].z), hf[5], s);
            s = fmaf(bf16_lo_f(g[i].w), hf[6], s); s = fmaf(bf16_hi_f(g[i].w), hf[7], s);
            acc[i * kMaxR + j] = s;
          }
        }
      }
    }
  }
}

// Backward of k_aggregate on dense rows (B images x R rows) with the caller's mask, which may be asymmetric, non-binary
// and have self-loops:  ada[b,j] = e[b,j] + sum_i mask[b,i,j] da[b,i].  kGrad: also dmask[b,i,j] += sum_d da[b,i,d] h[b,j,d]
// (h = the state operand that entered the step).  8 columns per thread per chunk.  Without kGrad the grid strides over
// (image, chunk) pairs.  With kGrad one block owns an image (grid-stride over images): the R*R dot products are reduced
// in a fixed order -- a warp butterfly, then the warps in index order -- and added by the owning block, so dmask is
// deterministic without atomics.
template <bool kGrad>
__global__ void __launch_bounds__(kGrad ? 128 : 256, kGrad ? 1 : 4)
k_aggregate_t(const bf16* __restrict__ da, const bf16* __restrict__ e, const float* __restrict__ mask,
              const bf16* __restrict__ h, int B, int R, int D, bf16* __restrict__ ada, float* __restrict__ dmask) {
  if constexpr (!kGrad) {
    const int D8 = D / 8;
    const int64_t total = static_cast<int64_t>(B) * D8;
    for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
      const int b = static_cast<int>(t / D8);
      const int d = static_cast<int>(t % D8) * 8;
      aggregate_t_chunk<false>(da, e, mask + static_cast<int64_t>(b) * R * R, nullptr,
                               static_cast<int64_t>(b) * R * D + d, R, D, ada, nullptr);
    }
  } else {
    constexpr int kAcc = kMaxR * kMaxR;
    __shared__ float red[4][kAcc];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
      const float* mb = mask + static_cast<int64_t>(b) * R * R;
      float acc[kAcc];
#pragma unroll
      for (int k = 0; k < kAcc; ++k) acc[k] = 0.f;
      for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8)
        aggregate_t_chunk<true>(da, e, mb, h, static_cast<int64_t>(b) * R * D + d, R, D, ada, acc);
#pragma unroll
      for (int i = 0; i < kMaxR; ++i) {
#pragma unroll
        for (int j = 0; j < kMaxR; ++j) {
          if (i < R && j < R) {
            float v = acc[i * kMaxR + j];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0) red[w][i * R + j] = v;
          }
        }
      }
      __syncthreads();
      // R*R can exceed the block (32 threads at D = 256): each thread finishes every blockDim-th entry
      for (int k = threadIdx.x; k < R * R; k += blockDim.x) {
        float s = 0.f;
        for (int q = 0; q < static_cast<int>(blockDim.x >> 5); ++q) s += red[q][k];
        dmask[static_cast<int64_t>(b) * R * R + k] += s;
      }
      __syncthreads();   // red is reused by the block's next image
    }
  }
}

struct ColsumJobs {
  ColsumJob j[4];
};
// grid = (column chunks of 64, segments * row slabs, jobs).  The rows are nseg segments of `rows` rows each (rows_dev, when
// given, holds the number of valid rows per segment), segment s starting at row s * seg_stride of X.
__global__ void k_colsum_multi(ColsumJobs jobs, int64_t ld, int rows, const int* __restrict__ rows_dev, int nseg,
                               int64_t seg_stride, int n_cols) {
  __shared__ float2 red[8][32];
  ColsumJob job = jobs.j[blockIdx.z];
  if (rows_dev != nullptr) rows = __ldg(rows_dev);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + lane * 2;
  const int slabs = gridDim.y / nseg;
  const int seg = blockIdx.y / slabs, slab = blockIdx.y % slabs;
  job.X += static_cast<int64_t>(seg) * seg_stride * ld;
  const int rows_per = (rows + slabs - 1) / slabs;
  const int r0 = slab * rows_per, r1 = min(rows, r0 + rows_per);
  float2 acc = make_float2(0.f, 0.f);
  if (c < n_cols) {
    int r = r0 + w;
    for (; r + 24 < r1; r += 32) {   // 4 independent loads in flight per thread
      const __nv_bfloat162 v0 = *reinterpret_cast<const __nv_bfloat162*>(job.X + static_cast<int64_t>(r) * ld + c);
      const __nv_bfloat162 v1 = *reinterpret_cast<const __nv_bfloat162*>(job.X + static_cast<int64_t>(r + 8) * ld + c);
      const __nv_bfloat162 v2 = *reinterpret_cast<const __nv_bfloat162*>(job.X + static_cast<int64_t>(r + 16) * ld + c);
      const __nv_bfloat162 v3 = *reinterpret_cast<const __nv_bfloat162*>(job.X + static_cast<int64_t>(r + 24) * ld + c);
      const float2 f0 = __bfloat1622float2(v0), f1 = __bfloat1622float2(v1), f2 = __bfloat1622float2(v2),
                   f3 = __bfloat1622float2(v3);
      acc.x += (f0.x + f1.x) + (f2.x + f3.x);
      acc.y += (f0.y + f1.y) + (f2.y + f3.y);
    }
    for (; r < r1; r += 8) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(job.X + static_cast<int64_t>(r) * ld + c));
      acc.x += f.x;
      acc.y += f.y;
    }
  }
  red[w][lane] = acc;
  __syncthreads();
  if (w == 0 && c < n_cols) {
    float2 t = red[0][lane];
#pragma unroll
    for (int i = 1; i < 8; ++i) {
      t.x += red[i][lane].x;
      t.y += red[i][lane].y;
    }
    if (job.out1 != nullptr) {
      atomicAdd(job.out1 + c, t.x * job.scale);
      if (c + 1 < n_cols) atomicAdd(job.out1 + c + 1, t.y * job.scale);
    }
    if (job.out2 != nullptr) {
      atomicAdd(job.out2 + c, t.x * job.scale);
      if (c + 1 < n_cols) atomicAdd(job.out2 + c + 1, t.y * job.scale);
    }
    if (job.out3 != nullptr) {
      atomicAdd(job.out3 + c, t.x * job.scale3);
      if (c + 1 < n_cols) atomicAdd(job.out3 + c + 1, t.y * job.scale3);
    }
  }
}

__global__ void k_gru_bwd_pre_ld(const float* __restrict__ dh, const bf16* __restrict__ z, const bf16* __restrict__ hc,
                                 const bf16* __restrict__ h, int rows, const int* __restrict__ rows_dev,
                                 const int* __restrict__ row0_dev, int D, bf16* __restrict__ dpre_z,
                                 bf16* __restrict__ dpre_h, int64_t ld_out, float* __restrict__ dh_acc) {
  // rows [row0, rows): both ends may live on the device (the self-loop rows of a compact role-graph path)
  if (rows_dev != nullptr) rows = __ldg(rows_dev);
  const int row0 = (row0_dev != nullptr) ? __ldg(row0_dev) : 0;
  const int D4 = D / 4;
  const int64_t total = static_cast<int64_t>(rows - row0) * D4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = row0 + t / D4;
    const int col = static_cast<int>(t % D4) * 4;
    const int64_t i = row * D + col;
    const float4 g = *reinterpret_cast<const float4*>(dh + i);
    const uint2 zz = *reinterpret_cast<const uint2*>(z + i);
    const uint2 cc = *reinterpret_cast<const uint2*>(hc + i);
    const uint2 hh = *reinterpret_cast<const uint2*>(h + i);
    const float gv[4] = {g.x, g.y, g.z, g.w};
    const float zv[4] = {bf16_lo_f(zz.x), bf16_hi_f(zz.x), bf16_lo_f(zz.y), bf16_hi_f(zz.y)};
    const float cv[4] = {bf16_lo_f(cc.x), bf16_hi_f(cc.x), bf16_lo_f(cc.y), bf16_hi_f(cc.y)};
    const float hv[4] = {bf16_lo_f(hh.x), bf16_hi_f(hh.x), bf16_lo_f(hh.y), bf16_hi_f(hh.y)};
    float dz[4], dc[4], da[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      dz[k] = gv[k] * (cv[k] - hv[k]) * zv[k] * (1.f - zv[k]);
      dc[k] = gv[k] * zv[k] * (1.f - cv[k] * cv[k]);
      da[k] = gv[k] * (1.f - zv[k]);
    }
    *reinterpret_cast<uint2*>(dpre_z + row * ld_out + col) = pack4_bf16(dz[0], dz[1], dz[2], dz[3]);
    *reinterpret_cast<uint2*>(dpre_h + row * ld_out + col) = pack4_bf16(dc[0], dc[1], dc[2], dc[3]);
    *reinterpret_cast<float4*>(dh_acc + i) = make_float4(da[0], da[1], da[2], da[3]);
  }
}

// one warp per output row
__global__ void k_matvec(const float* __restrict__ W, const float* __restrict__ x, int rows, int cols,
                         float* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float acc = 0.f;
  for (int k = lane; k < cols; k += 32) acc = fmaf(W[static_cast<int64_t>(row) * cols + k], x[k], acc);
  acc = warp_sum(acc);
  if (lane == 0) y[row] = acc;
}

struct Mat3 {
  const float* W[3];
  float* dW[3];
};
// grid = (cols / 256, row slabs, 3 matrices); y[k] += sum over the slab of W_x[o,k] s[x*rows + o]
__global__ void k_matvec_t_acc3(Mat3 m, const float* __restrict__ sv, int rows, int cols, float* __restrict__ y) {
  const float* __restrict__ W = m.W[blockIdx.z];
  const float* __restrict__ s = sv + static_cast<int64_t>(blockIdx.z) * rows;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int rows_per = (rows + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * rows_per, r1 = min(rows, r0 + rows_per);
  if (k >= cols || W == nullptr) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;   // four independent loads in flight
  int o = r0;
  for (; o + 3 < r1; o += 4) {
    const float* w = W + static_cast<int64_t>(o) * cols + k;
    a0 = fmaf(w[0], s[o], a0);
    a1 = fmaf(w[cols], s[o + 1], a1);
    a2 = fmaf(w[2 * static_cast<int64_t>(cols)], s[o + 2], a2);
    a3 = fmaf(w[3 * static_cast<int64_t>(cols)], s[o + 3], a3);
  }
  for (; o < r1; ++o) a0 = fmaf(W[static_cast<int64_t>(o) * cols + k], s[o], a0);
  atomicAdd(y + k, (a0 + a1) + (a2 + a3));
}

// grid = (chunks, 3 matrices); dW_x[o,k] += s[x*rows + o] * b[k], four columns per thread.
// ATOMIC: the verb and noun backward passes may accumulate into the same dW from two streams.
template <bool ATOMIC>
__global__ void k_outer_acc3(Mat3 m, const float* __restrict__ sv, const float* __restrict__ b, int rows, int cols) {
  float* __restrict__ dW = m.dW[blockIdx.y];
  if (dW == nullptr) return;
  const float* __restrict__ s = sv + static_cast<int64_t>(blockIdx.y) * rows;
  const int c4 = cols >> 2;
  const int64_t total = static_cast<int64_t>(rows) * c4;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int o = static_cast<int>(t / c4), k = static_cast<int>(t % c4) * 4;
    const float so = s[o];
    const float4 bv = *reinterpret_cast<const float4*>(b + k);
    float4* dst = reinterpret_cast<float4*>(dW + static_cast<int64_t>(o) * cols + k);
    const float4 upd = make_float4(so * bv.x, so * bv.y, so * bv.z, so * bv.w);
    if constexpr (ATOMIC) {
      atomicAdd(dst, upd);
    } else {
      float4 v = *dst;
      v.x += upd.x; v.y += upd.y; v.z += upd.z; v.w += upd.w;
      *dst = v;
    }
  }
}

__global__ void k_pack_bias3(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                             float scale, int n, int n_pad, float* __restrict__ dst) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < n) v = a[i] + (b != nullptr ? b[i] : 0.f) + (c != nullptr ? scale * c[i] : 0.f);
    dst[i] = v;
  }
}

__global__ void k_sumsq(const float* __restrict__ g, int64_t n4, float* __restrict__ out) {
  __shared__ float red[kThreads / 32];
  float acc = 0.f;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n4;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 v = *reinterpret_cast<const float4*>(g + t * 4);
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < kThreads / 32; ++i) t += red[i];
    atomicAdd(out, t);
  }
}

// torch.nn.utils.clip_grad_norm_ (coef = min(1, max_norm / (norm + 1e-6)), grads scaled in place) followed by
// torch.optim.Adamax: exp_avg = b1*exp_avg + (1-b1)*g; exp_inf = max(b2*exp_inf, |g| + eps);
// p -= lr / (1 - b1^step) * exp_avg / exp_inf.   `step` holds the number of steps taken BEFORE this one.
__global__ void k_clip_adamax(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                              float* __restrict__ u, int64_t n4, float lr, float b1, float b2, float eps,
                              float max_norm, const float* __restrict__ norm_sq, const float* __restrict__ step) {
  const float norm = sqrtf(*norm_sq);
  const float coef = fminf(1.0f, max_norm / (norm + 1e-6f));
  const float t = *step + 1.0f;
  const float clr = lr / (1.0f - powf(b1, t));
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 gv = *reinterpret_cast<const float4*>(g + i * 4);
    float4 mv = *reinterpret_cast<const float4*>(m + i * 4);
    float4 uv = *reinterpret_cast<const float4*>(u + i * 4);
    float4 pv = *reinterpret_cast<const float4*>(p + i * 4);
    float* gp = reinterpret_cast<float*>(&gv);
    float* mp = reinterpret_cast<float*>(&mv);
    float* up = reinterpret_cast<float*>(&uv);
    float* pp = reinterpret_cast<float*>(&pv);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      gp[k] *= coef;
      mp[k] = b1 * mp[k] + (1.0f - b1) * gp[k];
      up[k] = fmaxf(b2 * up[k], fabsf(gp[k]) + eps);
      pp[k] -= clr * (mp[k] / up[k]);
    }
    *reinterpret_cast<float4*>(g + i * 4) = gv;
    *reinterpret_cast<float4*>(m + i * 4) = mv;
    *reinterpret_cast<float4*>(u + i * 4) = uv;
    *reinterpret_cast<float4*>(p + i * 4) = pv;
  }
}

__global__ void k_inc(float* x) { *x += 1.0f; }

// ------------------------------------------------------------------------------------------------ top-k decode
// (v, c) ranks before (w, d): larger value, ties to the lower column (torch.argmax / a stable descending sort)
__device__ __forceinline__ bool topk_before(float v, int c, float w, int d) { return v > w || (v == w && c < d); }

template <int KMAX>
__device__ __forceinline__ void topk_insert(float (&tv)[KMAX], int (&tc)[KMAX], float v, int c) {
  if (!topk_before(v, c, tv[KMAX - 1], tc[KMAX - 1])) return;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {   // carry insertion: the candidate swaps with every entry it ranks before
    if (topk_before(v, c, tv[j], tc[j])) {
      const float tvj = tv[j];
      const int tcj = tc[j];
      tv[j] = v; tc[j] = c;
      v = tvj; c = tcj;
    }
  }
}

// One warp per row.  Each lane keeps the KMAX best (value, column) pairs of the columns it reads, sorted, in registers
// (the insertion is unrolled, so the list never leaves them), and a running (max, sum exp(x - max)) of its columns.
// The row is read in chunks of kTopkChunk values per lane, all loads of a chunk in flight at once; the running sum is
// rescaled once per chunk, so every column costs one expf.  Then k rounds of a warp argmax over the lane heads; the
// winning lane pops its head.  The sentinel (-inf, INT_MAX) ranks after every real column, -inf entries included.
// Every column < n is read exactly once; columns >= n are never read.
constexpr int kTopkChunk = 64;

template <int KMAX>
__global__ void __launch_bounds__(kThreads)
k_row_topk_logsoftmax(const float* __restrict__ x, int64_t ldl, int rows, int n, int k, int64_t* __restrict__ idx,
                      float* __restrict__ logp) {
  const int lane = threadIdx.x & 31;
  const int warps = blockDim.x >> 5;
  const bool vec = (ldl & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  for (int row = blockIdx.x * warps + (threadIdx.x >> 5); row < rows; row += gridDim.x * warps) {
    const float* xr = x + static_cast<int64_t>(row) * ldl;
    float tv[KMAX];
    int tc[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) { tv[j] = -INFINITY; tc[j] = INT_MAX; }
    float m = -INFINITY, se = 0.f;
    float v[kTopkChunk];
    // v[i] holds column col(i) of the current chunk (-inf where the column is >= n); fold the chunk into the state
    auto fold = [&](auto col) {
      float cm = -INFINITY;
#pragma unroll
      for (int i = 0; i < kTopkChunk; ++i) {
        cm = fmaxf(cm, v[i]);
        topk_insert<KMAX>(tv, tc, v[i], col(i));
      }
      const float mn = fmaxf(m, cm);
      if (mn > -INFINITY) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < kTopkChunk; ++i) acc += expf(v[i] - mn);   // -inf -> 0
        se = se * expf(m - mn) + acc;                                  // m = -inf: se is 0
        m = mn;
      }
    };
    if (vec) {   // 16-byte loads: lane reads float4 q = q0 + 32 i + lane of the row
      const int n4 = (n + 3) >> 2;
      for (int q0 = 0; q0 < n4; q0 += 32 * (kTopkChunk / 4)) {
#pragma unroll
        for (int i = 0; i < kTopkChunk / 4; ++i) {
          const int q = q0 + 32 * i + lane;
          float4 f = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
          if (4 * q + 3 < n) {
            f = __ldg(reinterpret_cast<const float4*>(xr) + q);
          } else if (4 * q < n) {   // the row's last, partial float4: scalar loads of the columns < n only
            f.x = __ldg(xr + 4 * q);
            if (4 * q + 1 < n) f.y = __ldg(xr + 4 * q + 1);
            if (4 * q + 2 < n) f.z = __ldg(xr + 4 * q + 2);
          }
          v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
        }
        fold([&](int i) { const int c = 4 * (q0 + 32 * (i >> 2) + lane) + (i & 3); return c < n ? c : INT_MAX; });
      }
    } else {     // any pitch / alignment: 4-byte loads, lane reads column c0 + 32 i + lane
      for (int c0 = 0; c0 < n; c0 += 32 * kTopkChunk) {
#pragma unroll
        for (int i = 0; i < kTopkChunk; ++i) {
          const int c = c0 + 32 * i + lane;
          v[i] = (c < n) ? __ldg(xr + c) : -INFINITY;
        }
        fold([&](int i) { const int c = c0 + 32 * i + lane; return c < n ? c : INT_MAX; });
      }
    }
    // log-sum-exp of the row from the per-lane (max, sum) pairs
    float M = m;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
    float S = (m > -INFINITY) ? se * expf(m - M) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) S += __shfl_xor_sync(0xffffffffu, S, o);
    const float log_s = logf(S);
    for (int j = 0; j < k; ++j) {
      float bv = tv[0];
      int bc = tc[0];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
        if (topk_before(ov, oc, bv, bc)) { bv = ov; bc = oc; }
      }
      if (tc[0] == bc) {                 // columns are unique within a row: exactly one lane pops its head
#pragma unroll
        for (int i = 0; i + 1 < KMAX; ++i) { tv[i] = tv[i + 1]; tc[i] = tc[i + 1]; }
        tv[KMAX - 1] = -INFINITY;
        tc[KMAX - 1] = INT_MAX;
      }
      if (lane == 0) {
        idx[static_cast<int64_t>(row) * k + j] = bc;
        logp[static_cast<int64_t>(row) * k + j] = (bv - M) - log_s;
      }
    }
  }
}

__global__ void k_situation_finish(const int64_t* __restrict__ verb, const int32_t* __restrict__ role_count,
                                   int n_verbs, int R, int n_cand, const float* __restrict__ verb_logp,
                                   int64_t* __restrict__ labels, float* __restrict__ label_logp,
                                   float* __restrict__ score) {
  for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < n_cand; u += gridDim.x * blockDim.x) {
    int64_t v = verb[u];
    if (v < 0 || v >= n_verbs) v = 0;    // clamped as in the role graph (k_prep_rows raised the flag)
    const int n = role_count[v];
    float s = (verb_logp != nullptr) ? verb_logp[u] : 0.f;
    for (int r = 0; r < R; ++r) {
      const int64_t o = static_cast<int64_t>(u) * R + r;
      if (r < n) {
        s += label_logp[o];
      } else {
        labels[o] = -1;
        label_logp[o] = 0.f;
      }
    }
    score[u] = s;
  }
}

#define SRG_LAUNCH_CHECK()                                                                      \
  do {                                                                                          \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                         \
    cudaError_t _e = cudaGetLastError();                                                        \
    if (_e != cudaSuccess)                                                                      \
      return set_error(SRG_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

}  // namespace

// ------------------------------------------------------------------------------------------------ launchers
int launch_gather_mask(const int32_t* verb2roles, const int32_t* role_count, int n_verbs, int R, const int64_t* verb,
                       int B, int64_t* role_idx, float* mask, int* bad, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  k_gather_mask<<<grid_for(static_cast<int64_t>(B) * R * R), kThreads, 0, s>>>(verb2roles, role_count, n_verbs, R,
                                                                              verb, B, role_idx, mask, bad);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_node_init_verb(const float* feat, int B, int D, float* h32, bf16* hb_hi, bf16* hb_mid, bf16* hb_lo,
                          cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  const int64_t n4 = static_cast<int64_t>(B) * D / 4;
  k_node_init_verb<<<grid_for(n4), kThreads, 0, s>>>(feat, n4, h32, hb_hi, Parts{hb_mid, hb_lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_split_cast(const float* x, int64_t n, bf16* hi, bf16* mid, bf16* lo, cudaStream_t s) {
  if (n <= 0) return SRG_OK;
  k_split_cast<<<grid_for(n / 4), kThreads, 0, s>>>(x, n / 4, hi, Parts{mid, lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_aggregate(const float* h32, const float* mask, int B, int R, int D, bf16* a_hi, bf16* a_mid, bf16* a_lo,
                     cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (R > kMaxR) return set_error(SRG_ERR_UNSUPPORTED, "max_role_count %d > %d", R, kMaxR);
  k_aggregate<<<grid_for(static_cast<int64_t>(B) * D / 4), kThreads, 0, s>>>(h32, mask, B, R, D, a_hi,
                                                                             Parts{a_mid, a_lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_pack_weight_multi(const PackJob* jobs, int n_jobs, int cols, cudaStream_t s) {
  for (int j0 = 0; j0 < n_jobs; j0 += kMaxPackJobs) {
    const int n = (n_jobs - j0 < kMaxPackJobs) ? n_jobs - j0 : kMaxPackJobs;
    PackJobs js;
    for (int i = 0; i < kMaxPackJobs; ++i) js.j[i] = jobs[j0 + (i < n ? i : 0)];
    dim3 grid(296, n);
    k_pack_weight_multi<<<grid, kThreads, 0, s>>>(js, cols);
    SRG_LAUNCH_CHECK();
  }
  return SRG_OK;
}

int launch_pack_bias(const float* a, const float* b, int n, int n_pad, float* dst, cudaStream_t s) {
  k_pack_bias<<<grid_for(n_pad), kThreads, 0, s>>>(a, b, n, n_pad, dst);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_count_targets(const int64_t* gt, int B, int R, int ignore_index, float* counts, cudaStream_t s) {
  SRG_CUDA(cudaMemsetAsync(counts, 0, 3 * sizeof(float), s));
  if (B <= 0) return SRG_OK;
  k_count_targets<<<grid_for(static_cast<int64_t>(B) * 3 * R, kThreads, 148), kThreads, 0, s>>>(gt, B, R, ignore_index,
                                                                                               counts);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_nouns_ce(const float* logits, int64_t ldl, int n_labels, const int64_t* gt, int B, int R,
                    const float* counts, float* loss, float* dlogits, float grad_scale, const float* gscale_dev,
                    const float* stats, int stats_tiles, bf16* dlb, int n_pad, int accumulate, cudaStream_t s) {
  const int rows = B * R;
  if (rows <= 0) return SRG_OK;
  int blocks = (rows + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (stats_tiles > 32) stats = nullptr;
  k_cross_entropy<3><<<blocks, kThreads, 0, s>>>(logits, ldl, n_labels, rows, gt, R, n_labels, counts, 0.f, loss,
                                                dlogits, grad_scale, gscale_dev,
                                                reinterpret_cast<const float2*>(stats), stats_tiles, nullptr, dlb, n_pad,
                                                n_pad, accumulate);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_verb_ce(const float* logits, int64_t ldl, int n_verbs, const int64_t* gt, int B, float inv_batch,
                   float* loss, float* dlogits, float grad_scale, const float* gscale_dev, const float* stats,
                   int stats_tiles, const float* batch_total, bf16* dlb, int n_pad, int accumulate, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  int blocks = (B + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (stats_tiles > 32) stats = nullptr;
  k_cross_entropy<1><<<blocks, kThreads, 0, s>>>(logits, ldl, n_verbs, B, gt, 1, -100, nullptr, inv_batch, loss,
                                                dlogits, grad_scale, gscale_dev,
                                                reinterpret_cast<const float2*>(stats), stats_tiles, batch_total, dlb,
                                                n_pad, n_pad, accumulate);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_row_topk_logsoftmax(const float* x, int64_t ldl, int rows, int n, int k, int64_t* idx, float* logp,
                               cudaStream_t s) {
  if (rows <= 0) return SRG_OK;
  if (k < 1 || k > 16 || n < k || ldl < n)
    return set_error(SRG_ERR_ARG, "topk_logsoftmax: need 1 <= k <= 16, k <= n <= ldl (k=%d, n=%d, ldl=%lld)", k, n,
                     (long long)ldl);
  const int blocks = grid_for(static_cast<int64_t>(rows) * 32);   // one warp per row
  if (k == 1) k_row_topk_logsoftmax<1><<<blocks, kThreads, 0, s>>>(x, ldl, rows, n, k, idx, logp);
  else if (k <= 4) k_row_topk_logsoftmax<4><<<blocks, kThreads, 0, s>>>(x, ldl, rows, n, k, idx, logp);
  else if (k <= 8) k_row_topk_logsoftmax<8><<<blocks, kThreads, 0, s>>>(x, ldl, rows, n, k, idx, logp);
  else k_row_topk_logsoftmax<16><<<blocks, kThreads, 0, s>>>(x, ldl, rows, n, k, idx, logp);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_situation_finish(const int64_t* verb, const int32_t* role_count, int n_verbs, int R, int n_cand,
                            const float* verb_logp, int64_t* labels, float* label_logp, float* score, cudaStream_t s) {
  if (n_cand <= 0) return SRG_OK;
  k_situation_finish<<<grid_for(n_cand), kThreads, 0, s>>>(verb, role_count, n_verbs, R, n_cand, verb_logp, labels,
                                                          label_logp, score);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_cast_pad(const float* src, int64_t ld, int rows, int n_valid, int n_pad, bf16* dst, int accumulate,
                    cudaStream_t s) {
  if (rows <= 0) return SRG_OK;
  if (n_pad % 8 != 0) return set_error(SRG_ERR_ARG, "cast_pad: padded width %d must be a multiple of 8", n_pad);
  k_cast_pad<<<grid_for(static_cast<int64_t>(rows) * n_pad / 8), kThreads, 0, s>>>(src, ld, rows, n_valid, n_pad, dst,
                                                                                   accumulate);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_colsum(const bf16* X, int64_t ld, int rows, int n_cols, float* out1, float scale1, float* out2,
                  float scale2, cudaStream_t s) {
  if (rows <= 0 || n_cols <= 0) return SRG_OK;
  int slabs = (rows + 255) / 256;
  if (slabs > 64) slabs = 64;
  dim3 grid((n_cols + 63) / 64, slabs);
  k_colsum<<<grid, kThreads, 0, s>>>(X, ld, rows, n_cols, out1, scale1, out2, scale2);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_prep_rows(const int32_t* role_count, int n_verbs, int R, const int64_t* verb, int B, int compact,
                     RowMap rm, int* bad, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  k_prep_rows<<<1, 1024, 0, s>>>(role_count, n_verbs, R, verb, B, compact, const_cast<int*>(rm.cnt),
                                 const_cast<int*>(rm.off), const_cast<int*>(rm.meta), bad);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_node_init_noun(const float* feat, const float* role_emb, const float* verb_emb, const int64_t* verb,
                          const int32_t* verb2roles, int n_verbs, int B, int R, int D, RowMap rm, int feat_rep,
                          float* h32, bf16* hb_hi, bf16* hb_mid, bf16* hb_lo, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (R > kMaxR) return set_error(SRG_ERR_UNSUPPORTED, "max_role_count %d > %d", R, kMaxR);
  if (feat_rep < 1) return set_error(SRG_ERR_ARG, "node_init_noun: feat_rep %d < 1", feat_rep);
  k_node_init_noun<<<grid_for(static_cast<int64_t>(B + kSelfRows) * D / 4), kThreads, 0, s>>>(
      feat, role_emb, verb_emb, verb, verb2roles, n_verbs, B, R, D, rm, feat_rep, h32, hb_hi, Parts{hb_mid, hb_lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_aggregate_rows(const float* h32, RowMap rm, int B, int R, int D, bf16* a_hi, bf16* a_mid, bf16* a_lo,
                          cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (R > kMaxR) return set_error(SRG_ERR_UNSUPPORTED, "max_role_count %d > %d", R, kMaxR);
  k_aggregate_rows<<<grid_for(static_cast<int64_t>(B + kSelfRows) * D / 4), kThreads, 0, s>>>(h32, rm, B, R, D, a_hi,
                                                                                            Parts{a_mid, a_lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_aggregate_t_rows(const bf16* da, const bf16* e, RowMap rm, int B, int R, int D, bf16* ada, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (R > kMaxR) return set_error(SRG_ERR_UNSUPPORTED, "max_role_count %d > %d", R, kMaxR);
  const int64_t units = (rm.cnt == nullptr) ? B : B + kSelfRows;
  k_aggregate_t_rows<<<grid_for(units * D / 8), kThreads, 0, s>>>(da, e, rm, B, R, D, ada);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_aggregate_t(const bf16* da, const bf16* e, const float* mask, const bf16* h, int B, int R, int D,
                       bf16* ada, float* dmask, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (R > kMaxR) return set_error(SRG_ERR_UNSUPPORTED, "max_role_count %d > %d", R, kMaxR);
  if (D % 256 != 0) return set_error(SRG_ERR_ARG, "aggregate_t: D=%d must be a multiple of 256", D);
  if (dmask != nullptr) {
    if (h == nullptr) return set_error(SRG_ERR_ARG, "aggregate_t: dmask needs the step's state operand");
    const int blocks = B < 148 * 16 ? B : 148 * 16;
    k_aggregate_t<true><<<blocks, D / 8 < 128 ? D / 8 : 128, 0, s>>>(da, e, mask, h, B, R, D, ada, dmask);
  } else {
    k_aggregate_t<false><<<grid_for(static_cast<int64_t>(B) * D / 8), kThreads, 0, s>>>(da, e, mask, nullptr, B, R, D,
                                                                                       ada, nullptr);
  }
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_classifier_input(const float* h32, RowMap rm, int R, int64_t rows, int D, DropSpec ds, bf16* x_hi,
                            bf16* x_mid, bf16* x_lo, cudaStream_t s) {
  if (rows <= 0) return SRG_OK;
  if (D % 8 != 0) return set_error(SRG_ERR_ARG, "classifier_input: D=%d must be a multiple of 8", D);
  k_classifier_input<<<grid_for(rows * D / 8), kThreads, 0, s>>>(h32, rm, R, rows, D, ds, x_hi, Parts{x_mid, x_lo});
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_classifier_input_bwd(const float* dx, RowMap rm, int B, int R, int D, DropSpec ds, float* dh, GruPre gp,
                                cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  if (D % 8 != 0) return set_error(SRG_ERR_ARG, "classifier_input_bwd: D=%d must be a multiple of 8", D);
  if (rm.meta != nullptr) {   // the shared pad row (and the rest of its tile) is accumulated into: clear it first
    k_zero_self_rows<<<grid_for(static_cast<int64_t>(kSelfRows) * D / 4), kThreads, 0, s>>>(dh, rm, D);
    SRG_LAUNCH_CHECK();
  }
  const int D8 = D / 8;
  const int threads = D8 < kThreads ? D8 : kThreads;
  const int chunks = (D8 + threads - 1) / threads;
  int slabs = (148 * 8) / chunks;
  if (slabs > B) slabs = B;
  if (slabs < 1) slabs = 1;
  dim3 grid(chunks, slabs);
  k_classifier_input_bwd<<<grid, threads, 0, s>>>(dx, rm, B, R, D, ds, dh, gp);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_dropout_mask(DropSpec ds, int64_t rows, int D, uint8_t* out, cudaStream_t s) {
  if (rows <= 0) return SRG_OK;
  if (D % 8 != 0) return set_error(SRG_ERR_ARG, "dropout_mask: D=%d must be a multiple of 8", D);
  k_dropout_mask<<<grid_for(rows * D / 8), kThreads, 0, s>>>(ds, rows, D, out);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_node_init_bwd(const float* dh0, const bf16* h0b, const float* feat, const float* role_emb,
                         const float* verb_emb, const int64_t* verb, const int32_t* verb2roles, int n_verbs,
                         int n_roles, int B, int R, int D, RowMap rm, float* d_role_emb, float* d_verb_emb,
                         float* dfeat, cudaStream_t s) {
  const bool emb = (d_role_emb != nullptr && d_verb_emb != nullptr);
  if (B <= 0 || (!emb && dfeat == nullptr)) return SRG_OK;
  auto kern = emb ? (dfeat ? k_node_init_bwd<true, true> : k_node_init_bwd<true, false>) : k_node_init_bwd<false, true>;
  kern<<<grid_for(static_cast<int64_t>(B) * D / 4), kThreads, 0, s>>>(
      dh0, h0b, feat, role_emb, verb_emb, verb, verb2roles, n_verbs, n_roles, B, R, D, rm, d_role_emb, d_verb_emb,
      dfeat);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_node_init_verb_bwd(const float* dh0, const bf16* h0b, int B, int D, float* dfeat, cudaStream_t s) {
  if (B <= 0) return SRG_OK;
  const int64_t n4 = static_cast<int64_t>(B) * D / 4;
  k_node_init_verb_bwd<<<grid_for(n4), kThreads, 0, s>>>(dh0, h0b, n4, dfeat);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_colsum_multi(const ColsumJob* jobs, int n_jobs, int64_t ld, int rows, const int* rows_dev, int nseg,
                        int64_t seg_stride, int n_cols, cudaStream_t s) {
  if (rows <= 0 || n_cols <= 0 || n_jobs <= 0 || nseg <= 0) return SRG_OK;
  if (n_jobs > 4) return set_error(SRG_ERR_ARG, "colsum_multi: at most 4 jobs");
  ColsumJobs js;
  for (int i = 0; i < 4; ++i) js.j[i] = jobs[i < n_jobs ? i : 0];
  int slabs = (rows + 511) / 512;                 // per segment
  if (slabs * nseg > 40) slabs = 40 / nseg;
  if (slabs < 1) slabs = 1;
  dim3 grid((n_cols + 63) / 64, slabs * nseg, n_jobs);
  k_colsum_multi<<<grid, kThreads, 0, s>>>(js, ld, rows, rows_dev, nseg, seg_stride, n_cols);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_gru_bwd_pre_ld(const float* dh, const bf16* z, const bf16* hc, const bf16* h, int rows, const int* rows_dev,
                          const int* row0_dev, int D, bf16* dpre_z, bf16* dpre_h, int64_t ld_out, float* dh_acc,
                          cudaStream_t s) {
  if (rows <= 0) return SRG_OK;
  k_gru_bwd_pre_ld<<<grid_for(static_cast<int64_t>(rows) * D / 4), kThreads, 0, s>>>(
      dh, z, hc, h, rows, rows_dev, row0_dev, D, dpre_z, dpre_h, ld_out, dh_acc);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_matvec(const float* W, const float* x, int rows, int cols, float* y, cudaStream_t s) {
  k_matvec<<<(rows + 7) / 8, kThreads, 0, s>>>(W, x, rows, cols, y);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_matvec_t_acc3(const float* const W[3], const float* sv, int rows, int cols, float* y, cudaStream_t s) {
  Mat3 m;
  for (int i = 0; i < 3; ++i) { m.W[i] = W[i]; m.dW[i] = nullptr; }
  int slabs = (rows + 31) / 32;
  if (slabs > 128) slabs = 128;
  dim3 grid((cols + kThreads - 1) / kThreads, slabs, 3);
  k_matvec_t_acc3<<<grid, kThreads, 0, s>>>(m, sv, rows, cols, y);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_outer_acc3(const float* sv, const float* b, int rows, int cols, float* const dW[3], bool atomic,
                      cudaStream_t s) {
  if (cols % 4 != 0) return set_error(SRG_ERR_ARG, "outer_acc3: cols=%d must be a multiple of 4", cols);
  Mat3 m;
  for (int i = 0; i < 3; ++i) { m.W[i] = nullptr; m.dW[i] = dW[i]; }
  dim3 grid(grid_for(static_cast<int64_t>(rows) * cols / 4, kThreads, 148 * 8), 3);
  if (atomic) k_outer_acc3<true><<<grid, kThreads, 0, s>>>(m, sv, b, rows, cols);
  else k_outer_acc3<false><<<grid, kThreads, 0, s>>>(m, sv, b, rows, cols);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_pack_bias3(const float* a, const float* b, const float* c, float scale, int n, int n_pad, float* dst,
                      cudaStream_t s) {
  k_pack_bias3<<<grid_for(n_pad), kThreads, 0, s>>>(a, b, c, scale, n, n_pad, dst);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_sumsq(const float* x, int64_t n, float* out, cudaStream_t s) {
  if (n % 4 != 0) return set_error(SRG_ERR_ARG, "sumsq: length %lld must be a multiple of 4", (long long)n);
  SRG_CUDA(cudaMemsetAsync(out, 0, sizeof(float), s));
  if (n <= 0) return SRG_OK;
  k_sumsq<<<grid_for(n / 4, kThreads, 148 * 4), kThreads, 0, s>>>(x, n / 4, out);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_adamax_step(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                       float beta2, float eps, float max_norm, const float* norm_sq, float* step, cudaStream_t s) {
  if (n % 4 != 0) return set_error(SRG_ERR_ARG, "adamax: flat length %lld must be a multiple of 4", (long long)n);
  if (n > 0) {
    k_clip_adamax<<<grid_for(n / 4), kThreads, 0, s>>>(params, grads, exp_avg, exp_inf, n / 4, lr, beta1, beta2, eps,
                                                       max_norm, norm_sq, step);
    SRG_LAUNCH_CHECK();
  }
  k_inc<<<1, 1, 0, s>>>(step);
  SRG_LAUNCH_CHECK();
  return SRG_OK;
}

int launch_clip_adamax(float* params, float* grads, float* exp_avg, float* exp_inf, int64_t n, float lr, float beta1,
                       float beta2, float eps, float max_norm, float* norm_sq, float* step, cudaStream_t s) {
  if (n <= 0) return SRG_OK;
  SRG_TRY(launch_sumsq(grads, n, norm_sq, s));
  return launch_adamax_step(params, grads, exp_avg, exp_inf, n, lr, beta1, beta2, eps, max_norm, norm_sq, step, s);
}

}  // namespace srg
