// Persistent, warp-specialised tcgen05 GEMM for sm_100a with fused GGNN epilogues.
//
//   D[M,N] = sum_s A_s[M, K_s] * B[N, koff_s : koff_s + K_s]^T        (bf16 operands, fp32 accumulate in TMEM)
//
// * A may be a list of K-segments (each with its own TMA descriptor): this is how the GRU's
//   "concatenated message and state" operands ([m | h], [m | r*h]) and the 3-term bf16 split used for
//   fp32 parity are fed without ever materialising a concatenated matrix.
// * Operands are K-major (row-major, K contiguous: activations x and nn.Linear weights W[out,in]) or
//   MN-major (the transposed view, used by dgrad/wgrad) -- selected at compile time.
// * CG == 2: the two CTAs of a cluster issue ONE tcgen05.mma.cta_group::2 of M=256; each CTA stages its
//   own 128 rows of A and half of the B tile.
// * Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (leader CTA), warp 2 = TMEM allocator,
//   warps 4..7 = epilogue (one TMEM lane quarter each). Accumulators are double-buffered in TMEM so the
//   epilogue of tile i overlaps the main loop of tile i+1.
// * Epilogue I/O goes through TMA (SWIZZLE_128B / SWIZZLE_64B boxes), so no global LSU traffic and no uncoalesced
//   access: per warp [32 rows x 128 B] in the store/logits epilogues, per CTA [128 rows x 32 columns] boxes issued by
//   one thread in the pipelined GRU epilogues (epilogue_pipe.cuh).
#pragma once
#include "ptx.cuh"

namespace srg {

constexpr int kBlockK = 64;     // bf16 elements per k-block = one 128 B swizzle span
constexpr int kUmmaK = 16;
constexpr int kTileM = 128;     // rows per CTA
constexpr int kNumThreads = 256;
constexpr int kEpiWarp0 = 4;
constexpr int kSlotBytes = 4096;  // 32 rows x 128 B
constexpr int kMaxSeg = 12;
constexpr int kMaxAMaps = 6;
constexpr int kMaxIoMaps = 7;

enum EpiKind : int {
  EPI_STORE_BF16 = 0,  // io0 = out hi (bf16); FLAG_LO: io1 = mid, io2 = lo  (3-way bf16 split x = hi + mid + lo)
  EPI_STORE_F32 = 1,   // io0 = out fp32 (FLAG_REDUCE: += via TMA reduce-add)
  EPI_ZR = 2,          // GRU update/reset gates:  z = sig(.), r = sig(.), rh = r*h
  EPI_H = 3,           // GRU candidate + state update: hc = tanh(.), h' = h + z*(hc - h)
  EPI_LOGITS = 4,      // classifier: logits + per-tile row softmax statistics
  EPI_DRH = 5,         // backward: drh = acc; dpre_r = drh*h*r*(1-r); e = drh*r
  EPI_DH = 6,          // backward: g = acc + dh_acc = dL/dh_{t-1}'; fused GRU-gate derivatives of step t-1
};

// FLAG_BK_A: the K coordinate of B follows A's (both operands are row blocks of equally laid out activations: the
// weight-gradient GEMMs over K segments), instead of running contiguously through a packed B
enum : int { FLAG_LO = 1, FLAG_STASH = 2, FLAG_REDUCE = 4, FLAG_NEXT = 8, FLAG_ADD = 16, FLAG_BK_A = 32 };

struct GemmMaps {
  CUtensorMap a[kMaxAMaps];
  CUtensorMap b;
  CUtensorMap io[kMaxIoMaps];
};

struct GemmArgs {
  int M, N;
  // Device-resident problem sizes (nullable).  The compact role-node layout makes the number of node rows a function of
  // the batch's verbs, which for the predicted-verb path only exist on the device: the host sizes descriptors, buffers
  // and the grid for the upper bound and the kernel reads the actual count, so a step needs no host synchronisation and
  // can be replayed from a CUDA graph.
  const int* m_dev;   // rows of D (overrides M; M stays the upper bound the tensor maps were built for)
  const int* k_dev;   // rows of EVERY K segment (overrides seg_kb / total_kb; rounded up to whole k-blocks)
  int nseg;
  int seg_map[kMaxSeg];
  int seg_acol[kMaxSeg];  // start coordinate along K inside the A map (elements)
  int seg_kb[kMaxSeg];    // k-blocks in this segment
  int total_kb;
  int corr_kb_begin;  // F32 instantiations: k-blocks >= this accumulate into the correction accumulator
  int k_splits;
  float alpha;
  const float* bias;  // [N] or nullptr
  float bias_scale;
  int n_split;   // EPI_ZR: first column of the r half
  int n_valid;   // EPI_LOGITS: number of real columns (the rest is padding)
  float* stats;  // EPI_LOGITS: [M][N / BLOCK_N][2] (row max, row sum-exp) per column tile
  int flags;
  // L2 eviction-priority hint of the B operand loads (0 = none).  The host sets evict_last when B is a weight matrix:
  // 16-50 MB that every CTA re-reads for the whole launch while GBs of activations stream through the 126 MB L2
  // (measured: H +4 %, DH +7 %, gate kernel +2 %, step -1.3 %).  evict_first on the epilogue traffic was also tried: it
  // costs the next kernel its L2 hits on what this one just wrote (DRH -6 %).
  unsigned long long b_hint;
#ifdef SRG_EPI_TIMING
  unsigned long long* epi_t;  // debug build: [8 kinds][8] clock counters (see tools/epi_timing.py)
#endif
};

template <int EPI, bool F32>
struct EpiTraits {
  static constexpr int kSlots = (EPI == EPI_STORE_BF16) ? (F32 ? 6 : 2)
                                : (EPI == EPI_STORE_F32) ? 4
                                : (EPI == EPI_ZR)        ? (F32 ? 6 : 4)
                                : (EPI == EPI_H)         ? (F32 ? 7 : 4)
                                : (EPI == EPI_LOGITS)    ? 4
                                : (EPI == EPI_DH)        ? 6
                                                         : 2;   // EPI_DRH
  // bf16 training instantiations of the fused GRU epilogues run the software-pipelined path (epilogue_pipe.cuh)
  static constexpr bool kPipe = !F32 && (EPI == EPI_ZR || EPI == EPI_H || EPI == EPI_DH || EPI == EPI_DRH);
};

template <int CG, int BLOCK_N, int EPI, bool F32>
struct GemmCfg {
  static constexpr int kABytes = kTileM * kBlockK * 2;
  static constexpr int kBBytes = (BLOCK_N / CG) * kBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kEpiBytes = 4 * EpiTraits<EPI, F32>::kSlots * kSlotBytes;
  static constexpr int kBarBytes = 1024;
  static constexpr int kSmemBudget = 232448 - 1024;  // 227 KB minus slack for the 1024 B alignment
  static constexpr int kStagesRaw = (kSmemBudget - kEpiBytes - kBarBytes) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kSmemBytes = kStages * kStageBytes + kEpiBytes + kBarBytes + 1024;
  static constexpr int kTmemCols = 2 * BLOCK_N;
  static_assert(kStages >= 3, "not enough shared memory for the main loop");
  static_assert(kTmemCols <= 512, "accumulators do not fit TMEM");
};

// ------------------------------------------------------------------------------------------------
// activation helpers
template <bool F32>
__device__ __forceinline__ float act_sigmoid(float x) {
  if constexpr (F32) {
    return 1.0f / (1.0f + expf(-x));
  } else {
    // one MUFU op instead of two (ex2 + rcp): sigmoid(x) = 0.5 + 0.5 tanh(x / 2); |error| <= 2.5e-4, below the
    // bf16 rounding of the stored gate (the epilogue warps are issue/latency bound, see profiles/r01_epi_timing.md)
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
    return fmaf(0.5f, t, 0.5f);
  }
}
// The reset gate as the training forward stashes it for the backward: r folded to min(r, 1 - r), negated when r > 1/2
// (r - 1 is exact there, and -0 stands for r = 1).  The backward needs r (1 - r); rebuilt from a bf16 r, 1 - r loses
// its relative precision as r saturates (bf16 values in [0.5, 1) are 2^-8 apart: 1 - r = 0.01 comes back to +-20 %).
// The folded value keeps 1 - r to bf16's 2^-9 plus the 2.5e-4 absolute error of act_sigmoid, at no extra MUFU op.
__device__ __forceinline__ float gate_fold(float r) { return r > 0.5f ? copysignf(1.0f - r, -1.0f) : r; }
__device__ __forceinline__ void gate_unfold(float f, float& g, float& one_minus_g) {
  const bool hi = signbit(f);
  g = hi ? 1.0f + f : f;
  one_minus_g = hi ? -f : 1.0f - f;
}
template <bool F32>
__device__ __forceinline__ float act_tanh(float x) {
  if constexpr (F32) {
    return tanhf(x);
  } else {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
  }
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo_f(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16_hi_f(uint32_t p) { return __uint_as_float(p & 0xFFFF0000u); }

// Swizzle-128B address of 16-byte chunk `c` (0..7) of row `r` (0..31) inside a 4 KB slot.
__device__ __forceinline__ uint32_t slot_addr(uint32_t slot_base, int r, int c) {
  return slot_base + r * 128 + ((c ^ (r & 7)) << 4);
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void lds128(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}

// 8 consecutive fp32 columns [8g, 8g+8) of this lane's row inside a 32-column fp32 slot (g = 0..3).
__device__ __forceinline__ void slot_ld_f32x8(uint32_t slot, int lane, int g, float (&v)[8]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  lds128(slot_addr(slot, lane, 2 * g), u[0], u[1], u[2], u[3]);
  lds128(slot_addr(slot, lane, 2 * g + 1), u[4], u[5], u[6], u[7]);
}
__device__ __forceinline__ void slot_st_f32x8(uint32_t slot, int lane, int g, const float (&v)[8]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  sts128(slot_addr(slot, lane, 2 * g), u[0], u[1], u[2], u[3]);
  sts128(slot_addr(slot, lane, 2 * g + 1), u[4], u[5], u[6], u[7]);
}
// 8 consecutive bf16 columns [8c, 8c+8) of this lane's row inside a 64-column bf16 slot (c = 0..7).
__device__ __forceinline__ void slot_ld_bf16x8(uint32_t slot, int lane, int c, float (&v)[8]) {
  uint32_t u[4];
  lds128(slot_addr(slot, lane, c), u[0], u[1], u[2], u[3]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = bf16_lo_f(u[i]);
    v[2 * i + 1] = bf16_hi_f(u[i]);
  }
}
__device__ __forceinline__ void slot_st_bf16x8(uint32_t slot, int lane, int c, const float (&v)[8]) {
  sts128(slot_addr(slot, lane, c), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]),
         pack_bf16(v[6], v[7]));
}
// 3-way split store: hi = bf16(v), mid = bf16(v - hi), lo = bf16(v - hi - mid)  (24 significant bits in total)
__device__ __forceinline__ void slot_st_bf16x8_split(uint32_t slot_hi, uint32_t slot_mid, uint32_t slot_lo, int lane,
                                                     int c, const float (&v)[8]) {
  uint32_t hi[4], mid[4];
  float r1[8], r2[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    hi[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
    r1[2 * i] = v[2 * i] - bf16_lo_f(hi[i]);
    r1[2 * i + 1] = v[2 * i + 1] - bf16_hi_f(hi[i]);
    mid[i] = pack_bf16(r1[2 * i], r1[2 * i + 1]);
    r2[2 * i] = r1[2 * i] - bf16_lo_f(mid[i]);
    r2[2 * i + 1] = r1[2 * i + 1] - bf16_hi_f(mid[i]);
  }
  sts128(slot_addr(slot_hi, lane, c), hi[0], hi[1], hi[2], hi[3]);
  sts128(slot_addr(slot_mid, lane, c), mid[0], mid[1], mid[2], mid[3]);
  slot_st_bf16x8(slot_lo, lane, c, r2);
}

__device__ __forceinline__ void load_bias8(const float* bias, int col, float scale, float (&b)[8]) {
  if (bias == nullptr) {
#pragma unroll
    for (int i = 0; i < 8; ++i) b[i] = 0.f;
    return;
  }
  const float4 x = __ldg(reinterpret_cast<const float4*>(bias + col));
  const float4 y = __ldg(reinterpret_cast<const float4*>(bias + col + 4));
  b[0] = x.x * scale; b[1] = x.y * scale; b[2] = x.z * scale; b[3] = x.w * scale;
  b[4] = y.x * scale; b[5] = y.y * scale; b[6] = y.z * scale; b[7] = y.w * scale;
}

// Debug build (-DSRG_EPI_TIMING, tools/epi_timing.py): SM-clock breakdown of the pipelined epilogues, summed over all
// epilogue warps per EPI kind: {tiles, chunks, tile total, wait accumulator, wait inputs, wait stores + issue,
// tmem ld + math, store issue}.
#ifdef SRG_EPI_TIMING
#define SRG_T(var) const long long var = clock64()
#define SRG_TACC(i, a, b) tacc_[i] += static_cast<unsigned long long>((b) - (a))
#else
#define SRG_T(var)
#define SRG_TACC(i, a, b)
#endif

}  // namespace srg
#include "epilogue_pipe.cuh"
namespace srg {

// ------------------------------------------------------------------------------------------------
template <int CG, int BLOCK_N, bool A_MN, bool B_MN, int EPI, bool F32>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_kernel(const __grid_constant__ GemmMaps maps, const GemmArgs args) {
  using Cfg = GemmCfg<CG, BLOCK_N, EPI, F32>;
  constexpr int STAGES = Cfg::kStages;
  constexpr int A_BYTES = Cfg::kABytes;
  constexpr int B_BYTES = Cfg::kBBytes;
  constexpr int B_ROWS = BLOCK_N / CG;  // B rows staged by this CTA
  constexpr int SLOTS = EpiTraits<EPI, F32>::kSlots;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (smem_base - ptx::smem_u32(smem_raw));

  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * A_BYTES;
  uint8_t* smem_epi = smem + STAGES * (A_BYTES + B_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + Cfg::kEpiBytes);
  uint64_t* full_bar = bars;                      // [STAGES]  (used in the leader CTA)
  uint64_t* empty_bar = bars + STAGES;            // [STAGES]
  uint64_t* tmem_full_bar = bars + 2 * STAGES;    // [2]
  uint64_t* tmem_empty_bar = bars + 2 * STAGES + 2;  // [2]     (used in the leader CTA)
  uint64_t* epi_in_bar = bars + 2 * STAGES + 4;   // [8] two per epilogue warp (ping-pong input sets)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 12);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  const bool is_leader = (cta_rank == 0);
  const int cluster_id = (CG == 2) ? static_cast<int>(ptx::cluster_id_x()) : static_cast<int>(blockIdx.x);
  const int num_clusters = (CG == 2) ? static_cast<int>(ptx::num_clusters_x()) : static_cast<int>(gridDim.x);

  // work decomposition (the sizes may live on the device, see GemmArgs)
  const int M_rt = (args.m_dev != nullptr) ? __ldg(args.m_dev) : args.M;
  const int seg_kb_rt = (args.k_dev != nullptr) ? (__ldg(args.k_dev) + kBlockK - 1) / kBlockK : 0;
  const int total_kb = (args.k_dev != nullptr) ? seg_kb_rt * args.nseg : args.total_kb;
  const int num_m_tiles = (M_rt + kTileM * CG - 1) / (kTileM * CG);
  const int num_n_tiles = args.N / BLOCK_N;
  const int kb_per_split = (total_kb + args.k_splits - 1) / args.k_splits;
  const int k_splits = (total_kb + kb_per_split - 1) / max(kb_per_split, 1);   // every split owns >= 1 k-block
  const int tiles_mn = num_m_tiles * num_n_tiles;
  const int total_work = tiles_mn * k_splits;

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int i = 0; i < kMaxAMaps; ++i) ptx::prefetch_tmap(&maps.a[i]);
    ptx::prefetch_tmap(&maps.b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], CG);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], CG * 128);
    }
    for (int i = 0; i < 8; ++i) ptx::mbar_init(&epi_in_bar[i], 1);
    ptx::fence_barrier_init();
  }
  if constexpr (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  if (warp == 2) ptx::tmem_alloc<CG>(tmem_ptr_smem, Cfg::kTmemCols);
  ptx::tcgen05_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_smem);

  if (warp == 0) {
    // =========================================================== TMA producer
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = cluster_id; w < total_work; w += num_clusters) {
        const int ks = w / tiles_mn;
        const int nt = (w % tiles_mn) % num_n_tiles;
        const int mt = (w % tiles_mn) / num_n_tiles;
        const int m0 = mt * kTileM * CG + static_cast<int>(cta_rank) * kTileM;
        const int nb0 = nt * BLOCK_N + static_cast<int>(cta_rank) * B_ROWS;
        const int kb_begin = ks * kb_per_split;
        const int kb_end = min(total_kb, kb_begin + kb_per_split);
        // locate the first segment (device-resident K: equally long segments of seg_kb_rt k-blocks)
        int seg = 0, seg_first = 0;
        if (seg_kb_rt != 0) {
          seg = kb_begin / seg_kb_rt;
          seg_first = seg * seg_kb_rt;
        } else {
          while (seg < args.nseg - 1 && kb_begin >= seg_first + args.seg_kb[seg]) {
            seg_first += args.seg_kb[seg];
            ++seg;
          }
        }
        int seg_len = (seg_kb_rt != 0) ? seg_kb_rt : args.seg_kb[seg];
        int seg_col = args.seg_acol[seg];
        const CUtensorMap* amap = &maps.a[args.seg_map[seg]];
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          while (seg < args.nseg - 1 && kb >= seg_first + seg_len) {   // next segment: once per segment, not per k-block
            seg_first += seg_len;
            ++seg;
            seg_len = (seg_kb_rt != 0) ? seg_kb_rt : args.seg_kb[seg];
            seg_col = args.seg_acol[seg];
            amap = &maps.a[args.seg_map[seg]];
          }
          const int ka = seg_col + (kb - seg_first) * kBlockK;
          const int kbcoord = (args.flags & FLAG_BK_A) ? ka : kb * kBlockK;
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
          uint8_t* sa = smem_a + stage * A_BYTES;
          uint8_t* sb = smem_b + stage * B_BYTES;
          if constexpr (CG == 2) {
            if constexpr (!A_MN) {
              ptx::tma_load_2d_pair(amap, &full_bar[stage], sa, ka, m0);
            } else {
#pragma unroll
              for (int g = 0; g < kTileM / 64; ++g)
                ptx::tma_load_2d_pair(amap, &full_bar[stage], sa + g * (kBlockK * 128), m0 + g * 64, ka);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d_pair(&maps.b, &full_bar[stage], sb, kbcoord, nb0, args.b_hint);
            } else {
#pragma unroll
              for (int g = 0; g < B_ROWS / 64; ++g)
                ptx::tma_load_2d_pair(&maps.b, &full_bar[stage], sb + g * (kBlockK * 128), nb0 + g * 64, kbcoord,
                                      args.b_hint);
            }
            if (is_leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2u * (A_BYTES + B_BYTES));
            else ptx::mbar_arrive_cluster(&full_bar[stage], 0);
          } else {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], A_BYTES + B_BYTES);
            if constexpr (!A_MN) {
              ptx::tma_load_2d(amap, &full_bar[stage], sa, ka, m0);
            } else {
#pragma unroll
              for (int g = 0; g < kTileM / 64; ++g)
                ptx::tma_load_2d(amap, &full_bar[stage], sa + g * (kBlockK * 128), m0 + g * 64, ka);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d(&maps.b, &full_bar[stage], sb, kbcoord, nb0, args.b_hint);
            } else {
#pragma unroll
              for (int g = 0; g < B_ROWS / 64; ++g)
                ptx::tma_load_2d(&maps.b, &full_bar[stage], sb + g * (kBlockK * 128), nb0 + g * 64, kbcoord,
                                 args.b_hint);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // =========================================================== MMA issuer (leader CTA only)
    if (is_leader && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(kTileM * CG, BLOCK_N, A_MN, B_MN);
      // K-major: atoms of 8 rows x 128 B, stacked every 1024 B; k-step inside the 128 B span = 32 B.
      // MN-major: 64-element groups every kBlockK*128 B, 8-k atoms every 1024 B; k-step = 16 rows = 2048 B.
      constexpr uint32_t A_LBO = A_MN ? kBlockK * 128 : 0, B_LBO = B_MN ? kBlockK * 128 : 0;
      constexpr uint32_t A_KSTEP = A_MN ? kUmmaK * 128 : kUmmaK * 2, B_KSTEP = B_MN ? kUmmaK * 128 : kUmmaK * 2;
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int w = cluster_id; w < total_work; w += num_clusters, ++iter) {
        const int ks = w / tiles_mn;
        const int kb_begin = ks * kb_per_split;
        const int kb_end = min(total_kb, kb_begin + kb_per_split);
        // F32 (parity) instantiations use the two TMEM accumulators of ONE tile: the leading hi*hi terms go to the
        // first, the small split-correction terms to the second (they are summed in fp32 in the epilogue).  The tensor
        // core truncates when it adds into the accumulator, so keeping the ~2^-9-sized corrections out of the large
        // running sum keeps that bias proportional to K/16 and not to 6K/16.
        const int acc = F32 ? 0 : (iter & 1);
        const uint32_t acc_phase = F32 ? (iter & 1) : ((iter >> 1) & 1);
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1u);
        ptx::tcgen05_fence_after();
        const uint32_t tmem_main = tmem_base + acc * BLOCK_N;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          const bool corr = F32 && kb >= args.corr_kb_begin;
          const uint32_t tmem_d = corr ? tmem_base + BLOCK_N : tmem_main;
          const int first_kb = corr ? args.corr_kb_begin : kb_begin;
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tcgen05_fence_after();
          const uint32_t sa = ptx::smem_u32(smem_a + stage * A_BYTES);
          const uint32_t sb = ptx::smem_u32(smem_b + stage * B_BYTES);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            const uint64_t da = ptx::make_smem_desc(sa + k * A_KSTEP, A_LBO, 1024);
            const uint64_t db = ptx::make_smem_desc(sb + k * B_KSTEP, B_LBO, 1024);
            ptx::umma_bf16<CG>(tmem_d, da, db, idesc, (kb > first_kb || k > 0) ? 1u : 0u);
          }
          ptx::umma_commit<CG>(&empty_bar[stage]);  // frees this smem stage (both CTAs) when the MMAs retire
          if (kb == kb_end - 1) ptx::umma_commit<CG>(&tmem_full_bar[acc]);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= kEpiWarp0) {
    // =========================================================== epilogue warps
    const int ew = warp - kEpiWarp0;  // == warp % 4: TMEM lane quarter
    const uint32_t slot0 = ptx::smem_u32(smem_epi + ew * SLOTS * kSlotBytes);
    auto slot = [&](int i) -> uint32_t { return slot0 + i * kSlotBytes; };
    auto slot_ptr = [&](int i) -> void* { return smem_epi + (ew * SLOTS + i) * kSlotBytes; };
    uint64_t* in_bar = &epi_in_bar[ew * 2];
    uint32_t in_phase = 0;
    int iter = 0;
    int store_set = 0;  // ping-pong for pure store epilogues
    (void)in_bar; (void)in_phase; (void)store_set;

    if constexpr (EpiTraits<EPI, F32>::kPipe) {
      // ---------------------------------------------------------------- software-pipelined path (epilogue_pipe.cuh)
      // The four epilogue warps drain a tile together; `leader` issues every TMA operation of the CTA's epilogue.
      constexpr int NCH = BLOCK_N / 32;
      constexpr int SETB = PipeTraits<EPI>::kSetBytes;
      static_assert(NCH % 2 == 0, "ping-pong sets assume an even number of chunks per tile");
      static_assert(2 * SETB <= Cfg::kEpiBytes, "epilogue sets do not fit their shared-memory region");
      uint8_t* wsm = smem_epi;
      uint64_t* bar2 = &epi_in_bar[0];
      const PipeCtx ctx{&maps, &args, lane, ew};
      const bool leader = (ew == 0 && lane == 0);
      auto epi_sync = [&]() { ptx::named_bar_sync(1, 128); };
      auto row_of = [&](int w_) {   // first row of this CTA's half of the tile
        return ((w_ % tiles_mn) / num_n_tiles) * kTileM * CG + static_cast<int>(cta_rank) * kTileM;
      };
      auto n0_of = [&](int w_) { return ((w_ % tiles_mn) % num_n_tiles) * BLOCK_N; };
      auto needs_in = [&](int n0_) { return EPI != EPI_ZR || n0_ >= args.n_split; };
      int set = 0;
      uint32_t ph = 0;
      bool issued = false;   // the loads of the chunk about to be processed are already in flight
#ifdef SRG_EPI_TIMING
      unsigned long long tacc_[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
      for (int w = cluster_id; w < total_work; w += num_clusters, ++iter) {
        const int row0 = row_of(w), n0 = n0_of(w);
        const int acc = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        const bool active = row0 < M_rt;         // CTA-uniform: TMA clips a partially valid tile itself
        const bool tin = needs_in(n0);
        const bool r_tile = (EPI == EPI_ZR) && tin;
        const uint32_t tacc = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BLOCK_N;
        // this lane's share of the tile's bias (columns [8*lane, 8*lane+8)), fetched while the main loop still runs
        float breg[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if constexpr (EPI == EPI_ZR || EPI == EPI_H) {
          if (active && lane * 8 < BLOCK_N) load_bias8(args.bias, n0 + lane * 8, 1.0f, breg);
        }
        SRG_T(tile_t0);
        if (!active) {
          ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
        } else {
#pragma unroll 1
          for (int cc = 0; cc < NCH; ++cc) {
            uint8_t* sp = wsm + set * SETB;
            // the chunk after this one: next chunk of the tile, or chunk 0 of this CTA's next (active) tile
            int nw = w, ncc = cc + 1;
            bool nvalid = true;
            if (ncc == NCH) {
              nw = w + num_clusters;
              ncc = 0;
              nvalid = (nw < total_work) && (row_of(nw) < M_rt);
            }
            const bool pre = nvalid && needs_in(n0_of(nw));
            SRG_T(c0);
            if (leader && tin && !issued) {   // only the first chunk of a run is not prefetched
              ptx::tma_wait_group_read<0>();
              pipe_issue<EPI>(ctx, sp, &bar2[set], n0, cc, row0);
            }
            SRG_T(c1);
            if (cc == 0) {
              ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
              ptx::tcgen05_fence_after();
            }
            SRG_T(c2);
            if (tin) {
              ptx::mbar_wait(&bar2[set], (ph >> set) & 1u);
              ph ^= (1u << set);
            }
            SRG_T(c3);
            if (leader) {
              if (pre) {     // the other set's last stores were committed one iteration ago
                ptx::tma_wait_group_read<0>();
                pipe_issue<EPI>(ctx, wsm + (set ^ 1) * SETB, &bar2[set ^ 1], n0_of(nw), ncc, row_of(nw));
              } else {
                ptx::tma_wait_group_read<1>();   // this set's stores of two chunks ago
              }
            }
            issued = pre;
            if (!tin) epi_sync();                // output-only chunk: nobody may overwrite the set before that wait
            SRG_T(c4);
            float accv[32];
            ptx::tmem_ld_32x32(tacc + cc * 32, accv);
            ptx::tmem_ld_wait();
            pipe_compute<EPI>(ctx, ptx::smem_u32(sp), accv, breg, cc, r_tile);
            ptx::fence_proxy_async_smem();
            epi_sync();                          // the results of all four warps are in the set
            SRG_T(c5);
            if (leader) {
              pipe_store<EPI>(ctx, sp, n0, cc, row0, r_tile);
              ptx::tma_commit_group();
            }
            SRG_T(c6);
            SRG_TACC(1, 0, 1);
            SRG_TACC(3, c1, c2);
            SRG_TACC(4, c2, c3);
            SRG_TACC(5, c0, c1);
            SRG_TACC(5, c3, c4);
            SRG_TACC(6, c4, c5);
            SRG_TACC(7, c5, c6);
            set ^= 1;
          }
        }
        ptx::tcgen05_fence_before();
        if constexpr (CG == 2) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        else ptx::mbar_arrive(&tmem_empty_bar[acc]);
        SRG_T(tile_t1);
        SRG_TACC(0, 0, 1);
        SRG_TACC(2, tile_t0, tile_t1);
      }
#ifdef SRG_EPI_TIMING
      if (lane == 0 && args.epi_t != nullptr)
        for (int i = 0; i < 8; ++i) atomicAdd(&args.epi_t[EPI * 8 + i], tacc_[i]);
#endif
      if (leader) ptx::tma_wait_group<0>();
      __syncwarp();
    } else
    for (int w = cluster_id; w < total_work; w += num_clusters, ++iter) {
      const int nt = (w % tiles_mn) % num_n_tiles;
      const int mt = (w % tiles_mn) / num_n_tiles;
      const int cta_row0 = mt * kTileM * CG + static_cast<int>(cta_rank) * kTileM;
      const int row0 = cta_row0 + ew * 32;  // first row of this warp
      const int n0 = nt * BLOCK_N;
      const int acc = F32 ? 0 : (iter & 1);
      const uint32_t acc_phase = F32 ? (iter & 1) : ((iter >> 1) & 1);
      // Static M: the tensor maps end at row M, TMA clips partially valid boxes itself and a warp whose rows all lie
      // beyond M has nothing to do.  Device-resident M: the maps cover the allocated upper bound, and every row of a CTA
      // tile that holds at least one valid row is written -- downstream kernels treat the rows up to the tile boundary
      // as defined (zero-gradient "self-loop" rows of the compact role-node layout, see k_prep_rows).
      const bool warp_active = (args.m_dev != nullptr) ? (cta_row0 < M_rt) : (row0 < M_rt);

      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tcgen05_fence_after();
      const uint32_t tacc = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BLOCK_N;
      const bool has_corr = F32 && args.corr_kb_begin < total_kb;
      // 32 accumulator columns of this lane's row (main + correction accumulator in the parity instantiations)
      auto load_acc = [&](int col, float (&v)[32]) {
        ptx::tmem_ld_32x32(tacc + col, v);
        ptx::tmem_ld_wait();
        if constexpr (F32) {
          if (has_corr) {
            float c2[32];
            ptx::tmem_ld_32x32(tacc + BLOCK_N + col, c2);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] += c2[i];
          }
        }
      };

      // per-row softmax statistics (EPI_LOGITS)
      float st_max = -INFINITY, st_sum = 0.f;
      (void)st_max; (void)st_sum;

#pragma unroll 1
      for (int cc = 0; warp_active && cc < BLOCK_N / 64; ++cc) {
        const int gcol = n0 + cc * 64;
        float accv[32];

        if constexpr (EPI == EPI_STORE_BF16) {
          constexpr int kPer = F32 ? 3 : 1;   // the 3-way split output exists only in the F32 instantiation
          const int s_hi = store_set * kPer, s_mid = s_hi + (F32 ? 1 : 0), s_lo = s_hi + (F32 ? 2 : 0);
          if (lane == 0) ptx::tma_wait_group_read<1>();
          __syncwarp();
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            load_acc(cc * 64 + half * 32, accv);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float b[8], v[8];
              load_bias8(args.bias, gcol + half * 32 + g * 8, args.bias_scale, b);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = fmaf(accv[g * 8 + i], args.alpha, b[i]);
              if (F32 && (args.flags & FLAG_LO)) slot_st_bf16x8_split(slot(s_hi), slot(s_mid), slot(s_lo), lane, half * 4 + g, v);
              else slot_st_bf16x8(slot(s_hi), lane, half * 4 + g, v);
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (warp_active) {
              ptx::tma_store_2d(&maps.io[0], slot_ptr(s_hi), gcol, row0);
              if (F32 && (args.flags & FLAG_LO)) {
                ptx::tma_store_2d(&maps.io[1], slot_ptr(s_mid), gcol, row0);
                ptx::tma_store_2d(&maps.io[2], slot_ptr(s_lo), gcol, row0);
              }
            }
            ptx::tma_commit_group();
          }
          store_set ^= 1;
        } else if constexpr (EPI == EPI_STORE_F32) {
          const int s0 = store_set * 2;
          if (lane == 0) ptx::tma_wait_group_read<1>();
          __syncwarp();
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            load_acc(cc * 64 + half * 32, accv);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float b[8], v[8];
              load_bias8(args.bias, gcol + half * 32 + g * 8, args.bias_scale, b);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = fmaf(accv[g * 8 + i], args.alpha, b[i]);
              slot_st_f32x8(slot(s0 + half), lane, g, v);
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (warp_active) {
              if (args.flags & FLAG_REDUCE) {
                ptx::tma_reduce_add_2d(&maps.io[0], slot_ptr(s0), gcol, row0);
                ptx::tma_reduce_add_2d(&maps.io[0], slot_ptr(s0 + 1), gcol + 32, row0);
              } else {
                ptx::tma_store_2d(&maps.io[0], slot_ptr(s0), gcol, row0);
                ptx::tma_store_2d(&maps.io[0], slot_ptr(s0 + 1), gcol + 32, row0);
              }
            }
            ptx::tma_commit_group();
          }
          store_set ^= 1;
        } else if constexpr (EPI == EPI_LOGITS) {
          const int s0 = store_set * 2;
          if (lane == 0) ptx::tma_wait_group_read<1>();
          __syncwarp();
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            load_acc(cc * 64 + half * 32, accv);
            float hmax = -INFINITY;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float b[8], v[8];
              const int c0 = gcol + half * 32 + g * 8;
              load_bias8(args.bias, c0, 1.0f, b);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                v[i] = accv[g * 8 + i] + b[i];
                accv[g * 8 + i] = (c0 + i < args.n_valid) ? v[i] : -INFINITY;
                hmax = fmaxf(hmax, accv[g * 8 + i]);
              }
              slot_st_f32x8(slot(s0 + half), lane, g, v);
            }
            if (hmax > -INFINITY) {
              const float nmax = fmaxf(st_max, hmax);
              float s = 0.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) s += __expf(accv[i] - nmax);
              st_sum = st_sum * __expf(st_max - nmax) + s;
              st_max = nmax;
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (warp_active) {
              ptx::tma_store_2d(&maps.io[0], slot_ptr(s0), gcol, row0);
              ptx::tma_store_2d(&maps.io[0], slot_ptr(s0 + 1), gcol + 32, row0);
            }
            ptx::tma_commit_group();
          }
          store_set ^= 1;
        } else if constexpr (EPI == EPI_ZR) {
          if (n0 < args.n_split) {
            // ---- update gate z = sigmoid(acc + b): io0 (bf16, or fp32 in F32 mode)
            if (lane == 0) ptx::tma_wait_group_read<0>();
            __syncwarp();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              load_acc(cc * 64 + half * 32, accv);
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                float b[8], v[8];
                load_bias8(args.bias, gcol + half * 32 + g * 8, 1.0f, b);
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = act_sigmoid<F32>(accv[g * 8 + i] + b[i]);
                if constexpr (F32) slot_st_f32x8(slot(half), lane, g, v);
                else slot_st_bf16x8(slot(0), lane, half * 4 + g, v);
              }
            }
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (warp_active) {
                if constexpr (F32) {
                  ptx::tma_store_2d(&maps.io[0], slot_ptr(0), gcol, row0);
                  ptx::tma_store_2d(&maps.io[0], slot_ptr(1), gcol + 32, row0);
                } else {
                  ptx::tma_store_2d(&maps.io[0], slot_ptr(0), gcol, row0);
                }
              }
              ptx::tma_commit_group();
            }
          } else {
            // ---- reset gate r = sigmoid(acc + b); rh = r * h.  in: io1 = h (fp32); out: io2 = rh hi, io3/io5 = rh mid/lo,
            //      io4 = r (bf16 stash for the backward pass)
            const int hcol = gcol - args.n_split;
            if (lane == 0) {
              ptx::tma_wait_group_read<0>();
              ptx::mbar_arrive_expect_tx(in_bar, 2 * kSlotBytes);
              ptx::tma_load_2d(&maps.io[1], in_bar, slot_ptr(0), hcol, row0);
              ptx::tma_load_2d(&maps.io[1], in_bar, slot_ptr(1), hcol + 32, row0);
            }
            ptx::mbar_wait(in_bar, in_phase);
            in_phase ^= 1u;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              load_acc(cc * 64 + half * 32, accv);
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                float b[8], r[8], h[8], rh[8];
                load_bias8(args.bias, gcol + half * 32 + g * 8, 1.0f, b);
                slot_ld_f32x8(slot(half), lane, g, h);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  r[i] = act_sigmoid<F32>(accv[g * 8 + i] + b[i]);
                  rh[i] = r[i] * h[i];
                }
                if (args.flags & FLAG_LO) slot_st_bf16x8_split(slot(2), slot(3), slot(5), lane, half * 4 + g, rh);
                else slot_st_bf16x8(slot(2), lane, half * 4 + g, rh);
                if (args.flags & FLAG_STASH) slot_st_bf16x8(slot(4), lane, half * 4 + g, r);
              }
            }
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (warp_active) {
                ptx::tma_store_2d(&maps.io[2], slot_ptr(2), hcol, row0);
                if (args.flags & FLAG_LO) {
                  ptx::tma_store_2d(&maps.io[3], slot_ptr(3), hcol, row0);
                  ptx::tma_store_2d(&maps.io[5], slot_ptr(5), hcol, row0);
                }
                if (args.flags & FLAG_STASH) ptx::tma_store_2d(&maps.io[4], slot_ptr(4), hcol, row0);
              }
              ptx::tma_commit_group();
            }
          }
        } else if constexpr (EPI == EPI_H) {
          // hc = tanh(acc + b); h' = h + z * (hc - h)
          // io0 = h fp32 (read, then overwritten in place with h'), io1 = z (bf16 | fp32 in F32 mode),
          // io2 = h' hi (bf16), io3 / io5 = h' mid / lo (F32 mode), io4 = hc (bf16 stash)
          constexpr int S_H = 0, S_Z = 2, S_HB = F32 ? 4 : 3, S_HM = 5, S_HL = 6;
          if (lane == 0) {
            ptx::tma_wait_group_read<0>();
            ptx::mbar_arrive_expect_tx(in_bar, (F32 ? 4 : 3) * kSlotBytes);
            ptx::tma_load_2d(&maps.io[0], in_bar, slot_ptr(S_H), gcol, row0);
            ptx::tma_load_2d(&maps.io[0], in_bar, slot_ptr(S_H + 1), gcol + 32, row0);
            ptx::tma_load_2d(&maps.io[1], in_bar, slot_ptr(S_Z), gcol, row0);
            if constexpr (F32) ptx::tma_load_2d(&maps.io[1], in_bar, slot_ptr(S_Z + 1), gcol + 32, row0);
          }
          ptx::mbar_wait(in_bar, in_phase);
          in_phase ^= 1u;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            load_acc(cc * 64 + half * 32, accv);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float b[8], h[8], z[8], hc[8], hn[8];
              load_bias8(args.bias, gcol + half * 32 + g * 8, 1.0f, b);
              slot_ld_f32x8(slot(S_H + half), lane, g, h);
              if constexpr (F32) slot_ld_f32x8(slot(S_Z + half), lane, g, z);
              else slot_ld_bf16x8(slot(S_Z), lane, half * 4 + g, z);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                hc[i] = act_tanh<F32>(accv[g * 8 + i] + b[i]);
                hn[i] = fmaf(z[i], hc[i] - h[i], h[i]);
              }
              slot_st_f32x8(slot(S_H + half), lane, g, hn);
              if constexpr (F32) {
                slot_st_bf16x8_split(slot(S_HB), slot(S_HM), slot(S_HL), lane, half * 4 + g, hn);
              } else {
                slot_st_bf16x8(slot(S_HB), lane, half * 4 + g, hn);
                if (args.flags & FLAG_STASH) slot_st_bf16x8(slot(S_Z), lane, half * 4 + g, hc);
              }
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (warp_active) {
              ptx::tma_store_2d(&maps.io[0], slot_ptr(S_H), gcol, row0);
              ptx::tma_store_2d(&maps.io[0], slot_ptr(S_H + 1), gcol + 32, row0);
              ptx::tma_store_2d(&maps.io[2], slot_ptr(S_HB), gcol, row0);
              if constexpr (F32) {
                ptx::tma_store_2d(&maps.io[3], slot_ptr(S_HM), gcol, row0);
                ptx::tma_store_2d(&maps.io[5], slot_ptr(S_HL), gcol, row0);
              }
              else if (args.flags & FLAG_STASH) ptx::tma_store_2d(&maps.io[4], slot_ptr(S_Z), gcol, row0);
            }
            ptx::tma_commit_group();
          }
        }
      }  // column chunks

      // all TMEM reads of this accumulator are complete: hand it back to the MMA warp
      ptx::tcgen05_fence_before();
      if constexpr (CG == 2) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
      else ptx::mbar_arrive(&tmem_empty_bar[acc]);

      if constexpr (EPI == EPI_LOGITS) {
        const int row = row0 + lane;
        if (row < M_rt) {
          float2* st = reinterpret_cast<float2*>(args.stats) + static_cast<size_t>(row) * num_n_tiles + nt;
          *st = make_float2(st_max, st_sum);
        }
      }
    }
    if (lane == 0) ptx::tma_wait_group<0>();
    __syncwarp();
  }

  // teardown
  ptx::tcgen05_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  if (warp == 2) ptx::tmem_dealloc<CG>(tmem_base, Cfg::kTmemCols);
}

}  // namespace srg
