// Software-pipelined epilogue of the fused GRU kernels (bf16 training instantiations of EPI_ZR, EPI_H, EPI_DH, EPI_DRH).
//
// A CTA tile (128 rows x BLOCK_N columns) is drained in 32-column chunks by the four epilogue warps together.  The
// operands of a chunk live in one "set" of shared memory, one region per tensor:
//   fp32 tensors as [128 rows x 128 B] SWIZZLE_128B boxes (16 KB), bf16 tensors as [128 rows x 64 B] SWIZZLE_64B boxes
//   (8 KB); warp w owns rows [32w, 32w+32) of every region.
// ONE thread (warp 0 of the epilogue group, lane 0) issues every TMA load and store of the CTA, so a chunk costs 2-8
// TMA operations per CTA instead of per warp (40-64 per tile instead of 160-256, against 128 operand boxes of the main
// loop).  Measured against per-warp boxes this is neutral at B=6144 -- the number of TMA operations is not what
// starves the H / DH main loops (profiles/r01_epi_timing.md) -- and, together with the bias values being fetched once
// per tile before the accumulator is waited for, +8 % on the gate kernels of a 768-image shard.
// Two sets ping-pong: the loads of the NEXT chunk (of this tile, or the first chunk of the CTA's next tile) are issued
// before the current chunk is processed; outputs overwrite their inputs in place where shapes match.
#pragma once

namespace srg {

// 16-byte chunk c (0..3) of row r inside a [rows x 64 B] SWIZZLE_64B box: bits [4,5] ^= bits [7,8]
__device__ __forceinline__ uint32_t u64_addr(uint32_t base, int r, int c) {
  return base + r * 64 + ((c ^ ((r >> 1) & 3)) << 4);
}
__device__ __forceinline__ void u64_ld_bf16x8(uint32_t base, int lane, int c, float (&v)[8]) {
  uint32_t u[4];
  lds128(u64_addr(base, lane, c), u[0], u[1], u[2], u[3]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = bf16_lo_f(u[i]);
    v[2 * i + 1] = bf16_hi_f(u[i]);
  }
}
__device__ __forceinline__ void u64_st_bf16x8(uint32_t base, int lane, int c, const float (&v)[8]) {
  sts128(u64_addr(base, lane, c), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]),
         pack_bf16(v[6], v[7]));
}

constexpr int kF32Box = 16384;   // [128 x 32] fp32
constexpr int kB16Box = 8192;    // [128 x 32] bf16
constexpr int kF32Warp = 4096;   // one warp's 32 rows of an fp32 box
constexpr int kB16Warp = 2048;   // one warp's 32 rows of a bf16 box

// Region offsets inside a set (bytes).  fp32 regions first, so that every region base is a multiple of 1024.
//   EPI_ZR : r tiles: [h f32 | rh | r]       z tiles: [z]
//   EPI_H  : [h f32 -> h' f32 | z -> hc | h' bf16]
//   EPI_DH : [dh f32 | z -> dpre_z | hc -> dpre_h | h | add]
//   EPI_DRH: [h -> dpre_r | r -> e]
template <int EPI>
struct PipeTraits {
  static constexpr int kSetBytes = (EPI == EPI_ZR)   ? kF32Box + 2 * kB16Box
                                   : (EPI == EPI_H)  ? kF32Box + 2 * kB16Box
                                   : (EPI == EPI_DH) ? kF32Box + 4 * kB16Box
                                                     : 2 * kB16Box;
};
constexpr int kRegB0 = kF32Box;                // first bf16 region after the fp32 one
constexpr int kRegB1 = kF32Box + kB16Box;
constexpr int kRegB2 = kF32Box + 2 * kB16Box;
constexpr int kRegB3 = kF32Box + 3 * kB16Box;

// Everything the epilogue group needs to know about its place in the kernel.
struct PipeCtx {
  const GemmMaps* maps;
  const GemmArgs* args;
  int lane;
  int ew;   // warp within the epilogue group = TMEM lane quarter
};

// ---- per-EPI: issue the loads of one chunk into set `sp` (one thread per CTA) --------------------------------------
// row0 = first row of the CTA tile
template <int EPI>
__device__ __forceinline__ void pipe_issue(const PipeCtx& c, uint8_t* sp, uint64_t* bar, int n0, int cc, int row0) {
  const GemmMaps& m = *c.maps;
  const GemmArgs& a = *c.args;
  const int gcol = n0 + cc * 32;
  if constexpr (EPI == EPI_ZR) {
    // r-tiles only: io1 = h fp32
    ptx::mbar_arrive_expect_tx(bar, kF32Box);
    ptx::tma_load_2d(&m.io[1], bar, sp, gcol - a.n_split, row0);
  } else if constexpr (EPI == EPI_H) {
    ptx::mbar_arrive_expect_tx(bar, kF32Box + kB16Box);
    ptx::tma_load_2d(&m.io[0], bar, sp, gcol, row0);                   // h fp32
    ptx::tma_load_2d(&m.io[1], bar, sp + kRegB0, gcol, row0);          // z bf16
  } else if constexpr (EPI == EPI_DH) {
    const bool next = (a.flags & FLAG_NEXT) != 0, has_add = (a.flags & FLAG_ADD) != 0;
    ptx::mbar_arrive_expect_tx(bar, kF32Box + (next ? 3 : 0) * kB16Box + (has_add ? kB16Box : 0));
    ptx::tma_load_2d(&m.io[0], bar, sp, gcol, row0);                   // dh_acc fp32
    if (next) {
      ptx::tma_load_2d(&m.io[1], bar, sp + kRegB0, gcol, row0);        // z
      ptx::tma_load_2d(&m.io[2], bar, sp + kRegB1, gcol, row0);        // hc
      ptx::tma_load_2d(&m.io[3], bar, sp + kRegB2, gcol, row0);        // h
    }
    if (has_add) ptx::tma_load_2d(&m.io[6], bar, sp + kRegB3, gcol, row0);
  } else {  // EPI_DRH
    ptx::mbar_arrive_expect_tx(bar, 2 * kB16Box);
    ptx::tma_load_2d(&m.io[0], bar, sp, gcol, row0);                   // h
    ptx::tma_load_2d(&m.io[1], bar, sp + kB16Box, gcol, row0);         // r
  }
}

// ---- per-EPI: compute one chunk (all lanes of all four warps) and write the results into the set -------------------
// s = shared address of the set; breg = this lane's 8 bias values of the tile (columns [8*lane, 8*lane+8) of it).
// Each lane owns one row: 32 columns = 4 groups of 8.  The shared-memory accesses are volatile asm, which the compiler
// keeps in program order, so the code is written in phases -- all loads of a batch of groups, then the math, then the
// stores -- to have the load latencies overlap instead of paying one per group (a single warp per scheduler runs this,
// there is nobody to switch to).  GB = groups per batch (register budget: EPI_DH holds five inputs per element).
template <int EPI>
__device__ __forceinline__ void pipe_compute(const PipeCtx& c, uint32_t s, const float (&acc)[32],
                                             const float (&breg)[8], int cc, bool r_tile) {
  const GemmArgs& a = *c.args;
  const int lane = c.lane;
  const uint32_t sf = s + c.ew * kF32Warp;                       // this warp's rows of the fp32 region (offset 0)
  auto sb = [&](int region_off) -> uint32_t { return s + region_off + c.ew * kB16Warp; };
  if constexpr (EPI == EPI_ZR) {
    float b[4][8];
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int i = 0; i < 8; ++i) b[g][i] = __shfl_sync(0xffffffffu, breg[i], cc * 4 + g);
    if (!r_tile) {   // z = sigmoid(acc + b) -> bf16 in region 0 (bf16 layout)
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float z[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) z[i] = act_sigmoid<false>(acc[g * 8 + i] + b[g][i]);
        u64_st_bf16x8(s + c.ew * kB16Warp, lane, g, z);
      }
    } else {         // r = sigmoid(acc + b); rh = r * h; the stash keeps r folded (gate_fold)
      const bool stash = (a.flags & FLAG_STASH) != 0;
      float h[4][8];
#pragma unroll
      for (int g = 0; g < 4; ++g) slot_ld_f32x8(sf, lane, g, h[g]);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float r[8], rh[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          r[i] = act_sigmoid<false>(acc[g * 8 + i] + b[g][i]);
          rh[i] = r[i] * h[g][i];
        }
        u64_st_bf16x8(sb(kRegB0), lane, g, rh);
        if (stash) {
#pragma unroll
          for (int i = 0; i < 8; ++i) r[i] = gate_fold(r[i]);
          u64_st_bf16x8(sb(kRegB1), lane, g, r);
        }
      }
    }
  } else if constexpr (EPI == EPI_H) {
    float h[4][8], z[4][8];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      slot_ld_f32x8(sf, lane, g, h[g]);
      u64_ld_bf16x8(sb(kRegB0), lane, g, z[g]);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float hc[8], hn[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float bi = __shfl_sync(0xffffffffu, breg[i], cc * 4 + g);
        hc[i] = act_tanh<false>(acc[g * 8 + i] + bi);
        hn[i] = fmaf(z[g][i], hc[i] - h[g][i], h[g][i]);
      }
      slot_st_f32x8(sf, lane, g, hn);                                      // h' fp32, in place
      u64_st_bf16x8(sb(kRegB1), lane, g, hn);                              // h' bf16 operand copy
      if (a.flags & FLAG_STASH) u64_st_bf16x8(sb(kRegB0), lane, g, hc);    // hc over z
    }
  } else if constexpr (EPI == EPI_DH) {
    const bool next = (a.flags & FLAG_NEXT) != 0, has_add = (a.flags & FLAG_ADD) != 0;
#pragma unroll
    for (int g0 = 0; g0 < 4; g0 += 2) {   // two batches of two groups
      float dh[2][8], ad[2][8], z[2][8], hc[2][8], h[2][8];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        slot_ld_f32x8(sf, lane, g0 + j, dh[j]);
        if (has_add) u64_ld_bf16x8(sb(kRegB3), lane, g0 + j, ad[j]);
        if (next) {
          u64_ld_bf16x8(sb(kRegB0), lane, g0 + j, z[j]);
          u64_ld_bf16x8(sb(kRegB1), lane, g0 + j, hc[j]);
          u64_ld_bf16x8(sb(kRegB2), lane, g0 + j, h[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int g = g0 + j;
#pragma unroll
        for (int i = 0; i < 8; ++i) dh[j][i] += acc[g * 8 + i];
        if (has_add) {
#pragma unroll
          for (int i = 0; i < 8; ++i) dh[j][i] += ad[j][i];
        }
        if (next) {
          float dz[8], dc[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            dz[i] = dh[j][i] * (hc[j][i] - h[j][i]) * z[j][i] * (1.0f - z[j][i]);
            dc[i] = dh[j][i] * z[j][i] * (1.0f - hc[j][i] * hc[j][i]);
            dh[j][i] = dh[j][i] * (1.0f - z[j][i]);
          }
          u64_st_bf16x8(sb(kRegB0), lane, g, dz);
          u64_st_bf16x8(sb(kRegB1), lane, g, dc);
        }
        slot_st_f32x8(sf, lane, g, dh[j]);
      }
    }
  } else {  // EPI_DRH (two bf16 regions, no fp32 one)
    const uint32_t s0 = s + c.ew * kB16Warp, s1 = s + kB16Box + c.ew * kB16Warp;
    float h[4][8], r[4][8];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      u64_ld_bf16x8(s0, lane, g, h[g]);
      u64_ld_bf16x8(s1, lane, g, r[g]);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float e[8], dp[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float d = acc[g * 8 + i];
        float rv, rc;
        gate_unfold(r[g][i], rv, rc);     // r and 1 - r from the folded stash
        dp[i] = d * h[g][i] * rv * rc;
        e[i] = d * rv;
      }
      u64_st_bf16x8(s0, lane, g, dp);
      u64_st_bf16x8(s1, lane, g, e);
    }
  }
}

// ---- per-EPI: TMA stores of one chunk (one thread per CTA) ---------------------------------------------------------
template <int EPI>
__device__ __forceinline__ void pipe_store(const PipeCtx& c, uint8_t* sp, int n0, int cc, int row0, bool r_tile) {
  const GemmMaps& m = *c.maps;
  const GemmArgs& a = *c.args;
  const int gcol = n0 + cc * 32;
  if constexpr (EPI == EPI_ZR) {
    if (!r_tile) {
      ptx::tma_store_2d(&m.io[0], sp, gcol, row0);
    } else {
      ptx::tma_store_2d(&m.io[2], sp + kRegB0, gcol - a.n_split, row0);
      if (a.flags & FLAG_STASH) ptx::tma_store_2d(&m.io[4], sp + kRegB1, gcol - a.n_split, row0);
    }
  } else if constexpr (EPI == EPI_H) {
    ptx::tma_store_2d(&m.io[0], sp, gcol, row0);
    ptx::tma_store_2d(&m.io[2], sp + kRegB1, gcol, row0);
    if (a.flags & FLAG_STASH) ptx::tma_store_2d(&m.io[4], sp + kRegB0, gcol, row0);
  } else if constexpr (EPI == EPI_DH) {
    ptx::tma_store_2d(&m.io[0], sp, gcol, row0);
    if (a.flags & FLAG_NEXT) {
      ptx::tma_store_2d(&m.io[4], sp + kRegB0, gcol, row0);
      ptx::tma_store_2d(&m.io[5], sp + kRegB1, gcol, row0);
    }
  } else {
    ptx::tma_store_2d(&m.io[2], sp, gcol, row0);
    ptx::tma_store_2d(&m.io[3], sp + kB16Box, gcol, row0);
  }
}

}  // namespace srg
