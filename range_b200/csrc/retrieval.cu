// K2 - fused retrieval over the database (reference: range/range.py:213-238).
//
//   S = q16 . Kh^T            (tcgen05.mma kind::f16, fp32 accumulators in TMEM)
//   G = qxyz . xyz^T          (3 FFMA per pair on CUDA cores, fp32: the x40 geo logit needs fp32)
//   RANGE :  P = softmax(15 S)                              O = P V
//   RANGE+:  P = beta softmax(12 S) + (1-beta) softmax(40 G) O = P V     ((1-b) Pg V + b Ps V == (..) V)
//
// The N x M similarity matrix never exists in memory.  Two passes, both streaming the database once.  This file holds
// the kernels for SMALL batches (fewer than 24 query-tile pairs; database split over CTAs to fill the SMs) and the
// geo-skip mask; large batches run the role-specialised kernels of retrieval_pc.cu.
//
//   range_stats_kernel   per query row: sum_j exp(t (s_j - 1)), max_j s_j (and the same for g).  Because
//                        |s|,|g| <= 1 the offset "-1" is a fixed, data-independent softmax max, so partial
//                        results over database splits / ranks merge with plain SUM and MAX.
//   range_apply_kernel   P'(row, j) = 2^(a s + cs_row) + 2^(gam g + cg_row)  in fp16, scaled per row so its
//                        largest entry is <= 2^13 (fp16 range) using the row statistics, then
//                        O(128 x 256 slice) += P' . Vt  on the tensor cores; epilogue rescales.
//
// Shared-memory bandwidth (128 B/clk/SM, shared by TMA writes, UMMA operand reads and LDS/STS) is scarce
// (profiles/r1a_summary.md), so P' never touches it: the softmax warps write it with tcgen05.st over the S
// columns it was computed from (S fp32 -> P' fp16 in place) and P.V runs in TS mode (A operand from TMEM).
// The stats kernel keeps Q in TMEM as well (TS-mode Q.K^T).
//
// TMEM (512 columns): apply  [0,128) S/P buf 0 | [128,256) S/P buf 1 | [256,512) O slice    (Q in smem)
//                     stats  [0,128) Q | [128,256) S buf 0 | [256,384) S buf 1
// CTA = 128 queries (x one 256-wide slice of the 1024 value dims for apply).  Warp roles: warps 0-7
// softmax/epilogue (warp w owns TMEM lanes 32 (w%4)..+31, group w/4 owns half of a tile's key columns),
// warp 8 TMA producer, warp 9 MMA issuer + TMEM allocator.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <cuda.h>
#include <cuda_runtime.h>

#include "ptx.cuh"
#include "range_kernels.h"

namespace {

constexpr int kBlockQ = 128;        // queries per CTA (UMMA M)
constexpr int kSliceV = 256;        // value dims per CTA (UMMA N of P.V)
constexpr int kStageBytes = 32768;  // one pipeline stage: a [.. x 64 fp16] SWIZZLE_128B tile set
constexpr int kNumSoftmaxWarps = 8;
constexpr int kThreads = (kNumSoftmaxWarps + 2) * 32;
// exponentials evaluated on the FMA pipe instead of MUFU (ptx::ex2_poly): every k-th element, 0 = none.
// Measured on B200: any offload is slower (the softmax warps are issue-bound, not MUFU-bound).
#ifndef RANGE_POLY_APPLY
#define RANGE_POLY_APPLY 0
#endif
#ifndef RANGE_POLY_STATS
#define RANGE_POLY_STATS 0
#endif
constexpr int kPolyModApply = RANGE_POLY_APPLY;
constexpr int kPolyModStats = RANGE_POLY_STATS;
constexpr uint32_t kTmemQ = 0;      // column offsets
constexpr uint32_t kTmemS = 128;

template <int NS, int NX, int kXyzBytes>
struct SmemLayout {
  static constexpr int stages = 0;
  static constexpr int xyz = stages + NS * kStageBytes;
  static constexpr int bars = xyz + NX * kXyzBytes;
  static constexpr int b_stage_full = 0;
  static constexpr int b_stage_empty = b_stage_full + NS;
  static constexpr int b_s_full = b_stage_empty + NS;
  static constexpr int b_s_empty = b_s_full + 2;      // stats only
  static constexpr int b_p_full = b_s_empty + 2;      // apply only
  static constexpr int b_xyz_full = b_p_full + 2;
  static constexpr int b_xyz_empty = b_xyz_full + NX;
  static constexpr int b_o_full = b_xyz_empty + NX;
  static constexpr int n_bars = b_o_full + 1;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int red = (tmem_slot + 16 + 15) / 16 * 16;  // stats cross-group reduction scratch
  static constexpr int total = red + kBlockQ * 16;
  static constexpr int dynamic_bytes = total + 1024;  // slack for the manual 1024-B alignment
};

struct PipeState {
  int idx = 0;
  uint32_t phase = 0;
  template <int N>
  __device__ __forceinline__ void advance() {
    if (++idx == N) {
      idx = 0;
      phase ^= 1;
    }
  }
};

__device__ __forceinline__ void named_bar_sync_softmax() {
  asm volatile("bar.sync 1, %0;" ::"n"(kNumSoftmaxWarps * 32) : "memory");
}

// ---------------------------------------------------------------------------------------------------
// K2a: row statistics.  Tile = 128 entries = two 32 KB stages (dims 0-127 | 128-255); Q in TMEM (TS-mode).
// 16 softmax warps (warp w: TMEM lanes 32 (w%4).., 32-entry column group w/4) + producer + MMA issuer.
// The xyz bytes of a tile are credited to the barrier its S tile arrives on (one wait per tile).
// ---------------------------------------------------------------------------------------------------
constexpr int kStatsWarps = 16;
constexpr int kStatsThreads = (kStatsWarps + 2) * 32;
struct StatsSmem {
  static constexpr int NS = 6, kKeys = 128, kXyzBytes = kKeys * 16;
  static constexpr int stages = 0;
  static constexpr int xyz = stages + NS * kStageBytes;            // 2 slots
  static constexpr int bars = xyz + 2 * kXyzBytes;
  static constexpr int b_stage_full = 0;
  static constexpr int b_stage_empty = b_stage_full + NS;
  static constexpr int b_s_full = b_stage_empty + NS;
  static constexpr int b_s_empty = b_s_full + 2;
  static constexpr int b_xyz_empty = b_s_empty + 2;
  static constexpr int n_bars = b_xyz_empty + 2;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int red = (tmem_slot + 16 + 15) / 16 * 16;      // cross-group reduction scratch [3][128] float4
  static constexpr int total = red + 3 * kBlockQ * 16;
  static constexpr int dynamic_bytes = total + 1024;
};

template <bool kGeo>
__global__ void __launch_bounds__(kStatsThreads, 1)
range_stats_kernel(const __grid_constant__ CUtensorMap tmK, const __half* __restrict__ q16,
                   const float4* __restrict__ db_xyz, const float4* __restrict__ q_xyz, int N, int M,
                   int tiles_per_split, float a_sem, float a_geo, float* __restrict__ part_sum,
                   float* __restrict__ part_max, const uint32_t* __restrict__ geo_mask, int mask_words) {
  using L = StatsSmem;
  constexpr int NS = L::NS, kKeys = L::kKeys, kXyzBytes = L::kXyzBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * kBlockQ;
  const int split = blockIdx.y;
  const int total_tiles = (M + kKeys - 1) / kKeys;
  const int t_begin = split * tiles_per_split;
  const int t_end = min(total_tiles, t_begin + tiles_per_split);
  const int T = t_end - t_begin;
  // geo-skip bit of database tile t for this query tile (see geo_mask_kernel); warp-uniform
  const uint32_t* mask_row = (kGeo && geo_mask) ? geo_mask + size_t(blockIdx.x) * mask_words : nullptr;
  auto skip_geo = [&](int t) { return mask_row != nullptr && ((__ldg(mask_row + (t >> 5)) >> (t & 31)) & 1u); };

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(&bars[L::b_stage_full + i], 1);
      ptx::mbar_init(&bars[L::b_stage_empty + i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars[L::b_s_full + i], kGeo ? 2 : 1);     // MMA commit (+ the tile's xyz bytes)
      ptx::mbar_init(&bars[L::b_s_empty + i], kStatsWarps);
      ptx::mbar_init(&bars[L::b_xyz_empty + i], kStatsWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kStatsWarps + 1) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  // warp-uniform copies (see ptx::umma_commit_u32) for the MMA-issuing warp
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
  const uint32_t bars_u = smem_u + L::bars;
  if (warp < kStatsWarps) ptx::load_q_to_tmem16(q16, q0, N, tmem_base + kTmemQ, warp, lane);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();

  if (warp == kStatsWarps) {
    // ===== TMA producer =====
    if (lane == 0) {
      ptx::prefetch_tmap(&tmK);
      PipeState st;
      for (int j = 0; j < T; ++j) {
        const int key0 = (t_begin + j) * kKeys;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          ptx::mbar_wait(&bars[L::b_stage_empty + st.idx], st.phase ^ 1);
          uint8_t* dst = smem + L::stages + st.idx * kStageBytes;
          ptx::mbar_expect_tx(&bars[L::b_stage_full + st.idx], kStageBytes);
          ptx::tma_load_2d(dst, &tmK, &bars[L::b_stage_full + st.idx], (2 * half) * 64, key0);
          ptx::tma_load_2d(dst + 16384, &tmK, &bars[L::b_stage_full + st.idx], (2 * half + 1) * 64, key0);
          st.advance<NS>();
        }
        if (kGeo) {      // xyz(j) -> slot j&1 (free once the softmax warps are done with tile j-2), last in the iteration
          ptx::mbar_wait(&bars[L::b_xyz_empty + (j & 1)], ((j >> 1) & 1) ^ 1);
          if (skip_geo(t_begin + j)) {
            ptx::mbar_arrive(&bars[L::b_s_full + (j & 1)]);                       // nothing to load for this tile
          } else {
            ptx::mbar_expect_tx(&bars[L::b_s_full + (j & 1)], kXyzBytes);
            ptx::bulk_load_1d(smem + L::xyz + (j & 1) * kXyzBytes, db_xyz + key0, kXyzBytes, &bars[L::b_s_full + (j & 1)]);
          }
        }
      }
    }
  } else if (warp == kStatsWarps + 1) {
    // ===== MMA issuer: S[b] = Q (TMEM) . K^T =====
    constexpr uint32_t idesc = ptx::umma_idesc_f16(kBlockQ, kKeys);
    PipeState st;
    for (int j = 0; j < T; ++j) {
      const int b = j & 1;
      ptx::mbar_wait(&bars[L::b_s_empty + b], ((j >> 1) & 1) ^ 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        ptx::mbar_wait(&bars[L::b_stage_full + st.idx], st.phase);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t b_base = smem_u + L::stages + st.idx * kStageBytes;
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              ptx::umma_f16_ts(tmem_base + kTmemS + b * kKeys, tmem_base + kTmemQ + (2 * half + c) * 32 + kk * 8,
                               ptx::umma_desc_kmajor_sw128(b_base + c * 16384 + kk * 32), idesc, (half | c | kk) != 0);
          ptx::umma_commit_u32(bars_u + 8 * (L::b_stage_empty + st.idx));
        }
        __syncwarp();
        st.advance<NS>();
      }
      if (ptx::elect_one()) ptx::umma_commit_u32(bars_u + 8 * (L::b_s_full + b));
      __syncwarp();
    }
  } else {
    // ===== softmax statistics =====
    const int grp = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int n = q0 + row;
    float4 qx = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kGeo && n < N) qx = q_xyz[n];
    const float gx = qx.x * a_geo, gy = qx.y * a_geo, gz = qx.z * a_geo;
    float sum_s = 0.f, sum_g = 0.f, max_s = -2.f, max_g = -3.0e38f;
    for (int j = 0; j < T; ++j) {
      const int b = j & 1;
      const int key0 = (t_begin + j) * kKeys + grp * 32;
      ptx::mbar_wait(&bars[L::b_s_full + b], (j >> 1) & 1);      // S(j) in TMEM and xyz(j) in smem
      ptx::tc_fence_after();
      uint32_t s0[32];
      ptx::tmem_ld32(tmem_base + (uint32_t(quarter * 32) << 16) + kTmemS + b * kKeys + grp * 32, s0);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars[L::b_s_empty + b]);
      const uint32_t kxyz = ptx::smem_u32(smem + L::xyz + b * kXyzBytes) + grp * 32 * 16;
      const int nvalid = M - key0;            // >= 32 except in the last tile
      const bool with_geo = kGeo && !skip_geo(t_begin + j);
      // the geo part is selected per TILE (warp-uniform): two straight-line bodies, no branch inside the unrolled loop
      auto body = [&](auto masked, auto geo) {
        constexpr bool kM = decltype(masked)::value, kG = decltype(geo)::value;
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float sv[2], gv[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float s = __uint_as_float(s0[i + u]);
            const bool valid = !kM || (i + u < nvalid);
            float es = ptx::ex2(fmaf(s, a_sem, -a_sem));
            if (!valid) es = 0.f;
            sum_s += es;
            sv[u] = valid ? s : -2.f;
            if (kG) {
              const float4 k = ptx::lds_f4(kxyz + (i + u) * 16);
              const float g = fmaf(gx, k.x, fmaf(gy, k.y, fmaf(gz, k.z, -a_geo)));   // a_geo (g - 1)
              float eg = ptx::ex2(g);
              if (!valid) eg = 0.f;
              sum_g += eg;
              gv[u] = valid ? g : -3.0e38f;
            }
          }
          max_s = ptx::max3(max_s, sv[0], sv[1]);
          if (kG) max_g = ptx::max3(max_g, gv[0], gv[1]);
        }
      };
      if (nvalid >= 32) {
        if (with_geo) body(std::false_type{}, std::true_type{}); else body(std::false_type{}, std::false_type{});
      } else {
        if (with_geo) body(std::true_type{}, std::true_type{}); else body(std::true_type{}, std::false_type{});
      }
      if (kGeo) {
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&bars[L::b_xyz_empty + b]);
      }
    }
    // combine the four column groups, write this split's partials
    float4* red = reinterpret_cast<float4*>(smem + L::red);
    if (grp > 0) red[(grp - 1) * kBlockQ + row] = make_float4(sum_s, sum_g, max_s, max_g);
    asm volatile("bar.sync 1, %0;" ::"n"(kStatsWarps * 32) : "memory");
    if (grp == 0 && n < N) {
#pragma unroll
      for (int g2 = 0; g2 < 3; ++g2) {
        const float4 o = red[g2 * kBlockQ + row];
        sum_s += o.x;
        sum_g += o.y;
        max_s = fmaxf(max_s, o.z);
        max_g = fmaxf(max_g, o.w);
      }
      // max_g holds a_geo (g - 1); store the raw cosine
      const float raw_g = kGeo ? (max_g / a_geo + 1.f) : 0.f;
      float2* ps = reinterpret_cast<float2*>(part_sum) + size_t(split) * N + n;
      float2* pm = reinterpret_cast<float2*>(part_max) + size_t(split) * N + n;
      *ps = make_float2(sum_s, sum_g);
      *pm = make_float2(max_s, raw_g);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kStatsWarps + 1) ptx::tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------
// K2b: apply  (O slice = P' . Vt).  Tile = 128 entries.  SS-mode Q.K^T with Q resident in shared memory,
// TS-mode P.V with P' in TMEM.  Measured dead ends: a 64-entry tile with Q in TMEM
// (a TS-mode MMA fetches its 128x16 A tile from TMEM in ~64 clk, which dominates UMMA_N = 64), sharing P'
// between the four value-slice CTAs over DSMEM (9 B/clk/SM with the whole chip active).
// rowc[n] = {cs, cg, qx*a_geo, qy*a_geo, qz*a_geo, out_scale, -, -}
// ---------------------------------------------------------------------------------------------------
// kProf: per-role wait-cycle accounting for tools/time_apply.py (prof[role * 8 + counter], CTA (0,1,0) only)
#define PROF_T0() long long _t0 = kProf ? clock64() : 0
#define PROF_ADD(role, k) do { if (kProf && prof_on) { long long _t1 = clock64(); prof_acc[k] += _t1 - _t0; _t0 = _t1; } } while (0)
struct ApplySmem {
  static constexpr int NS = 4, NX = 4, kKeys = 128, kXyzBytes = kKeys * 16;
  static constexpr int q = 0;                                   // 4 x [128 rows x 64 dims] SW128
  static constexpr int stages = q + 65536;
  static constexpr int xyz = stages + NS * kStageBytes;
  static constexpr int bars = xyz + NX * kXyzBytes;
  static constexpr int b_q_full = 0;
  static constexpr int b_stage_full = 1;
  static constexpr int b_stage_empty = b_stage_full + NS;
  static constexpr int b_s_full = b_stage_empty + NS;
  static constexpr int b_p_full = b_s_full + 2;
  static constexpr int b_xyz_full = b_p_full + 2;
  static constexpr int b_xyz_empty = b_xyz_full + NX;
  static constexpr int b_o_full = b_xyz_empty + NX;
  static constexpr int n_bars = b_o_full + 1;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16;
  static constexpr int dynamic_bytes = total + 1024;
};

// ---------------------------------------------------------------------------------------------------
// CTA pairs (cta_group::2): two CTAs of a cluster = two adjacent query tiles x the same value slice run ONE
// 256-row UMMA.  Each CTA loads only half of every B tile (64 of the 128 entries of a K tile,
// 128 of the 256 value dims of a Vt tile), which halves TMA writes and UMMA B-operand reads per SM - the
// shared-memory bandwidth that bounds the single-CTA kernel - and doubles the pipeline depth in tiles.
// Leader (cluster rank 0) issues every MMA; completions are multicast to both CTAs' barriers; the peer's
// softmax warps signal "P' ready" on the leader's barrier through DSMEM.
// ---------------------------------------------------------------------------------------------------
struct PairSmem : ApplySmem {
  static constexpr int b_q_pair = ApplySmem::n_bars;
  static constexpr int n_bars2 = b_q_pair + 1;
  static constexpr int tmem_slot = ApplySmem::bars + n_bars2 * 8;
  static constexpr int total = tmem_slot + 16;
  static constexpr int dynamic_bytes = total + 1024;
};

// 16 softmax warps (4 per SM sub-partition; warp w owns TMEM lanes 32 (w%4).. and the 32-entry column group
// w/4 of every tile) keep the MUFU pipe - the RANGE+ bottleneck: 2 ex2 per pair, 16/clk/SM - fed.  Measured
// alternatives: two 8-warp sets ping-ponging over tiles (same speed: one set alone cannot saturate MUFU) and
// evaluating part of the exponentials on the FMA pipe (slower: register spills under the 112-register cap).
// Per tile a warp passes ONE barrier: the entries' xyz bytes are credited to the same mbarrier the MMA
// completion arrives on.  (Prefetching S(j+1) into a second register array was measured slower: spills.)
constexpr int kPairSoftmaxWarps = 16;
constexpr int kPairThreads = (kPairSoftmaxWarps + 2) * 32;

template <bool kGeo, bool kProf = false>
__global__ void __launch_bounds__(kPairThreads, 1)
range_apply_pair_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK64,
                        const __grid_constant__ CUtensorMap tmV128, const float4* __restrict__ db_xyz,
                        const float4* __restrict__ rowc, int N, int M, int tiles_per_split, float a_sem,
                        float* __restrict__ out, size_t out_split_stride, const uint32_t* __restrict__ geo_mask,
                        int mask_words, long long* __restrict__ prof = nullptr) {
  using L = PairSmem;
  constexpr int NS = L::NS, NX = L::NX, kKeys = L::kKeys, kXyzBytes = L::kXyzBytes;
  long long prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const bool prof_on = kProf && prof != nullptr && blockIdx.x == 2 && blockIdx.y == 0 && blockIdx.z == 0;
  const long long prof_start = kProf ? clock64() : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int slice = blockIdx.y;
  const int q0 = blockIdx.x * kBlockQ;          // cluster = (2,1,1): blockIdx.x = 2 * pair + rank
  const int split = blockIdx.z;
  const int total_tiles = (M + kKeys - 1) / kKeys;
  const int t_begin = split * tiles_per_split;
  const int t_end = min(total_tiles, t_begin + tiles_per_split);
  const int T = t_end - t_begin;
  // geo-skip bit of database tile t for THIS CTA's query tile (see geo_mask_kernel); warp-uniform
  const uint32_t* mask_row = (kGeo && geo_mask) ? geo_mask + size_t(blockIdx.x) * mask_words : nullptr;
  auto skip_geo = [&](int t) { return mask_row != nullptr && ((__ldg(mask_row + (t >> 5)) >> (t & 31)) & 1u); };

  if (threadIdx.x == 0) {
    ptx::mbar_init(&bars[L::b_q_full], 1);
    ptx::mbar_init(&bars[L::b_q_pair], 2);
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(&bars[L::b_stage_full + i], 1);
      ptx::mbar_init(&bars[L::b_stage_empty + i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars[L::b_s_full + i], kGeo ? 2 : 1);            // MMA commit (+ this CTA's xyz bytes)
      ptx::mbar_init(&bars[L::b_p_full + i], 2 * kPairSoftmaxWarps);  // 16 warps x 2 CTAs
    }
    for (int i = 0; i < 2; ++i) ptx::mbar_init(&bars[L::b_xyz_empty + i], kPairSoftmaxWarps);
    ptx::mbar_init(&bars[L::b_o_full], 1);
    ptx::fence_mbar_init();
  }
  if (warp == kPairSoftmaxWarps + 1) ptx::tmem_alloc_2sm<512>(tmem_slot);
  ptx::tc_fence_before();
  ptx::cluster_sync();                           // barriers of BOTH CTAs initialised before any remote arrive
  ptx::tc_fence_after();
  // warp-uniform copies (see ptx::umma_commit_u32) for the MMA-issuing warp
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
  const uint32_t bars_u = smem_u + L::bars;         // [0,128) S/P buf 0 | [128,256) S/P buf 1 | [256,512) O
  const uint32_t tmem_o = tmem_base + 256;

  if (warp == kPairSoftmaxWarps) {
    // ===== TMA producer (both CTAs): own Q; own half of K(j) / Vt(j); bytes credited to the leader =====
    if (lane == 0 && T > 0) {
      ptx::prefetch_tmap(&tmQ);
      ptx::prefetch_tmap(&tmK64);
      ptx::prefetch_tmap(&tmV128);
      ptx::mbar_expect_tx(&bars[L::b_q_full], 65536);
      for (int c = 0; c < 4; ++c) ptx::tma_load_2d(smem + L::q + c * 16384, &tmQ, &bars[L::b_q_full], c * 64, q0);
      PipeState st;
      for (int j = 0; j <= T; ++j) {
        if (j < T) {
          const int key0 = (t_begin + j) * kKeys;
          PROF_T0();
          ptx::mbar_wait(&bars[L::b_stage_empty + st.idx], st.phase ^ 1);
          PROF_ADD(0, 0);
          uint8_t* dst = smem + L::stages + st.idx * kStageBytes;
          if (leader) ptx::mbar_expect_tx(&bars[L::b_stage_full + st.idx], 2 * kStageBytes);
#pragma unroll
          for (int c = 0; c < 4; ++c)     // this CTA's 64 entries x 256 dims, as 4 [64 x 64] boxes
            ptx::tma_load_2d_2sm(dst + c * 8192, &tmK64, &bars[L::b_stage_full + st.idx], c * 64, key0 + int(rank) * 64);
          st.advance<NS>();
        }
        if (j >= 1) {
          const int key0 = (t_begin + j - 1) * kKeys;
          PROF_T0();
          ptx::mbar_wait(&bars[L::b_stage_empty + st.idx], st.phase ^ 1);
          PROF_ADD(0, 1);
          uint8_t* dst = smem + L::stages + st.idx * kStageBytes;
          if (leader) ptx::mbar_expect_tx(&bars[L::b_stage_full + st.idx], 2 * kStageBytes);
#pragma unroll
          for (int h = 0; h < 2; ++h)     // this CTA's 128 value dims x 128 entries, as 2 [128 x 64] boxes
            ptx::tma_load_2d_2sm(dst + h * 16384, &tmV128, &bars[L::b_stage_full + st.idx], key0 + h * 64,
                                 slice * kSliceV + int(rank) * 128);
          st.advance<NS>();
        }
        if (kGeo && j < T) {
          // xyz(j) -> slot j&1, bytes credited to s_full[j&1] (the barrier S(j) arrives on).  Issued LAST in the
          // iteration: the slot frees only when softmax(j-2) is done, and nothing the MMA warp is about to need
          // may queue behind that wait.
          ptx::mbar_wait(&bars[L::b_xyz_empty + (j & 1)], ((j >> 1) & 1) ^ 1);
          if (skip_geo(t_begin + j)) {
            ptx::mbar_arrive(&bars[L::b_s_full + (j & 1)]);                       // nothing to load for this tile
          } else {
            ptx::mbar_expect_tx(&bars[L::b_s_full + (j & 1)], kXyzBytes);
            ptx::bulk_load_1d(smem + L::xyz + (j & 1) * kXyzBytes, db_xyz + (t_begin + j) * kKeys, kXyzBytes,
                              &bars[L::b_s_full + (j & 1)]);
          }
        }
      }
      if (prof_on) { prof[0] = prof_acc[0]; prof[1] = prof_acc[1]; prof[2] = clock64() - prof_start; }
    }
  } else if (warp == kPairSoftmaxWarps + 1) {
    if (T > 0) {
      // both CTAs: tell the leader when this CTA's Q tile has landed
      ptx::mbar_wait(&bars[L::b_q_full], 0);
      if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars[L::b_q_pair]), 0));
      __syncwarp();
    }
    if (leader && T > 0) {
      // ===== MMA issuer (leader only) =====
      constexpr uint32_t idesc_qk = ptx::umma_idesc_f16(2 * kBlockQ, kKeys);
      constexpr uint32_t idesc_pv = ptx::umma_idesc_f16(2 * kBlockQ, kSliceV);
      ptx::mbar_wait_cluster(&bars[L::b_q_pair], 0);
      PipeState st;
      for (int j = 0; j <= T; ++j) {
        if (j < T) {
          const uint32_t tmem_s = tmem_base + (j & 1) * kKeys;
          PROF_T0();
          ptx::mbar_wait(&bars[L::b_stage_full + st.idx], st.phase);
          PROF_ADD(1, 0);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t b_base = smem_u + L::stages + st.idx * kStageBytes;
            const uint32_t a_base = smem_u + L::q;
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                ptx::umma_f16_ss_2sm(tmem_s, ptx::umma_desc_kmajor_sw128(a_base + c * 16384 + kk * 32),
                                     ptx::umma_desc_kmajor_sw128(b_base + c * 8192 + kk * 32), idesc_qk, (c | kk) != 0);
            ptx::umma_commit_2sm_u32(bars_u + 8 * (L::b_stage_empty + st.idx));
            ptx::umma_commit_2sm_u32(bars_u + 8 * (L::b_s_full + (j & 1)));
          }
          __syncwarp();
          PROF_ADD(1, 1);
          st.advance<NS>();
        }
        if (j >= 1) {
          const int jj = j - 1, b = jj & 1;
          PROF_T0();
          ptx::mbar_wait_cluster(&bars[L::b_p_full + b], (jj >> 1) & 1);
          PROF_ADD(1, 2);
          ptx::mbar_wait(&bars[L::b_stage_full + st.idx], st.phase);
          PROF_ADD(1, 3);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t b_base = smem_u + L::stages + st.idx * kStageBytes;
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                // P'(jj): column group g = 32 entries, written as 16 packed columns at S-buffer column 32 g
                ptx::umma_f16_ts_2sm(tmem_o, tmem_base + b * kKeys + (2 * h + (kk >> 1)) * 32 + (kk & 1) * 8,
                                     ptx::umma_desc_kmajor_sw128(b_base + h * 16384 + kk * 32), idesc_pv,
                                     (jj > 0) || (h | kk) != 0);
            ptx::umma_commit_2sm_u32(bars_u + 8 * (L::b_stage_empty + st.idx));
          }
          __syncwarp();
          PROF_ADD(1, 4);
          st.advance<NS>();
        }
      }
      if (ptx::elect_one()) ptx::umma_commit_2sm_u32(bars_u + 8 * (L::b_o_full));
      __syncwarp();
      if (prof_on && lane == 0) { for (int k = 0; k < 5; ++k) prof[8 + k] = prof_acc[k]; prof[8 + 5] = clock64() - prof_start; }
    }
  } else {
    // ===== softmax: S (TMEM fp32) -> P' (TMEM fp16, in place) ; then epilogue =====
    const int grp = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int n = q0 + row;
    float cs = -INFINITY, cg = -INFINITY, gx = 0.f, gy = 0.f, gz = 0.f, out_scale = 0.f;
    if (n < N) {
      const float4 c0 = rowc[2 * n], c1 = rowc[2 * n + 1];
      cs = c0.x; cg = c0.y; gx = c0.z; gy = c0.w; gz = c1.x; out_scale = c1.y;
    }
    const uint32_t p_full_leader[2] = {ptx::mapa(ptx::smem_u32(&bars[L::b_p_full]), 0),
                                       ptx::mapa(ptx::smem_u32(&bars[L::b_p_full + 1]), 0)};
    const uint32_t lane_col = (uint32_t(quarter * 32) << 16) + grp * 32;
    for (int j = 0; j < T; ++j) {
      const int b = j & 1;
      const uint32_t taddr = tmem_base + lane_col + b * kKeys;
      uint32_t cur[32];
      PROF_T0();
      ptx::mbar_wait(&bars[L::b_s_full + b], (j >> 1) & 1);      // S(j) in TMEM and xyz(j) in smem
      ptx::tc_fence_after();
      ptx::tmem_ld32(taddr, cur);
      PROF_ADD(2, 0);
      ptx::tmem_ld_wait();
      PROF_ADD(2, 1);
      const int key0 = (t_begin + j) * kKeys + grp * 32;
      const uint32_t kxyz = ptx::smem_u32(smem + L::xyz + b * kXyzBytes) + grp * 32 * 16;
      const int nvalid = M - key0;            // >= 32 except in the last tile
      const bool with_geo = kGeo && !skip_geo(t_begin + j);
      uint32_t packed[16];
      // the geo part is selected per TILE (warp-uniform): separate straight-line bodies
      auto body = [&](auto masked, auto geo) {
        constexpr bool kM = decltype(masked)::value, kG = decltype(geo)::value;
#pragma unroll
        for (int w = 0; w < 16; ++w) {
          float pv[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int i = 2 * w + u;
            float p = ptx::ex2(fmaf(__uint_as_float(cur[i]), a_sem, cs));
            if (kG) {
              const float4 k = ptx::lds_f4(kxyz + i * 16);
              p += ptx::ex2(fmaf(gx, k.x, fmaf(gy, k.y, fmaf(gz, k.z, cg))));
            }
            if (kM && i >= nvalid) p = 0.f;
            pv[u] = p;
          }
          packed[w] = ptx::pack_half2(pv[0], pv[1]);
        }
      };
      if (nvalid >= 32) {
        if (with_geo) body(std::false_type{}, std::true_type{}); else body(std::false_type{}, std::false_type{});
      } else {
        if (with_geo) body(std::true_type{}, std::true_type{}); else body(std::true_type{}, std::false_type{});
      }
      PROF_ADD(2, 3);
      // P'(row, 32 entries) as 16 packed columns over the first half of the 32 S columns it came from
      ptx::tmem_st16(taddr, packed);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        // the leader's MMA warp waits for both CTAs; the payload is in TMEM, so no memory release is needed
        if (leader) ptx::mbar_arrive(&bars[L::b_p_full + b]);
        else ptx::mbar_arrive_cluster_relaxed(p_full_leader[b]);
        if (kGeo) ptx::mbar_arrive(&bars[L::b_xyz_empty + b]);
      }
      PROF_ADD(2, 4);
    }
    if (prof_on && threadIdx.x == 0) { for (int k = 0; k < 5; ++k) prof[16 + k] = prof_acc[k]; prof[16 + 5] = clock64() - prof_start; prof[16 + 6] = T; }
    if (T > 0) {
      ptx::mbar_wait(&bars[L::b_o_full], 0);
      ptx::tc_fence_after();
      float* orow = out + size_t(split) * out_split_stride + size_t(n) * 1024 + slice * kSliceV + grp * 64;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        uint32_t v[32];
        ptx::tmem_ld32(tmem_o + (uint32_t(quarter * 32) << 16) + grp * 64 + cc * 32, v);
        ptx::tmem_ld_wait();
        if (n < N) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float4 o;
            o.x = __uint_as_float(v[i]) * out_scale;
            o.y = __uint_as_float(v[i + 1]) * out_scale;
            o.z = __uint_as_float(v[i + 2]) * out_scale;
            o.w = __uint_as_float(v[i + 3]) * out_scale;
            *reinterpret_cast<float4*>(orow + cc * 32 + i) = o;
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync();                           // neither CTA may free TMEM / exit while the pair is in flight
  if (warp == kPairSoftmaxWarps + 1) ptx::tmem_dealloc_2sm<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------
// Geographic tile skipping.  The geo weight of an entry is exp(T (g - 1)) / l_g with l_g >= exp(T (g_max - 1)),
// so an entry with g <= g_max - D carries at most exp(-T D) of the row's normaliser; with
// D = (ln M_total + 24 ln 2) / T every such entry of the WHOLE database together is < 2^-24 relative - below
// fp32 resolution.  When the database is stored in a spatially sorted order (range_b200/database.py) and the
// queries of a tile are close to each other (rasters; range.py sorts scattered queries), whole 128-entry
// tiles satisfy the bound for all 128 queries and skip the geo exponential, its 3 FFMA and the xyz load.
// caps[t] = (unit centre, angular radius) of database tile t.  mask bit (qtile, t) = 1 -> skip.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block128_reduce(float v, bool is_max, float* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float w = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, w) : v + w;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  const float a = scratch[0], b = scratch[1], c = scratch[2], d = scratch[3];
  return is_max ? fmaxf(fmaxf(a, b), fmaxf(c, d)) : (a + b) + (c + d);
}

// Once the statistics pass has run, the row normalisers l_g are KNOWN (sums[n].y = sum_j exp(T (g_j - 1))): an entry
// carries at most 2^-24 / M_total of the row's geo mass iff g <= 1 + (ln l_g - ln M_total - 24 ln 2) / T, which is at
// least as tight as the bound from the nearest entry alone (l_g >= exp(T (g_max - 1))) and much tighter where the
// database is dense around the query.  `sums` != null selects it (apply pass); thr_ln = ln M_total + 24 ln 2.
__global__ void __launch_bounds__(128)
geo_mask_kernel(const float4* __restrict__ q_xyz, int N, const float4* __restrict__ caps, int n_tiles, int M, float delta,
                const float2* __restrict__ sums, float thr_ln, float geo_temp, uint32_t* __restrict__ mask, int words) {
  __shared__ float scratch[4];
  const int n = blockIdx.x * 128 + threadIdx.x;
  const bool valid = n < N;
  float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) x = q_xyz[n];
  const float sx = block128_reduce(x.x, false, scratch);
  const float sy = block128_reduce(x.y, false, scratch);
  const float sz = block128_reduce(x.z, false, scratch);
  const float norm = sqrtf(sx * sx + sy * sy + sz * sz);
  const float kPi = 3.14159274f, kEps = 2e-4f;       // eps covers acosf / fp32 dot rounding
  float cx = 0.f, cy = 0.f, cz = 1.f, r_q = kPi;       // degenerate tile (antipodal points): never skip
  if (norm > 1e-3f) {
    cx = sx / norm; cy = sy / norm; cz = sz / norm;
    const float d = valid ? acosf(fminf(1.f, fmaxf(-1.f, cx * x.x + cy * x.y + cz * x.z))) : 0.f;
    r_q = block128_reduce(d, true, scratch) + kEps;
  }
  // Lower bounds valid for every row of the tile: g_max >= cos(far) of the closest database tile, and the geo
  // normaliser l_g = sum_j exp(T (g_j - 1)) >= sum over tiles of (entries in the tile) exp(T (cos(far_t) - 1)).
  float glb = -1.f, llb = 0.f;
  for (int t = threadIdx.x; t < n_tiles; t += 128) {
    const float4 c = caps[t];
    const float far = acosf(fminf(1.f, fmaxf(-1.f, cx * c.x + cy * c.y + cz * c.z))) + r_q + c.w + kEps;
    if (far < kPi) {
      const float cf = cosf(far);
      glb = fmaxf(glb, cf);
      llb += float(min(128, M - t * 128)) * __expf(geo_temp * (cf - 1.f));
    }
  }
  glb = block128_reduce(glb, true, scratch);
  llb = block128_reduce(llb, false, scratch);
  float thr = glb - delta;
  if (llb > 0.f) thr = fmaxf(thr, 1.f + (logf(llb) - thr_ln) / geo_temp - 1e-6f);
  if (sums != nullptr) {
    // smallest normaliser of the tile's rows (padding rows do not count); -(max of -l)
    const float lmin = -block128_reduce(valid ? -sums[n].y : -3.0e38f, true, scratch);
    if (lmin > 0.f && lmin < 3.0e38f) thr = fmaxf(thr, 1.f + (logf(lmin) - thr_ln) / geo_temp - 1e-6f);
  }
  for (int w = threadIdx.x; w < words; w += 128) {
    uint32_t bits = 0;
    for (int b = 0; b < 32; ++b) {
      const int t = w * 32 + b;
      if (t < n_tiles) {
        const float4 c = caps[t];
        const float near = acosf(fminf(1.f, fmaxf(-1.f, cx * c.x + cy * c.y + cz * c.z))) - r_q - c.w - kEps;
        if (near > 0.f && cosf(near) <= thr) bits |= 1u << b;
      }
    }
    mask[size_t(blockIdx.x) * words + w] = bits;
  }
}

// ---------------------------------------------------------------------------------------------------
// small helper kernels
// ---------------------------------------------------------------------------------------------------
// partials [splits][N][2] -> [N][2]
__global__ void reduce_stats_kernel(const float2* __restrict__ part_sum, const float2* __restrict__ part_max,
                                    int N, int splits, float2* __restrict__ sums, float2* __restrict__ maxs) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float2 s = part_sum[n], m = part_max[n];
  for (int k = 1; k < splits; ++k) {
    const float2 a = part_sum[size_t(k) * N + n], b = part_max[size_t(k) * N + n];
    s.x += a.x; s.y += a.y;
    m.x = fmaxf(m.x, b.x); m.y = fmaxf(m.y, b.y);
  }
  sums[n] = s;
  maxs[n] = m;
}

// row constants of the apply kernel from the (global) row statistics
//   sem weight of entry j:  ws 2^(a_s (s_j - 1)) / l_s ,  geo: wg 2^(a_g (g_j - 1)) / l_g   (ws = beta, wg = 1 - beta)
//   B = upper bound of the largest blended weight; P' = weight * 2^13 / B; out = acc * B / 2^13 / vscale
__global__ void row_constants_kernel(const float2* __restrict__ sums, const float2* __restrict__ maxs,
                                     const float4* __restrict__ q_xyz, int N, int geo, float beta, float a_sem,
                                     float a_geo, float inv_vscale, float4* __restrict__ rowc) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float2 l = sums[n], m = maxs[n];
  const float ws = geo ? beta : 1.f, wg = geo ? 1.f - beta : 0.f;
  const float top_s = ws * exp2f(a_sem * (m.x - 1.f)) / l.x;
  const float top_g = geo ? wg * exp2f(a_geo * (m.y - 1.f)) / l.y : 0.f;
  const float B = top_s + top_g;
  const float C = 8192.f;
  const float cs = (ws > 0.f) ? -a_sem + log2f(ws * C / (B * l.x)) : -INFINITY;
  const float cg = (wg > 0.f) ? -a_geo + log2f(wg * C / (B * l.y)) : -INFINITY;
  float4 q = geo ? q_xyz[n] : make_float4(0.f, 0.f, 0.f, 0.f);
  rowc[2 * n] = make_float4(cs, cg, q.x * a_geo, q.y * a_geo);
  rowc[2 * n + 1] = make_float4(q.z * a_geo, B / C * inv_vscale, 0.f, 0.f);
}

// out[n][:] = sum over splits of part[split][n][:]
__global__ void reduce_out_kernel(const float4* __restrict__ part, size_t split_stride4, int splits, size_t total4,
                                  float4* __restrict__ out) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  float4 a = part[i];
  for (int k = 1; k < splits; ++k) {
    const float4 b = part[size_t(k) * split_stride4 + i];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
  }
  out[i] = a;
}

template <class K>
cudaError_t set_smem(K kernel, int bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

}  // namespace

namespace rangeb200 {

long long* g_prof_buffer = nullptr;
void set_profile_buffer(long long* p) { g_prof_buffer = p; }

int retrieval_stats_smem_bytes() { return StatsSmem::dynamic_bytes; }
int retrieval_apply_smem_bytes() { return PairSmem::dynamic_bytes; }

cudaError_t launch_stats(const RetrievalArgs& a, float* part_sum, float* part_max, cudaStream_t stream) {
  const int bytes = retrieval_stats_smem_bytes();
  cudaError_t e;
  if ((e = set_smem(range_stats_kernel<true>, bytes)) != cudaSuccess) return e;
  if ((e = set_smem(range_stats_kernel<false>, bytes)) != cudaSuccess) return e;
  dim3 grid((a.N + kBlockQ - 1) / kBlockQ, a.stats_splits, 1);
  if (a.geo)
    range_stats_kernel<true><<<grid, kStatsThreads, bytes, stream>>>(a.tmK128, a.q16, a.db_xyz, a.q_xyz, a.N, a.M,
                                                               a.stats_tiles_per_split, a.a_sem, a.a_geo, part_sum,
                                                               part_max, a.geo_mask, a.mask_words);
  else
    range_stats_kernel<false><<<grid, kStatsThreads, bytes, stream>>>(a.tmK128, a.q16, a.db_xyz, a.q_xyz, a.N, a.M,
                                                                a.stats_tiles_per_split, a.a_sem, a.a_geo, part_sum,
                                                                part_max, nullptr, 0);
  return cudaGetLastError();
}

cudaError_t launch_geo_mask(const float* q_xyz, int N, int rows, const float* caps, int n_tiles, int M, float delta,
                            const float* sums, float thr_ln, float geo_temp, uint32_t* mask, int words,
                            cudaStream_t stream) {
  // rows >= ceil(N / 128): all-padding query tiles (the CTA-pair grid is rounded up to even) get an all-zero row
  geo_mask_kernel<<<rows, 128, 0, stream>>>(reinterpret_cast<const float4*>(q_xyz), N,
                                                       reinterpret_cast<const float4*>(caps), n_tiles, M, delta,
                                            reinterpret_cast<const float2*>(sums), thr_ln, geo_temp, mask, words);
  return cudaGetLastError();
}

cudaError_t launch_reduce_stats(const float* part_sum, const float* part_max, int N, int splits, float* sums,
                                float* maxs, cudaStream_t stream) {
  reduce_stats_kernel<<<(N + 255) / 256, 256, 0, stream>>>(
      reinterpret_cast<const float2*>(part_sum), reinterpret_cast<const float2*>(part_max), N, splits,
      reinterpret_cast<float2*>(sums), reinterpret_cast<float2*>(maxs));
  return cudaGetLastError();
}

cudaError_t launch_row_constants(const float* sums, const float* maxs, const float* q_xyz, int N, int geo,
                                 float beta, float a_sem, float a_geo, float inv_vscale, float* rowc,
                                 cudaStream_t stream) {
  row_constants_kernel<<<(N + 255) / 256, 256, 0, stream>>>(
      reinterpret_cast<const float2*>(sums), reinterpret_cast<const float2*>(maxs),
      reinterpret_cast<const float4*>(q_xyz), N, geo, beta, a_sem, a_geo, inv_vscale, reinterpret_cast<float4*>(rowc));
  return cudaGetLastError();
}

template <class Kern, class... Args>
cudaError_t launch_pair(Kern kern, dim3 grid, int bytes, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kPairThreads);
  cfg.dynamicSmemBytes = size_t(bytes);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
  if (e != cudaSuccess) {
    int nclusters = -1;
    cudaError_t e2 = cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg);
    fprintf(stderr, "range_b200: cluster launch failed (%s); grid (%u,%u,%u) smem %d; max active clusters %d (%s)\n",
            cudaGetErrorString(e), grid.x, grid.y, grid.z, bytes, nclusters, cudaGetErrorString(e2));
  }
  return e;
}

cudaError_t launch_apply(const RetrievalArgs& a, const float* rowc, float* out, size_t out_split_stride,
                         cudaStream_t stream) {
  cudaError_t e;
  const float4* rc = reinterpret_cast<const float4*>(rowc);
  const int qtiles = (a.N + kBlockQ - 1) / kBlockQ;
  long long* no_prof = nullptr;
  const uint32_t* no_mask = nullptr;
  // CTA pairs: cluster (2,1,1) over the query-tile axis (an odd tile count gets one all-padding CTA)
  const int bytes = PairSmem::dynamic_bytes;
  dim3 grid((qtiles + 1) / 2 * 2, 1024 / kSliceV, a.apply_splits);
  if (g_prof_buffer) {   // instrumented build of the same kernel (tools/time_apply.py)
    if ((e = set_smem(range_apply_pair_kernel<true, true>, bytes)) != cudaSuccess) return e;
    return launch_pair(range_apply_pair_kernel<true, true>, grid, bytes, stream, a.tmQ, a.tmK64, a.tmV128, a.db_xyz,
                       rc, a.N, a.M, a.apply_tiles_per_split, a.a_sem, out, out_split_stride, a.geo_mask, a.mask_words,
                       g_prof_buffer);
  }
  if ((e = set_smem(range_apply_pair_kernel<true>, bytes)) != cudaSuccess) return e;
  if ((e = set_smem(range_apply_pair_kernel<false>, bytes)) != cudaSuccess) return e;
  if (a.geo)
    return launch_pair(range_apply_pair_kernel<true>, grid, bytes, stream, a.tmQ, a.tmK64, a.tmV128, a.db_xyz, rc,
                       a.N, a.M, a.apply_tiles_per_split, a.a_sem, out, out_split_stride, a.geo_mask, a.mask_words,
                       no_prof);
  return launch_pair(range_apply_pair_kernel<false>, grid, bytes, stream, a.tmQ, a.tmK64, a.tmV128, a.db_xyz, rc,
                     a.N, a.M, a.apply_tiles_per_split, a.a_sem, out, out_split_stride, no_mask, 0, no_prof);
}

cudaError_t launch_reduce_out(const float* part, size_t split_stride, int splits, size_t total, float* out,
                              cudaStream_t stream) {
  const size_t total4 = total / 4;
  reduce_out_kernel<<<unsigned((total4 + 255) / 256), 256, 0, stream>>>(
      reinterpret_cast<const float4*>(part), split_stride / 4, splits, total4, reinterpret_cast<float4*>(out));
  return cudaGetLastError();
}

}  // namespace rangeb200
