// Retrieval neighbours: the k database entries with the largest retrieval weight per query - the coefficients the
// reference multiplies V[j] by (range/range.py:213-238), which it computes as a dense matrix P and drops.
//
//   RANGE :  w_j = 2^(a_s (s_j - 1)) / l_s
//   RANGE+:  w_j = ws 2^(a_s (s_j - 1)) / l_s + wg 2^(a_g (g_j - 1)) / l_g          ws = beta, wg = 1 - beta
// with a = temperature * log2(e) and the row sums l_s, l_g of the statistics pass (retrieval.cu: fixed offset -1).
//
// A separate pass: the statistics / apply kernels are untouched.
//   range_topk_kernel    S = Q . K^T as in range_stats_kernel (Q in TMEM, TS-mode tcgen05.mma, K tiles by TMA, the
//                        tile's xyz by bulk copy; same geo-skip mask as the apply pass), grid (query tiles, database
//                        splits).  8 softmax warps: warp w owns TMEM lanes 32 (w%4).. and the 64-entry half w/4 of every
//                        128-entry tile.  Each thread keeps a descending list of K (key, entry) pairs in registers and
//                        tests every entry against the k-th key before anything else:
//                          RANGE  key = s (the weight is monotone in s; only the final k are exponentiated)
//                          RANGE+ key = w, evaluated only when the log-domain bound max(ts, tg) + 1 >= log2(k-th w)
//                        Entries that pass are handed to a one-copy insertion loop through a per-thread row of shared
//                        memory (no dynamic register indexing; a warp waits for its busiest lane, not for the union).
//   topk_merge_kernel    one warp per query: a k-round merge of the (split, half) lists [parts][N][k]; row n -> perm[n].
//                        Also merges the lists the shards of an M-sharded database send to a query's owner
//                        (range_topk_merge: one part per rank, entries already in rows of the whole database).
#include <cstdint>
#include <cstdio>
#include <type_traits>
#include <cuda.h>
#include <cuda_runtime.h>

#include "ptx.cuh"
#include "range_kernels.h"

namespace {

constexpr int kBlockQ = 128;        // queries per CTA (UMMA M)
constexpr int kKeys = 128;          // database entries per tile (UMMA N)
constexpr int kStageBytes = 32768;  // one pipeline stage: [128 entries x 128 dims] fp16 as two SWIZZLE_128B boxes
constexpr int kTopkWarps = 8;
constexpr int kTopkThreads = (kTopkWarps + 2) * 32;
constexpr int kKeyRow = 36;         // floats per thread in the pass-on buffer (32 keys, 16-byte aligned rows)
constexpr uint32_t kTmemQ = 0;      // TMEM columns: [0,128) Q | [128,256) S buf 0 | [256,384) S buf 1
constexpr uint32_t kTmemS = 128;

struct TopkSmem {
  static constexpr int NS = 5, kXyzBytes = kKeys * 16;
  static constexpr int stages = 0;
  static constexpr int xyz = stages + NS * kStageBytes;             // 2 slots
  static constexpr int keys = xyz + 2 * kXyzBytes;                  // [softmax threads][kKeyRow] fp32
  static constexpr int bars = keys + kTopkWarps * 32 * kKeyRow * 4;
  static constexpr int b_stage_full = 0;
  static constexpr int b_stage_empty = b_stage_full + NS;
  static constexpr int b_s_full = b_stage_empty + NS;
  static constexpr int b_s_empty = b_s_full + 2;
  static constexpr int b_xyz_empty = b_s_empty + 2;
  static constexpr int n_bars = b_xyz_empty + 2;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16;
  static constexpr int dynamic_bytes = total + 1024;                // slack for the manual 1024-B alignment
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

// part_w / part_idx: [2 * splits][N][k], part = 2 * split + half; unfilled slots have entry -1
template <bool kGeo, int K>
__global__ void __launch_bounds__(kTopkThreads, 1)
range_topk_kernel(const __grid_constant__ CUtensorMap tmK, const __half* __restrict__ q16,
                  const float4* __restrict__ db_xyz, const float4* __restrict__ q_xyz, const float2* __restrict__ sums,
                  int N, int M, int tiles_per_split, float a_sem, float a_geo, float beta, int k,
                  const uint32_t* __restrict__ geo_mask, int mask_words, float* __restrict__ part_w,
                  int32_t* __restrict__ part_idx) {
  using L = TopkSmem;
  constexpr int NS = L::NS, kXyzBytes = L::kXyzBytes;
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
  // geo-skip bit of database tile t for this query tile (geo_mask_kernel, apply-pass bound); warp-uniform
  const uint32_t* mask_row = (kGeo && geo_mask) ? geo_mask + size_t(blockIdx.x) * mask_words : nullptr;
  auto skip_geo = [&](int t) { return mask_row != nullptr && ((__ldg(mask_row + (t >> 5)) >> (t & 31)) & 1u); };

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(&bars[L::b_stage_full + i], 1);
      ptx::mbar_init(&bars[L::b_stage_empty + i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars[L::b_s_full + i], kGeo ? 2 : 1);     // MMA commit (+ the tile's xyz bytes)
      ptx::mbar_init(&bars[L::b_s_empty + i], kTopkWarps);
      ptx::mbar_init(&bars[L::b_xyz_empty + i], kTopkWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kTopkWarps + 1) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
  const uint32_t bars_u = smem_u + L::bars;
  if (warp < kTopkWarps) {        // the 16-warp Q loader, two column groups per warp
    ptx::load_q_to_tmem16(q16, q0, N, tmem_base + kTmemQ, warp, lane);
    ptx::load_q_to_tmem16(q16, q0, N, tmem_base + kTmemQ, warp + kTopkWarps, lane);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();

  if (warp == kTopkWarps) {
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
            ptx::mbar_arrive(&bars[L::b_s_full + (j & 1)]);
          } else {
            ptx::mbar_expect_tx(&bars[L::b_s_full + (j & 1)], kXyzBytes);
            ptx::bulk_load_1d(smem + L::xyz + (j & 1) * kXyzBytes, db_xyz + key0, kXyzBytes, &bars[L::b_s_full + (j & 1)]);
          }
        }
      }
    }
  } else if (warp == kTopkWarps + 1) {
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
    // ===== selection =====
    const int grp = warp >> 2, quarter = warp & 3;          // grp: entries [64 grp, 64 grp + 64) of every tile
    const int row = quarter * 32 + lane;
    const int n = q0 + row;
    // RANGE+: ts = a_s s + cs, tg = a_g q.x + cg with w = 2^ts + 2^tg;  RANGE: cs only for the final exponentials
    float cs = 0.f, cg = -INFINITY, gx = 0.f, gy = 0.f, gz = 0.f;
    if (n < N) {
      const float2 l = sums[n];
      if (kGeo) {
        cs = beta > 0.f ? log2f(beta / l.x) - a_sem : -INFINITY;
        cg = beta < 1.f ? log2f((1.f - beta) / l.y) - a_geo : -INFINITY;
        const float4 qx = q_xyz[n];
        gx = qx.x * a_geo; gy = qx.y * a_geo; gz = qx.z * a_geo;
      } else {
        cs = -a_sem - log2f(l.x);
      }
    }
    float val[K];
    int idx[K];
#pragma unroll
    for (int p = 0; p < K; ++p) { val[p] = -INFINITY; idx[p] = -1; }
    float thr = -INFINITY;       // key of the k-th entry: a candidate must beat it
    float lthr = -INFINITY;      // RANGE+: log2(thr), -inf while the list is not full
    auto insert = [&](float v, int j) {
#pragma unroll
      for (int p = K - 1; p > 0; --p) {        // ties: the entry already listed (smaller index) stays ahead
        const bool up = val[p - 1] < v, here = val[p] < v;
        const float nv = up ? val[p - 1] : (here ? v : val[p]);
        const int ni = up ? idx[p - 1] : (here ? j : idx[p]);
        val[p] = nv; idx[p] = ni;
      }
      if (val[0] < v) { val[0] = v; idx[0] = j; }
      // thr = val[k - 1] as a minimum: a selection by index would be compiled to a local-memory array
      thr = val[0];
#pragma unroll
      for (int p = 1; p < K; ++p) thr = p < k ? fminf(thr, val[p]) : thr;
      if (kGeo) lthr = thr > 0.f ? log2f(thr) : -INFINITY;
    };
    float* keyrow = reinterpret_cast<float*>(smem + L::keys) + threadIdx.x * kKeyRow;
    for (int j = 0; j < T; ++j) {
      const int b = j & 1;
      ptx::mbar_wait(&bars[L::b_s_full + b], (j >> 1) & 1);      // S(j) in TMEM and xyz(j) in smem
      ptx::tc_fence_after();
      const bool with_geo = kGeo && !skip_geo(t_begin + j);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const int col = grp * 64 + h * 32;
        const int key0 = (t_begin + j) * kKeys + col;
        uint32_t s0[32];
        ptx::tmem_ld32(tmem_base + (uint32_t(quarter * 32) << 16) + kTmemS + b * kKeys + col, s0);
        ptx::tmem_ld_wait();
        if (h == 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&bars[L::b_s_empty + b]);
        }
        const uint32_t kxyz = ptx::smem_u32(smem + L::xyz + b * kXyzBytes) + col * 16;
        const int nvalid = M - key0;            // >= 32 except in the last tile
        // keys in place of s; bit i = entry key0 + i beats the k-th key (the geo part is selected per tile)
        uint32_t pass = 0;
        auto body = [&](auto masked, auto geo) {
          constexpr bool kM = decltype(masked)::value, kG = decltype(geo)::value;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float s = __uint_as_float(s0[i]);
            const bool valid = !kM || i < nvalid;
            bool hit;
            if (kGeo) {
              const float ts = fmaf(s, a_sem, cs);
              float tg = -INFINITY;
              if (kG) {
                const float4 kx = ptx::lds_f4(kxyz + i * 16);
                tg = fmaf(gx, kx.x, fmaf(gy, kx.y, fmaf(gz, kx.z, cg)));
              }
              // w <= 2^(max + 1); the slack covers the approximate ex2 / lg2
              hit = valid && fmaxf(ts, tg) + 1.001f >= lthr;
              if (hit) {
                const float w = ptx::ex2(ts) + ptx::ex2(tg);
                s0[i] = __float_as_uint(w);
                hit = w > thr;
              }
            } else {
              hit = valid && s > thr;
            }
            pass |= uint32_t(hit) << i;
          }
        };
        if (nvalid >= 32) {
          if (with_geo) body(std::false_type{}, std::true_type{}); else body(std::false_type{}, std::false_type{});
        } else {
          if (with_geo) body(std::true_type{}, std::true_type{}); else body(std::true_type{}, std::false_type{});
        }
        if (pass) {
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<uint4*>(keyrow + i) = make_uint4(s0[i], s0[i + 1], s0[i + 2], s0[i + 3]);
          do {
            const int i = __ffs(pass) - 1;
            pass &= pass - 1;
            const float v = keyrow[i];
            if (v > thr) insert(v, key0 + i);
          } while (pass);
        }
      }
      if (kGeo) {
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&bars[L::b_xyz_empty + b]);
      }
    }
    if (n < N) {
      if (!kGeo) {
        // keys -> weights (monotone: the order holds), then equal weights by entry (odd-even transposition sort)
#pragma unroll
        for (int p = 0; p < K; ++p) val[p] = idx[p] >= 0 ? ptx::ex2(fmaf(val[p], a_sem, cs)) : -INFINITY;
#pragma unroll
        for (int pass2 = 0; pass2 < K; ++pass2)
#pragma unroll
          for (int p = pass2 & 1; p + 1 < K; p += 2) {
            const int i0 = idx[p], i1 = idx[p + 1];
            const bool swap = val[p] == val[p + 1] && unsigned(i0) > unsigned(i1);
            idx[p] = swap ? i1 : i0;
            idx[p + 1] = swap ? i0 : i1;
          }
      }
      const size_t o = (size_t(2 * split + grp) * N + n) * k;
#pragma unroll
      for (int p = 0; p < K; ++p)
        if (p < k) {
          part_w[o + p] = val[p];
          part_idx[o + p] = idx[p];
        }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kTopkWarps + 1) ptx::tmem_dealloc<512>(tmem_base);
}

// One warp per query: lane l holds the heads of parts l, l + 32, .. (sorted by weight descending, then entry); k rounds
// of a warp arg-max (larger weight, then smaller entry) - the parts are disjoint, so no duplicates.  A found entry is
// stored as row0 + entry (a shard's rows in the whole database: the order of ties is kept, shards are ascending ranges).
constexpr int kMergeSlots = 4;      // parts per lane: parts <= 128
__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ part_w, const int32_t* __restrict__ part_idx, int parts, int N, int k,
                  const int32_t* __restrict__ perm, int row0, int32_t* __restrict__ idx, float* __restrict__ weight) {
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (n >= N) return;
  int head[kMergeSlots];
#pragma unroll
  for (int s = 0; s < kMergeSlots; ++s) head[s] = 0;
  const int dst = perm ? perm[n] : n;
  for (int r = 0; r < k; ++r) {
    float bw = -INFINITY;
    int bi = 0x7fffffff, bs = -1;
#pragma unroll
    for (int s = 0; s < kMergeSlots; ++s) {
      const int part = lane + 32 * s;
      if (part < parts && head[s] < k) {
        const size_t o = (size_t(part) * N + n) * k + head[s];
        const int i = part_idx[o];
        const float w = part_w[o];
        if (i >= 0 && (w > bw || (w == bw && i < bi))) { bw = w; bi = i; bs = s; }
      }
    }
    float w = bw;
    int i = bi;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float w2 = __shfl_xor_sync(0xffffffffu, w, off);
      const int i2 = __shfl_xor_sync(0xffffffffu, i, off);
      if (w2 > w || (w2 == w && i2 < i)) { w = w2; i = i2; }
    }
    if (bs >= 0 && bi == i) {
#pragma unroll
      for (int s = 0; s < kMergeSlots; ++s) head[s] += (s == bs);
    }
    if (lane == 0) {
      const bool found = i != 0x7fffffff;
      idx[size_t(dst) * k + r] = found ? row0 + i : -1;
      weight[size_t(dst) * k + r] = found ? w : 0.f;
    }
  }
}

template <class Kern>
cudaError_t launch_one(Kern kern, dim3 grid, const rangeb200::RetrievalArgs& a, int tiles_per_split, const float* sums,
                       float beta, int k, float* part_w, int32_t* part_idx, cudaStream_t s) {
  const int bytes = TopkSmem::dynamic_bytes;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  kern<<<grid, kTopkThreads, bytes, s>>>(a.tmK128, a.q16, a.db_xyz, a.q_xyz, reinterpret_cast<const float2*>(sums),
                                         a.N, a.M, tiles_per_split, a.a_sem, a.a_geo, beta, k, a.geo_mask, a.mask_words,
                                         part_w, part_idx);
  return cudaGetLastError();
}

template <int K>
cudaError_t launch_bucket(dim3 grid, const rangeb200::RetrievalArgs& a, int tiles_per_split, const float* sums,
                          float beta, int k, float* part_w, int32_t* part_idx, cudaStream_t s) {
  if (a.geo) return launch_one(range_topk_kernel<true, K>, grid, a, tiles_per_split, sums, beta, k, part_w, part_idx, s);
  return launch_one(range_topk_kernel<false, K>, grid, a, tiles_per_split, sums, beta, k, part_w, part_idx, s);
}

}  // namespace

namespace rangeb200 {

cudaError_t launch_topk(const RetrievalArgs& a, int splits, int tiles_per_split, const float* sums, float beta, int k,
                        float* part_w, int32_t* part_idx, const int32_t* perm, int row0, int32_t* idx, float* weight,
                        cudaStream_t s) {
  if (k < 1 || k > kTopkMax || 2 * splits > 32 * kMergeSlots) return cudaErrorInvalidValue;
  const dim3 grid((a.N + kBlockQ - 1) / kBlockQ, splits, 1);
  cudaError_t e;
  if (k <= 8) e = launch_bucket<8>(grid, a, tiles_per_split, sums, beta, k, part_w, part_idx, s);
  else if (k <= 16) e = launch_bucket<16>(grid, a, tiles_per_split, sums, beta, k, part_w, part_idx, s);
  else e = launch_bucket<32>(grid, a, tiles_per_split, sums, beta, k, part_w, part_idx, s);
  if (e != cudaSuccess) return e;
  return launch_topk_merge(part_w, part_idx, 2 * splits, a.N, k, perm, row0, idx, weight, s);
}

cudaError_t launch_topk_merge(const float* part_w, const int32_t* part_idx, int parts, int N, int k,
                              const int32_t* perm, int row0, int32_t* idx, float* weight, cudaStream_t s) {
  if (k < 1 || k > kTopkMax || parts < 1 || parts > 32 * kMergeSlots) return cudaErrorInvalidValue;
  topk_merge_kernel<<<(N + 7) / 8, 256, 0, s>>>(part_w, part_idx, parts, N, k, perm, row0, idx, weight);
  return cudaGetLastError();
}

}  // namespace rangeb200
