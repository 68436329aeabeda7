// Merging partial retrieved features (no kernel counterpart in the reference: range/range.py:217,236-238 compute one
// dense product per softmax on one device).
//
//   combine_concat_kernel   out[perm[n]] = [ sum_k w_k part_k[n] | q64[n] ]  - the last step of
//                             * an M-sharded database: part_k = the partial rows rank k wrote into this rank's receive
//                               buffer (fixed summation order: results do not depend on arrival order), w_k = 1
//                             * a beta sweep: parts = (O_geo, O_sem), w = (1 - beta, beta)   (range.py:238 is linear in beta)
//   sweep_concat_kernel     out_b[perm[n]] = [ (1 - beta_b) G[n] + beta_b S[n] | q64[n] ] for up to 8 beta at once - the
//                           last step of a beta sweep on an M-sharded database: G / S = the sums of the partial slots of
//                           the geographic (beta 0) and semantic (beta 1) ends; every slot is read once for all beta
//   *_any_kernel            the two above for a value width D other than 1024: parts (N,D), rows [D | 256]
//   reduce_route_kernel     an M-sharded database, apply pass on CTA pairs (small batches, value widths other than
//                           1024): one query chunk's split partials summed and each row stored once into its owner's
//                           receive buffer over NVLink (large 1024-wide batches: the apply kernel's epilogue stores there)
//   peer memory             receive buffers are plain cudaMalloc allocations exported / opened with CUDA IPC handles
#include <cstdint>
#include <cuda_runtime.h>

#include "range_kernels.h"

namespace {

using rangeb200::CombineParts;
using rangeb200::RowRoute;
using rangeb200::SweepParts;

// one CTA of 256 threads per row: thread t handles feature columns [4t, 4t+4) and location column t
template <int kDtype>      // 0: fp64 (N,1280); 1: fp32 (N,1280); 2: packed (fp32 features, fp64 location columns: 6144 B per row)
__global__ void __launch_bounds__(256)
combine_concat_kernel(const CombineParts parts, const double* __restrict__ q64, int N, const int* __restrict__ perm,
                      void* __restrict__ out) {
  const int n = blockIdx.x;
  const int t = threadIdx.x;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int k = 0; k < parts.n; ++k) {
    const float4 v = __ldcs(reinterpret_cast<const float4*>(parts.p[k] + size_t(n) * 1024) + t);
    const float w = parts.w[k];
    a.x = fmaf(w, v.x, a.x); a.y = fmaf(w, v.y, a.y); a.z = fmaf(w, v.z, a.z); a.w = fmaf(w, v.w, a.w);
  }
  const double q = q64[size_t(n) * 256 + t];
  const size_t r = perm ? size_t(perm[n]) : size_t(n);
  if (kDtype == 0) {
    double* o = reinterpret_cast<double*>(out) + r * 1280;
    __stcs(reinterpret_cast<double2*>(o + 4 * t), make_double2(double(a.x), double(a.y)));
    __stcs(reinterpret_cast<double2*>(o + 4 * t + 2), make_double2(double(a.z), double(a.w)));
    o[1024 + t] = q;
  } else if (kDtype == 1) {
    float* o = reinterpret_cast<float*>(out) + r * 1280;
    __stcs(reinterpret_cast<float4*>(o) + t, a);
    o[1024 + t] = float(q);
  } else {
    char* o = reinterpret_cast<char*>(out) + r * 6144;
    __stcs(reinterpret_cast<float4*>(o) + t, a);
    reinterpret_cast<double*>(o + 4096)[t] = q;
  }
}

// one CTA of 256 threads per row, like combine_concat_kernel.  Per column fmaf(w_sem, s, w_geo * g): with one slot per
// end this is bit for bit what combine_concat_kernel computes for parts (G, S), weights (w_geo, w_sem).
template <int kDtype>      // 0: fp64 (N,1280); 1: fp32 (N,1280)
__global__ void __launch_bounds__(256)
sweep_concat_kernel(const SweepParts parts, const double* __restrict__ q64, int N, const int* __restrict__ perm) {
  const int n = blockIdx.x;
  const int t = threadIdx.x;
  const size_t off = size_t(n) * 256 + t;           // float4 index of columns [4t, 4t+4) of row n
  float4 g = __ldcs(reinterpret_cast<const float4*>(parts.geo[0]) + off);
  float4 s = __ldcs(reinterpret_cast<const float4*>(parts.sem[0]) + off);
  for (int k = 1; k < parts.n_slots; ++k) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(parts.geo[k]) + off);
    const float4 b = __ldcs(reinterpret_cast<const float4*>(parts.sem[k]) + off);
    g.x += a.x; g.y += a.y; g.z += a.z; g.w += a.w;
    s.x += b.x; s.y += b.y; s.z += b.z; s.w += b.w;
  }
  const double q = q64[size_t(n) * 256 + t];
  const size_t r = perm ? size_t(perm[n]) : size_t(n);
  for (int b = 0; b < parts.n_betas; ++b) {
    const float wg = parts.w_geo[b], ws = parts.w_sem[b];
    const float4 v = make_float4(fmaf(ws, s.x, wg * g.x), fmaf(ws, s.y, wg * g.y), fmaf(ws, s.z, wg * g.z),
                                 fmaf(ws, s.w, wg * g.w));
    if (kDtype == 0) {
      double* o = reinterpret_cast<double*>(parts.out[b]) + r * 1280;
      __stcs(reinterpret_cast<double2*>(o + 4 * t), make_double2(double(v.x), double(v.y)));
      __stcs(reinterpret_cast<double2*>(o + 4 * t + 2), make_double2(double(v.z), double(v.w)));
      __stcs(o + 1024 + t, q);
    } else {
      float* o = reinterpret_cast<float*>(parts.out[b]) + r * 1280;
      __stcs(reinterpret_cast<float4*>(o) + t, v);
      __stcs(o + 1024 + t, float(q));
    }
  }
}

// The two kernels above for a value width D != 1024 (the 1024-wide launches keep them): one CTA of 256 threads per row,
// thread t handles feature columns t, t + 256, ... and location column t.  Per column the same arithmetic.
// Row of `out`: dtype 0 fp64 / 1 fp32: D + 256 columns; 2 packed: packed_row_bytes(D), fp32 columns [D, round_up(D, 4))
// written as zero.
template <int kDtype>
__device__ __forceinline__ void store_row(void* out, size_t r, int D, int c, float v) {
  if (kDtype == 0) __stcs(reinterpret_cast<double*>(out) + r * size_t(D + 256) + c, double(v));
  else if (kDtype == 1) __stcs(reinterpret_cast<float*>(out) + r * size_t(D + 256) + c, v);
  else __stcs(reinterpret_cast<float*>(reinterpret_cast<char*>(out) + r * rangeb200::packed_row_bytes(D)) + c, v);
}

template <int kDtype>
__device__ __forceinline__ void store_q(void* out, size_t r, int D, int t, double q) {
  if (kDtype == 0) __stcs(reinterpret_cast<double*>(out) + r * size_t(D + 256) + D + t, q);
  else if (kDtype == 1) __stcs(reinterpret_cast<float*>(out) + r * size_t(D + 256) + D + t, float(q));
  else __stcs(reinterpret_cast<double*>(reinterpret_cast<char*>(out) + r * rangeb200::packed_row_bytes(D) +
                                        size_t((D + 3) / 4 * 4) * 4) + t, q);
}

template <int kDtype>
__global__ void __launch_bounds__(256)
combine_concat_any_kernel(const CombineParts parts, const double* __restrict__ q64, int N, int D,
                          const int* __restrict__ perm, void* __restrict__ out) {
  const int n = blockIdx.x;
  const int t = threadIdx.x;
  const size_t r = perm ? size_t(perm[n]) : size_t(n);
  const int cols = kDtype == 2 ? (D + 3) / 4 * 4 : D;
  for (int c = t; c < cols; c += 256) {
    float a = 0.f;
    if (c < D)
      for (int k = 0; k < parts.n; ++k) a = fmaf(parts.w[k], __ldcs(parts.p[k] + size_t(n) * D + c), a);
    store_row<kDtype>(out, r, D, c, a);
  }
  store_q<kDtype>(out, r, D, t, q64[size_t(n) * 256 + t]);
}

template <int kDtype>      // 0: fp64, 1: fp32
__global__ void __launch_bounds__(256)
sweep_concat_any_kernel(const SweepParts parts, const double* __restrict__ q64, int N, int D,
                        const int* __restrict__ perm) {
  const int n = blockIdx.x;
  const int t = threadIdx.x;
  const size_t r = perm ? size_t(perm[n]) : size_t(n);
  for (int c = t; c < D; c += 256) {
    const size_t off = size_t(n) * D + c;
    float g = __ldcs(parts.geo[0] + off), s = __ldcs(parts.sem[0] + off);
    for (int k = 1; k < parts.n_slots; ++k) {
      g += __ldcs(parts.geo[k] + off);
      s += __ldcs(parts.sem[k] + off);
    }
    for (int b = 0; b < parts.n_betas; ++b)
      store_row<kDtype>(parts.out[b], r, D, c, fmaf(parts.w_sem[b], s, parts.w_geo[b] * g));
  }
  const double q = q64[size_t(n) * 256 + t];
  for (int b = 0; b < parts.n_betas; ++b) store_q<kDtype>(parts.out[b], r, D, t, q);
}

// One thread per 4 columns of a row of the chunk [n0, n0 + rows): the row's split partials part[k][n][0:D] summed in
// split order 0 .. splits-1 with the additions of reduce_out_kernel (the same bits), then stored once at
//   peer[g / slab] + ((size_t)rank * slab + g % slab) * D,   g = n0 + n,
// the owner computed per row (a chunk of 256-row multiples may span several 128-row-multiple slabs).  D % 4 == 0 and
// 16-byte aligned buffers (range_retrieve_apply_routed_values checks both).
__global__ void __launch_bounds__(256)
reduce_route_kernel(const float4* __restrict__ part, size_t split_stride4, int splits, long long n0, int rows, int D,
                    const RowRoute route) {
  const int D4 = D / 4;
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= size_t(rows) * D4) return;
  float4 a = __ldcs(part + i);
  for (int k = 1; k < splits; ++k) {
    const float4 b = __ldcs(part + size_t(k) * split_stride4 + i);
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
  }
  const long long g = n0 + (long long)(i / D4);
  const int c4 = int(i % D4);
  const int owner = int(g / route.slab);
  float* peer = route.peer[0];
#pragma unroll
  for (int r = 1; r < rangeb200::kMaxRanks; ++r) peer = owner == r ? route.peer[r] : peer;   // no local copy of peer[]
  float* row = peer + (size_t(route.rank) * size_t(route.slab) + size_t(g - owner * route.slab)) * D;
  reinterpret_cast<float4*>(row)[c4] = a;
}

}  // namespace

namespace rangeb200 {

cudaError_t launch_combine_concat(const CombineParts& parts, const double* q64, int N, int D, const int* perm, void* out,
                                  int dtype, cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  if (D != 1024) {
    if (dtype == 0) combine_concat_any_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, D, perm, out);
    else if (dtype == 1) combine_concat_any_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, D, perm, out);
    else combine_concat_any_kernel<2><<<N, 256, 0, s>>>(parts, q64, N, D, perm, out);
    return cudaGetLastError();
  }
  if (dtype == 0) combine_concat_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  else if (dtype == 1) combine_concat_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  else combine_concat_kernel<2><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  return cudaGetLastError();
}

cudaError_t launch_sweep_concat(const SweepParts& parts, const double* q64, int N, int D, const int* perm, int dtype,
                                cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  if (D != 1024) {
    if (dtype == 0) sweep_concat_any_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, D, perm);
    else sweep_concat_any_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, D, perm);
    return cudaGetLastError();
  }
  if (dtype == 0) sweep_concat_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, perm);
  else sweep_concat_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, perm);
  return cudaGetLastError();
}

cudaError_t launch_reduce_route(const float* part, size_t split_stride, int splits, long long n0, int rows, int D,
                                const RowRoute& route, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  const size_t total4 = size_t(rows) * (D / 4);
  reduce_route_kernel<<<unsigned((total4 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const float4*>(part),
                                                                     split_stride / 4, splits, n0, rows, D, route);
  return cudaGetLastError();
}

}  // namespace rangeb200
