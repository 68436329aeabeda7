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
//   route_rows_kernel       small batches of an M-sharded database: this rank's (N,1024) partial rows -> the owners'
//                           receive buffers over NVLink (large batches: the apply kernel's epilogue stores there itself)
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

__global__ void __launch_bounds__(256)
route_rows_kernel(const float4* __restrict__ O, int N, const RowRoute route) {
  const int n = blockIdx.x;
  if (n >= N) return;
  reinterpret_cast<float4*>(rangeb200::route_row(route, n))[threadIdx.x] = O[size_t(n) * 256 + threadIdx.x];
}

}  // namespace

namespace rangeb200 {

cudaError_t launch_combine_concat(const CombineParts& parts, const double* q64, int N, const int* perm, void* out,
                                  int dtype, cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  if (dtype == 0) combine_concat_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  else if (dtype == 1) combine_concat_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  else combine_concat_kernel<2><<<N, 256, 0, s>>>(parts, q64, N, perm, out);
  return cudaGetLastError();
}

cudaError_t launch_sweep_concat(const SweepParts& parts, const double* q64, int N, const int* perm, int dtype,
                                cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  if (dtype == 0) sweep_concat_kernel<0><<<N, 256, 0, s>>>(parts, q64, N, perm);
  else sweep_concat_kernel<1><<<N, 256, 0, s>>>(parts, q64, N, perm);
  return cudaGetLastError();
}

cudaError_t launch_route_rows(const float* O, int N, const RowRoute& route, cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  route_rows_kernel<<<N, 256, 0, s>>>(reinterpret_cast<const float4*>(O), N, route);
  return cudaGetLastError();
}

}  // namespace rangeb200
