// Host-side half of the device -> host hand-over of model(locs) (range/range.py:222,240: np.concatenate of the fp32
// retrieved feature with the fp64 location embedding promotes everything to float64).
//
// The fp32 feature columns carry 4 bytes of information each; widening them on the device makes the PCIe copy move
// 10 240 B per query of which 4 096 B are padding.  The device therefore emits PACKED rows (RANGE_OUT_PACKED: 1024
// fp32 + 256 fp64 = 6 144 B; D fp32 + 256 fp64 for a database of value width D), they cross PCIe as they are, and
// range_host_unpack_rows widens them into the caller's (N,D+256) float64 array on the host cores: a small thread team
// of its own (independent of OMP_NUM_THREADS, which torchrun pins to 1), AVX2 conversion with non-temporal stores when
// the CPU has it.
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "../../include/range_b200.h"

namespace {

constexpr int kLoc = 256;

// packed row of a database with value width D: D fp32 feature columns padded to a multiple of 4 (so that the fp64 part
// stays 16-byte aligned), then kLoc fp64 location columns; 6 144 B for D = 1024
size_t packed_row(int D) { return size_t((D + 3) / 4 * 4) * 4 + kLoc * 8; }

void unpack_rows_scalar(const unsigned char* src, double* dst, int D, int64_t lo, int64_t hi) {
  const size_t row = packed_row(D);
  for (int64_t n = lo; n < hi; ++n) {
    const float* f = reinterpret_cast<const float*>(src + size_t(n) * row);
    double* o = dst + size_t(n) * (D + kLoc);
    for (int i = 0; i < D; ++i) o[i] = double(f[i]);
    memcpy(o + D, src + size_t(n) * row + row - kLoc * 8, kLoc * 8);
  }
}

#if defined(__x86_64__)
__attribute__((target("avx2"))) void unpack_rows_avx2(const unsigned char* src, double* dst, int D, int64_t lo,
                                                      int64_t hi) {
  // rows of the result start (D + 256) * 8 B apart: 32-byte aligned whenever the array is and D % 4 == 0 (checked by
  // the caller)
  const size_t row = packed_row(D);
  const int D8 = D / 8 * 8;
  for (int64_t n = lo; n < hi; ++n) {
    const float* f = reinterpret_cast<const float*>(src + size_t(n) * row);
    double* o = dst + size_t(n) * (D + kLoc);
    for (int i = 0; i < D8; i += 8) {
      const __m256 v = _mm256_loadu_ps(f + i);
      _mm256_stream_pd(o + i, _mm256_cvtps_pd(_mm256_castps256_ps128(v)));
      _mm256_stream_pd(o + i + 4, _mm256_cvtps_pd(_mm256_extractf128_ps(v, 1)));
    }
    if (D8 < D) _mm256_stream_pd(o + D8, _mm256_cvtps_pd(_mm_loadu_ps(f + D8)));     // D % 8 == 4
    const double* q = reinterpret_cast<const double*>(src + size_t(n) * row + row - kLoc * 8);
    for (int i = 0; i < kLoc; i += 4) _mm256_stream_pd(o + D + i, _mm256_loadu_pd(q + i));
  }
  _mm_sfence();
}
#endif

}  // namespace

extern "C" int range_host_unpack_rows(const void* packed, int64_t N, int value_dim, double* out, int n_threads) {
  if (N < 0 || value_dim < 1 || value_dim > RANGE_MAX_VALUE_DIM || (N > 0 && (!packed || !out))) return RANGE_ERR_INVALID;
  if (N == 0) return RANGE_OK;
  void (*fn)(const unsigned char*, double*, int, int64_t, int64_t) = unpack_rows_scalar;
#if defined(__x86_64__)
  if (__builtin_cpu_supports("avx2") && (reinterpret_cast<uintptr_t>(out) & 31) == 0 && value_dim % 4 == 0)
    fn = unpack_rows_avx2;
#endif
  const unsigned char* src = static_cast<const unsigned char*>(packed);
  int64_t t = n_threads < 1 ? 1 : n_threads;
  if (t > (N + 255) / 256) t = (N + 255) / 256;          // at least 256 rows (1.5 MB at D = 1024) per thread
  if (t <= 1) {
    fn(src, out, value_dim, 0, N);
    return RANGE_OK;
  }
  std::vector<std::thread> team;
  team.reserve(size_t(t - 1));
  for (int64_t k = 1; k < t; ++k) team.emplace_back(fn, src, out, value_dim, N * k / t, N * (k + 1) / t);
  fn(src, out, value_dim, 0, N / t);
  for (auto& th : team) th.join();
  return RANGE_OK;
}

extern "C" int range_host_unpack(const void* packed, int64_t N, double* out, int n_threads) {
  return range_host_unpack_rows(packed, N, 1024, out, n_threads);
}
