// C-ABI layer: argument checking, workspace carving, tensor-map construction, kernel sequencing.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>

#include "../../include/range_b200.h"
#include "range_kernels.h"

using namespace rangeb200;

namespace {

thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return fail(RANGE_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

constexpr int kDimK = 256, kDimV = 1024, kBlockQ = 128, kBlockKeys = 128;
constexpr int64_t kEncodeChunk = 131072;   // queries per encoder pass (bounds the feature workspace)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// 2-D tensor [rows][cols] row-major (fp16, or fp32 when f32), box [box_rows][128 B inner], SWIZZLE_128B
int make_tmap(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows, bool f32 = false) {
  auto fn = get_encode_fn();
  if (!fn) return fail(RANGE_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {cols * (f32 ? 4u : 2u)};
  cuuint32_t box[2] = {f32 ? 32u : 64u, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                  const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RANGE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", int(r));
  return RANGE_OK;
}

// 2-D view [rows][2048 B] (256 x uint64) of a byte buffer, box [8 rows][2048 B], no swizzle: the P' ring of the
// producer/consumer apply kernel (one row = one 8-entry key chunk of a tile: [128 query rows][16 B])
int make_tmap_rows2k(CUtensorMap* m, const void* base, uint64_t rows) {
  auto fn = get_encode_fn();
  if (!fn) return fail(RANGE_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t gdim[2] = {256, rows};
  cuuint64_t gstr[1] = {2048};
  cuuint32_t box[2] = {256, 8};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RANGE_ERR_CUDA, "cuTensorMapEncodeTiled (ring) failed (%d)", int(r));
  return RANGE_OK;
}

}  // namespace

struct range_ctx {
  int device = 0;
  int sm_count = 148;
  ShTable sh;
  int n_layers = 0;
  std::vector<int> dims;
  std::vector<const double*> W, b;
  double w0_first = 30.0, w0_hidden = 1.0;
  int64_t M = 0, Mpad = 0;
  const void* Kh = nullptr;
  const void* Vt = nullptr;
  const float* xyz = nullptr;
  float vscale = 1.f;
  CUtensorMap tmK128, tmK64, tmV128;
  const float* caps = nullptr;     // (Mpad / 128, 4) bounding caps of the database tiles, or null
  int64_t M_total = 0;             // entries of the whole (unsharded) database: sets the geo-skip threshold
  // tensor-core encoder (split fp16): prepared weights live in a caller-provided buffer
  int enc_precision = RANGE_ENC_F64;
  bool enc_prepared = false;
  const int* perm = nullptr;
  std::vector<CUtensorMap> tmWh, tmWl;         // weights hi / lo, box [256 rows x 64] (siren_tc_kernel)
  std::vector<CUtensorMap> tmWh2, tmWl2;       // the same arrays, box [128 rows x 64] (siren_pair_kernel: half a tile per CTA)
  std::vector<int> sh_off, sh_par;     // host copies of the harmonics table's chain offsets / parities (layout planning)
};

namespace {

// ---- feature layout of the tensor-core encoder's first layer (ShTable::K0 / fmap, range_kernels.h) --------------------
// Rounds layout: the (l, |m|) Horner chains sorted by length (longest first; ties by |m|, then l), 32 per round.
struct ShLayout {
  int rounds = 0, K0 = 0;
  std::vector<int> order;              // rounds layout: slot (32 r + lane) -> entry, -1 for an unused slot
  std::vector<int> roff;               // [rounds + 1] offsets (doubles) into the round table
  std::vector<int> perm, fmap;         // [K0]: column -> reference feature index l*l + l +- |m| (-1: zero column) / entry map
};

void entry_lm(int L, std::vector<int>& el, std::vector<int>& em) {
  for (int am = 0; am < L; ++am)
    for (int l = am; l < L; ++l) { el.push_back(l); em.push_back(am); }
}

// want_rounds == false: production order (for am: for l >= am: cos, then sin when am > 0), K0 = L*L
ShLayout plan_sh_layout(int L, const std::vector<int>& off, bool want_rounds) {
  ShLayout y;
  const int E = L * (L + 1) / 2;
  std::vector<int> el, em;
  entry_lm(L, el, em);
  if (!want_rounds) {
    y.K0 = L * L;
    for (int e = 0; e < E; ++e) {
      y.perm.push_back(el[e] * el[e] + el[e] + em[e]);
      y.fmap.push_back(em[e] == 0 ? e : (e | em[e] << 16));
      if (em[e]) {
        y.perm.push_back(el[e] * el[e] + el[e] - em[e]);
        y.fmap.push_back(e | em[e] << 16 | 1 << 24);
      }
    }
    return y;
  }
  std::vector<int> idx(E);
  for (int e = 0; e < E; ++e) idx[e] = e;
  std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) {
    const int la = off[a + 1] - off[a], lb = off[b + 1] - off[b];
    return la != lb ? la > lb : a < b;             // entries are already ordered by |m|, then l
  });
  y.rounds = (E + 31) / 32;
  y.K0 = 64 * y.rounds;
  y.order.assign(size_t(y.rounds) * 32, -1);
  for (int i = 0; i < E; ++i) y.order[i] = idx[i];
  y.roff.push_back(0);
  for (int r = 0; r < y.rounds; ++r) {
    int nst = 1;
    for (int i = 0; i < 32; ++i) {
      const int e = y.order[r * 32 + i];
      if (e >= 0) nst = std::max(nst, off[e + 1] - off[e]);
      if (e < 0) {
        y.perm.push_back(-1); y.perm.push_back(-1);
        y.fmap.push_back(kShZeroSlot); y.fmap.push_back(kShZeroSlot);
      } else {
        y.perm.push_back(el[e] * el[e] + el[e] + em[e]);
        y.fmap.push_back(em[e] == 0 ? e : (e | em[e] << 16));
        y.perm.push_back(em[e] ? el[e] * el[e] + el[e] - em[e] : -1);
        y.fmap.push_back(em[e] ? (e | em[e] << 16 | 1 << 24) : kShZeroSlot);
      }
    }
    y.roff.push_back(y.roff.back() + 32 * (1 + nst));
  }
  return y;
}

// rounds layout only when its table and the kernel's scratch fit in shared memory
bool sh_rounds_fit(int L, const ShLayout& y) {
  return y.rounds > 0 && sh_rounds_smem_bytes(L, y.rounds, y.roff.back()) <= size_t(200) * 1024;
}

ShLayout choose_sh_layout(const range_ctx* c) {
  if (!c->sh.closed_form && !c->sh_off.empty()) {
    ShLayout y = plan_sh_layout(c->sh.L, c->sh_off, true);
    if (sh_rounds_fit(c->sh.L, y)) return y;
  }
  return plan_sh_layout(c->sh.L, c->sh_off, false);
}

size_t sh_layout_bytes(const ShLayout& y) {      // perm + fmap (+ round table, meta, offsets) inside the prepared buffer
  size_t b = 2 * align_up(size_t(y.K0) * 4, 256);
  if (y.rounds) b += align_up(size_t(y.roff.back()) * 8, 256) + align_up(size_t(y.rounds) * 128, 256) + align_up(size_t(y.rounds + 1) * 4, 256);
  return b;
}

struct RetrievalPlan {
  int splits, tiles_per_split;              // apply kernel
  int stats_splits, stats_tiles_per_split;  // stats kernel
  int mask_rows, mask_words;                // geo-skip mask: [even-padded query tiles][ceil(tiles / 32)]
  bool pc;                                  // apply with the producer/consumer kernel (retrieval_pc.cu)
  bool stats_pc;                            // statistics with the CTA-pair / four-group kernel (retrieval_pc.cu)
  size_t off_part_sum, off_part_max, off_sums, off_maxs, off_rowc, off_mask, off_ring, off_flags, off_pc_part, off_pc_scratch, off_part_out, off_O, total;
};

// RANGE_SIREN_KERNEL=cta: the one-tile-per-CTA layer kernel (siren_tc_kernel) instead of the persistent CTA pairs
int siren_kernel_override() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RANGE_SIREN_KERNEL");
    v = (e && !strcmp(e, "cta")) ? 1 : 0;
  }
  return v;
}

// 0 = choose by batch size, 1 = always the single-role CTA-pair kernel, 2 = producer/consumer whenever possible
int apply_kernel_override() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RANGE_APPLY_KERNEL");
    v = !e ? 0 : (!strcmp(e, "pair") ? 1 : (!strcmp(e, "pc") ? 2 : 0));
  }
  return v;
}

// Database splits: enough CTAs to fill the SMs when there are few query tiles.
RetrievalPlan plan_retrieval(const range_ctx* c, int64_t N) {
  RetrievalPlan p{};
  const int64_t qtiles = (N + kBlockQ - 1) / kBlockQ;
  const int64_t tiles = (c->M + kBlockKeys - 1) / kBlockKeys;
  int64_t want = 1;
  const int64_t ctas = qtiles * 4;
  if (ctas < 2 * c->sm_count) want = (2 * c->sm_count + ctas - 1) / ctas;
  int64_t max_splits = tiles / 8 > 0 ? tiles / 8 : 1;      // at least 8 tiles per split
  if (want > max_splits) want = max_splits;
  if (want > 64) want = 64;
  // the tensor core's fp32 accumulation truncates (retrieval_pc.cu: kAccWindow): at most 256 tiles per accumulator
  const int64_t for_accuracy = (tiles + 255) / 256 < 256 ? (tiles + 255) / 256 : 256;
  if (want < for_accuracy) want = for_accuracy;
  p.tiles_per_split = int((tiles + want - 1) / want);
  p.splits = int((tiles + p.tiles_per_split - 1) / p.tiles_per_split);
  // stats kernel: one CTA per (query tile, split).  Its partials are tiny, so choose the split count that
  // minimises wave quantisation: waves(s) / s with waves(s) = ceil(qtiles * s / SMs), keeping >= 32 tiles per split.
  int64_t best = want;
  double best_cost = 1e30;
  for (int64_t sp = want; sp <= 16 && sp <= (tiles / 32 > 0 ? tiles / 32 : 1); ++sp) {
    const double waves = double((qtiles * sp + c->sm_count - 1) / c->sm_count);
    const double cost = waves / double(sp) * (1.0 + 0.004 * double(sp));      // small per-CTA fixed cost
    if (cost < best_cost - 1e-9) { best_cost = cost; best = sp; }
  }
  // large batches: CTA pairs (two query tiles per cluster) -> waves are counted in clusters
  const int64_t qpairs0 = (qtiles + 1) / 2, slots = c->sm_count / 2;
  p.stats_pc = apply_kernel_override() != 1 && slots > 0 && qpairs0 >= apply_pc_units(c->sm_count);
  if (p.stats_pc) {
    best = 1;
    best_cost = 1e30;
    for (int64_t sp = 1; sp <= 16 && sp <= (tiles / 32 > 0 ? tiles / 32 : 1); ++sp) {
      const double waves = double((qpairs0 * sp + slots - 1) / slots);
      const double cost = waves / double(sp) * (1.0 + 0.004 * double(sp));
      if (cost < best_cost - 1e-9) { best_cost = cost; best = sp; }
    }
  }
  p.stats_tiles_per_split = int((tiles + best - 1) / best);
  p.stats_splits = int((tiles + p.stats_tiles_per_split - 1) / p.stats_tiles_per_split);
  size_t o = 0;
  p.off_part_sum = o; o += align_up(size_t(p.stats_splits) * N * 8, 256);
  p.off_part_max = o; o += align_up(size_t(p.stats_splits) * N * 8, 256);
  p.off_sums = o;     o += align_up(size_t(N) * 8, 256);
  p.off_maxs = o;     o += align_up(size_t(N) * 8, 256);
  p.off_rowc = o;     o += align_up(size_t(N) * 32, 256);
  p.mask_rows = int((qtiles + 1) / 2 * 2);
  p.mask_words = int((tiles + 31) / 32);
  p.off_mask = o;     o += c->caps ? align_up(size_t(p.mask_rows) * p.mask_words * 4, 256) : 0;
  // producer/consumer apply: enough query-tile pairs to give every unit (2 producer + 4 consumer SMs) a full round
  const int units = apply_pc_units(c->sm_count);
  const int64_t qpairs = (qtiles + 1) / 2;
  const int ov = apply_kernel_override();
  p.pc = units > 0 && ov != 1 && (ov == 2 || qpairs >= units);
  p.off_ring = o;     o += p.pc ? align_up(apply_pc_ring_bytes(c->sm_count), 1024) : 0;
  p.off_flags = o;    o += p.pc ? align_up(apply_pc_flag_bytes(c->sm_count, N, c->M), 256) : 0;
  p.off_pc_part = o;  o += p.pc ? align_up(apply_pc_part_bytes(c->sm_count, N, c->M), 256) : 0;
  p.off_pc_scratch = o; o += p.pc ? align_up(apply_pc_scratch_bytes(c->sm_count), 256) : 0;
  p.off_part_out = o; o += (p.splits > 1 && !p.pc) ? align_up(size_t(p.splits) * N * kDimV * 4, 256) : 0;
  p.off_O = o;        o += p.pc ? 0 : align_up(size_t(N) * kDimV * 4, 256);   // scratch O of range_retrieve_apply_concat (small batches)
  p.total = o;
  return p;
}

// ws: aligned workspace base; when the database carries bounding caps the geo-skip mask is (re)computed here
int fill_args(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp, float geo_temp,
              const RetrievalPlan& p, char* ws, cudaStream_t stream, RetrievalArgs* a, const float* sums = nullptr) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (mode != RANGE_MODE_RANGE && mode != RANGE_MODE_RANGE_PLUS) return fail(RANGE_ERR_INVALID, "unknown mode %d", mode);
  if (N <= 0 || N > (int64_t(1) << 30)) return fail(RANGE_ERR_INVALID, "N out of range");
  int r = make_tmap(&a->tmQ, q16, uint64_t(N), kDimK, kBlockQ);
  if (r) return r;
  a->tmK128 = c->tmK128;
  a->tmK64 = c->tmK64;
  a->tmV128 = c->tmV128;
  a->q16 = reinterpret_cast<const __half*>(q16);
  a->db_xyz = reinterpret_cast<const float4*>(c->xyz);
  a->q_xyz = reinterpret_cast<const float4*>(qxyz);
  a->N = int(N);
  a->M = int(c->M);
  a->geo = mode == RANGE_MODE_RANGE_PLUS;
  a->apply_splits = p.splits;
  a->apply_tiles_per_split = p.tiles_per_split;
  a->stats_splits = p.stats_splits;
  a->stats_tiles_per_split = p.stats_tiles_per_split;
  const float log2e = 1.4426950408889634f;
  a->a_sem = temp * log2e;
  a->a_geo = geo_temp * log2e;
  a->geo_mask = nullptr;
  a->mask_words = 0;
  if (a->geo && c->caps && geo_temp > 0.f) {
    // entries with g <= g_max - delta together carry < 2^-24 of the row's geo normaliser (retrieval.cu)
    const float thr_ln = logf(float(c->M_total)) + 24.f * 0.6931471805599453f;
    const float delta = thr_ln / geo_temp;
    uint32_t* mask = reinterpret_cast<uint32_t*>(ws + p.off_mask);
    // apply pass: the (global) row normalisers are known and tighten the bound
    CUDA_TRY(launch_geo_mask(qxyz, int(N), p.mask_rows, c->caps, int(c->Mpad / kBlockKeys), int(c->M), delta, sums, thr_ln,
                             geo_temp, mask, p.mask_words, stream));
    g_launches += 1;
    a->geo_mask = mask;
    a->mask_words = p.mask_words;
  }
  return RANGE_OK;
}

// Neighbours pass: the statistics plan's database splits (at most kTopkMaxSplits: the merge takes 2 lists per split and
// CTA), its geo-skip mask, then the partial lists [2 * splits][N][k] (weight, entry).
struct TopkPlan {
  RetrievalPlan ret;                        // only the mask fields are used; ret.off_mask is relative to this workspace
  int splits, tiles_per_split;
  size_t off_w, off_idx, total;
};

TopkPlan plan_topk(const range_ctx* c, int64_t N, int k) {
  TopkPlan t;
  t.ret = plan_retrieval(c, N);
  const int64_t tiles = (c->M + kBlockKeys - 1) / kBlockKeys;
  const int64_t want = std::min<int64_t>(t.ret.stats_splits, kTopkMaxSplits);
  t.tiles_per_split = int((tiles + want - 1) / want);
  t.splits = int((tiles + t.tiles_per_split - 1) / t.tiles_per_split);
  const size_t lists = size_t(2 * t.splits) * size_t(N) * size_t(k) * 4;
  size_t o = 0;
  t.ret.off_mask = o; o += c->caps ? align_up(size_t(t.ret.mask_rows) * t.ret.mask_words * 4, 256) : 0;
  t.off_w = o;        o += align_up(lists, 256);
  t.off_idx = o;      o += align_up(lists, 256);
  t.total = o;
  return t;
}

}  // namespace

extern "C" {

const char* range_last_error(void) { return g_err; }
int range_version(void) { return 100; }
int64_t range_launch_count(void) { return g_launches.load(); }
// not in the public header: work decomposition of the producer/consumer apply kernel (tests/test_capi.py; host code only)
void range_debug_apply_plan(int sm_count, int64_t N, int64_t M, int32_t* out7) { apply_pc_describe_plan(sm_count, N, M, out7); }
// not in the public header: feature layout of the tensor-core encoder's first layer for a harmonics table with these
// chain offsets (tests/test_capi.py; host code only).  off: n_entries + 1 host ints; perm / fmap: K0 ints each (cap >= K0).
// Returns K0 (<= 0 on bad arguments or cap too small); *rounds = 0 for the production-order layout.
int range_debug_sh_layout(int L, const int32_t* off, int want_rounds, int32_t* rounds, int32_t* round_table_doubles,
                          int32_t* perm, int32_t* fmap, int cap) {
  if (L <= 0 || !off || !rounds || !round_table_doubles || !perm || !fmap) return -1;
  const int E = L * (L + 1) / 2;
  const ShLayout y = plan_sh_layout(L, std::vector<int>(off, off + E + 1), want_rounds != 0);
  if (y.K0 > cap) return -1;
  *rounds = y.rounds;
  *round_table_doubles = y.rounds ? y.roff.back() : 0;
  std::copy(y.perm.begin(), y.perm.end(), perm);
  std::copy(y.fmap.begin(), y.fmap.end(), fmap);
  return y.K0;
}
// not in the public header: developer hook used by tools/time_apply.py
void range_debug_set_profile_buffer(void* device_buffer) { set_profile_buffer(reinterpret_cast<long long*>(device_buffer)); }

int range_ctx_create(int device, range_ctx** out) {
  if (!out) return fail(RANGE_ERR_INVALID, "out is null");
  int count = 0;
  CUDA_TRY(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(RANGE_ERR_INVALID, "device %d out of range (%d devices)", device, count);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(RANGE_ERR_UNSUPPORTED, "range_b200 needs an sm_100 device, found sm_%d%d", prop.major, prop.minor);
  range_ctx* c = new range_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  *out = c;
  return RANGE_OK;
}

int range_ctx_destroy(range_ctx* ctx) {
  delete ctx;
  return RANGE_OK;
}

int range_ctx_set_sh_table(range_ctx* c, int L, int n_entries, const double* pref, const int32_t* off,
                           const double* coef, const int32_t* par) {
  if (!c || L <= 0 || n_entries != L * (L + 1) / 2 || !pref || !off || !coef || !par)
    return fail(RANGE_ERR_INVALID, "bad spherical-harmonics table (L=%d, entries=%d)", L, n_entries);
  c->sh = ShTable{L, n_entries, pref, off, coef, par};
  c->sh_off.assign(size_t(n_entries) + 1, 0);
  c->sh_par.assign(size_t(n_entries), 0);
  CUDA_TRY(cudaMemcpy(c->sh_off.data(), off, c->sh_off.size() * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(c->sh_par.data(), par, c->sh_par.size() * 4, cudaMemcpyDeviceToHost));
  for (int e = 0; e < n_entries; ++e)
    if (c->sh_off[e + 1] <= c->sh_off[e] || c->sh_off[e + 1] - c->sh_off[e] > 255) {
      c->sh = ShTable{};
      return fail(RANGE_ERR_INVALID, "spherical-harmonics table: entry %d has %d coefficients", e, c->sh_off[e + 1] - c->sh_off[e]);
    }
  c->enc_prepared = false;
  c->enc_precision = RANGE_ENC_F64;    // the prepared feature layout belonged to the previous table
  return RANGE_OK;
}

int range_ctx_set_sh_closed_form(range_ctx* c, int L, int n_entries, const double* norm) {
  if (!c || L <= 0 || n_entries != L * (L + 1) / 2 || !norm)
    return fail(RANGE_ERR_INVALID, "bad closed-form harmonics arguments (L=%d, entries=%d)", L, n_entries);
  c->sh = ShTable{};
  c->sh.L = L;
  c->sh.n_entries = n_entries;
  c->sh.pref = norm;              // "a table is set" marker for the entry checks; unused by the closed-form kernels
  c->sh.closed_form = 1;
  c->sh.norm = norm;
  c->sh_off.clear(); c->sh_par.clear();
  c->enc_prepared = false;
  c->enc_precision = RANGE_ENC_F64;
  return RANGE_OK;
}

int range_ctx_set_encoder(range_ctx* c, int n_layers, const int32_t* dims, const double* const* W,
                          const double* const* b, double w0_first, double w0_hidden) {
  if (!c || n_layers < 1 || !dims || !W || !b) return fail(RANGE_ERR_INVALID, "bad encoder arguments");
  for (int i = 0; i < n_layers; ++i) {
    if (dims[i] % 16 || dims[i + 1] % 64)
      return fail(RANGE_ERR_UNSUPPORTED, "layer %d: (%d -> %d) needs in %% 16 == 0 and out %% 64 == 0", i, dims[i],
                  dims[i + 1]);
    if (!W[i] || !b[i]) return fail(RANGE_ERR_INVALID, "layer %d has null weights", i);
  }
  if (dims[n_layers] != kDimK)
    return fail(RANGE_ERR_UNSUPPORTED, "embedding dim must be %d, got %d", kDimK, dims[n_layers]);
  c->n_layers = n_layers;
  c->dims.assign(dims, dims + n_layers + 1);
  c->W.assign(W, W + n_layers);
  c->b.assign(b, b + n_layers);
  c->w0_first = w0_first;
  c->w0_hidden = w0_hidden;
  c->enc_prepared = false;
  c->enc_precision = RANGE_ENC_F64;
  return RANGE_OK;
}

int range_ctx_set_db(range_ctx* c, int64_t M, int64_t Mpad, const void* Kh, const void* Vt, const float* xyz,
                     float vscale) {
  if (!c || M <= 0 || Mpad < M || Mpad % kBlockKeys || !Kh || !Vt || !xyz || !(vscale > 0.f))
    return fail(RANGE_ERR_INVALID, "bad database arguments (M=%lld, Mpad=%lld)", (long long)M, (long long)Mpad);
  if (M > (int64_t(1) << 30)) return fail(RANGE_ERR_UNSUPPORTED, "M too large");
  CUDA_TRY(cudaSetDevice(c->device));
  int r = make_tmap(&c->tmK128, Kh, uint64_t(Mpad), kDimK, 128);
  if (r) return r;
  r = make_tmap(&c->tmK64, Kh, uint64_t(Mpad), kDimK, 64);
  if (r) return r;
  r = make_tmap(&c->tmV128, Vt, kDimV, uint64_t(Mpad), 128);
  if (r) return r;
  c->M = M; c->Mpad = Mpad; c->Kh = Kh; c->Vt = Vt; c->xyz = xyz; c->vscale = vscale;
  c->caps = nullptr; c->M_total = M;
  return RANGE_OK;
}

int range_ctx_set_db_caps(range_ctx* c, int64_t n_tiles, const float* caps, int64_t M_total) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (!caps) { c->caps = nullptr; c->M_total = c->M; return RANGE_OK; }
  if (n_tiles != c->Mpad / kBlockKeys || M_total < c->M)
    return fail(RANGE_ERR_INVALID, "caps: %lld tiles for Mpad=%lld, M_total=%lld", (long long)n_tiles,
                (long long)c->Mpad, (long long)M_total);
  c->caps = caps;
  c->M_total = M_total;
  return RANGE_OK;
}

int range_geo_mask_shape(range_ctx* c, int64_t N, int32_t* rows, int32_t* words) {
  if (!c || !c->Kh || N <= 0 || !rows || !words) return fail(RANGE_ERR_INVALID, "bad arguments");
  const RetrievalPlan p = plan_retrieval(c, N);
  *rows = p.mask_rows;
  *words = p.mask_words;
  return RANGE_OK;
}

int range_geo_mask(range_ctx* c, int64_t N, const float* qxyz, float geo_temp, const float* sums, uint32_t* mask,
                   void* stream) {
  if (!c || !c->Kh || !c->caps) return fail(RANGE_ERR_INVALID, "database caps not set");
  if (N <= 0 || !qxyz || !mask || !(geo_temp > 0.f)) return fail(RANGE_ERR_INVALID, "bad arguments");
  const RetrievalPlan p = plan_retrieval(c, N);
  const float thr_ln = logf(float(c->M_total)) + 24.f * 0.6931471805599453f;
  CUDA_TRY(launch_geo_mask(qxyz, int(N), p.mask_rows, c->caps, int(c->Mpad / kBlockKeys), int(c->M), thr_ln / geo_temp, sums, thr_ln,
                           geo_temp, mask, p.mask_words, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

size_t range_sort_workspace_bytes(range_ctx* c, int64_t N) {
  if (!c || N <= 0 || N > (int64_t(1) << 30)) return 0;
  return sort_workspace_bytes(int(N));
}

int range_sort_queries(range_ctx* c, int64_t N, const double* lonlat, double* lonlat_sorted, int32_t* perm,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!c || N <= 0 || N > (int64_t(1) << 30) || !lonlat || !lonlat_sorted || !perm || !workspace)
    return fail(RANGE_ERR_INVALID, "bad arguments");
  if (workspace_bytes < sort_workspace_bytes(int(N))) return fail(RANGE_ERR_WORKSPACE, "sort workspace too small");
  CUDA_TRY(launch_sort_queries(lonlat, int(N), lonlat_sorted, perm, workspace, cudaStream_t(stream)));
  g_launches += sort_launches(int(N));
  return RANGE_OK;
}

int range_sh_features(range_ctx* c, int64_t N, const double* lonlat, double* Yt, int64_t ld, void* stream) {
  if (!c || !c->sh.pref) return fail(RANGE_ERR_INVALID, "spherical-harmonics table not set");
  if (N < 0 || ld < N || !lonlat || !Yt) return fail(RANGE_ERR_INVALID, "bad arguments");
  CUDA_TRY(launch_sh(c->sh, lonlat, int(N), Yt, size_t(ld), cudaStream_t(stream)));
  g_launches += N > 0;
  return RANGE_OK;
}

static bool tc_supported(const range_ctx* c) {
  if (!c || !c->n_layers) return false;
  for (int i = 0; i < c->n_layers; ++i)
    if (c->dims[i] % 64 || c->dims[i + 1] % 256) return false;
  return true;
}

size_t range_encoder_prepared_bytes(range_ctx* c) {
  if (!tc_supported(c) || !c->sh.pref || c->dims[0] != c->sh.L * c->sh.L) return 0;
  const ShLayout y = choose_sh_layout(c);
  size_t b = sh_layout_bytes(y);
  for (int i = 0; i < c->n_layers; ++i)
    b += 2 * align_up(size_t(i == 0 ? y.K0 : c->dims[i]) * c->dims[i + 1] * 2, 256);   // hi + lo fp16
  return b + 256;
}

int range_ctx_prepare_encoder(range_ctx* c, void* buf, size_t bytes, void* stream) {
  if (!c || !c->sh.pref || !c->n_layers) return fail(RANGE_ERR_INVALID, "encoder / SH table not set");
  if (!tc_supported(c)) return fail(RANGE_ERR_UNSUPPORTED, "tensor-core encoder needs layer widths %% 256 == 0 and inputs %% 64 == 0");
  if (!buf || bytes < range_encoder_prepared_bytes(c)) return fail(RANGE_ERR_WORKSPACE, "prepared-encoder buffer too small");
  const int L = c->sh.L, F = L * L;
  if (c->dims[0] != F) return fail(RANGE_ERR_INVALID, "encoder input dim %d != L*L", c->dims[0]);
  cudaStream_t s = cudaStream_t(stream);
  // feature layout of the first layer's input: column -> reference feature index l*l + l +- am (the weight columns
  // are permuted / zero-padded to match), column -> harmonics entry (raster combine), round table (sh_rounds_kernel)
  const ShLayout y = choose_sh_layout(c);
  char* p = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(buf), 256));
  int* dperm = reinterpret_cast<int*>(p); p += align_up(size_t(y.K0) * 4, 256);
  int* dfmap = reinterpret_cast<int*>(p); p += align_up(size_t(y.K0) * 4, 256);
  CUDA_TRY(cudaMemcpyAsync(dperm, y.perm.data(), size_t(y.K0) * 4, cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(dfmap, y.fmap.data(), size_t(y.K0) * 4, cudaMemcpyHostToDevice, s));
  c->sh.K0 = y.K0; c->sh.fmap = dfmap;
  c->sh.rounds = 0; c->sh.rtab = nullptr; c->sh.rtab_doubles = 0; c->sh.rmeta = nullptr; c->sh.rroff = nullptr;
  std::vector<double> tab;
  std::vector<int> meta;
  if (y.rounds) {
    const int E = c->sh.n_entries;
    std::vector<double> pref(E), coef(size_t(c->sh_off[E]));
    CUDA_TRY(cudaMemcpy(pref.data(), c->sh.pref, pref.size() * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(coef.data(), c->sh.coef, coef.size() * 8, cudaMemcpyDeviceToHost));
    std::vector<int> el, em;
    entry_lm(L, el, em);
    tab.assign(size_t(y.roff.back()), 0.0);
    meta.assign(size_t(y.rounds) * 32, 0);
    for (int r = 0; r < y.rounds; ++r) {
      const int nst = (y.roff[r + 1] - y.roff[r]) / 32 - 1;
      double* t = tab.data() + y.roff[r];
      for (int i = 0; i < 32; ++i) {
        const int e = y.order[r * 32 + i];
        if (e < 0) continue;                                   // unused slot: pref = 0, zero coefficients -> zero columns
        t[i] = em[e] == 0 ? 1.0 : pref[e];                     // |m| = 0: the per-query kernels emit the chain value itself
        const int len = c->sh_off[e + 1] - c->sh_off[e], pad = nst - len;
        for (int k = 0; k < len; ++k) t[32 * (1 + pad + k) + i] = coef[size_t(c->sh_off[e]) + k];
        meta[r * 32 + i] = em[e] | (c->sh_par[e] ? 0x100 : 0);
      }
    }
    double* dtab = reinterpret_cast<double*>(p); p += align_up(tab.size() * 8, 256);
    int* dmeta = reinterpret_cast<int*>(p); p += align_up(meta.size() * 4, 256);
    int* droff = reinterpret_cast<int*>(p); p += align_up(y.roff.size() * 4, 256);
    CUDA_TRY(cudaMemcpyAsync(dtab, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dmeta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(droff, y.roff.data(), y.roff.size() * 4, cudaMemcpyHostToDevice, s));
    c->sh.rounds = y.rounds; c->sh.rtab = dtab; c->sh.rtab_doubles = int(tab.size()); c->sh.rmeta = dmeta; c->sh.rroff = droff;
  }
  CUDA_TRY(cudaStreamSynchronize(s));          // the sources above are stack-lifetime host vectors
  c->perm = dperm;
  c->tmWh.assign(c->n_layers, CUtensorMap{}); c->tmWl.assign(c->n_layers, CUtensorMap{});
  c->tmWh2.assign(c->n_layers, CUtensorMap{}); c->tmWl2.assign(c->n_layers, CUtensorMap{});
  for (int i = 0; i < c->n_layers; ++i) {
    const int K_in = c->dims[i], K = i == 0 ? y.K0 : K_in, H = c->dims[i + 1];
    void* wh = p; p += align_up(size_t(K) * H * 2, 256);
    void* wl = p; p += align_up(size_t(K) * H * 2, 256);
    CUDA_TRY(launch_split_weights(c->W[i], H, K_in, K, i == 0 ? dperm : nullptr, wh, wl, s));
    g_launches += 1;
    int r = make_tmap(&c->tmWh[i], wh, uint64_t(H), uint64_t(K), 256);
    if (r) return r;
    r = make_tmap(&c->tmWl[i], wl, uint64_t(H), uint64_t(K), 256);
    if (r) return r;
    r = make_tmap(&c->tmWh2[i], wh, uint64_t(H), uint64_t(K), 128);
    if (r) return r;
    r = make_tmap(&c->tmWl2[i], wl, uint64_t(H), uint64_t(K), 128);
    if (r) return r;
  }
  c->enc_prepared = true;
  c->enc_precision = RANGE_ENC_F16X3;
  return RANGE_OK;
}

int range_ctx_set_encoder_precision(range_ctx* c, int mode) {
  if (!c) return fail(RANGE_ERR_INVALID, "null ctx");
  if (mode == RANGE_ENC_F16X3 && !c->enc_prepared) return fail(RANGE_ERR_INVALID, "call range_ctx_prepare_encoder first");
  if (mode != RANGE_ENC_F64 && mode != RANGE_ENC_F16X3) return fail(RANGE_ERR_INVALID, "unknown encoder precision %d", mode);
  c->enc_precision = mode;
  return RANGE_OK;
}

static size_t encode_ws_tc(const range_ctx* c, int64_t chunk) {
  size_t widest = 0;
  for (int i = 1; i < c->n_layers; ++i) widest = widest > size_t(c->dims[i]) ? widest : size_t(c->dims[i]);
  // features hi + lo, two ping-pong hidden buffers hi + lo (all fp16), row-major fp64 embedding
  return 2 * align_up(size_t(chunk) * c->sh.K0 * 2, 256) + 4 * align_up(size_t(chunk) * widest * 2, 256) +
         size_t(chunk) * kDimK * 8 + 1024;
}

size_t range_encode_workspace_bytes(range_ctx* c, int64_t N) {
  if (!c || !c->n_layers || N <= 0) return 0;
  if (c->enc_precision == RANGE_ENC_F16X3) return encode_ws_tc(c, N < kEncodeChunk ? N : kEncodeChunk);
  const int64_t chunk = N < kEncodeChunk ? N : kEncodeChunk;
  const size_t ld = align_up(size_t(chunk), 128);
  size_t widest = 0;
  for (int i = 1; i < c->n_layers; ++i) widest = widest > size_t(c->dims[i]) ? widest : size_t(c->dims[i]);
  // features + two ping-pong hidden buffers (feature-major) + row-major embedding
  return (size_t(c->dims[0]) + 2 * widest) * ld * 8 + size_t(chunk) * kDimK * 8 + 1024;
}

// Tensor-core encoder over N queries in chunks: features (per-point harmonics from `lonlat`, or - on a raster - the
// separable evaluation from `rt` / `ij`, which also writes the queries' coordinates to `lonlat_out`), SIREN, normalise.
static int encode_tc(range_ctx* c, int64_t N, const double* lonlat, const RasterTables* rt, const int32_t* ij,
                     double* lonlat_out, double* q64, void* q16, float* qxyz, void* workspace, cudaStream_t s) {
  const int64_t chunk = N < kEncodeChunk ? N : kEncodeChunk;
  size_t widest = 0;
  for (int i = 1; i < c->n_layers; ++i) widest = widest > size_t(c->dims[i]) ? widest : size_t(c->dims[i]);
  char* p = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  const int F = c->sh.K0;              // columns of the feature rows (ShTable::K0: L*L, or 64 per round)
  void* Yh = p; p += align_up(size_t(chunk) * F * 2, 256);
  void* Yl = p; p += align_up(size_t(chunk) * F * 2, 256);
  void* hid[2][2];
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) { hid[a][b] = p; p += align_up(size_t(chunk) * widest * 2, 256); }
  double* emb = reinterpret_cast<double*>(p);
  for (int64_t n0 = 0; n0 < N; n0 += chunk) {
    const int n = int(N - n0 < chunk ? N - n0 : chunk);
    const double* coords = rt ? lonlat_out + 2 * n0 : lonlat + 2 * n0;
    if (rt) CUDA_TRY(launch_raster_combine(c->sh, *rt, ij + 2 * n0, n, Yh, Yl, lonlat_out + 2 * n0, s));
    else CUDA_TRY(launch_sh_rowmajor(c->sh, coords, n, Yh, Yl, c->sm_count, s));
    const void *ah = Yh, *al = Yl;
    for (int i = 0; i < c->n_layers; ++i) {
      const bool last = i == c->n_layers - 1;
      const int K = i == 0 ? F : c->dims[i], H = c->dims[i + 1];
      CUtensorMap tmAh, tmAl;
      int r = make_tmap(&tmAh, ah, uint64_t(n), uint64_t(K), 128);
      if (r) return r;
      r = make_tmap(&tmAl, al, uint64_t(n), uint64_t(K), 128);
      if (r) return r;
      const double w0 = last ? 0.0 : (i == 0 ? c->w0_first : c->w0_hidden);
      void* oh = last ? nullptr : hid[i & 1][0];
      void* ol = last ? nullptr : hid[i & 1][1];
      if (siren_kernel_override() == 1)
        CUDA_TRY(launch_siren_tc(tmAh, tmAl, c->tmWh[i], c->tmWl[i], c->b[i], n, K, H, w0, oh, ol, last ? emb : nullptr, s));
      else
        CUDA_TRY(launch_siren_pair(tmAh, tmAl, c->tmWh2[i], c->tmWl2[i], c->b[i], n, K, H, w0, oh, ol, last ? emb : nullptr,
                                   c->sm_count, s));
      ah = hid[i & 1][0]; al = hid[i & 1][1];
    }
    CUDA_TRY(launch_normalize(emb, coords, n, kDimK, q64 + n0 * kDimK, kDimK,
                              reinterpret_cast<char*>(q16) + n0 * kDimK * 2, qxyz + n0 * 4, s));
    g_launches += 2 + c->n_layers;
  }
  return RANGE_OK;
}

int range_encode(range_ctx* c, int64_t N, const double* lonlat, double* q64, void* q16, float* qxyz,
                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!c || !c->sh.pref || !c->n_layers) return fail(RANGE_ERR_INVALID, "encoder not set");
  // the first layer may be zero-padded up to the next multiple of 16 input columns (L*L = 100 for SatCLIP-L10)
  const int F = c->sh.L * c->sh.L;
  if (c->dims[0] < F || c->dims[0] - F >= 16)
    return fail(RANGE_ERR_INVALID, "encoder input dim %d does not match L*L = %d", c->dims[0], F);
  if (c->dims[0] != F && c->enc_precision != RANGE_ENC_F64)
    return fail(RANGE_ERR_UNSUPPORTED, "padded first layer (%d > L*L = %d) needs the fp64 encoder", c->dims[0], F);
  if (N <= 0 || !lonlat || !q64 || !q16 || !qxyz) return fail(RANGE_ERR_INVALID, "bad arguments");
  if (workspace_bytes < range_encode_workspace_bytes(c, N) || !workspace)
    return fail(RANGE_ERR_WORKSPACE, "encode workspace too small");
  cudaStream_t s = cudaStream_t(stream);
  const int64_t chunk = N < kEncodeChunk ? N : kEncodeChunk;
  if (c->enc_precision == RANGE_ENC_F16X3)
    return encode_tc(c, N, lonlat, nullptr, nullptr, nullptr, q64, q16, qxyz, workspace, s);
  const size_t ld = align_up(size_t(chunk), 128);
  size_t widest = 0;
  for (int i = 1; i < c->n_layers; ++i) widest = widest > size_t(c->dims[i]) ? widest : size_t(c->dims[i]);
  double* Yt = reinterpret_cast<double*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  double* hid[2] = {Yt + size_t(c->dims[0]) * ld, Yt + (size_t(c->dims[0]) + widest) * ld};
  double* emb = Yt + (size_t(c->dims[0]) + 2 * widest) * ld;
  for (int64_t n0 = 0; n0 < N; n0 += chunk) {
    const int n = int(N - n0 < chunk ? N - n0 : chunk);
    CUDA_TRY(launch_sh(c->sh, lonlat + 2 * n0, n, Yt, ld, s));
    if (c->dims[0] > F)       // zero rows for the padded input columns of the first layer
      CUDA_TRY(cudaMemsetAsync(Yt + size_t(F) * ld, 0, size_t(c->dims[0] - F) * ld * sizeof(double), s));
    const double* in = Yt;
    for (int i = 0; i < c->n_layers; ++i) {
      const bool last = i == c->n_layers - 1;
      double* out = last ? emb : hid[i & 1];
      CUDA_TRY(launch_siren_layer(c->W[i], c->b[i], in, ld, c->dims[i + 1], c->dims[i], n,
                                  last ? 0.0 : (i == 0 ? c->w0_first : c->w0_hidden), out,
                                  last ? size_t(kDimK) : ld, last ? 1 : 0, s));
      in = out;
    }
    CUDA_TRY(launch_normalize(emb, lonlat + 2 * n0, n, kDimK, q64 + n0 * kDimK, kDimK,
                              reinterpret_cast<char*>(q16) + n0 * kDimK * 2, qxyz + n0 * 4, s));
    g_launches += 2 + c->n_layers;
  }
  return RANGE_OK;
}

static int raster_supported(const range_ctx* c) {
  if (!c || !c->sh.pref || !c->n_layers) return fail(RANGE_ERR_INVALID, "encoder not set");
  if (c->sh.closed_form)
    return fail(RANGE_ERR_UNSUPPORTED, "raster encoder: closed-form harmonics are not evaluated separably (use range_encode)");
  if (c->enc_precision != RANGE_ENC_F16X3 || c->dims[0] != c->sh.L * c->sh.L)
    return fail(RANGE_ERR_UNSUPPORTED, "raster encoder needs the tensor-core encoder (range_ctx_prepare_encoder)");
  return RANGE_OK;
}

size_t range_raster_tables_bytes(range_ctx* c, int64_t n_lat, int64_t n_lon) {
  if (!c || !c->sh.pref || n_lat <= 0 || n_lon <= 0) return 0;
  return raster_tables_bytes(c->sh.L, int(n_lat), int(n_lon)) + 256;
}

int range_raster_tables(range_ctx* c, int64_t n_lat, const double* lat, int64_t n_lon, const double* lon, void* tables,
                        size_t bytes, void* stream) {
  int r = raster_supported(c);
  if (r) return r;
  if (n_lat <= 0 || n_lon <= 0 || n_lat > (1 << 24) || n_lon > (1 << 24) || !lat || !lon || !tables)
    return fail(RANGE_ERR_INVALID, "bad arguments");
  if (bytes < range_raster_tables_bytes(c, n_lat, n_lon)) return fail(RANGE_ERR_WORKSPACE, "raster tables buffer too small");
  void* buf = reinterpret_cast<void*>(align_up(reinterpret_cast<size_t>(tables), 256));
  const RasterTables t = raster_tables_layout(c->sh.L, int(n_lat), int(n_lon), buf);
  CUDA_TRY(launch_raster_tables(c->sh, lat, lon, t, cudaStream_t(stream)));
  g_launches += 2;
  return RANGE_OK;
}

int range_raster_points(range_ctx* c, int64_t n_lat, int64_t n_lon, const void* tables, int64_t p0, int64_t N,
                        const int32_t* perm, int32_t* ij, double* lonlat, void* stream) {
  int r = raster_supported(c);
  if (r) return r;
  if (n_lat <= 0 || n_lon <= 0 || !tables || N <= 0 || N > (int64_t(1) << 30) || p0 < 0 || (!ij && !lonlat))
    return fail(RANGE_ERR_INVALID, "bad arguments");
  if (p0 + N > n_lat * n_lon) return fail(RANGE_ERR_INVALID, "points [%lld, %lld) outside the %lld x %lld raster", (long long)p0,
                                          (long long)(p0 + N), (long long)n_lat, (long long)n_lon);
  void* buf = reinterpret_cast<void*>(align_up(reinterpret_cast<size_t>(const_cast<void*>(tables)), 256));
  const RasterTables t = raster_tables_layout(c->sh.L, int(n_lat), int(n_lon), buf);
  CUDA_TRY(launch_raster_points(t, p0, int(N), perm, ij, lonlat, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

int range_encode_raster(range_ctx* c, int64_t n_lat, int64_t n_lon, const void* tables, int64_t N, const int32_t* ij,
                        double* lonlat, double* q64, void* q16, float* qxyz, void* workspace, size_t workspace_bytes,
                        void* stream) {
  int r = raster_supported(c);
  if (r) return r;
  if (n_lat <= 0 || n_lon <= 0 || !tables || N <= 0 || !ij || !lonlat || !q64 || !q16 || !qxyz)
    return fail(RANGE_ERR_INVALID, "bad arguments");
  if (workspace_bytes < range_encode_workspace_bytes(c, N) || !workspace)
    return fail(RANGE_ERR_WORKSPACE, "encode workspace too small");
  void* buf = reinterpret_cast<void*>(align_up(reinterpret_cast<size_t>(const_cast<void*>(tables)), 256));
  const RasterTables t = raster_tables_layout(c->sh.L, int(n_lat), int(n_lon), buf);
  return encode_tc(c, N, nullptr, &t, ij, lonlat, q64, q16, qxyz, workspace, cudaStream_t(stream));
}

size_t range_retrieve_workspace_bytes(range_ctx* c, int64_t N) {
  if (!c || !c->Kh || N <= 0) return 0;
  return plan_retrieval(c, N).total + 256;
}

int range_retrieve_stats(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                         float geo_temp, float* sums, float* maxs, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (!q16 || !qxyz || !sums || !maxs || !workspace) return fail(RANGE_ERR_INVALID, "null argument");
  if (N <= 0) return fail(RANGE_ERR_INVALID, "N must be positive");
  const RetrievalPlan p = plan_retrieval(c, N);
  if (workspace_bytes < p.total + 256) return fail(RANGE_ERR_WORKSPACE, "retrieve workspace too small");
  RetrievalArgs a;
  char* ws = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  cudaStream_t s = cudaStream_t(stream);
  int r = fill_args(c, mode, N, q16, qxyz, temp, geo_temp, p, ws, s, &a);
  if (r) return r;
  float* part_sum = p.stats_splits > 1 ? reinterpret_cast<float*>(ws + p.off_part_sum) : sums;
  float* part_max = p.stats_splits > 1 ? reinterpret_cast<float*>(ws + p.off_part_max) : maxs;
  if (p.stats_pc) CUDA_TRY(launch_stats_pc(a, part_sum, part_max, s));
  else CUDA_TRY(launch_stats(a, part_sum, part_max, s));
  g_launches += 1;
  if (p.stats_splits > 1) {
    CUDA_TRY(launch_reduce_stats(part_sum, part_max, int(N), p.stats_splits, sums, maxs, s));
    g_launches += 1;
  }
  return RANGE_OK;
}

// apply pass; the result goes either to O (N,1024) fp32 or, fused with the concat of range/range.py:222,240, to the
// caller's (N,1280) array `out` (rows through `perm`, fp32 or fp64) together with the location columns q64
static bool valid_out_dtype(int d) { return d == RANGE_OUT_F64 || d == RANGE_OUT_F32 || d == RANGE_OUT_PACKED; }

static int check_route(const range_route* r, int64_t N, RowRoute* out) {
  if (!r) return RANGE_OK;
  if (r->n_ranks < 1 || r->n_ranks > RANGE_MAX_RANKS || r->rank < 0 || r->rank >= r->n_ranks || r->slab_rows < 1)
    return fail(RANGE_ERR_INVALID, "route: %d ranks (max %d), rank %d, %lld rows per rank", r->n_ranks, RANGE_MAX_RANKS,
                r->rank, (long long)r->slab_rows);
  if (r->slab_rows % kBlockQ)
    return fail(RANGE_ERR_INVALID, "route: slab_rows (%lld) must be a multiple of %d (a query tile has one owner)",
                (long long)r->slab_rows, kBlockQ);
  if (N > int64_t(r->n_ranks) * r->slab_rows)
    return fail(RANGE_ERR_INVALID, "route: %lld rows do not fit %d ranks x %lld rows", (long long)N, r->n_ranks,
                (long long)r->slab_rows);
  out->n_ranks = r->n_ranks;
  out->rank = r->rank;
  out->slab = r->slab_rows;
  for (int i = 0; i < r->n_ranks; ++i) {
    if (!r->peer[i]) return fail(RANGE_ERR_INVALID, "route: receive buffer of rank %d is null", i);
    out->peer[i] = r->peer[i];
  }
  return RANGE_OK;
}

static int apply_impl(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp, float geo_temp,
                      float beta, const float* sums, const float* maxs, float* O, const double* q64, const int32_t* perm,
                      void* out, int out_dtype, const range_route* route, void* workspace, size_t workspace_bytes,
                      void* stream) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (!q16 || !qxyz || !sums || !maxs || !workspace || (!O && !(out && q64) && !route))
    return fail(RANGE_ERR_INVALID, "null argument");
  if (N <= 0) return fail(RANGE_ERR_INVALID, "N must be positive");
  if (mode == RANGE_MODE_RANGE_PLUS && !(beta >= 0.f && beta <= 1.f))
    return fail(RANGE_ERR_INVALID, "beta must be in [0,1]");
  if (out && !valid_out_dtype(out_dtype)) return fail(RANGE_ERR_INVALID, "unknown out dtype");
  RowRoute rr;
  if (int r0 = check_route(route, N, &rr)) return r0;
  const RetrievalPlan p = plan_retrieval(c, N);
  if (workspace_bytes < p.total + 256) return fail(RANGE_ERR_WORKSPACE, "retrieve workspace too small");
  RetrievalArgs a;
  char* ws = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  cudaStream_t s = cudaStream_t(stream);
  int r = fill_args(c, mode, N, q16, qxyz, temp, geo_temp, p, ws, s, &a, sums);
  if (r) return r;
  float* rowc = reinterpret_cast<float*>(ws + p.off_rowc);
  CUDA_TRY(launch_row_constants(sums, maxs, qxyz, int(N), a.geo, beta, a.a_sem, a.a_geo, 1.f / c->vscale, rowc, s));
  const size_t stride = size_t(N) * kDimV;
  const int W = kDimV + kDimK;
  if (p.pc) {
    CUtensorMap tmP;
    void* ring = ws + p.off_ring;
    r = make_tmap_rows2k(&tmP, ring, uint64_t(apply_pc_ring_rows(c->sm_count)));
    if (r) return r;
    if (route) {    // M-sharded: consumers store this shard's partial rows into the owner ranks' receive buffers
      CUDA_TRY(launch_apply_pc(a, tmP, rowc, nullptr, kDimV, 0, nullptr, &rr, ring, ws + p.off_flags, ws + p.off_pc_part,
                               ws + p.off_pc_scratch, c->sm_count, s));
    } else if (out) {      // consumers write straight into the (N,1280) result; the location columns follow
      if (out_dtype == RANGE_OUT_PACKED) {     // rows of 6144 B: 1024 fp32 features, then 256 fp64 location columns
        CUDA_TRY(launch_apply_pc(a, tmP, rowc, out, 1536, 0, perm, nullptr, ring, ws + p.off_flags, ws + p.off_pc_part,
                                 ws + p.off_pc_scratch, c->sm_count, s));
        CUDA_TRY(launch_concat_q(q64, int(N), kDimK, perm, out, 768, 512, RANGE_OUT_F64, s));
      } else {
        CUDA_TRY(launch_apply_pc(a, tmP, rowc, out, W, out_dtype == RANGE_OUT_F64, perm, nullptr, ring, ws + p.off_flags,
                                 ws + p.off_pc_part, ws + p.off_pc_scratch, c->sm_count, s));
        CUDA_TRY(launch_concat_q(q64, int(N), kDimK, perm, out, W, kDimV, out_dtype, s));
      }
      g_launches += 1;
    } else {
      CUDA_TRY(launch_apply_pc(a, tmP, rowc, O, kDimV, 0, nullptr, nullptr, ring, ws + p.off_flags, ws + p.off_pc_part,
                               ws + p.off_pc_scratch, c->sm_count, s));
    }
    g_launches += 2 + (apply_pc_part_bytes(c->sm_count, N, c->M) > 0);
    return RANGE_OK;
  }
  float* Odst = O ? O : reinterpret_cast<float*>(ws + p.off_O);
  float* part_out = p.splits > 1 ? reinterpret_cast<float*>(ws + p.off_part_out) : Odst;
  CUDA_TRY(launch_apply(a, rowc, part_out, stride, s));
  g_launches += 2;
  if (p.splits > 1) {
    CUDA_TRY(launch_reduce_out(part_out, stride, p.splits, stride, Odst, s));
    g_launches += 1;
  }
  if (route) {
    CUDA_TRY(launch_route_rows(Odst, int(N), rr, s));
    g_launches += 1;
  } else if (out) {
    CombineParts one;
    one.n = 1; one.p[0] = Odst; one.w[0] = 1.f;
    CUDA_TRY(launch_combine_concat(one, q64, int(N), perm, out, out_dtype, s));
    g_launches += 1;
  }
  return RANGE_OK;
}

int range_retrieve_apply(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                         float geo_temp, float beta, const float* sums, const float* maxs, float* O,
                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!O) return fail(RANGE_ERR_INVALID, "null argument");
  return apply_impl(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, maxs, O, nullptr, nullptr, nullptr, 0, nullptr,
                    workspace, workspace_bytes, stream);
}

int range_retrieve_apply_concat(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                                float geo_temp, float beta, const float* sums, const float* maxs, const double* q64,
                                const int32_t* perm, void* out, int out_dtype, void* workspace, size_t workspace_bytes,
                                void* stream) {
  if (!out || !q64) return fail(RANGE_ERR_INVALID, "null argument");
  return apply_impl(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, maxs, nullptr, q64, perm, out, out_dtype, nullptr,
                    workspace, workspace_bytes, stream);
}

int range_retrieve_concat(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp, float geo_temp,
                          float beta, const double* q64, const int32_t* perm, void* out, int out_dtype, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (!workspace) return fail(RANGE_ERR_INVALID, "null workspace");
  if (N <= 0) return fail(RANGE_ERR_INVALID, "N must be positive");
  const RetrievalPlan p = plan_retrieval(c, N);
  if (workspace_bytes < p.total + 256) return fail(RANGE_ERR_WORKSPACE, "retrieve workspace too small");
  char* ws = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  float* sums = reinterpret_cast<float*>(ws + p.off_sums);
  float* maxs = reinterpret_cast<float*>(ws + p.off_maxs);
  int r = range_retrieve_stats(c, mode, N, q16, qxyz, temp, geo_temp, sums, maxs, workspace, workspace_bytes, stream);
  if (r) return r;
  return range_retrieve_apply_concat(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, maxs, q64, perm, out, out_dtype,
                                     workspace, workspace_bytes, stream);
}

size_t range_topk_workspace_bytes(range_ctx* c, int64_t N, int k) {
  if (!c || !c->Kh || N <= 0 || N > (int64_t(1) << 30) || k < 1 || k > RANGE_TOPK_MAX) return 0;
  return plan_topk(c, N, k).total + 256;
}

// range_retrieve_topk (perm, k <= M, device rows) and range_retrieve_topk_rows (no perm, k past M, rows row0 + j)
static int topk_impl(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp, float geo_temp,
                     float beta, const float* sums, int k, const int32_t* perm, int64_t row0, int32_t* idx,
                     float* weight, void* workspace, size_t workspace_bytes, void* stream) {
  if (!q16 || !qxyz || !sums || !idx || !weight || !workspace) return fail(RANGE_ERR_INVALID, "null argument");
  if (N <= 0) return fail(RANGE_ERR_INVALID, "N must be positive");
  if (mode == RANGE_MODE_RANGE_PLUS && !(beta >= 0.f && beta <= 1.f))
    return fail(RANGE_ERR_INVALID, "beta must be in [0,1]");
  if (workspace_bytes < range_topk_workspace_bytes(c, N, k)) return fail(RANGE_ERR_WORKSPACE, "top-k workspace too small");
  const TopkPlan t = plan_topk(c, N, k);
  RetrievalArgs a;
  char* ws = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  cudaStream_t s = cudaStream_t(stream);
  int r = fill_args(c, mode, N, q16, qxyz, temp, geo_temp, t.ret, ws, s, &a, sums);     // apply-pass geo-skip mask
  if (r) return r;
  CUDA_TRY(launch_topk(a, t.splits, t.tiles_per_split, sums, beta, k, reinterpret_cast<float*>(ws + t.off_w),
                       reinterpret_cast<int32_t*>(ws + t.off_idx), perm, int(row0), idx, weight, s));
  g_launches += 2;
  return RANGE_OK;
}

int range_retrieve_topk(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                        float geo_temp, float beta, const float* sums, int k, const int32_t* perm, int32_t* idx,
                        float* weight, void* workspace, size_t workspace_bytes, void* stream) {
  static_assert(RANGE_TOPK_MAX == kTopkMax, "topk.cu list buckets");
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (k < 1 || k > RANGE_TOPK_MAX || k > c->M)
    return fail(RANGE_ERR_INVALID, "k = %d: need 1 <= k <= %d and k <= M = %lld", k, RANGE_TOPK_MAX, (long long)c->M);
  return topk_impl(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, k, perm, 0, idx, weight, workspace,
                   workspace_bytes, stream);
}

int range_retrieve_topk_rows(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                             float geo_temp, float beta, const float* sums, int k, int64_t row0, int32_t* idx,
                             float* weight, void* workspace, size_t workspace_bytes, void* stream) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (k < 1 || k > RANGE_TOPK_MAX) return fail(RANGE_ERR_INVALID, "k = %d: need 1 <= k <= %d", k, RANGE_TOPK_MAX);
  if (row0 < 0 || row0 + c->M > int64_t(INT32_MAX))
    return fail(RANGE_ERR_INVALID, "row0 = %lld: rows row0 .. row0 + M - 1 must be int32", (long long)row0);
  return topk_impl(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, k, nullptr, row0, idx, weight, workspace,
                   workspace_bytes, stream);
}

int range_topk_merge(range_ctx* c, int n_parts, int64_t N, int k, const float* part_w, const int32_t* part_idx,
                     const int32_t* perm, int32_t* idx, float* weight, void* stream) {
  if (!c || !part_w || !part_idx || !idx || !weight) return fail(RANGE_ERR_INVALID, "null argument");
  if (n_parts < 1 || n_parts > RANGE_MAX_RANKS) return fail(RANGE_ERR_INVALID, "n_parts must be in [1, %d]", RANGE_MAX_RANKS);
  if (N <= 0 || N > (int64_t(1) << 30)) return fail(RANGE_ERR_INVALID, "N must be in [1, 2^30]");
  if (k < 1 || k > RANGE_TOPK_MAX) return fail(RANGE_ERR_INVALID, "k = %d: need 1 <= k <= %d", k, RANGE_TOPK_MAX);
  CUDA_TRY(launch_topk_merge(part_w, part_idx, n_parts, int(N), k, perm, 0, idx, weight, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

int range_retrieve_apply_routed(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                                float geo_temp, float beta, const float* sums, const float* maxs, const range_route* route,
                                void* workspace, size_t workspace_bytes, void* stream) {
  if (!route) return fail(RANGE_ERR_INVALID, "null route");
  return apply_impl(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, maxs, nullptr, nullptr, nullptr, nullptr, 0, route,
                    workspace, workspace_bytes, stream);
}

int range_combine_concat(range_ctx* c, int64_t N, int n_parts, const float* const* parts, const float* weights,
                         const double* q64, const int32_t* perm, void* out, int out_dtype, void* stream) {
  if (!c || N <= 0 || N > (int64_t(1) << 30) || !parts || !q64 || !out) return fail(RANGE_ERR_INVALID, "bad arguments");
  if (n_parts < 1 || n_parts > kMaxParts) return fail(RANGE_ERR_INVALID, "n_parts must be in [1, %d]", kMaxParts);
  if (!valid_out_dtype(out_dtype)) return fail(RANGE_ERR_INVALID, "unknown out dtype");
  CombineParts cp;
  cp.n = n_parts;
  for (int k = 0; k < n_parts; ++k) {
    if (!parts[k]) return fail(RANGE_ERR_INVALID, "part %d is null", k);
    cp.p[k] = parts[k];
    cp.w[k] = weights ? weights[k] : 1.f;
  }
  CUDA_TRY(launch_combine_concat(cp, q64, int(N), perm, out, out_dtype, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

int range_sweep_concat(range_ctx* c, int64_t N, int n_slots, const float* const* geo, const float* const* sem,
                       int n_betas, const float* w_geo, const float* w_sem, const double* q64, const int32_t* perm,
                       void* const* outs, int out_dtype, void* stream) {
  static_assert(RANGE_MAX_RANKS == kMaxRanks && RANGE_SWEEP_MAX_BETAS == kSweepMaxBetas, "merge.cu: SweepParts");
  if (!c || !geo || !sem || !w_geo || !w_sem || !q64 || !outs) return fail(RANGE_ERR_INVALID, "null argument");
  if (N <= 0 || N > (int64_t(1) << 30)) return fail(RANGE_ERR_INVALID, "N must be in [1, 2^30]");
  if (n_slots < 1 || n_slots > RANGE_MAX_RANKS) return fail(RANGE_ERR_INVALID, "n_slots must be in [1, %d]", RANGE_MAX_RANKS);
  if (n_betas < 1 || n_betas > RANGE_SWEEP_MAX_BETAS)
    return fail(RANGE_ERR_INVALID, "n_betas must be in [1, %d]", RANGE_SWEEP_MAX_BETAS);
  if (out_dtype != RANGE_OUT_F64 && out_dtype != RANGE_OUT_F32)
    return fail(RANGE_ERR_INVALID, "out dtype must be RANGE_OUT_F64 or RANGE_OUT_F32");
  SweepParts sp;
  sp.n_slots = n_slots;
  sp.n_betas = n_betas;
  for (int k = 0; k < n_slots; ++k) {
    if (!geo[k] || !sem[k]) return fail(RANGE_ERR_INVALID, "slot %d is null", k);
    sp.geo[k] = geo[k];
    sp.sem[k] = sem[k];
  }
  for (int b = 0; b < n_betas; ++b) {
    if (!outs[b]) return fail(RANGE_ERR_INVALID, "output %d is null", b);
    sp.w_geo[b] = w_geo[b];
    sp.w_sem[b] = w_sem[b];
    sp.out[b] = outs[b];
  }
  CUDA_TRY(launch_sweep_concat(sp, q64, int(N), perm, out_dtype, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

/* ---- peer memory (receive buffers of an M-sharded database) ---- */
int range_peer_alloc(size_t bytes, void** dptr, unsigned char* handle64) {
  if (!bytes || !dptr || !handle64) return fail(RANGE_ERR_INVALID, "bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return fail(RANGE_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
  }
  memcpy(handle64, &h, 64);
  *dptr = p;
  return RANGE_OK;
}

int range_peer_open(const unsigned char* handle64, void** dptr) {
  if (!handle64 || !dptr) return fail(RANGE_ERR_INVALID, "bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  CUDA_TRY(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RANGE_OK;
}

int range_peer_close(void* dptr) {
  if (!dptr) return fail(RANGE_ERR_INVALID, "null pointer");
  CUDA_TRY(cudaIpcCloseMemHandle(dptr));
  return RANGE_OK;
}

int range_peer_free(void* dptr) {
  if (!dptr) return fail(RANGE_ERR_INVALID, "null pointer");
  CUDA_TRY(cudaFree(dptr));
  return RANGE_OK;
}

int range_retrieve(range_ctx* c, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                   float geo_temp, float beta, float* O, void* workspace, size_t workspace_bytes, void* stream) {
  if (!c || !c->Kh) return fail(RANGE_ERR_INVALID, "database not set");
  if (!workspace) return fail(RANGE_ERR_INVALID, "null workspace");
  if (N <= 0) return fail(RANGE_ERR_INVALID, "N must be positive");
  const RetrievalPlan p = plan_retrieval(c, N);
  if (workspace_bytes < p.total + 256) return fail(RANGE_ERR_WORKSPACE, "retrieve workspace too small");
  char* ws = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 256));
  float* sums = reinterpret_cast<float*>(ws + p.off_sums);
  float* maxs = reinterpret_cast<float*>(ws + p.off_maxs);
  int r = range_retrieve_stats(c, mode, N, q16, qxyz, temp, geo_temp, sums, maxs, workspace, workspace_bytes, stream);
  if (r) return r;
  return range_retrieve_apply(c, mode, N, q16, qxyz, temp, geo_temp, beta, sums, maxs, O, workspace,
                              workspace_bytes, stream);
}

int range_concat_scatter(range_ctx* c, int64_t N, const float* O, const double* q64, const int32_t* perm, void* out,
                         int out_dtype, void* stream) {
  if (!c || N <= 0 || !O || !q64 || !out) return fail(RANGE_ERR_INVALID, "bad arguments");
  if (!valid_out_dtype(out_dtype)) return fail(RANGE_ERR_INVALID, "unknown out dtype");
  CombineParts one;
  one.n = 1; one.p[0] = O; one.w[0] = 1.f;
  CUDA_TRY(launch_combine_concat(one, q64, int(N), perm, out, out_dtype, cudaStream_t(stream)));
  g_launches += 1;
  return RANGE_OK;
}

int range_concat(range_ctx* c, int64_t N, const float* O, const double* q64, void* out, int out_dtype,
                 void* stream) {
  return range_concat_scatter(c, N, O, q64, nullptr, out, out_dtype, stream);
}

}  // extern "C"
