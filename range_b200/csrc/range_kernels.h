// Internal launch interface between the C-ABI layer (capi.cu) and the kernels.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace rangeb200 {

// ---- K1: spherical harmonics (encoder.cu) -----------------------------------------------------
struct ShTable {
  int L = 0;
  int n_entries = 0;
  const double* pref = nullptr;   // [n_entries]           entries ordered |m|-major: for am: for l >= am
  const int* off = nullptr;       // [n_entries + 1]
  const double* coef = nullptr;   // Horner coefficients in c^2, highest power first
  const int* par = nullptr;       // [n_entries] polynomial parity
  // harmonics_calculation == 'closed-form' (spherical_harmonics_closed_form.py): no polynomial table, only the
  // normalisation factors (sqrt(2) *) SH_renormalization(l, |m|), |m|-major like the entries above
  int closed_form = 0;
  const double* norm = nullptr;   // [n_entries]
  // ---- set by range_ctx_prepare_encoder (tensor-core encoder): the feature layout of the first layer's input ----
  // K0 columns per query row (a multiple of 64); fmap[f] = entry | |m| << 16 | is_sin << 24, or kShZeroSlot for a
  // column that is always zero.  Two layouts:
  //   production order (closed-form harmonics, or a table too large for shared memory): K0 = L*L, for am: for l >= am:
  //     cos, then sin (am > 0);
  //   rounds (sh_rounds_kernel): the entries sorted by Horner-chain length, 32 per round; round r, lane i owns columns
  //     64 r + 2 i (cos) and 64 r + 2 i + 1 (sin): K0 = 64 * ceil(n_entries / 32), one 128-byte k-block per round.
  int K0 = 0;
  const int* fmap = nullptr;      // [K0]
  int rounds = 0;                 // > 0: rounds layout
  const double* rtab = nullptr;   // per round: pref[32], then coef[nsteps][32] (leading zeros pad shorter chains)
  int rtab_doubles = 0;
  const int* rmeta = nullptr;     // [rounds][32]  |m| | parity << 8
  const int* rroff = nullptr;     // [rounds + 1]  offsets into rtab (doubles)
};
constexpr int kShZeroSlot = 1 << 25;
// dynamic shared memory sh_rounds_kernel needs for this table (0: no rounds layout)
size_t sh_rounds_smem_bytes(int L, int rounds, int rtab_doubles);
// Yt[f * ld + n] for f < L*L, n < N   (feature-major so a thread per query writes coalesced)
cudaError_t launch_sh(const ShTable& t, const double* lonlat, int N, double* Yt, size_t ld, cudaStream_t s);

// ---- K1b: SIREN layer  out = act(W . Xt + b) (encoder.cu) ---------------------------------------
// W [H][K] row-major, Xt [K][ldx] feature-major.  out_rowmajor == 0: out[h * ldo + n]; 1: out[n * ldo + h].
// act_w0 > 0: sin(act_w0 * v); act_w0 == 0: identity.   Requires H % 64 == 0, K % 16 == 0.
cudaError_t launch_siren_layer(const double* W, const double* b, const double* Xt, size_t ldx, int H, int K, int N,
                               double act_w0, double* out, size_t ldo, int out_rowmajor, cudaStream_t s);

// ---- K1/K1b on the tensor cores: split-precision (3 x fp16) tcgen05 GEMMs (encoder_tc.cu) ------------------
// features as hi/lo fp16, row-major [N][t.K0], in the layout t.fmap describes (rounds or production order)
cudaError_t launch_sh_rowmajor(const ShTable& t, const double* lonlat, int N, void* Yh, void* Yl, int sm_count,
                               cudaStream_t s);
// W fp64 [H][K_in] -> hi/lo fp16 of 2^10 W, [H][K]; output column f = input column perm[f] (zero when perm[f] < 0;
// perm == null: K == K_in, identity)
cudaError_t launch_split_weights(const double* W, int H, int K_in, int K, const int* perm, void* Wh, void* Wl,
                                 cudaStream_t s);
// out = act(A . B^T + bias): A hi/lo [N][K], B hi/lo [H][K] (tensor maps: fp16, box [rows x 64], SWIZZLE_128B);
// act_w0 > 0 -> sin(act_w0 x) written as hi/lo fp16 [N][H]; out_f64 != null -> plain fp64 [N][H]
cudaError_t launch_siren_tc(const CUtensorMap& tmAh, const CUtensorMap& tmAl, const CUtensorMap& tmBh,
                            const CUtensorMap& tmBl, const double* bias, int N, int K, int H, double act_w0,
                            void* out_hi, void* out_lo, double* out_f64, cudaStream_t s);
// the same layer on persistent CTA pairs (cta_group::2): B tensor maps with box [128 rows x 64], A as above
cudaError_t launch_siren_pair(const CUtensorMap& tmAh, const CUtensorMap& tmAl, const CUtensorMap& tmBh,
                              const CUtensorMap& tmBl, const double* bias, int N, int K, int H, double act_w0,
                              void* out_hi, void* out_lo, double* out_f64, int sm_count, cudaStream_t s);

// ---- K1 on a lat/lon raster: separable evaluation, bit-identical to launch_sh_rowmajor (encoder_raster.cu) ----
struct RasterTables {
  int H = 0, W = 0;               // distinct latitudes / longitudes
  double* leg = nullptr;          // [H][L(L+1)/2]   latitude factor of every (l, |m|), |m|-major
  void* trig = nullptr;           // [W][L] double2  (cos |m| phi, sin |m| phi)
  double* lat = nullptr;          // [H] degrees
  double* lon = nullptr;          // [W] degrees
};
size_t raster_tables_bytes(int L, int H, int W);
RasterTables raster_tables_layout(int L, int H, int W, void* buf);     // buf 256-byte aligned
cudaError_t launch_raster_tables(const ShTable& sh, const double* lat, const double* lon, const RasterTables& t,
                                 cudaStream_t s);
// raster points p0 + (perm ? perm[n] : n), n < N (point p = i * W + j): ij (N,2) and / or lonlat (N,2), either may be null
cudaError_t launch_raster_points(const RasterTables& t, long long p0, int N, const int32_t* perm, int32_t* ij,
                                 double* lonlat, cudaStream_t s);
// ij (N,2) int32 = (latitude index, longitude index) -> features hi/lo fp16 [N][sh.K0] (layout sh.fmap), lonlat (N,2) fp64
cudaError_t launch_raster_combine(const ShTable& sh, const RasterTables& t, const int32_t* ij, int N, void* Yh, void* Yl,
                                  double* lonlat, cudaStream_t s);

// ---- K3: normalise / concat (encoder.cu) ----------------------------------------------------------
// e [N][D] fp64 row-major -> q64 [N][D] (ld = ldq), q16 [N][D] fp16, qxyz [N][4] fp32 from lonlat
cudaError_t launch_normalize(const double* e, const double* lonlat, int N, int D, double* q64, size_t ldq,
                             void* q16, float* qxyz, cudaStream_t s);
// only the location columns: out[perm ? perm[n] : n][col0 .. col0 + DQ) = q64[n]  (row length ld)
cudaError_t launch_concat_q(const double* q64, int N, int DQ, const int* perm, void* out, int ld, int col0, int dtype,
                            cudaStream_t s);

// ---- merging partial retrieved features: M-sharded databases, beta sweeps (merge.cu) ------------------------
constexpr int kMaxRanks = 8, kMaxParts = 8;
// Where the rows of an M-sharded apply pass go: row n belongs to rank n / slab and is stored (fp32, D wide) in that
// rank's receive buffer [n_ranks][slab][D] at slot `rank` - peer[r] is rank r's buffer as mapped into this process
// (NVLink peer memory; for r == rank the local buffer).  n_ranks == 0: no routing.  route_row: D = 1024 (the
// producer/consumer epilogue); launch_reduce_route takes D as an argument.
struct RowRoute {
  int n_ranks = 0, rank = 0;
  long long slab = 0;
  float* peer[kMaxRanks] = {};
};
__device__ __forceinline__ float* route_row(const RowRoute& r, int n) {
  int owner = int(n / r.slab);
  owner = owner < r.n_ranks ? owner : r.n_ranks - 1;            // padding rows (never stored) must not index past peer[]
  return r.peer[owner] + (size_t(r.rank) * size_t(r.slab) + size_t(n - owner * r.slab)) * 1024;
}
struct CombineParts {
  int n = 0;
  const float* p[kMaxParts] = {};
  float w[kMaxParts] = {};
};
// value width D, parts (N,D) fp32: out[perm ? perm[n] : n] = [sum_k w[k] p[k][n][0:D] | q64[n][0:256]]; dtype 0: fp64
// (N,D+256), 1: fp32 (N,D+256), 2: packed rows of packed_row_bytes(D) (D fp32 padded to a multiple of 4, 256 fp64)
__host__ __device__ inline size_t packed_row_bytes(int D) { return size_t((D + 3) / 4 * 4) * 4 + 256 * 8; }
cudaError_t launch_combine_concat(const CombineParts& parts, const double* q64, int N, int D, const int* perm, void* out,
                                  int dtype, cudaStream_t s);
// rows [n0, n0 + rows) of an apply pass, value width D (D % 4 == 0): part [splits][rows][D] fp32 (split k at
// part + k * split_stride floats) summed in split order (reduce_out's additions) -> the owners' receive buffers
cudaError_t launch_reduce_route(const float* part, size_t split_stride, int splits, long long n0, int rows, int D,
                                const RowRoute& route, cudaStream_t s);
// a beta sweep's last step: the geographic (beta 0) and semantic (beta 1) ends, each as n_slots partial slots
constexpr int kSweepMaxBetas = 8;
struct SweepParts {
  int n_slots = 0, n_betas = 0;
  const float* geo[kMaxRanks] = {};
  const float* sem[kMaxRanks] = {};
  float w_geo[kSweepMaxBetas] = {};
  float w_sem[kSweepMaxBetas] = {};
  void* out[kSweepMaxBetas] = {};
};
// G = sum of the geo slots, S = sum of the sem slots (slot order); for every b < n_betas:
// out[b][perm ? perm[n] : n] = [fmaf(w_sem[b], S[n], w_geo[b] * G[n]) | q64[n]]; slots (N,D) fp32; dtype 0: fp64
// (N,D+256), 1: fp32 (N,D+256)
cudaError_t launch_sweep_concat(const SweepParts& parts, const double* q64, int N, int D, const int* perm, int dtype,
                                cudaStream_t s);

// ---- spatial batching of the queries (sort.cu) ----------------------------------------------------
size_t sort_workspace_bytes(int N);
int sort_launches(int N);     // kernels launch_sort_queries issues
// perm[i] = caller's row of sorted row i; lonlat_sorted[i] = lonlat[perm[i]]  (stable sort by cell: a pure function of lonlat)
cudaError_t launch_sort_queries(const double* lonlat, int N, double* lonlat_sorted, int32_t* perm, void* workspace,
                                cudaStream_t s);

// ---- K2: retrieval (retrieval.cu) ---------------------------------------------------------------
struct RetrievalArgs {
  CUtensorMap tmQ;      // queries, box [128 rows x 64 dims]
  CUtensorMap tmK128;   // keys, box [128 entries x 64 dims]
  CUtensorMap tmK64;    // keys, box [64 entries x 64 dims]          (CTA-pair kernel: half a K tile per CTA)
  CUtensorMap tmV128;   // values^T, box [128 dims x 64 entries]    (CTA-pair kernel: half a Vt tile per CTA)
  // split-fp16 retrieval (split != 0): the lo halves Kl / Vtl with the same boxes as tmK128 / tmK64 / tmV128;
  // q16 rows are then 512 halves [hi | lo] and tmQ covers all 512 columns
  CUtensorMap tmKl128, tmKl64, tmVl128;
  int split;
  const __half* q16;
  const float4* db_xyz;
  const float4* q_xyz;
  int N, M;
  int geo;
  int stats_splits, stats_tiles_per_split;   // 128-entry tiles
  int apply_splits, apply_tiles_per_split;   // 128-entry tiles
  float a_sem, a_geo;   // temperature * log2(e)
  const uint32_t* geo_mask;   // [query tiles][mask_words] skip bits per 128-entry database tile, or null
  int mask_words;
};
void set_profile_buffer(long long* device_buffer_of_64);   // debug: wait-cycle accounting of the apply kernel
int retrieval_stats_smem_bytes();
int retrieval_apply_smem_bytes();
cudaError_t launch_stats(const RetrievalArgs& a, float* part_sum, float* part_max, cudaStream_t s);
// skip bits from the query tiles' and database tiles' bounding caps (retrieval.cu: geo_mask_kernel)
// sums (N,2) != null: use the known geo normalisers (apply pass), thr_ln = ln M_total + 24 ln 2
cudaError_t launch_geo_mask(const float* q_xyz, int N, int rows, const float* caps, int n_tiles, int M, float delta,
                            const float* sums, float thr_ln, float geo_temp, uint32_t* mask, int words, cudaStream_t s);
cudaError_t launch_reduce_stats(const float* part_sum, const float* part_max, int N, int splits, float* sums,
                                float* maxs, cudaStream_t s);
cudaError_t launch_row_constants(const float* sums, const float* maxs, const float* q_xyz, int N, int geo,
                                 float beta, float a_sem, float a_geo, float inv_vscale, float* rowc, cudaStream_t s);
// the CTA-pair apply kernel over ceil(dim_v / 256) value slices (Vt padded to whole slices); row n of split k's
// result at out + k * out_split_stride + n * out_ld, columns >= dim_v not stored
cudaError_t launch_apply(const RetrievalArgs& a, const float* rowc, float* out, size_t out_split_stride, int out_ld,
                         int dim_v, cudaStream_t s);
// role-specialised persistent apply kernel for large batches (retrieval_pc.cu): P' computed once per tile pair by
// producer CTAs, handed to the value-slice consumers through an L2-resident ring
int apply_pc_units(int sm_count);
size_t apply_pc_ring_bytes(int sm_count);
size_t apply_pc_flag_bytes(int sm_count, int64_t N, int64_t M);
int apply_pc_ring_rows(int sm_count);          // ring as a 2-D tensor [rows][2 KB]
size_t apply_pc_part_bytes(int sm_count, int64_t N, int64_t M);
void apply_pc_describe_plan(int sm_count, int64_t N, int64_t M, int32_t out[7]);   // test hook   // partial outputs of the split tail pairs
// row n of the result goes to out + (perm ? perm[n] : n) * out_ld (+ column), fp32 or fp64
// (out_ld in elements of the output type); route != null: rows go to the owners' receive buffers instead (fp32)
cudaError_t launch_apply_pc(const RetrievalArgs& a, const CUtensorMap& tmP, const float* rowc, void* out, int out_ld,
                            int out_f64, const int* perm, const RowRoute* route, void* ring, void* flags, void* part,
                            void* scratch, int sm_count, cudaStream_t s);
size_t apply_pc_scratch_bytes(int sm_count);   // consumers' accumulation-window scratch
// statistics pass with the producer's structure (retrieval_pc.cu); same partials as launch_stats
cudaError_t launch_stats_pc(const RetrievalArgs& a, float* part_sum, float* part_max, cudaStream_t s);
cudaError_t launch_reduce_out(const float* part, size_t split_stride, int splits, size_t total, float* out,
                              cudaStream_t s);
// q64 (N,256) fp64 -> q16x2 (N,512) fp16 rows [hi | lo]: hi = rn_f16(q) (range_encode's q16), lo = rn_f16(q - hi)
cudaError_t launch_split_queries(const double* q64, int N, void* q16x2, cudaStream_t s);

// ---- retrieval neighbours: the k largest retrieval weights per query (topk.cu) ------------------------------------
constexpr int kTopkMax = 32, kTopkMaxSplits = 64;
// a.geo selects RANGE+ (a.geo_mask: the apply-pass mask or null); sums (N,2) from the statistics pass.  Database split
// `split` covers tiles [split * tiles_per_split, ..); partial lists part_w / part_idx [2 * splits][N][k]; result row n
// (k entries, descending weight, then ascending entry) -> idx / weight row perm[n] (perm null: n); a found entry j is
// stored as row0 + j, an unfilled slot (fewer than k entries) as -1 with weight 0
cudaError_t launch_topk(const RetrievalArgs& a, int splits, int tiles_per_split, const float* sums, float beta, int k,
                        float* part_w, int32_t* part_idx, const int32_t* perm, int row0, int32_t* idx, float* weight,
                        cudaStream_t s);
// the merge step alone: `parts` lists [parts][N][k], each sorted by weight descending then entry, -1 entries last
cudaError_t launch_topk_merge(const float* part_w, const int32_t* part_idx, int parts, int N, int k,
                              const int32_t* perm, int row0, int32_t* idx, float* weight, cudaStream_t s);

}  // namespace rangeb200
