/* range_b200 - C ABI of the B200-native RANGE / RANGE+ embedding hot path.
 *
 * The reference (mvrl/RANGE) has no FFI: the path sits behind the Python API
 *     load_model(model_name, pretrained_path, device, db_path=..., beta=...)   range/load_model.py:16-51
 *     model(locs) -> np.ndarray (N, 1280) float64                              range/range.py:206-242
 * range_b200/load_model.py keeps that API and binds this library with ctypes (INTEGRATION.md shows the
 * stub).  Each entry point below names the reference lines it replaces.
 *
 * Conventions: extern "C", plain pointers and sizes only.  Every function returns 0 on success or a
 * negative RANGE_ERR_* code; range_last_error() gives the thread-local message.  All data pointers are
 * DEVICE pointers owned by the caller (e.g. the PyTorch allocator) unless marked "host".  `stream` is a
 * cudaStream_t passed as void*.  The library allocates no device memory: scratch comes from the caller
 * (range_*_workspace_bytes).  One ctx per device; calls on one ctx must be serialised by the caller.
 */
#ifndef RANGE_B200_H
#define RANGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RANGE_OK 0
#define RANGE_ERR_INVALID (-1)     /* bad argument / state (e.g. database not set)   */
#define RANGE_ERR_CUDA (-2)        /* a CUDA runtime / driver call failed            */
#define RANGE_ERR_WORKSPACE (-3)   /* workspace too small                            */
#define RANGE_ERR_UNSUPPORTED (-4) /* shape outside what the kernels are built for   */

#define RANGE_MODE_RANGE 0      /* one softmax, temperature 15        range/range.py:102-105 */
#define RANGE_MODE_RANGE_PLUS 1 /* semantic (12) + geographic (40)     range/range.py:107-112 */

#define RANGE_OUT_F64 0
#define RANGE_OUT_F32 1
#define RANGE_OUT_PACKED 2 /* rows of 6144 B: 1024 fp32 feature columns, then 256 fp64 location columns - every bit of
                              information of the reference's float64 row (its feature columns are fp32 values widened,
                              range/range.py:222,240) in 60 % of the bytes; range_host_unpack widens on the host.
                              For a database of value width D (range_ctx_set_db_values) a row is 4 round_up(D, 4) bytes
                              of fp32 features (D columns, then zero padding: the fp64 part stays 16-byte aligned),
                              then 256 fp64 location columns - 6144 B for D = 1024 */

typedef struct range_ctx range_ctx;

const char* range_last_error(void);
int range_version(void);

/* lifetime */
int range_ctx_create(int device, range_ctx** out);
int range_ctx_destroy(range_ctx* ctx);

/* Spherical-harmonics coefficient table (range_b200/sh_table.py:build_table) - replaces the generated
 * spherical_harmonics_ylm.py the reference imports at positional_encoding/spherical_harmonics.py:3.
 * Borrowed device arrays; entries ordered |m|-major. */
int range_ctx_set_sh_table(range_ctx* ctx, int L, int n_entries, const double* pref, const int32_t* off,
                           const double* coef, const int32_t* par);

/* harmonics_calculation == 'closed-form' checkpoints (positional_encoding/spherical_harmonics_closed_form.py:8-40):
 * associated-Legendre recurrence instead of the generated polynomials.  norm: device array of L (L + 1) / 2
 * factors, |m|-major (for am: for l >= am): SH_renormalization(l, am), times sqrt(2) for am > 0.  Borrowed. */
int range_ctx_set_sh_closed_form(range_ctx* ctx, int L, int n_entries, const double* norm);

/* SIREN weights - replaces SirenNet's parameters, location_encoder.py:73-112 (checkpoint keys
 * model.location.nnet.layers.{i}.{weight,bias}, model.location.nnet.last_layer.{weight,bias}).
 * dims: host array of n_layers+1 ints (dims[0] == L*L); W, b: host arrays of n_layers device pointers,
 * W[i] is (dims[i+1], dims[i]) row-major fp64.  All but the last layer apply sin(w0 * x), w0 = w0_first
 * for layer 0 and w0_hidden after (location_encoder.py:80-83,119). */
int range_ctx_set_encoder(range_ctx* ctx, int n_layers, const int32_t* dims, const double* const* W,
                          const double* const* b, double w0_first, double w0_hidden);

/* Optional tensor-core encoder: the SIREN layers as split-precision tcgen05 GEMMs - every operand as hi + lo fp16,
 * three kind::f16 products per term, fp32 accumulation (fp32-class accuracy; the reference's fp64 SIREN sits on
 * spherical-harmonic input that carries >= 1e-3 of its own rounding noise).
 * Needs every layer width % 256 == 0 and input width % 64 == 0; call after range_ctx_set_sh_table / _closed_form and
 * range_ctx_set_encoder (setting either again requires a new prepare).  `buf`, a device buffer of
 * range_encoder_prepared_bytes() the caller keeps alive, receives the split weights - the first layer's columns permuted
 * and zero-padded to the order in which the harmonics kernel emits features (analytic tables: Horner chains sorted by
 * length, 64 columns per round of 32 chains; closed form: |m|-major) - and that kernel's tables.  After a successful
 * prepare the ctx encodes in RANGE_ENC_F16X3 until range_ctx_set_encoder_precision(ctx, RANGE_ENC_F64). */
#define RANGE_ENC_F64 0
#define RANGE_ENC_F16X3 1
#define RANGE_ENC_TF32X3 RANGE_ENC_F16X3 /* earlier name of the same mode */
size_t range_encoder_prepared_bytes(range_ctx* ctx);
int range_ctx_prepare_encoder(range_ctx* ctx, void* buf, size_t bytes, void* stream);
int range_ctx_set_encoder_precision(range_ctx* ctx, int mode);

/* Device-resident database (range_b200/database.py) - replaces the tensors built at range/range.py:78-100.
 *   Kh  (Mpad, 256) fp16 row-major: row-normalised keys, rows >= M zero
 *   Vt  (Dp, Mpad) fp16: values transposed (entries contiguous) times vscale, columns >= M zero;
 *       D = value_dim (1 <= D <= RANGE_MAX_VALUE_DIM; RANGE_ERR_INVALID otherwise), Dp = round_up(D, 256), rows >= D zero
 *   xyz (Mpad, 4) fp32: unit vectors (x, y, z, 0)
 * Mpad is a multiple of 128.  Borrowed; must outlive the ctx or the next set_db.  The value width D sets the shapes
 * of every entry point below that reads or writes value rows: O and the parts of range_combine_concat /
 * range_sweep_concat are (N, D) fp32, results are (N, D + 256) or packed rows of 4 round_up(D, 4) + 2048 bytes.
 * A ctx with no database has D = 1024.  range_ctx_set_db is range_ctx_set_db_values with value_dim = 1024. */
#define RANGE_MAX_VALUE_DIM 4096
int range_ctx_set_db_values(range_ctx* ctx, int64_t M, int64_t Mpad, int value_dim, const void* Kh, const void* Vt,
                            const float* xyz, float vscale);
int range_ctx_set_db(range_ctx* ctx, int64_t M, int64_t Mpad, const void* Kh, const void* Vt, const float* xyz,
                     float vscale);

/* Optional: bounding caps of the database's 128-entry tiles, caps (Mpad/128, 4) fp32 device = (unit centre x, y, z,
 * angular radius in radians), borrowed.  With caps set, RANGE+ retrieval skips the geographic term of every
 * (128-query tile, 128-entry tile) whose entries all lie so far from all the tile's queries that together they
 * carry < 2^-24 of each row's geo normaliser (the geo softmax of range/range.py:231-234 has temperature 40:
 * exp(40 (cos d - 1))).  Effective when the database is stored in a spatially sorted order
 * (range_b200/database.py) and queries are batched spatially (range_sort_queries).  M_total = entries of the
 * whole database when this ctx holds one shard of it.  caps = NULL disables.  Reset by range_ctx_set_db. */
int range_ctx_set_db_caps(range_ctx* ctx, int64_t n_tiles, const float* caps, int64_t M_total);

/* Optional split-fp16 retrieval: Q.K^T and P'.V with every operand as hi + lo fp16 (x = hi + lo, 22 significant bits)
 * and three kind::f16 products per term (hi.hi + hi.lo + lo.hi), fp32 accumulation - about three times the tensor
 * work of the default fp16 operands, which keep 11 significant bits of q, K, P' and V.
 *   Kl  (Mpad, 256) fp16: rn_f16(K - Kh) of the fp32 keys Kh was rounded from, rows >= M zero
 *   Vtl (Dp, Mpad)  fp16: rn_f16(vscale V - Vt), the same layout as Vt
 * Borrowed like Kh / Vt (must outlive the ctx or the next set_db); both null clears them.  Reset by range_ctx_set_db.
 * range_ctx_set_retrieval_precision(ctx, RANGE_RET_F16X3) then switches every retrieval entry point (stats, apply, the
 * concat wrappers, topk, topk_rows, the routed applies) to the split operands: their `q16` argument becomes the
 * (N, 512) fp16 row [hi (256) | lo (256)] that range_split_queries builds from q64 (its hi half is range_encode's q16,
 * bit for bit), and the workspace functions size for that mode.  RANGE_RET_F16X3 without lo halves is
 * RANGE_ERR_INVALID.  The statistics and apply passes then always run the single-role kernels, the apply pass in query
 * chunks as for a value width != 1024. */
#define RANGE_RET_F16 0
#define RANGE_RET_F16X3 1
int range_ctx_set_db_lo(range_ctx* ctx, const void* Kl, const void* Vtl);
int range_ctx_set_retrieval_precision(range_ctx* ctx, int mode);
/* q64 (N,256) fp64 -> q16x2 (N,512) fp16: [rn_f16(q) | rn_f16(q - rn_f16(q))] */
int range_split_queries(range_ctx* ctx, int64_t N, const double* q64, void* q16x2, void* stream);

/* Diagnostic: the skip mask the RANGE+ kernels would use for these queries - mask [rows][words] uint32, bit t of
 * row r set = query tile r (128 rows of qxyz) skips the geo term of database tile t.  Shape from
 * range_geo_mask_shape (rows = query tiles rounded up to even).  sums = NULL: the mask of the statistics pass (bound
 * from the nearest database tile); sums = the (N,2) output of range_retrieve_stats: the tighter mask of the apply
 * pass (the geo normalisers are known: an entry is negligible iff exp(T (g - 1)) <= 2^-24 l_g / M_total). */
int range_geo_mask_shape(range_ctx* ctx, int64_t N, int32_t* rows, int32_t* words);
int range_geo_mask(range_ctx* ctx, int64_t N, const float* qxyz, float geo_temp, const float* sums, uint32_t* mask,
                   void* stream);

/* Spatial batching of a query batch (no reference counterpart: rows are independent, range/range.py:213-240).
 * perm[i] = caller's row index of sorted row i, lonlat_sorted[i] = lonlat[perm[i]]; cube-map Hilbert cells,
 * deterministic.  Run the encoder / retrieval on lonlat_sorted and hand perm to range_concat_scatter. */
size_t range_sort_workspace_bytes(range_ctx* ctx, int64_t N);
int range_sort_queries(range_ctx* ctx, int64_t N, const double* lonlat, double* lonlat_sorted, int32_t* perm,
                       void* workspace, size_t workspace_bytes, void* stream);

/* K1: features Yt[f * ld + n] = Y_f(lonlat[n]) for f < L*L - SphericalHarmonics.forward,
 * positional_encoding/spherical_harmonics.py:27-42.  lonlat (N,2) fp64 (lon, lat) degrees. */
int range_sh_features(range_ctx* ctx, int64_t N, const double* lonlat, double* Yt, int64_t ld, void* stream);

/* K1 + K1b + K3: LocationEncoder.forward (location_encoder.py:273-275) then the L2 normalisation of
 * range/range.py:212 and the query unit vector of range/range.py:225-229.
 *   q64 (N,256) fp64, q16 (N,256) fp16, qxyz (N,4) fp32 */
size_t range_encode_workspace_bytes(range_ctx* ctx, int64_t N);
int range_encode(range_ctx* ctx, int64_t N, const double* lonlat, double* q64, void* q16, float* qxyz,
                 void* workspace, size_t workspace_bytes, void* stream);

/* Dense lat/lon rasters (BASELINE config 5; the reference evaluates grids built like
 * range/evaluation/visualize_embeddings.py:29-45 point by point through spherical_harmonics.py:27-42).  Every analytic
 * harmonic is (latitude factor) x (longitude factor): range_raster_tables evaluates the latitude factors once per
 * distinct latitude and the trigonometric factors once per distinct longitude into `tables` (a device buffer of
 * range_raster_tables_bytes() the caller keeps alive); range_encode_raster then encodes queries given as
 * ij (N,2) int32 = (latitude index, longitude index) - any subset of the raster in any order, e.g. after
 * range_sort_queries - and also writes their coordinates lonlat (N,2) fp64 (lon, lat); an index outside the raster
 * gives a NaN row.  Same outputs, workspace and
 * bit-identical values as range_encode on those coordinates.  Needs the tensor-core encoder and the analytic
 * harmonics (RANGE_ERR_UNSUPPORTED otherwise: call range_encode on the coordinates instead). */
size_t range_raster_tables_bytes(range_ctx* ctx, int64_t n_lat, int64_t n_lon);
int range_raster_tables(range_ctx* ctx, int64_t n_lat, const double* lat, int64_t n_lon, const double* lon,
                        void* tables, size_t bytes, void* stream);
/* index and coordinate rows of the raster points p0 + (perm ? perm[n] : n), n < N (point p = i * n_lon + j, lat-major like
 * coord_grid): ij (N,2) int32 for range_encode_raster and / or lonlat (N,2) fp64 for range_sort_queries (either may be
 * NULL) - the host builds neither list.  perm (from range_sort_queries on a chunk's coordinates) is chunk-local. */
int range_raster_points(range_ctx* ctx, int64_t n_lat, int64_t n_lon, const void* tables, int64_t p0, int64_t N,
                        const int32_t* perm, int32_t* ij, double* lonlat, void* stream);
int range_encode_raster(range_ctx* ctx, int64_t n_lat, int64_t n_lon, const void* tables, int64_t N,
                        const int32_t* ij, double* lonlat, double* q64, void* q16, float* qxyz, void* workspace,
                        size_t workspace_bytes, void* stream);

/* K2: retrieval, range/range.py:213-217 (RANGE) and :213-238 (RANGE+).
 *   stats: sums (N,2) = {sum_j exp(temp (s_j-1)), sum_j exp(geo_temp (g_j-1))}, maxs (N,2) = {max s, max g}
 *          over THIS ctx's database shard; shards merge with SUM / MAX (M-sharding across GPUs).
 *   apply: O (N,D) fp32 = this shard's contribution to the retrieved feature, normalised with the given
 *          (global) sums; shards merge with SUM.
 *   retrieve = stats + apply for an unsharded database.
 * The workspace size depends on the database's value width D; for D != 1024 the apply pass runs in query chunks that
 * keep its largest scratch arrays (the partial results of the database splits) within 1 GiB. */
size_t range_retrieve_workspace_bytes(range_ctx* ctx, int64_t N);
int range_retrieve_stats(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                         float geo_temp, float* sums, float* maxs, void* workspace, size_t workspace_bytes,
                         void* stream);
int range_retrieve_apply(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                         float geo_temp, float beta, const float* sums, const float* maxs, float* O,
                         void* workspace, size_t workspace_bytes, void* stream);
int range_retrieve(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                   float geo_temp, float beta, float* O, void* workspace, size_t workspace_bytes, void* stream);

/* K2 apply + K3 in one call: this shard-less variant writes the retrieved feature straight into the caller's
 * (N,D+256) result - row n to out row perm[n] (perm from range_sort_queries, NULL = identity), as fp64
 * (RANGE_OUT_F64, what range/range.py:222,240 returns) or fp32 - followed by the location columns q64.  For
 * large batches of a 1024-wide database the apply kernel's epilogue does the concat itself (no (N,1024)
 * intermediate); small batches and other widths run apply + range_concat_scatter internally. */
int range_retrieve_apply_concat(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                                float geo_temp, float beta, const float* sums, const float* maxs, const double* q64,
                                const int32_t* perm, void* out, int out_dtype, void* workspace, size_t workspace_bytes,
                                void* stream);

/* K2 + K3 in ONE call for an unsharded database: range_retrieve_stats + range_retrieve_apply_concat with the statistics
 * kept in the workspace.  Same result layout as range_retrieve_apply_concat. */
int range_retrieve_concat(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                          float geo_temp, float beta, const double* q64, const int32_t* perm, void* out, int out_dtype,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Retrieval neighbours: which database entries an embedding is made of.  The weight of entry j for a query is the
 * coefficient range/range.py:213-238 multiplies V[j] by - RANGE: softmax(temp S)_j; RANGE+: (1-beta) softmax(geo_temp G)_j
 * + beta softmax(temp S)_j - computed with the row sums `sums` (N,2) of range_retrieve_stats.  For every query: the k
 * (1 <= k <= RANGE_TOPK_MAX, k <= M) largest weights over THIS ctx's database rows, descending, equal fp32 weights by
 * smaller row; idx (N,k) int32 = device database rows 0..M-1 of this ctx (the caller maps them to its own row order),
 * weight (N,k) fp32.  Row n of the result goes to row perm[n] (perm from range_sort_queries; NULL = identity).  With
 * the global sums of an M-sharded database each shard returns its local top k, which merge by weight
 * (range_retrieve_topk_rows, range_topk_merge below).  A separate pass over the database: range_retrieve_* are
 * unaffected. */
#define RANGE_TOPK_MAX 32
size_t range_topk_workspace_bytes(range_ctx* ctx, int64_t N, int k);
int range_retrieve_topk(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                        float geo_temp, float beta, const float* sums, int k, const int32_t* perm, int32_t* idx,
                        float* weight, void* workspace, size_t workspace_bytes, void* stream);

/* A shard's list for an M-sharded database: range_retrieve_topk without perm (row n of the result is query n), with
 * two differences.  Entry j is reported as row0 + j - with row0 = the shard's first row, a row of the whole database,
 * so equal weights still order by the smaller (global) row: shards are ascending contiguous ranges of it.  k is only
 * bounded by RANGE_TOPK_MAX: when the shard holds fewer than k entries the tail of each list is entry -1, weight 0.
 * Needs row0 >= 0 and row0 + M <= INT32_MAX.  Same workspace as range_retrieve_topk. */
int range_retrieve_topk_rows(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                             float geo_temp, float beta, const float* sums, int k, int64_t row0, int32_t* idx,
                             float* weight, void* workspace, size_t workspace_bytes, void* stream);

/* Merge of n_parts (1 <= n_parts <= RANGE_MAX_RANKS) lists of k entries per query, laid out [n_parts][N][k] (part_w
 * fp32, part_idx int32), each sorted by weight descending and then by entry, -1 entries (weight 0) allowed at the tail;
 * the parts hold disjoint entries.  Result: the k entries with the largest weights, same order and same -1 tail, row n
 * to idx / weight row perm[n] (NULL = identity).  This is what the owner of a query receives from the P shards'
 * range_retrieve_topk_rows lists.  Device pointers; no workspace. */
int range_topk_merge(range_ctx* ctx, int n_parts, int64_t N, int k, const float* part_w, const int32_t* part_idx,
                     const int32_t* perm, int32_t* idx, float* weight, void* stream);

/* ---- M-sharded database (one process per GPU, rank r holds rows [r M/P, (r+1) M/P) of the database) ----
 * The softmax-weighted sums of range/range.py:213-217,231-238 are associative in the database axis: with the fixed
 * offset (|s|,|g| <= 1) the per-shard exp-sums of range_retrieve_stats merge by SUM (one all-reduce of 8 B per query),
 * the per-shard maxima stay local (they only scale the fp16 weights), and the per-shard outputs of the apply pass,
 * normalised with the global sums, merge by SUM.  range_retrieve_apply_routed_values is range_retrieve_apply whose
 * result rows go straight to their owners: row n belongs to rank n / slab_rows and is stored as D fp32 (D the ctx's
 * value width) at
 *       route->peer[n / slab_rows] + ((size_t)route->rank * slab_rows + n % slab_rows) * D,
 * (slab_rows a multiple of 128: a 128-query tile has one owner) peer[r] being rank r's receive buffer
 * [n_ranks][slab_rows][D] fp32 mapped into this process (range_peer_open; peer[rank] = the local buffer; 16-byte
 * aligned).  Large batches of a 1024-wide database store from the apply kernel's epilogue (warp-transposed into full
 * 128-byte lines), so the partial rows cross NVLink while the tensor cores work on the next tiles; otherwise one kernel
 * per query chunk sums the database splits' partial rows and stores each row once, in 16-byte vectors.  No collective
 * moves them.  After a barrier across the ranks, the owner sums its n_ranks slots in rank order (range_combine_concat:
 * deterministic) and appends the location columns.  Needs D % 4 == 0 (RANGE_ERR_UNSUPPORTED otherwise): the slots
 * stay contiguous (slab_rows, D) arrays that range_combine_concat / range_sweep_concat read as they are. */
#define RANGE_MAX_RANKS 8
typedef struct range_route {
  int32_t n_ranks, rank;
  int64_t slab_rows;
  float* peer[RANGE_MAX_RANKS];
} range_route;
int range_retrieve_apply_routed_values(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz,
                                       float temp, float geo_temp, float beta, const float* sums, const float* maxs,
                                       const range_route* route, void* workspace, size_t workspace_bytes, void* stream);
/* range_retrieve_apply_routed_values for a 1024-wide database (rows 1024 floats apart): RANGE_ERR_UNSUPPORTED for any
 * other value width. */
int range_retrieve_apply_routed(range_ctx* ctx, int mode, int64_t N, const void* q16, const float* qxyz, float temp,
                                float geo_temp, float beta, const float* sums, const float* maxs,
                                const range_route* route, void* workspace, size_t workspace_bytes, void* stream);

/* out row perm[n] (NULL = identity) = [ sum_k weights[k] * parts[k][n][0:D] | q64[n][0:256] ] in out_dtype, D the ctx's
 * value width: (N,D+256) fp64 / fp32 or packed rows.
 * parts: host array of n_parts (<= 8) device pointers to (N,D) fp32; weights: host array or NULL (all 1).
 * Uses: the slots of an M-sharded receive buffer (weights 1); a beta sweep - range/range.py:238 is linear in beta,
 * so O(beta) = (1-beta) O(0) + beta O(1) serves any number of beta from two apply passes (Readme.md:27-31). */
int range_combine_concat(range_ctx* ctx, int64_t N, int n_parts, const float* const* parts, const float* weights,
                         const double* q64, const int32_t* perm, void* out, int out_dtype, void* stream);

/* The last step of a beta sweep on an M-sharded database, for up to RANGE_SWEEP_MAX_BETAS beta at once:
 *   outs[b] row perm[n] (NULL = identity) = [ w_sem[b] * S[n] + w_geo[b] * G[n] | q64[n][0:256] ]
 * G = sum of the n_slots geo slots, S = sum of the n_slots sem slots, each summed in slot order 0 .. n_slots-1 (the
 * partial rows of the geographic end, beta 0, and of the semantic end, beta 1, that the ranks sent this owner); per
 * column fmaf(w_sem, s, w_geo * g).  geo / sem: host arrays of n_slots (1 <= n_slots <= RANGE_MAX_RANKS) device pointers
 * to (N,D) fp32 (D the ctx's value width); w_geo / w_sem: host arrays of n_betas (1 <= n_betas <= RANGE_SWEEP_MAX_BETAS) weights, normally
 * 1 - beta and beta rounded on the host; outs: host array of n_betas device pointers to (N,D+256) results in out_dtype
 * (RANGE_OUT_F64 or RANGE_OUT_F32).  Every slot is read once, whatever n_betas.  With n_slots = 1 the rows are bit for bit
 * those of range_combine_concat with parts (G, S) and weights (w_geo, w_sem). */
#define RANGE_SWEEP_MAX_BETAS 8
int range_sweep_concat(range_ctx* ctx, int64_t N, int n_slots, const float* const* geo, const float* const* sem,
                       int n_betas, const float* w_geo, const float* w_sem, const double* q64, const int32_t* perm,
                       void* const* outs, int out_dtype, void* stream);

/* Receive buffers must be mappable by the other ranks' processes: the one place where the library allocates device
 * memory itself (cudaMalloc + CUDA IPC handle, 64 opaque bytes to hand to the peers, e.g. with all_gather_object).
 * range_peer_open maps a peer's buffer into this process (enables peer access over NVLink), range_peer_close unmaps
 * it, range_peer_free releases an allocation of range_peer_alloc. */
int range_peer_alloc(size_t bytes, void** dptr, unsigned char* handle64);
int range_peer_open(const unsigned char* handle64, void** dptr);
int range_peer_close(void* dptr);
int range_peer_free(void* dptr);

/* HOST function (no CUDA): widen N packed rows (RANGE_OUT_PACKED, e.g. a pinned staging buffer a device->host copy
 * just filled) of a database of value width value_dim = D (1 <= D <= 4096) into the caller's (N,D+256) float64 array -
 * the array range/range.py:222,240 returns - with a thread team of n_threads of its own.  range_host_unpack is
 * range_host_unpack_rows with value_dim = 1024. */
int range_host_unpack_rows(const void* packed, int64_t N, int value_dim, double* out, int n_threads);
int range_host_unpack(const void* packed, int64_t N, double* out, int n_threads);

/* K3: out (N,D+256) = [O | q64] (O (N,D), D the ctx's value width) as fp64 (RANGE_OUT_F64, what the reference returns: range/range.py:222,240)
 * or fp32. */
int range_concat(range_ctx* ctx, int64_t N, const float* O, const double* q64, void* out, int out_dtype,
                 void* stream);

/* as range_concat, writing row n to out row perm[n] (perm from range_sort_queries; NULL = identity) */
int range_concat_scatter(range_ctx* ctx, int64_t N, const float* O, const double* q64, const int32_t* perm,
                         void* out, int out_dtype, void* stream);

/* number of kernels this library launched since process start (bench.py's gpu_launches) */
int64_t range_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RANGE_B200_H */
