// csrc/internal.h -- host-side declarations shared between the obboot translation units.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <string>
#include <vector>

#include "../../include/obboot.h"

namespace ob {

// ---- tile geometry of the Gram contraction (gram.cu) ----
constexpr int BM = 128;        // replicate slots per panel (M tile)
constexpr int BN = 128;        // sufficient-statistic columns per N tile
constexpr int KT = 32;         // rows (contraction) per pipeline stage
constexpr int GRAM_THREADS = 256;   // consumer threads of the Gram CTA (8 warps); + one producer warpgroup

struct CudaError { cudaError_t code; const char* what; const char* file; int line; };

#define OB_CUDA(expr)                                                          \
    do {                                                                       \
        cudaError_t e__ = (expr);                                              \
        if (e__ != cudaSuccess) throw ::ob::CudaError{e__, #expr, __FILE__, __LINE__}; \
    } while (0)

struct StatusError { ob_status code; std::string msg; };

// A packed design row holds the K design columns followed by T >= 1 outcome columns (T = 1 for run(); a quantile
// sweep carries one RIF outcome per tau, ob_design_apply_rif_multi).  Sufficient-statistic columns of the Gram
// contraction, in this order: for j = 0..K-1 the pairs (j,j) (j,j+1) .. (j,K-1) (upper triangle of X'WX, row-major),
// then (j, y_0) .. (j, y_{T-1}) (X'Wy per outcome); one trailing (y_0, y_0) cell keeps the T = 1 layout equal to the
// row-major upper triangle of [x|y][x|y]^T.  P' = K(K+1)/2 + K T + 1, of which P = K(K+1)/2 + K T are algorithmic.
inline int64_t num_pairs(int K, int T) { return (int64_t)K * (K + 1) / 2 + (int64_t)K * T + 1; }
// row stride (in doubles) of the packed design: >= K + T, congruent to 4 mod 8 so that the
// B-fragment shared-memory loads of gram.cu are bank-conflict free
inline int design_ldx(int V) { int l = V; while ((l & 7) != 4) ++l; return l; }
// index of the first pair of design column j; pair (j,l), l < K, sits at pair_base + (l - j), pair (j, y_t) at
// pair_base + (K - j) + t
inline int64_t pair_base(int K, int T, int j) { return (int64_t)j * (K + T) - (int64_t)j * (j - 1) / 2; }

// ---- fixed row segmentation of a group (the summation tree of the split-n Gram) ----
// A group's padded rows are cut into `segs` <= MAX_SEGS leaf segments of seg_rows rows each (the last one
// may be short).  Both numbers depend on the group's GLOBAL row count only -- never on panels, batches, grid
// shape or the number of GPUs.  A tile's leaf partials are summed by the aligned binary tree over the leaf
// index space [0, MAX_SEGS) (absent leaves are skipped), see gram_reduce in gram.cu.  Under row sharding
// (SURVEY.md 8e, mode N) rank r of a power-of-two world owns the aligned leaf range
// [r * MAX_SEGS / world, (r+1) * MAX_SEGS / world): a complete subtree, so the per-rank sums combine to
// bit-identical results for any world size.
// 256 leaves keep the work units small enough for an even split over 148 persistent CTAs even when a launch covers
// only one or two panels (replicate sharding over 8 GPUs, panel batches of a 1e8-row problem): with 64 leaves config 3
// on 8 GPUs ran 20 units on the busiest CTA against 19.03 on average (5 % idle), now 77 against 76.1.
constexpr int MAX_SEGS = 256;
constexpr int MAX_WORLD = 64;    // row shards (a power of two): every rank owns an aligned subtree of >= 4 leaves
inline int64_t pad_rows(int64_t n) { return n <= KT ? KT : (n + KT - 1) / KT * KT; }
inline void segment_rows(int64_t n_pad, int& segs, int& seg_rows) {
    const int64_t stages = n_pad / KT;
    int64_t s = stages / 4 < 1 ? 1 : (stages / 4 > MAX_SEGS ? MAX_SEGS : stages / 4);
    const int64_t per = (stages + s - 1) / s;     // stages per segment
    s = (stages + per - 1) / per;
    segs = (int)s; seg_rows = (int)(per * KT);
}
struct RowShard {
    int64_t n_global = 0;        // rows of the whole group
    int64_t row_begin = 0;       // position (within the group, frame order) of this shard's first row
    int64_t n_local = 0;         // valid rows held here
    int segs = 1, seg_rows = KT; // global segmentation
    int leaf_lo = 0, leaf_hi = 1;// leaves owned here: [leaf_lo, leaf_hi) (possibly empty), leaf_lo aligned to MAX_SEGS / world
    int leaf_span = MAX_SEGS;    // MAX_SEGS / world
};
inline RowShard row_shard(int64_t n_global, int rank, int world) {
    RowShard r;
    r.n_global = n_global;
    const int64_t n_pad = pad_rows(n_global);
    segment_rows(n_pad, r.segs, r.seg_rows);
    r.leaf_span = MAX_SEGS / world;
    r.leaf_lo = rank * r.leaf_span < r.segs ? rank * r.leaf_span : r.segs;
    r.leaf_hi = (rank + 1) * r.leaf_span < r.segs ? (rank + 1) * r.leaf_span : r.segs;
    const int64_t lo = (int64_t)r.leaf_lo * r.seg_rows, hi = (int64_t)r.leaf_hi * r.seg_rows;
    r.row_begin = lo < n_global ? lo : n_global;
    const int64_t row_end = hi < n_global ? hi : n_global;
    r.n_local = row_end - r.row_begin;
    return r;
}

struct GroupData {               // one group's packed design in HBM (the rows this GPU holds)
    int64_t n = 0;               // valid rows held here
    int64_t n_pad = 0;           // rows padded to a multiple of KT (zero rows)
    RowShard shard;              // how these rows sit inside the whole group (world = 1: everything)
    double* X = nullptr;         // [n_pad][ldx]: cols 0..K-1 design (intercept first), col K outcome, rest 0
    double* w = nullptr;         // [n_pad] sample weights (0 on padding) or nullptr
    double* Xs = nullptr;        // weighted only: sqrt(w_i) * X[i][:] (ols.rs:68-78), the operand of the Gram contraction
    uint32_t* src = nullptr;     // [n] frame row each packed row came from (ob_design_update_outcome)
    double* y_raw = nullptr;     // [n] the untransformed outcome, saved by the first ob_design_apply_rif so that further
                                 // quantiles are computed from the raw y (a quantile sweep packs once)
    // Heckman selection equation (ob_design_attach_selection): Z [n][K1] row-major with the intercept first, sel [n] =
    // (selection outcome == 1), Xm [n_pad][ldx] = the design with unselected rows zeroed (operand of the outcome Gram)
    double* hk_Z = nullptr; uint8_t* hk_sel = nullptr; double* hk_Xm = nullptr;
    // clusters (ob_design_attach_clusters): [n] resampling unit of each packed row, or nullptr (rows are resampled)
    uint32_t* uid = nullptr;
    const double* gram_operand() const { return Xs ? Xs : X; }
};

// ---- resample.cu ----
// counts layout per group: [panels][n_pad][BM] of count_t (uint8_t or uint16_t); slot 0 of panel 0
// is the point estimate (all ones on valid rows).
struct CountsArgs {
    void* C; int count_bytes; int64_t n; int64_t n_pad; int panels;   // n, n_pad: rows held here
    int64_t n_global = 0;         // rows of the whole group (draws per replicate); row_begin: global position of local row 0
    int64_t row_begin = 0;
    int64_t slots;                // valid slots in this batch
    int first_slot;               // 1: slot 0 is the point estimate, replicates start at slot 1; 0: replicates from slot 0
    int64_t rep0;                 // global replicate id of local slot 0 (-1.. for the point slot)
    int group; uint64_t seed;
};
void counts_clear(const CountsArgs& a, cudaStream_t st);
// index-stream mode: idx [reps][n] u32 on device; overflow_flag (device int) set when a count saturates
void counts_from_indices(const CountsArgs& a, const uint32_t* d_idx, int* d_overflow, cudaStream_t st);
// native mode, two phases: Poisson(lambda) body over the local rows (accumulates the local column sums into
// d_colsum [panels*BM] int64, zeroed by the caller), then -- after d_colsum has been summed over all row shards --
// the exact fix-up draws.  d_flags[0] = body overshoot, d_flags[1] = count saturated.
// d_lut: counts_lut_bytes() of scratch per group (the inverse-CDF byte table, rebuilt by every call: 2 launches)
size_t counts_lut_bytes();
void counts_philox_body_launch(const CountsArgs& a, long long* d_colsum, unsigned char* d_lut, cudaStream_t st);
void counts_philox_fixup_launch(const CountsArgs& a, const long long* d_colsum, int* d_flags, cudaStream_t st);

// Bayesian bootstrap (Rubin 1981): C [panels][n_pad][BM] of fp32 E_i ~ iid Exp(1) per (row, replicate) -- the point slot
// holds 1.0 on valid rows, padding rows and slots outside [first_slot, slots) hold 0 -- and part [segs][panels*BM]: each
// (leaf segment, slot)'s sum of E in a fixed order (leaf_sum_launch then sums the leaves by the Gram's aligned tree).  Native
// stream: E = -log U, U in (0, 1) from Philox4x32-10 keyed by (seed; global row, group, global replicate id, stream tag);
// explicit stream: wt [replicates of the batch][n_global], the caller's E in the group's row order.
struct BayesArgs {
    float* C; int64_t n, n_pad; int panels;      // rows held here
    int64_t n_global, row_begin;
    int64_t slots; int first_slot; int64_t rep0; // as CountsArgs
    int group; uint64_t seed;
    int segs, seg_rows;                          // leaves held here (RowShard) and rows per leaf
    const float* wt;                             // explicit stream on the device, or null (native)
    double* part;                                // [segs][panels * BM]
    int* flags = nullptr;                        // flags[3] |= 1: an explicit weight that is not a positive normal float
};
void bayes_weights_launch(const BayesArgs& a, cudaStream_t st);

// ---- cluster.cu ----
// attach: uid[row] = codes_frame[src[row]], present[code] = 1 (d_flags[0] |= 1 on a code outside [0, n_codes)); then
// unit[code] = exclusive scan of present (*d_units = the stratum's unit count); then uid[row] = unit[uid[row]]
void cluster_gather_launch(const int32_t* d_codes_frame, const uint32_t* src, int64_t n, int32_t n_codes, uint32_t* uid,
                           uint8_t* present, int* d_flags, cudaStream_t st);
void cluster_scan_launch(const uint8_t* present, int32_t n_codes, uint32_t* unit, long long* d_units, cudaStream_t st);
void cluster_remap_launch(uint32_t* uid, int64_t n, const uint32_t* unit, cudaStream_t st);
// C [panels][n_pad][BM] = U [panels][u_pad][BM] gathered through uid (rows [n, n_pad) zero); rows[slot] += the slot's row
// count (zeroed by the caller; slots < `slots` only)
struct ExpandArgs {
    void* C; const void* U; const uint32_t* uid; int count_bytes;
    int64_t n, n_pad, u_pad; int panels; int64_t slots;
    long long* rows;
};
void counts_expand_launch(const ExpandArgs& a, cudaStream_t st);

// ---- gram.cu ----
constexpr int BQ = 32;            // column quantum of the Gram CTA tile: one 8-column DMMA sub-tile for each of the SM's four
                                  // schedulers (consumer warps w and w + 4 sit on the same one)
// The columns the contraction computes, in tile order.  P' minus the STRUCTURAL ZEROS: the product of two different
// dummies of one categorical predictor is 0 on every row (a row has one level), so those cells of X'WX are exactly 0.0
// whatever the multiplicities; they are not computed, the reduced Gram holds 0.0 there.  Everything downstream still
// sees the full row-major upper triangle (pair_base): `colmap` scatters computed column c to its place.
struct GramColumns {
    int Pc = 0;                        // computed columns
    int nfull = 0, tail_q = 0;         // column tiling of Pc: nfull tiles of BN columns + a tail tile of tail_q quanta (0 = none)
    int ntiles = 0;                    // nfull + (tail_q > 0)
    std::vector<uint16_t> pairs;       // [ntiles * BN][2] design-row offsets (j, l) of column c; padding columns: (K, K)
    std::vector<int32_t> colmap;       // [ntiles * BN] index in the row-major upper triangle of [x|y][x|y]^T, -1 = padding
};
// cat_levels: level counts (incl. the base level) of the design's categorical predictors, in column order, or empty
// when unknown (ob_design_from_dense): then nothing is dropped.
GramColumns gram_columns(int K, int T, int n_cont, const std::vector<int>& cat_levels);
// the outcome columns of gram_columns alone (the K T cells of X'Wy and (y_0, y_0)), same order, same colmap targets:
// the narrow contraction of a cached run whose X'WX is known (ob_bootstrap_run_cached)
GramColumns gram_outcome_columns(int K, int T);

// ---- per-replicate Gram cache (ob_gram_cache): compact layouts that do not depend on T ----
// xx [2][slots][K(K+1)/2]: the X'WX upper triangle, row-major; yy [2][slots][K T + 1]: the X'Wy cells (j, y_t) j-major, then
// (y_0, y_0).  gram_cache_map(K, T)[c] = position in a reduced-Gram row [Pld] of xx cell c (c < K(K+1)/2), else of yy cell
// c - K(K+1)/2.
inline int gram_cache_xx_cells(int K) { return K * (K + 1) / 2; }
inline int gram_cache_y_cells(int K, int T) { return K * T + 1; }
std::vector<int32_t> gram_cache_map(int K, int T);
struct GramCacheCopy {
    double* gram; int64_t slots_pad; int Pld;  // the batch's reduced Gram [2][slots_pad][Pld]
    int64_t slot_lo, nslots;                   // its slots are the run's slots [slot_lo, slot_lo + nslots)
    double* xx; double* yy; int64_t cslots;    // the cache, [2][cslots][nx] and [2][cslots][ny]
    const int32_t* map; int nx, ny;            // device gram_cache_map, nx = K(K+1)/2, ny = K T + 1
    int c_lo, c_hi;                            // cells [c_lo, c_hi) of the map are copied
};
// batch Gram -> cache (after gram_reduce_launch / gram_combine_launch)
void gram_cache_extract_launch(const GramCacheCopy& a, cudaStream_t st);
// cache -> batch Gram; after gram_reduce_launch / gram_combine_launch, which zero the whole buffer first
void gram_cache_assemble_launch(const GramCacheCopy& a, cudaStream_t st);
struct GramPlan {
    int K, T, ldx, panels, ntiles;
    int nfull, tail_q, Pld;       // column tiling of the computed columns and the row stride of the reduced Gram (gram_pld)
    int64_t n_pad[2];             // local padded rows
    int segs[2], seg_rows[2];     // leaves held here and rows per leaf (RowShard: function of the global row count only)
    int leaf_span;                // MAX_SEGS / world: size of the aligned subtree this GPU reduces
    int64_t units[2];             // panels * ntiles * segs
    int grid;
    int64_t num_partials;         // = units[0] + units[1]
    size_t smem_bytes; int ring;  // shared memory and pipeline depth of the Gram CTA
};
// Column tiling: tiles of BN = 128 columns (four quanta) and a tail tile of one to three quanta -- 32, 64 or 96 columns;
// the DMMA time of a tile is proportional to its quanta.  K = 17: 171 columns = 1.5 tiles; K = 31: 528 = 4.25; K = 51
// with two four-level categoricals: 1372 computed columns = 10.75.
inline void gram_col_tiling(int64_t Pc, int& nfull, int& tail_q) {
    const int64_t quanta = (Pc + BQ - 1) / BQ;
    nfull = (int)(quanta / 4); tail_q = (int)(quanta % 4);
}
// upper bound on the number of column tiles (structural zeros can only lower it): workspace sizing
inline int gram_ntiles(int K, int T) { int f, q; gram_col_tiling(num_pairs(K, T), f, q); return f + (q > 0); }
// row stride of the reduced Gram [slot][Pld]: all P' cells of the upper triangle
inline int gram_pld(int K, int T) { return (int)((num_pairs(K, T) + BQ - 1) / BQ * BQ); }
GramPlan gram_make_plan(int K, int T, int ldx, int panels, const GroupData g[2], int count_bytes, int num_sms,
                        const GramColumns& cols);
// whether the Gram CTA fits in shared memory at design row stride ldx with count_bytes-wide multiplicities: always at
// 8-bit (K + outcomes <= 280), up to ldx 268 at 16-bit, up to ldx 236 with fp32 Bayesian weights (count_bytes 4).  The
// drivers refuse or stop widening where it does not.
bool gram_fits(int ldx, int count_bytes);
struct GramArgs {
    const double* X[2]; const void* C[2];     // X: the (sqrt(w)-scaled when weighted) design
    int count_bytes;
    double* partials;            // [num_partials][BM*BN]
    const uint16_t* d_pairs;     // [ntiles*BN][2] column offsets (j,l) within a design row (GramColumns::pairs)
    const int32_t* d_colmap;     // [ntiles*BN] GramColumns::colmap
    double* gram;                // out: [2][panels*BM][Pld]
    int tail_mi = 16;            // 8-slot groups of the batch's last panel that hold valid slots, rounded up to a multiple
                                 // of 4 (16 = full): lets the kernel skip the DMMAs of slot groups that do not exist
};
void gram_launch(const GramPlan& plan, const GramArgs& args, cudaStream_t st, cudaEvent_t ev_main_begin = nullptr,
                 cudaEvent_t ev_main_end = nullptr);
// the two halves of gram_launch: the contraction over a sub-range of each group's leaves (null = all), and the
// fixed-tree reduction of the partial tiles (once every leaf has been contracted)
void gram_launch_leaves(const GramPlan& plan, const GramArgs& args, const int seg_lo[2], const int seg_n[2], cudaStream_t st);
void gram_reduce_launch(const GramPlan& plan, const GramArgs& args, cudaStream_t st);
// out [2][slots_pad] = per slot, the aligned-tree sum of part [segs[0] + segs[1]][slots_pad] over each group's leaves held
// here (span = MAX_SEGS / world); mode N then combines the per-rank sums with gram_combine_launch
void leaf_sum_launch(const double* part, const int segs[2], int64_t slots_pad, int span, double* out, cudaStream_t st);
// mode N: gram = aligned-tree sum over ranks of gathered [world][2][slots_pad*Pld] per-rank sums; ranks_with_rows[g]
// = number of leading ranks that hold leaves of group g
void gram_combine_launch(const double* gathered, int world, const int ranks_with_rows[2], int64_t per_group_elems,
                         double* gram, cudaStream_t st);
int64_t gram_schedule_debug(int K, int panels, int64_t slots_last_panel, const GroupData gd[2], int grid, int64_t* out8, int64_t cap);

// ---- solve.cu ----
struct SolveArgs {
    const double* gram;      // [2][slots_pad][Pld]
    int64_t slots_pad; int Pld;
    int64_t slots;           // valid slots in this batch (slot 0 = point estimate when has_point)
    int K, n_cont, ref_kind;
    int T = 1;               // outcome columns: stats [slots][T][S], beta_a / beta_b [slots][T][K], point_extra [T][5K+1]
    int n_norm; const int* d_norm_m; const int* d_norm_off; const int* d_norm_idx; const int* d_norm_has_base;
    int n_base; int S;
    int weighted;
    double na, nb;           // group row counts (n_obs)
    const long long* rows = nullptr;   // clustered designs: [2][slots_pad] row counts per slot (replace na / nb), else null
    const double* esum = nullptr;      // Bayesian bootstrap: [2][slots_pad] sums of the raw weights E per slot, else null
    // outputs
    double* stats;           // [slots][S]
    int* status;             // [slots]
    double* beta_a; double* beta_b;    // [slots][K] (post-Yun) or nullptr
    double* point_extra;     // slot 0 only: [xa_mean K | xb_mean K | beta_star K | raw beta_a K | raw beta_b K | total_gap] or nullptr
    double* scratch = nullptr;   // solve_scratch_bytes(..) of device memory when that is non-zero (designs wider than ~160 columns)
};
void solve_launch(const SolveArgs& a, cudaStream_t st);
size_t solve_smem_bytes(int K, bool pooled, int n_norm);
// 0 while a (K+1) x (K+1) system fits shared memory; else the bytes of per-slot global scratch solve_launch needs
size_t solve_scratch_bytes(int K, bool pooled, int n_norm, int T, int64_t slots);

// ---- reduce_stats.cu ----
// stats [reps][S] + status [reps] (device) -> se,p,lo,hi,t [S] each (device, contiguous 5*S) and n_ok
// up to REDUCE_MAX_REPS replicates the per-statistic sort runs in shared memory; beyond that in d_scratch
// (reduce_stats_scratch_bytes(reps, S) bytes of device memory)
constexpr int64_t REDUCE_MAX_REPS = 16384;
void reduce_stats_launch(const double* stats, const int* status, int64_t reps, int S,
                         const double* point_stats, double* out5S, long long* n_ok, cudaStream_t st,
                         double* d_scratch = nullptr);
size_t reduce_stats_scratch_bytes(int64_t reps, int S);

// ---- pack.cu ----
struct PackArgs {
    int64_t n; int n_cont, n_cat;
    const double* const* d_cont;     // device array of device column pointers
    const int32_t* const* d_cat;     // device array of device code-column pointers
    const int32_t* d_cat_levels;     // [n_cat]
    const int32_t* d_dummy_start;    // [n_cat] first design column of each categorical
    const double* d_y; const double* d_w; const uint8_t* d_group;
    int K, ldx;
};
// pass 1+2: per-block group counts and their exclusive scan (d_block_counts [nblocks][2] becomes the
// per-block base rank; d_totals[2] = group sizes); flags[0] = negative weight seen, flags[1] = bad code
int pack_num_blocks(int64_t n);
void pack_count_scan(const PackArgs& a, long long* d_block_counts, long long* d_totals, int* d_flags, cudaStream_t st);
// pass 3: staged transpose/scatter of the rows into the packed per-group designs
// Row-shard window of a pack (ob_design_pack_row_shard_async): the packed frame slice's row q of group g belongs at shard
// row pos = q + shift[g]; rows outside [0, n_local[g]) are exported for the exchange: low side (pos < 0) at export row
// pos + lo_add[g] (= q), high side at hi_base[g] + (pos - n_local[g]).
struct PackWindow {
    long long shift[2], n_local[2], lo_add[2], hi_base[2];
    double* EX[2]; double* Ew[2]; uint32_t* Esrc[2];
    uint32_t src_add;
};
// blocks [blk0, blk1) of PK_ROWS = 128 frame rows each (blk1 < 0: to the end)
void pack_scatter(const PackArgs& a, const long long* d_block_base, GroupData ga, GroupData gb, int* d_flags,
                  cudaStream_t st, int blk0 = 0, int blk1 = -1, const PackWindow* win = nullptr);
constexpr int PACK_BLOCK_ROWS = 128;
// src[i] = first + i (designs built from dense per-group matrices: the "frame" is group A's rows, then group B's)
void iota_launch(uint32_t* dst, int64_t n, uint32_t first, cudaStream_t st);
// p[i] += add (frame-row maps of frame slices become maps into the whole frame)
void add_u32_launch(uint32_t* p, int64_t n, uint32_t add, cudaStream_t st);
// outcome refresh: X[r][K] = y[src[r]] (and Xs[r][K] = sqrt(w[r]) * y[src[r]]) for every packed row of the group
void update_outcome_launch(const GroupData& g, int K, int ldx, const double* d_y_frame, cudaStream_t st);
// Xs[i][:] = sqrt(w[i]) * X[i][:] for all V = K+1 columns (WLS as OLS on sqrt(w)-scaled data, ols.rs:68-78)
void scale_rows_launch(const GroupData& g, int ldx, cudaStream_t st);
void scale_rows_range_launch(const GroupData& g, int ldx, int64_t row0, int64_t rows, cudaStream_t st);
// residuals of the point estimate: r = y - X beta (ols.rs:118-119) for one group; the outcome sits in column ycol
void residuals_launch(const GroupData& g, int K, int ycol, int ldx, const double* d_beta, double* d_out, cudaStream_t st);
// dst [rows][ld_dst] = design columns 0..K-1 of src [rows][ld_src], zeros from column K on
void relayout_launch(const double* src, int ld_src, double* dst, int ld_dst, int64_t rows, int K, cudaStream_t st);

// ---- ingest.cu ----
constexpr int INGEST_MAX_COLS = 288;
struct IngestScanArgs {
    long long n;
    int n_valid; const uint8_t* valid[INGEST_MAX_COLS];      // validity bytes of the numeric columns that carry nulls
    int n_nan; const double* nan_cols[INGEST_MAX_COLS];      // numeric columns in which a NaN counts as null (nan_is_null)
    int n_dict; const int32_t* codes[INGEST_MAX_COLS];       // dictionary columns: categoricals.., group last
    int dict_size[INGEST_MAX_COLS];
    uint8_t* present[INGEST_MAX_COLS];                       // [dict_size] per dictionary column, zeroed by the caller
    uint8_t* row_valid;                                      // [n] out
    long long* kept;                                         // out: rows kept (zeroed by the caller)
    int* flags;                                              // bit 0: code >= dict_size
};
struct IngestApplyArgs {
    long long n; int n_cat;
    const uint8_t* row_valid;
    const int32_t* group_codes; const int32_t* group_map;    // dictionary code -> 0 (A) / 1 (reference) / anything else
    int32_t* cat_codes[INGEST_MAX_COLS];                     // in place: dictionary code -> level code
    const int32_t* remap; int remap_off[INGEST_MAX_COLS];    // concatenated per-categorical tables
    uint8_t* group_out;                                      // [n]
    int* flags;                                              // bit 1: a valid row maps to an absent level
};
void ingest_scan_launch(const IngestScanArgs& a, cudaStream_t st);
void ingest_apply_launch(const IngestApplyArgs& a, cudaStream_t st);

// ---- comm.cu: collectives between the GPUs of one box (mode N row sharding) ----
// Two transports behind one interface: NCCL over NVLink/NVSwitch (one process per GPU; libnccl is dlopen'ed, the
// communicator is bootstrapped from an ncclUniqueId the host layer broadcasts), and an in-process transport for
// several contexts of ONE process (threads; device-to-device copies), used when a single host process drives
// all GPUs and by the single-GPU tests of the sharded path.
enum class CommDType { I32, I64, F64 };
enum class CommOp { SUM, MAX, MIN };
struct Comm {
    int rank = 0, world = 1;
    virtual ~Comm() = default;
    // in place, on device memory, ordered on stream st; returns only after the result is usable on st
    virtual void allreduce(void* buf, size_t count, CommDType dt, CommOp op, cudaStream_t st) = 0;
    // recv [world][bytes] <- every rank's send [bytes]
    virtual void allgather(const void* send, void* recv, size_t bytes, cudaStream_t st) = 0;
    // variable sizes: rank r's `sizes[r]` bytes (its `send`) land at recv + offsets[r] on every rank
    virtual void allgatherv(const void* send, void* recv, const size_t* offsets, const size_t* sizes, cudaStream_t st) = 0;
    // personalised exchange: bytes[src * world + dst] (the same table on every rank) travel from src's
    // send + send_off[dst] to dst's recv + recv_off[src]
    virtual void alltoallv(const void* send, const size_t* send_off, void* recv, const size_t* recv_off, const size_t* bytes,
                           cudaStream_t st) = 0;
};
struct LocalGroup;                       // shared state of an in-process group (ob_local_group)
LocalGroup* local_group_create(int world);
void local_group_destroy(LocalGroup* g);
Comm* comm_create_local(LocalGroup* g, int rank, int device);
void nccl_unique_id(uint8_t* id128);
Comm* comm_create_nccl(const uint8_t* id128, int rank, int world);

// ---- heckman.cu: Heckman two-step replicate (SURVEY 8f-4) ----
constexpr int HK_MAX_SEL = 8;        // selection-equation columns incl. the intercept
struct HkGroup { const double* Z; const uint8_t* sel; int64_t n, n_pad; };   // Z [n][K1] row-major (intercept first), sel [n]
int hk_num_chunks(int64_t n);
// frame-order selection columns -> packed group order through the frame-row map; flags[0] |= 1 on a NaN selection outcome
void hk_gather_launch(const uint32_t* src, int64_t n, int K1, const double* const* d_pred, const double* d_outcome, double* Z, uint8_t* sel,
                      int* d_flags, cudaStream_t st);
// Xm = X with the rows of unselected observations zeroed (all ldx columns)
void hk_mask_launch(const double* X, const uint8_t* sel, double* Xm, int64_t rows, int ldx, cudaStream_t st);
// one Fisher-scoring step of every active slot: partial [chunks][panels][K1 + K1(K1+1)/2][BM], then the per-slot update
void hk_probit_accum_launch(const HkGroup& g, int K1, const void* C, int count_bytes, int panels, const double* gamma, const int* active,
                            int64_t slots_pad, double* partial, cudaStream_t st);
void hk_probit_update_launch(const double* partial, int nchunks, int panels, int K1, int64_t slots, double tol, int last_iter, double* gamma,
                             int* active, int* pstatus, int* n_active, cudaStream_t st);
// IMR sums: partial [chunks][panels][K1 + 5][BM]; L [panels][n_pad][BM] = c * IMR
void hk_terms_launch(const HkGroup& g, const double* X, int ldx, int ycol, int K1, const void* C, int count_bytes, int panels, const double* gamma,
                     double* L, double* partial, cudaStream_t st);
void hk_xterm_launch(const HkGroup& g, const double* X, int ldx, int K, int panels, const double* L, double* partial, cudaStream_t st);
void hk_reduce_launch(const double* partial, int nchunks, int panels, int nacc, double* out, int64_t slots_pad, cudaStream_t st);
struct HkSolveArgs {
    const double* gram; int64_t slots_pad; int Pld; int64_t slots;
    int K, K1, ref_kind;
    const double* terms[2]; const double* xterm[2]; const double* gamma[2]; const int* pstatus[2];
    double na, nb; int S;
    double* stats; int* status; double* beta_a; double* beta_b; double* point_extra;
};
void hk_solve_launch(const HkSolveArgs& a, cudaStream_t st);

// ---- mm.cu: Machado-Mata quantile decomposition (SURVEY 8f-3) ----
constexpr int MM_MAX_COLS = 47;      // design columns incl. the intercept
constexpr int MM_MAX_SIMS = 4096;    // simulations per pass (the effects kernel sorts them in shared memory)
struct MmArgs {
    const double* X[2]; const void* C[2]; int64_t n[2], n_pad[2];   // unweighted designs, multiplicity matrices of this batch
    int ldx, K, count_bytes, sims;
    int64_t slots;                   // passes (columns of the multiplicity matrix) in this batch
    const double* taus;              // [slots][sims] the random quantiles of every pass
    double* state; int64_t state_stride;     // per block mm_state_vectors() vectors of state_stride doubles
    double* betas; int* info;        // [slots][sims][2][K], [slots][sims][2] (status | iterations << 8 | candidates << 16):
                                     // problem-major, problem = (slot sims + sim) 2 + group
    int* counter;                    // work queue (zeroed by the caller)
    int64_t p_begin, p_end;          // problems [p_begin, p_end) are solved by this launch (mode R: the rank's share)
};
int mm_state_vectors();
int mm_blocks_per_sm(int K, int64_t rows);      // rows = the larger group
// every (group, pass, simulation) quantile regression of the batch: interior point + vertex polish, one block per problem
void mm_qr_launch(const MmArgs& m, int grid, cudaStream_t st);
// native streams: taus [slots][sims], simulated original rows rows_a / rows_b [slots][sims]; global pass id of slot s =
// pass0 + s, except that slot 0 is pass 0 (the point estimates) when first_slot is set
void mm_streams_launch(const MmArgs& m, long long pass0, int first_slot, uint64_t seed, double* taus, uint32_t* rows_a, uint32_t* rows_b, cudaStream_t st);
// simulation + empirical quantiles + effects per pass: stats [slots][3 nq], status [slots], nsucc [slots] (may be null)
void mm_effects_launch(const MmArgs& m, const uint32_t* rows_a, const uint32_t* rows_b, int nq, const double* d_quantiles,
                       double* stats, int* status, int* nsucc, cudaStream_t st);

// ---- rif.cu ----
// RIF transform (math/rif.rs:14-88) of a packed group's raw outcome (g.y_raw if saved, else column ycol itself),
// written to column ycol
// comm: the row-sharding communicator when g is one rank's shard of the group (leaf partials and radix histograms are
// all-reduced; results bit-identical to the unsharded transform), else null
void rif_transform(const GroupData& g, int ycol, int ldx, double tau, void* d_scratch, size_t scratch_bytes,
                   cudaStream_t st, Comm* comm = nullptr);
size_t rif_scratch_bytes(int64_t n);

}  // namespace ob
