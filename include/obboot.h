/* include/obboot.h -- C ABI of libobboot: the B200-native bootstrap-inference path of
 * oaxaca_blinder (reference: dot-comma-hyphen/oaxaca-blinder-rs, crate oaxaca_blinder).
 *
 * This is the drop-in boundary: what a `build.rs`-linked `extern "C"` block in the reference
 * crate would bind to replace the body of OaxacaBuilder::run() from the group split to the
 * assembled results (builder.rs:808-950), and decompose_quantile()'s RIF pre-step
 * (builder.rs:721-737).  Plain pointers and sizes only; #[repr(C)]-compatible structs; no C++
 * or torch types.  INTEGRATION.md shows the Rust-side binding.
 *
 * Citations are file:line under oaxaca_blinder/src/ of the reference.
 *
 * There is NO CPU fallback: every compute entry point needs a CUDA device (sm_100a) and returns
 * OB_ERR_CUDA / OB_ERR_NO_DEVICE otherwise.
 */
#ifndef OBBOOT_H
#define OBBOOT_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OBBOOT_ABI_VERSION 6

/* ---- errors: OaxacaError variants (error.rs:6-19) + device errors ------------------------- */
typedef enum ob_status {
    OB_OK = 0,
    OB_ERR_POLARS = 1,            /* PolarsError: malformed frame / dtype */
    OB_ERR_COLUMN_NOT_FOUND = 2,  /* ColumnNotFound (builder.rs:776) */
    OB_ERR_INVALID_GROUP = 3,     /* InvalidGroupVariable: <2 groups (builder.rs:67-71), empty group
                                     (:431-435), negative weight (ols.rs:60-66), zero total weight (builder.rs:603-607) */
    OB_ERR_NALGEBRA = 4,          /* NalgebraError: Cholesky failed on the point estimate (ols.rs:107-111) */
    OB_ERR_DIAGNOSTIC = 5,        /* DiagnosticError (unused on this path) */
    OB_ERR_INSUFFICIENT_DATA = 6, /* InsufficientData: n_obs <= k (ols.rs:98-105) */
    OB_ERR_INVALID_ARG = 7,       /* null pointer / out-of-range option (no reference counterpart) */
    OB_ERR_CUDA = 8,
    OB_ERR_NCCL = 9,
    OB_ERR_NO_DEVICE = 10,
    OB_ERR_UNSUPPORTED = 11       /* shape outside what the kernels are built for (e.g. K + outcome columns > 280) */
} ob_status;

/* ReferenceCoefficients (decomposition.rs:5-20).  Neumark == Pooled, Cotton == Weighted. */
typedef enum ob_ref_kind { OB_REF_GROUP_A = 0, OB_REF_GROUP_B = 1, OB_REF_POOLED = 2, OB_REF_WEIGHTED = 3 } ob_ref_kind;

typedef struct ob_ctx ob_ctx;        /* device, streams, workspace; one per calling thread (run(&self) is re-entrant) */
typedef struct ob_design ob_design;  /* packed design of both groups, resident in HBM; owned by the context that
                                        created it: destroy designs before their context */

ob_status ob_device_count(int32_t* n_out);
/* Page-locked host memory for buffers the library copies to or from asynchronously (frame columns, residuals_b): DMA
 * goes straight to the caller's buffer instead of through the driver's staging copy.  Plain malloc'ed memory works
 * everywhere too, only slower.  ob_host_register pins an existing allocation (e.g. a Rust Vec) in place. */
ob_status ob_host_alloc(size_t bytes, void** out);
void ob_host_free(void* p);
ob_status ob_host_register(void* p, size_t bytes);
ob_status ob_host_unregister(void* p);
ob_status ob_ctx_create(int32_t device, ob_ctx** out);
void ob_ctx_destroy(ob_ctx* ctx);
/* message of the last failing call on this context (owned by the context) */
const char* ob_last_error(const ob_ctx* ctx);
uint32_t ob_abi_version(void);

/* ---- (1) design-matrix pack --------------------------------------------------------------
 * The cleaned frame as the reference holds it at builder.rs:808: nulls dropped (:760-784),
 * categorical levels sorted and coded (:380-418).  Column pointers are HOST memory (pinned or
 * pageable); the call copies them to the device and packs
 *   X_g = [__ob_intercept__ | continuous.. | dummies.. | outcome]   row-major, per group
 * (prepare_data, builder.rs:294-378; column order :325-327; dummy for code c>=1 of categorical
 * q sits at design column 1 + n_cont + sum_{q'<q}(levels[q']-1) + (c-1), code 0 is the base :402). */
typedef struct ob_frame_view {
    int64_t n;                         /* rows */
    int32_t n_cont;                    /* continuous predictors, user order */
    const double* const* cont;         /* [n_cont] columns of n doubles */
    int32_t n_cat;                     /* categorical predictors, user order */
    const int32_t* const* cat_codes;   /* [n_cat] columns of n codes in [0, cat_levels[q]) */
    const int32_t* cat_levels;         /* [n_cat] level count m incl. base */
    const double* outcome;             /* [n] */
    const double* weights;             /* [n] or NULL (builder.rs:355-370) */
    const uint8_t* group;              /* [n] 0 = group A, 1 = group B (reference_group), else ignored (builder.rs:73-94) */
} ob_frame_view;

ob_status ob_design_pack(ob_ctx* ctx, const ob_frame_view* frame, ob_design** out);

/* Asynchronous variant for frames in page-locked memory (ob_host_alloc / ob_host_register; pageable memory works but
 * overlaps nothing).  Returns as soon as the group split is known -- ob_design_shape answers -- while the columns are
 * still being uploaded and packed, in row chunks, on the context's copy stream.  ob_bootstrap_run may be called at
 * once: its replicate generation needs no design rows, and its Gram contraction starts on the rows that have arrived,
 * so the PCIe transfer disappears under the first kernels.  Contract: the frame's buffers stay valid and unmodified
 * until ob_design_wait() or the first call that uses the design (ob_bootstrap_run, ob_design_download, ...) has
 * returned.  Errors found late (negative weight, ols.rs:60-66; code outside its levels) are reported by that call,
 * and the design is unusable afterwards. */
ob_status ob_design_pack_async(ob_ctx* ctx, const ob_frame_view* frame, ob_design** out);
ob_status ob_design_wait(ob_ctx* ctx, ob_design* d);
/* The same for mode N (a collective: every rank of the context's communicator calls it, with ITS contiguous slice of
 * the frame, slices in rank order): the result is rank's ROW SHARD (as ob_design_redistribute_rows builds), but a
 * row is written straight to its place in the shard while the slice is still uploading, only the rows another rank
 * owns wait in an export buffer for one exchange over NVLink, and ob_bootstrap_run overlaps all of it with its
 * replicate generation and a first Gram launch over the rows already in place.  The first call that uses the design
 * performs the exchange and is therefore a collective too. */
ob_status ob_design_pack_row_shard_async(ob_ctx* ctx, const ob_frame_view* slice, ob_design** out);

/* ---- (0) ingest: cleaning and coding on the device --------------------------------------------
 * What the reference does on the host between run()'s clone of the frame (builder.rs:788) and the group split:
 * clean_dataframe (:760-784: drop every row with a null in any used column), create_dummies_manual (:380-418: levels =
 * sorted unique values of the CLEANED frame, first level = base) and split_groups' coding (:61-102).  String columns
 * arrive dictionary-encoded (Arrow DictionaryArray / polars Categorical physical codes / pandas Categorical): an int32
 * code per row (< 0 = null) and a dictionary the HOST keeps, in any order.  Two calls, because only the host can
 * compare strings:
 *   ob_ingest_begin   uploads the columns, computes row validity and which dictionary entries occur among valid rows
 *   (host)            sorts the present entries -> group map (0 = group A, 1 = reference_group, other = ignored) and,
 *                     per categorical, dictionary code -> level code (0 = base); rows_kept < 1 / < 2 groups -> errors
 *   ob_ingest_finish  applies the maps on the device and packs (== ob_design_pack of the cleaned, coded frame)
 * No O(n) work is left on the host. */
typedef struct ob_raw_f64 { const double* data; const uint8_t* valid; } ob_raw_f64;       /* valid NULL = no nulls; valid[i] == 0 = null */
typedef struct ob_raw_dict { const int32_t* codes; int32_t dict_size; } ob_raw_dict;      /* codes[i] < 0 = null */
typedef struct ob_raw_frame {
    int64_t n;
    int32_t n_cont; const ob_raw_f64* cont;
    int32_t n_cat;  const ob_raw_dict* cat;
    ob_raw_f64 outcome;
    ob_raw_f64 weights;          /* data NULL = unweighted */
    ob_raw_dict group;
    int32_t nan_is_null;         /* 1: a NaN in a numeric column is a null too (numpy / pandas frames), tested on the device */
} ob_raw_frame;
typedef struct ob_ingest ob_ingest;
ob_status ob_ingest_begin(ob_ctx* ctx, const ob_raw_frame* frame, ob_ingest** out);
ob_status ob_ingest_rows_kept(const ob_ingest* ing, int64_t* rows_kept);
/* present_out [dict_size]: 1 if the entry occurs in a kept row; column = categorical index, or -1 for the group column */
ob_status ob_ingest_presence(const ob_ingest* ing, int32_t column, uint8_t* present_out);
/* group_map [group dict_size]; cat_remap [n_cat][dict_size] (entries absent from the cleaned frame: any value < 0);
 * cat_levels [n_cat] level counts incl. base.  May be called once per ingest object (codes are remapped in place);
 * destroy the object afterwards. */
ob_status ob_ingest_finish(ob_ctx* ctx, ob_ingest* ing, const int32_t* group_map, const int32_t* const* cat_remap,
                           const int32_t* cat_levels, ob_design** out);
void ob_ingest_destroy(ob_ingest* ing);

/* Same, from the dense matrices get_data_matrices() returns (builder.rs:252-291): row-major
 * X_g [n_g x K] incl. the intercept column, y_g, optional w_g.  n_cont fixes the pooled
 * indicator position (builder.rs:560-564). */
ob_status ob_design_from_dense(ob_ctx* ctx, int32_t K, int32_t n_cont,
                               const double* Xa, const double* ya, const double* wa, int64_t na,
                               const double* Xb, const double* yb, const double* wb, int64_t nb,
                               ob_design** out);
void ob_design_destroy(ob_design* d);
ob_status ob_design_shape(const ob_design* d, int64_t* na, int64_t* nb, int32_t* K, int32_t* n_cont);
/* device time (CUDA events, ms) ob_design_pack spent uploading the columns and in the pack kernels; either may be NULL */
ob_status ob_design_pack_timings(const ob_design* d, double* ms_h2d, double* ms_pack_kernels);
/* get_data_matrices() equivalent: copies the packed design back (row-major [n_g x K]); any pointer may be NULL */
ob_status ob_design_download(ob_ctx* ctx, const ob_design* d, double* Xa, double* ya, double* wa,
                             double* Xb, double* yb, double* wb);
/* Outcome refresh for callers that re-run the decomposition on the SAME predictors with another outcome (JMP's two
 * runs, jmp.rs:44-106; the engine's perturbed-wage sweeps, engine/src/analysis.rs:871-914): replaces the outcome
 * column of the packed design by y_frame (host, one value per row of the frame the design was packed from, nulls
 * not allowed), keeping X, the weights and the group split resident.  8 n bytes over PCIe instead of the whole frame.
 * Undoes a previous ob_design_apply_rif.  For ob_design_from_dense designs the "frame" is [y_a ; y_b]. */
ob_status ob_design_update_outcome(ob_ctx* ctx, ob_design* d, const double* y_frame, int64_t n_frame);
/* decompose_quantile pre-step (builder.rs:721-737 -> math/rif.rs:14-88): replaces each group's
 * outcome by its RIF at quantile tau, computed on the device, unweighted, per group.  The raw outcome is kept, so a
 * quantile sweep (tau = 0.1, 0.5, 0.9 ...) packs once and calls apply_rif + ob_bootstrap_run per quantile: every call
 * transforms the RAW outcome, never an earlier RIF. */
ob_status ob_design_apply_rif(ob_ctx* ctx, ob_design* d, double tau);
/* Quantile sweep in one pass (decompose_quantile called for tau = 0.1, 0.5, 0.9 ..., builder.rs:711-757): the design
 * gets one RIF outcome column per quantile (1 <= n_tau <= 8), side by side.  ob_bootstrap_run then contracts X'WX once
 * and X'Wy once per quantile in the same pass (P = K(K+1)/2 + n_tau K Gram columns instead of n_tau (K(K+1)/2 + K)),
 * factors each replicate's Gram once and solves n_tau right-hand sides.  Every per-outcome array of ob_result grows a
 * leading quantile dimension: point_stats, std_err, p_value, ci_*, t_stat [n_tau x S]; beta_star, beta_a, beta_b
 * [n_tau x K]; rep_stats [rows x n_tau x S]; rep_beta_* [rows x n_tau x K]; residuals_b [n_tau x n_b];
 * total_gap_multi [n_tau].  All quantiles see the same resamples (the reference draws fresh ones per call; with a
 * fixed seed ours are the same per call anyway), so each quantile's results equal a single-quantile run bit for bit.
 * ob_design_apply_rif(tau) is the n_tau = 1 case; ob_design_update_outcome returns to one raw outcome.
 * On a row shard (mode N) both are collectives: the radix-select histograms and the leaf partial sums of mean, SD and
 * density are all-reduced over the context's communicator, and the RIF values are bit-identical to the unsharded ones. */
ob_status ob_design_apply_rif_multi(ob_ctx* ctx, ob_design* d, const double* taus, int32_t n_tau);
ob_status ob_design_num_outcomes(const ob_design* d, int32_t* n_out);

/* ---- Heckman selection (OaxacaBuilder::heckman_selection, builder.rs:236-246; HeckmanEstimator, estimation.rs:114-269) --
 * Attaches the selection equation to a packed design: the binary selection outcome and the selection predictors, one
 * value per row of the frame the design was packed from (host memory, frame order, nulls already dropped like every
 * used column, builder.rs:760-784).  ob_bootstrap_run then runs the two-step estimator on every replicate: probit of
 * the selection outcome on [1 | predictors] over all (resampled) rows of a group (math/probit.rs:25-175), inverse Mills
 * ratio on the rows with selection == 1, OLS of the outcome on [X | IMR] over those rows (heckman.rs:38-108).  All
 * coefficient and mean vectors get one more entry (IMR, last), and the statistics are
 *   S = 5 + 2 (K + 1) + K1:  [explained, unexplained, endowments, coefficients, interaction,
 *                            detailed_explained[K+1], detailed_unexplained[K+1], detailed_selection[K1]]
 * with K1 = 1 + n_pred (builder.rs:464-534; the first selection row is the intercept's).  As in the reference, Yun
 * normalisation is not applied under Heckman (estimation.rs:160-161, builder.rs:634) and residuals are zeros.
 * Refused (OB_ERR_UNSUPPORTED): Pooled | Neumark reference coefficients (the reference's pooled regression yields K
 * coefficients against K+1, builder.rs:548-589 vs estimation.rs:139-141), sample weights, row-sharded designs,
 * more than 7 selection predictors. */
typedef struct ob_selection_view {
    int32_t n_pred;                  /* selection predictors, user order */
    const double* const* pred;       /* [n_pred] columns of n_frame doubles */
    const double* outcome;           /* [n_frame] selection outcome: 1 = the outcome is observed */
} ob_selection_view;
ob_status ob_design_attach_selection(ob_ctx* ctx, ob_design* d, const ob_selection_view* sel, int64_t n_frame);
ob_status ob_design_selection_cols(const ob_design* d, int32_t* k1_out);     /* 0 = no selection equation attached */
int32_t ob_num_stats_heckman(int32_t K, int32_t K1);

/* ---- cluster bootstrap: resample whole clusters instead of rows ---------------------------------------------------
 * Rows nested in clusters (employees in firms, people in panels, households in PSUs) are not independent draws; under
 * intra-cluster correlation the row bootstrap understates every SE, p-value and CI width.  A clustered design resamples
 * UNITS with replacement, and a drawn unit brings all its rows; replicate b is the reference's run_single_pass
 * (builder.rs:420-699) on the frame made of the drawn units' rows, so group sizes vary by replicate:
 *   OB_CLUSTER_BY_GROUP  a unit is a (cluster, group) pair; each replicate draws M_A units from group A's and M_B from group
 *                        B's, independently (M_g = clusters with at least one row in group g).  With singleton clusters
 *                        this is the row bootstrap; coded in frame order, the native stream gives its counts bit for bit.
 *   OB_CLUSTER_JOINT     one stratum: a unit is a cluster with a row in group A or B, each replicate draws M of them and a
 *                        drawn unit contributes its rows of both groups.  A group can come out empty or too small; such a
 *                        replicate fails (OB_ERR_INVALID_GROUP / OB_ERR_INSUFFICIENT_DATA) and is dropped like any failed
 *                        replicate.
 * Units are numbered by ascending cluster code; an explicit index stream (ob_boot_opts.idx_a / idx_b) draws unit positions:
 * BY_GROUP idx_a [reps x M_A], idx_b [reps x M_B]; JOINT idx_a [reps x M] with idx_b = NULL.  The native stream is keyed
 * like the row stream by (seed; unit, stream tag, global replicate id), tag = the group under BY_GROUP and 2 under JOINT,
 * so results do not depend on batching or replicate sharding.  The point estimate and RIF outcomes use the full sample.
 * codes_frame [n_frame]: one code in [0, n_codes) per row of the frame the design was packed from (rows the cleaning
 * dropped are never read; a kept row's code out of range is OB_ERR_INVALID_ARG).  strata NONE detaches (codes may be NULL)
 * and the design resamples rows again.  Attaching or detaching invalidates a Gram cache's X'WX (the next cached run fills).
 * Refused (OB_ERR_UNSUPPORTED): row-sharded designs (mode N), designs with a selection equation (either order), and
 * ob_mm_run on a clustered design.  ob_debug_counts returns the expanded row counts of the native stream. */
typedef enum { OB_CLUSTER_NONE = 0, OB_CLUSTER_BY_GROUP = 1, OB_CLUSTER_JOINT = 2 } ob_cluster_strata;
ob_status ob_design_attach_clusters(ob_ctx* ctx, ob_design* d, const int32_t* codes_frame, int64_t n_frame,
                                    int32_t n_codes, int32_t strata);
/* strata and unit counts of a design (NONE, 0, 0 when unclustered; JOINT: units_a == units_b == M) */
ob_status ob_design_clusters(const ob_design* d, int32_t* strata, int64_t* units_a, int64_t* units_b);

/* ---- (2)-(5) bootstrap ---------------------------------------------------------------------*/
typedef struct ob_boot_opts {
    int32_t ref_kind;                /* ob_ref_kind; builder default is GROUP_A (builder.rs:123) */
    /* .normalize([...]) entries (normalization.rs:5-51), in user order */
    int32_t n_norm;
    const int32_t* norm_m;           /* [n_norm] level count incl. base (category_counts, builder.rs:799) */
    const int32_t* norm_off;         /* [n_norm+1] offsets into norm_idx */
    const int32_t* norm_idx;         /* design-column indices matched by the "{var}_" name prefix (normalization.rs:14-20) */
    const int32_t* norm_has_base;    /* [n_norm] 1 if a base-category row is emitted (builder.rs:636-640) */
    int64_t reps;                    /* bootstrap_reps; 0 is legal (all SE fields NaN, builder.rs:851-855) */
    uint64_t seed;                   /* Philox key of the native resampling stream */
    /* test-only explicit resample index stream (host memory): idx_a [reps x n_a], idx_b [reps x n_b],
     * row positions within the group in frame order; NULL = native Philox stream */
    const uint32_t* idx_a;
    const uint32_t* idx_b;
    /* replicate shard [rep_begin, rep_end) of the global replicate ids 0..reps-1 computed by this
     * call; rep_end = 0 means reps.  Streams are keyed by global id, so results do not depend on the sharding. */
    int64_t rep_begin;
    int64_t rep_end;
    int32_t skip_reduce;             /* 1: stop after per-replicate statistics (multi-GPU: gather first, then ob_reduce_stats) */
    int32_t count_bits;              /* 0 auto, 8 or 16: width of the multiplicity matrix.  16 needs K + outcomes <= 268
                                        (the Gram kernel's shared memory; wider designs are refused, OB_ERR_UNSUPPORTED);
                                        auto starts at 8 and widens to 16 when a count saturates, where 16 fits */
    int64_t max_workspace_bytes;     /* 0 = default (60% of free HBM); bounds the multiplicity-matrix batch */
    /* Mode R inside the library (replicate sharding; SURVEY 8e): 1 = the context carries a communicator of `world`
     * ranks (ob_comm_init_*), every rank holds the WHOLE design and makes this same call; the library computes the
     * contiguous balanced shard of the global replicate ids that belongs to its rank (rep_begin / rep_end must be 0),
     * all-gathers the replicate statistics device to device over the communicator (NVLink) and runs the reduction on
     * every rank: identical results everywhere, bit-identical to one GPU.  rep_* outputs then cover ALL reps rows.
     * An explicit index stream, if given, is the full [reps x n] stream on every rank. */
    int32_t shard_replicates;
} ob_boot_opts;

/* Caller-allocated outputs (host memory).  D = K + n_base rows in each detailed list, where n_base =
 * number of normalize entries with has_base; S = 5 + 2*D statistics per replicate, ordered
 *   [explained, unexplained, endowments, coefficients, interaction, detailed_explained[D], detailed_unexplained[D]]
 * (builder.rs:867-930).  Optional pointers may be NULL. */
typedef struct ob_result {
    /* point estimates (builder.rs:810-811, :932-950) */
    double total_gap;
    double* point_stats;     /* [S] */
    double* xa_mean;         /* [K] */
    double* xb_mean;         /* [K] */
    double* beta_star;       /* [K] */
    double* beta_a;          /* [K] optional: group coefficients after Yun */
    double* beta_b;          /* [K] optional */
    double* residuals_b;     /* [n_b] optional: OaxacaResults.residuals (builder.rs:946) */
    /* reduction over successful replicates (inference.rs:4-34, builder.rs:849-865) */
    int64_t n_ok;
    double* std_err;         /* [S] */
    double* p_value;         /* [S] */
    double* ci_lower;        /* [S] */
    double* ci_upper;        /* [S] */
    double* t_stat;          /* [S] */
    /* per-replicate detail for this call's shard, rows = rep_end - rep_begin (optional) */
    double* rep_stats;       /* [rows x S], NaN rows for failed replicates */
    int32_t* rep_status;     /* [rows] ob_status of each replicate (OB_OK / OB_ERR_NALGEBRA / ...) */
    double* rep_beta_a;      /* [rows x K] */
    double* rep_beta_b;      /* [rows x K] */
    /* device timings of the last call, milliseconds (CUDA events) */
    double ms_counts, ms_gram, ms_solve, ms_reduce, ms_total;
    double ms_gram_kernel;   /* the DMMA contraction kernel alone (ms_gram also covers the split-n partial reduction) */
    int32_t gpu_launches;    /* kernels launched by this call */
    double ms_comm;          /* row-sharded runs: time inside the collectives (also contained in ms_counts / ms_total) */
    double* total_gap_multi; /* [n_tau] optional: total gap per outcome of a multi-outcome design (total_gap = the first) */
    double* sel_gamma_a;     /* [K1] optional, Heckman designs: probit coefficients of the point estimate, group A */
    double* sel_gamma_b;     /* [K1] optional */
} ob_result;

int32_t ob_num_stats(int32_t K, int32_t n_norm, const int32_t* norm_has_base);

ob_status ob_bootstrap_run(ob_ctx* ctx, const ob_design* design, const ob_boot_opts* opts, ob_result* res);

/* ---- outcome sweeps over fixed resamples: the per-replicate Gram cache --------------------------------------------
 * The replicates of the native stream depend only on (seed, global replicate id, group sizes), so re-running the
 * bootstrap on the same design with a new outcome (ob_design_update_outcome, ob_design_apply_rif*) resamples exactly the
 * same rows: every replicate's X'WX is unchanged, only X'Wy is new.  A cache keeps, for every slot of a run (the point
 * estimate and this rank's replicates) and both groups, the reduced X'WX upper triangle and the X'Wy cells of the last
 * outcome.  ob_bootstrap_run_cached takes the same inputs and returns the same outputs as ob_bootstrap_run, bit for bit;
 * it contracts only what the cache does not hold:
 *   OB_CACHE_FILLED        nothing reusable (another design, X / weights / row shard changed, another seed, reps, replicate
 *                          range or sharding): the full contraction, the cache is (re)filled;
 *   OB_CACHE_OUTCOME_ONLY  X'WX reusable: only the K T + 1 outcome columns are contracted (also when T changed);
 *   OB_CACHE_SOLVE_ONLY    X'WX and the outcome unchanged (another ref_kind or normalisation): no resampling and no
 *                          contraction, only the solves and the reduction.
 * ref_kind, normalisation, skip_reduce, max_workspace_bytes and count_bits are not part of the key.  Explicit index
 * streams and designs with a selection equation are refused (OB_ERR_UNSUPPORTED); a cache belongs to the context that
 * created it (another context: OB_ERR_INVALID_ARG).  A call that fails leaves the cache empty.  Sharded runs (mode R and
 * mode N) agree on the use over the communicator, every rank takes the same path.  The device memory (about
 * 16 K(K+1)/2 + 16 (K T + 1) bytes per slot, from the context's design pool) is released by ob_gram_cache_destroy or by
 * ob_ctx_destroy, whichever comes first; a cache outliving its context only frees its host struct. */
typedef struct ob_gram_cache ob_gram_cache;
typedef enum { OB_CACHE_NONE = 0, OB_CACHE_FILLED = 1, OB_CACHE_OUTCOME_ONLY = 2, OB_CACHE_SOLVE_ONLY = 3 } ob_cache_use;
ob_status ob_gram_cache_create(ob_ctx* ctx, ob_gram_cache** out);
void ob_gram_cache_destroy(ob_gram_cache* c);
/* what the last ob_bootstrap_run_cached on c did (ob_cache_use; OB_CACHE_NONE before the first call or after a failed one)
 * and the device memory the cache holds */
ob_status ob_gram_cache_last_use(const ob_gram_cache* c, int32_t* use, int64_t* bytes);
ob_status ob_bootstrap_run_cached(ob_ctx* ctx, const ob_design* design, const ob_boot_opts* opts, ob_gram_cache* cache,
                                  ob_result* res);

/* ---- Bayesian bootstrap (Rubin 1981): Dirichlet-weighted replicates instead of multinomial counts ---------------------
 * Replicate b gives row i of group g the weight pi_i = n_g E_i / sum_{j in g} E_j with E_i ~ iid Exp(1): Dirichlet(1, .., 1)
 * scaled to n_g, stratified by group like the row bootstrap.  A replicate is the reference's single pass (builder.rs:420-699)
 * with the multiplicity c_i replaced by pi_i: WLS on the weights pi_i w_i, means sum(pi w x) / sum(pi w), Cotton / Weighted
 * omega from sum_g pi w when weighted and n_g when not, Pooled stacks the two pi-weighted groups, and the n-guards use n_g
 * (every row is present).  No replicate can lose a row, so none loses a categorical level the way a row-bootstrap draw can
 * (an all-zero dummy column makes X'WX singular and the replicate is dropped).  The point estimate (slot 0, weight 1) is the
 * unchanged point pass.
 * Native stream (wt_a = wt_b = NULL, or bayes = NULL): E = -log U, U in (0, 1) from Philox4x32-10 keyed by (seed; global
 * row, group, global replicate id, a stream tag of its own), E rounded to fp32: results do not depend on batching, grid shape,
 * replicate sharding (mode R) or row sharding (mode N).  Explicit stream (test-only, like idx_a / idx_b): wt_a [reps x n_a]
 * and wt_b [reps x n_b], positive unnormalised E in the group's frame order; the library applies the same normalisation.
 * The weights are fp32 A operands of the FP64 Gram contraction (4 bytes per row and replicate of workspace), which bounds
 * the design at K + outcomes <= 236.  opts->idx_a / idx_b must be NULL and count_bits 0 (OB_ERR_INVALID_ARG).  cache may be
 * NULL; with a cache the native stream fills and reuses it like ob_bootstrap_run_cached (the scheme is part of its key).
 * Refused (OB_ERR_UNSUPPORTED): clustered designs, designs with a selection equation, K + outcomes > 236, and a cache with
 * an explicit stream. */
typedef struct ob_bayes_opts {
    const float* wt_a;               /* [reps x n_a] or NULL (native stream) */
    const float* wt_b;               /* [reps x n_b] or NULL */
} ob_bayes_opts;
ob_status ob_bootstrap_run_bayes(ob_ctx* ctx, const ob_design* design, const ob_boot_opts* opts, const ob_bayes_opts* bayes,
                                 ob_gram_cache* cache, ob_result* res);

/* Reduction alone, on host arrays gathered from several shards, in replicate order
 * (process_component, builder.rs:849-865): out arrays [S] each. */
ob_status ob_reduce_stats(ob_ctx* ctx, const double* rep_stats, const int32_t* rep_status, int64_t reps, int32_t S,
                          const double* point_stats, int64_t* n_ok, double* std_err, double* p_value,
                          double* ci_lower, double* ci_upper, double* t_stat);

/* ---- Machado-Mata quantile decomposition (SURVEY 8f-3) ------------------------------------------------
 * QuantileDecompositionBuilder::run (quantile_decomposition.rs:281-421) from the group split on: the point pass and every
 * bootstrap pass (resample both groups with replacement, :337-354) fit `simulations` quantile regressions per group at
 * random quantiles tau ~ U(0.01, 0.99) (run_single_pass, :173-279; solve_qr, math/quantile_regression.rs:22-135), simulate
 * y_aa = x_a'beta_a(tau), y_bb = x_b'beta_b(tau), y_ab = x_a'beta_b(tau) on one randomly drawn row of each group per
 * simulation, and difference their empirical quantiles (:164-171) at the target quantiles:
 *   statistics per pass  S = 3 n_quantiles:  [gap = q_aa - q_bb, characteristics = q_ab - q_bb, coefficients = q_aa - q_ab]
 * per target quantile, reduced over the passes by bootstrap_stats (inference.rs:4-34; t = estimate / se when |se| > 1e-9).
 * A pass is a column of the multiplicity matrix ob_bootstrap_run builds; each regression is solved on the device to the
 * LP's optimal vertex (interior point + polish, csrc/mm.cu) -- the reference's clarabel solution is that vertex up to the
 * solver's tolerance.  A regression that does not converge is dropped like a non-Solved clarabel status (:227-236), a
 * pass with fewer than simulations / 2 fits in a group fails (:238-242) and is dropped from the reduction (:350-353);
 * on the point pass that is OB_ERR_NALGEBRA.  The design must be unweighted with one raw outcome (the Machado-Mata
 * builder has neither weights nor a RIF), K <= 47 columns; row-sharded designs are refused.
 * Test-only explicit streams (the reference's are unseeded thread_rng draws): idx_a / idx_b as in ob_boot_opts; taus
 * [(reps + 1) x simulations], pass 0 = point estimates; draw_a / draw_b [(reps + 1) x simulations] = position of the
 * simulated row in the pass's (resampled) group frame (needs idx_* when reps > 0).  NULL = native Philox streams. */
typedef struct ob_mm_opts {
    int32_t simulations;             /* builder default 200 (quantile_decomposition.rs:58), <= 4096 */
    int32_t n_quantiles;
    const double* quantiles;         /* builder default 0.1 0.25 0.5 0.75 0.9 (:57) */
    int64_t reps;                    /* bootstrap_reps, builder default 20 (:59) */
    uint64_t seed;
    const uint32_t* idx_a;
    const uint32_t* idx_b;
    const double* taus;
    const uint32_t* draw_a;
    const uint32_t* draw_b;
    int64_t rep_begin;               /* replicate shard as in ob_boot_opts (rep_end = 0: all) */
    int64_t rep_end;
    int32_t skip_reduce;
    int32_t count_bits;              /* 0 auto, 8 or 16 */
    int64_t max_workspace_bytes;     /* 0 = default (60% of free HBM) */
    int32_t shard_replicates;        /* mode R inside the library: every rank holds the design and makes this same call; the
                                        library splits each batch's (pass, simulation, group) regressions evenly over the
                                        ranks (finer than a pass-level split: 20 passes do not divide over 8 GPUs, 8400
                                        regressions do), all-gathers the coefficients device to device over the context's
                                        communicator and computes effects + reduction on every rank: identical results
                                        everywhere, bit-identical to one GPU */
} ob_mm_opts;

typedef struct ob_mm_result {
    double* point_stats;             /* [n_quantiles x 3] */
    int64_t n_ok;
    double* std_err;                 /* [n_quantiles x 3] each */
    double* p_value;
    double* ci_lower;
    double* ci_upper;
    double* t_stat;
    double* rep_stats;               /* [rows x n_quantiles x 3] optional, NaN rows for failed passes */
    int32_t* rep_status;             /* [rows] optional */
    double* point_betas_a;           /* [simulations x K] optional: the point pass's fitted coefficients (NaN rows = failed) */
    double* point_betas_b;
    int32_t* point_qr_info_a;        /* [simulations] optional: status (0 vertex verified, 1 interior-point solution only, */
    int32_t* point_qr_info_b;        /*   2 failed) | interior-point iterations << 8 | rows used by the polish << 16 */
    int64_t qr_total, qr_vertex, qr_approx, qr_failed, qr_iterations;   /* over the regressions of this call */
    double ms_counts, ms_qr, ms_effects, ms_reduce, ms_total;
    int32_t gpu_launches;
} ob_mm_result;

ob_status ob_mm_run(ob_ctx* ctx, const ob_design* design, const ob_mm_opts* opts, ob_mm_result* res);

/* ---- multi-GPU ---------------------------------------------------------------------------------
 * Mode R (replicate sharding, the default): every GPU holds the whole design.  With a communicator attached to the
 * context, ob_boot_opts.shard_replicates = 1 does everything inside the library: shard, device-to-device all-gather
 * of the statistics over NVLink, reduction on every rank.  Without one, each GPU runs ob_bootstrap_run on its
 * [rep_begin, rep_end) with skip_reduce = 1, the host gathers the replicate rows and calls ob_reduce_stats.
 *
 * Mode N (row sharding, for n too large for one HBM; BASELINE config 5): the rows of each group are cut
 * by ob_row_shard_plan into `world` contiguous ranges (world a power of two <= 64; the cut follows the
 * fixed summation tree of the Gram contraction, so results are bit-identical for every world size).  Rank r
 * packs only its rows, marks the design with ob_design_set_row_shard and attaches a communicator to its
 * context; ob_bootstrap_run then exchanges, per panel batch, the replicate column sums (all-reduce) and the
 * per-rank Gram sums (all-gather) and returns identical statistics on every rank (residuals_b covers the
 * local rows of group B only).  An explicit index stream, if given, holds GLOBAL row positions.
 *
 * Communicators: NCCL over NVLink/NVSwitch for one process per GPU (libnccl.so.2 is opened at run time;
 * rank 0 creates the id, the host broadcasts its 128 bytes), or an in-process group for several contexts
 * (threads) of one process. */
#define OB_COMM_ID_BYTES 128
/* replicate shard [begin, end) of `rank` under shard_replicates (contiguous, balanced: the first reps % world ranks
 * hold one replicate more) */
ob_status ob_replicate_shard(int64_t reps, int32_t world, int32_t rank, int64_t* rep_begin, int64_t* rep_end);
ob_status ob_comm_unique_id(uint8_t* id128);
ob_status ob_comm_init_nccl(ob_ctx* ctx, const uint8_t* id128, int32_t rank, int32_t world);
typedef struct ob_local_group ob_local_group;
ob_status ob_local_group_create(int32_t world, ob_local_group** out);
void ob_local_group_destroy(ob_local_group* group);
ob_status ob_comm_init_local(ob_ctx* ctx, ob_local_group* group, int32_t rank);
void ob_comm_destroy(ob_ctx* ctx);
/* rows [row_begin, row_end) of a group of n_group rows (positions within the group, frame order) that rank holds */
ob_status ob_row_shard_plan(int64_t n_group, int32_t world, int32_t rank, int64_t* row_begin, int64_t* row_end);
/* declares a packed design to be rank's shard of groups of n_a_global / n_b_global rows (its local row counts
 * must equal the plan's) */
ob_status ob_design_set_row_shard(ob_design* d, int64_t n_a_global, int64_t n_b_global, int32_t world, int32_t rank);

/* Mode R with a distributed upload: every rank packed a CONTIGUOUS SLICE of the frame (ob_design_pack on rows
 * [n r / world, n (r+1) / world), slices in rank order); assembles the full per-group designs on every rank with one
 * variable-size all-gather over the context's communicator (NVLink), so that a rank moves only 1/world of the frame
 * over PCIe.  The result equals ob_design_pack of the whole frame bit for bit. */
ob_status ob_design_allgather_rows(ob_ctx* ctx, const ob_design* local_slice, ob_design** out);

/* how a design sits inside the whole problem: global group sizes and (world, rank) of its row shard (1, 0 if unsharded) */
ob_status ob_design_row_shard(const ob_design* d, int64_t* n_a_global, int64_t* n_b_global, int32_t* world, int32_t* rank);

/* Mode N from frame slices: every rank packed a CONTIGUOUS SLICE of the frame (as for ob_design_allgather_rows);
 * re-cuts each group's rows along ob_row_shard_plan and exchanges them over the communicator (NVLink; point-to-point,
 * every row moves at most once, and hardly any when the groups are spread evenly over the frame).  The result is
 * rank's row shard, already marked as such (ob_design_set_row_shard is not needed), bit-identical to packing exactly
 * the plan's rows.  A rank then uploads 1/world of the frame and never holds more than 1/world of the design. */
ob_status ob_design_redistribute_rows(ob_ctx* ctx, const ob_design* local_slice, ob_design** out);

/* Host-only debugging aid (no device needed): the work-unit schedule of the Gram kernel for a problem shape -- out8
 * receives up to cap rows of (cta, group, panel, column tile, row segment, pipeline stages, 8-slot groups, quanta of a
 * tail tile or 0 for a full tile);
 * returns the total number of units or -1 on bad arguments.  The CPU tests use it to check that every
 * (group, panel, tile, segment) is computed exactly once and that the CTAs get equal shares. */
int64_t ob_debug_gram_schedule(int32_t K, int64_t n_a, int64_t n_b, int64_t slots, int32_t world, int32_t rank, int32_t grid,
                               int64_t* out8, int64_t cap);

/* Host-only debugging aid: the columns the Gram contraction computes for a design with n_cont continuous predictors
 * and the categorical predictors cat_levels [n_cat] (level counts incl. the base; K must equal 1 + n_cont + sum(m - 1),
 * else -- and for n_cat = 0 -- nothing is dropped) and T outcome columns: pairs_out [cap][2] = design-row offsets (j, l)
 * of computed column c, colmap_out [cap] = its index in the row-major upper triangle of [x|y][x|y]^T (-1 = padding).
 * The products of two different dummies of one categorical are structural zeros of X'WX and are not computed.
 * tiling_out[3] (may be NULL) = {computed columns, tiles of 128 columns, quanta of 32 columns in the tail tile}.
 * Returns the table length (tiles x 128) or -1 on bad arguments. */
int64_t ob_debug_gram_columns(int32_t K, int32_t T, int32_t n_cont, const int32_t* cat_levels, int32_t n_cat,
                              uint16_t* pairs_out, int32_t* colmap_out, int64_t cap, int32_t* tiling_out);
/* The same for the outcome-only contraction of ob_bootstrap_run_cached (OB_CACHE_OUTCOME_ONLY): the K T columns of X'Wy
 * and the (y_0, y_0) cell, in the order of the full table, tiled like it. */
int64_t ob_debug_gram_outcome_columns(int32_t K, int32_t T, uint16_t* pairs_out, int32_t* colmap_out, int64_t cap,
                                      int32_t* tiling_out);

/* Multiplicity counts of one replicate of the native stream (for the statistical validation
 * tests): counts_out [n] for group g (0 = A, 1 = B) of design d. */
ob_status ob_debug_counts(ob_ctx* ctx, const ob_design* d, uint64_t seed, int64_t rep, int32_t group,
                          uint16_t* counts_out);

/* The native Bayesian-bootstrap weights E (unnormalised, fp32) of global replicate `rep` of `group`, [n_group] in row
 * order, from the production kernel (tests; not on row-sharded designs). */
ob_status ob_debug_bayes_weights(ob_ctx* ctx, const ob_design* d, uint64_t seed, int64_t rep, int32_t group, float* out);
/* The multiplicity matrix ob_bootstrap_run builds from an explicit index stream (same kernel), read back for the
 * bit-exactness tests: idx [reps x n_global] (host; global row positions within the group), counts_out
 * [reps x n_local] (row-major by replicate; n_local = the rows of the group this design holds, all of them unless
 * row-sharded), count_bits 8 or 16.  flags_out (may be NULL): bit 0 = a count saturated at the width, bit 1 = an
 * index was >= n_global. */
ob_status ob_debug_counts_from_indices(ob_ctx* ctx, const ob_design* d, int32_t group, const uint32_t* idx, int64_t reps,
                                       int32_t count_bits, uint16_t* counts_out, int32_t* flags_out);

/* What the last successful ob_bootstrap_run_cached left in cache c (read-only; for the cell-by-cell tests of the Gram
 * contraction): shape_out[5] = {slots, K, T, count_bytes of the fill (1 or 2), 1 if row counts are held (clustered
 * designs) else 0}; xx_out [2][slots][K(K+1)/2] = the X'WX upper triangles, row-major; yy_out [2][slots][K T + 1] = the
 * cells (j, y_t), j-major, then (y_0, y_0); rows_out [2][slots] = each slot's group row counts (clustered designs only,
 * else untouched).  Slot 0 is the point estimate, slot s >= 1 replicate rep_begin + s - 1 of the run (under
 * shard_replicates: of this rank's shard).  Any output may be NULL.  An empty cache is OB_ERR_INVALID_ARG. */
ob_status ob_debug_gram_cache_read(ob_ctx* ctx, const ob_gram_cache* c, int64_t* shape_out, double* xx_out, double* yy_out,
                                   int64_t* rows_out);

#ifdef __cplusplus
}
#endif
#endif /* OBBOOT_H */
