/* include/obboot_builder.h -- C ABI of the host-side OaxacaBuilder mirror (csrc/host/builder.h).
 *
 * The reference's builder is Rust (builder.rs:37-246); this image has no Rust toolchain, so the host layer is C++
 * and is exported through these plain-C entry points for bindings (the Python mirror in
 * oaxaca_blinder_rs_b200/builder.py uses them through ctypes).  Method names and semantics follow the reference:
 *   OaxacaBuilder::new / from_formula            builder.rs:114-160
 *   .predictors .categorical_predictors .bootstrap_reps .normalize .weights .reference_coefficients
 *   .heckman_selection                           builder.rs:165-246
 *   .run() .decompose_quantile(q) .get_data_matrices()   builder.rs:787, :711, :252
 * Results come back as the JSON the reference's to_json() produces (serde layout of types.rs:10-47), plus the
 * #[serde(skip)] vectors when with_extra != 0.
 */
#ifndef OBBOOT_BUILDER_H
#define OBBOOT_BUILDER_H
#include "obboot.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ob_frame ob_frame;       /* minimal columnar table: f64 / string columns with validity */
typedef struct ob_builder ob_builder;
typedef struct ob_results ob_results;

ob_frame* ob_frame_new(void);
void ob_frame_free(ob_frame* f);
/* valid may be NULL (no nulls); valid[i] == 0 marks a null */
ob_status ob_frame_add_f64(ob_frame* f, const char* name, const double* data, const uint8_t* valid, int64_t n);
/* values[i] == NULL marks a null */
ob_status ob_frame_add_str(ob_frame* f, const char* name, const char* const* values, int64_t n);
/* LazyCsvReader::new(path).with_has_header(true) (main.rs:161-165); on failure *out = NULL and err receives the message */
ob_status ob_frame_read_csv(const char* path, ob_frame** out, char* err, size_t err_len);

/* the frame is copied (run() clones it too, builder.rs:788) */
ob_builder* ob_builder_new(const ob_frame* f, const char* outcome, const char* group, const char* reference_group);
ob_status ob_builder_from_formula(const ob_frame* f, const char* formula, const char* group, const char* reference_group,
                                  ob_builder** out, char* err, size_t err_len);
void ob_builder_free(ob_builder* b);
ob_status ob_builder_predictors(ob_builder* b, const char* const* names, int32_t n);
ob_status ob_builder_categorical_predictors(ob_builder* b, const char* const* names, int32_t n);
ob_status ob_builder_normalize(ob_builder* b, const char* const* names, int32_t n);
ob_status ob_builder_weights(ob_builder* b, const char* column);
ob_status ob_builder_bootstrap_reps(ob_builder* b, int64_t reps);
/* ReferenceCoefficients in declaration order (decomposition.rs:5-20): 0 GroupA 1 GroupB 2 Pooled 3 Weighted 4 Cotton 5 Neumark */
ob_status ob_builder_reference_coefficients(ob_builder* b, int32_t kind);
ob_status ob_builder_heckman_selection(ob_builder* b, const char* outcome, const char* const* predictors, int32_t n);
/* additions of the GPU path: Philox seed, CUDA device, test-only explicit index stream ([reps x n_a], [reps x n_b]) */
ob_status ob_builder_seed(ob_builder* b, uint64_t seed);
ob_status ob_builder_device(ob_builder* b, int32_t device);
ob_status ob_builder_index_stream(ob_builder* b, const uint32_t* idx_a, const uint32_t* idx_b);
/* cluster bootstrap (ob_design_attach_clusters): resample whole clusters of `column` (string or numeric labels, coded in
 * their sorted order; the column joins the null filter) with ob_cluster_strata `strata`; OB_CLUSTER_NONE resamples rows
 * again.  run, run_outcomes and decompose_quantile honour it; an index stream then draws units (joint: idx_b = NULL).
 * The results gain a summary line and a "clusters" JSON key {strata, units_a, units_b}. */
ob_status ob_builder_cluster(ob_builder* b, const char* column, int32_t strata);
/* Bayesian bootstrap (ob_bootstrap_run_bayes) when on != 0: Dirichlet row weights instead of multinomial counts; run,
 * run_outcomes and decompose_quantile honour it.  The results gain a summary line and "bootstrap_scheme": "bayes" in JSON. */
ob_status ob_builder_bayesian(ob_builder* b, int32_t on);

ob_status ob_builder_run(ob_builder* b, ob_results** out);
/* run() once per outcome column names[n] (f64 columns) on ONE ingest: rows are cleaned over every listed column (plus the
 * configured ones), the first run fills a per-replicate Gram cache and the others contract only their outcome columns
 * (ob_bootstrap_run_cached).  outs[n] receives one results object per outcome, each equal to run() with that column as
 * the outcome when the columns share their nulls.  Unsupported with heckman_selection or index_stream. */
ob_status ob_builder_run_outcomes(ob_builder* b, const char* const* names, int32_t n, ob_results** outs);
ob_status ob_builder_decompose_quantile(ob_builder* b, double quantile, ob_results** out);
/* get_data_matrices(): sizes first (any out pointer may be NULL), then the row-major copies */
ob_status ob_builder_get_data_matrices(ob_builder* b, int64_t* n_a, int64_t* n_b, int32_t* k,
                                       double* x_a, double* y_a, double* x_b, double* y_b);
/* Host-only description of the cleaned / coded frame (state at builder.rs:808) as JSON: rows kept, n_a, n_b,
 * design column names, base-category names, categorical level counts, the .normalize index lists.  No device needed. */
const char* ob_builder_describe(ob_builder* b);
/* message of the last failure on this builder: the reference's Display text (error.rs:27-38) */
const char* ob_builder_last_error(const ob_builder* b);
ob_status ob_builder_last_status(const ob_builder* b);   /* status of the last failing call */

void ob_results_free(ob_results* r);
/* to_json(); strings are owned by the results object */
const char* ob_results_json(ob_results* r, int32_t with_residuals, int32_t with_extra);
const char* ob_results_summary(ob_results* r);       /* summary() text (display.rs:9-79) */
const char* ob_results_markdown(ob_results* r);
int64_t ob_results_residuals(const ob_results* r, double* out);   /* returns n_b; copies when out != NULL */

/* ---- Machado-Mata: QuantileDecompositionBuilder (quantile_decomposition.rs:21-100), run() (:281-421),
 * QuantileDecompositionResults (:425-505).  Defaults as in the reference: quantiles 0.1 0.25 0.5 0.75 0.9, 200 simulations,
 * 20 bootstrap replications.  Results as JSON: {"results_by_quantile": {"q25": {"total_gap": {name, estimate, std_err,
 * t_stat, p_value, ci_lower, ci_upper}, "characteristics_effect": {..}, "coefficients_effect": {..}}, ..}, "n_a", "n_b", ..}
 * with the reference's keys "q{(tau * 100) as u32}" (:277). */
typedef struct ob_qd_builder ob_qd_builder;
typedef struct ob_qd_results ob_qd_results;
ob_qd_builder* ob_qd_builder_new(const ob_frame* f, const char* outcome, const char* group, const char* reference_group);
void ob_qd_builder_free(ob_qd_builder* b);
ob_status ob_qd_builder_predictors(ob_qd_builder* b, const char* const* names, int32_t n);
ob_status ob_qd_builder_categorical_predictors(ob_qd_builder* b, const char* const* names, int32_t n);
ob_status ob_qd_builder_quantiles(ob_qd_builder* b, const double* q, int32_t n);
ob_status ob_qd_builder_simulations(ob_qd_builder* b, int64_t reps);
ob_status ob_qd_builder_bootstrap_reps(ob_qd_builder* b, int64_t reps);
/* additions of the GPU path: seed of the native Philox streams, CUDA device, test-only explicit streams (ob_mm_opts) */
ob_status ob_qd_builder_seed(ob_qd_builder* b, uint64_t seed);
ob_status ob_qd_builder_device(ob_qd_builder* b, int32_t device);
ob_status ob_qd_builder_streams(ob_qd_builder* b, const uint32_t* idx_a, const uint32_t* idx_b, const double* taus,
                                const uint32_t* draw_a, const uint32_t* draw_b);
ob_status ob_qd_builder_run(ob_qd_builder* b, ob_qd_results** out);
/* the key of a target quantile in results_by_quantile: format!("q{}", (tau * 100.0) as u32) (quantile_decomposition.rs:277);
 * returns its length */
int32_t ob_qd_quantile_key(double tau, char* out, size_t out_len);
const char* ob_qd_builder_last_error(const ob_qd_builder* b);
ob_status ob_qd_builder_last_status(const ob_qd_builder* b);
void ob_qd_results_free(ob_qd_results* r);
const char* ob_qd_results_json(ob_qd_results* r);
const char* ob_qd_results_summary(ob_qd_results* r);      /* summary() text (quantile_decomposition.rs:441-505) */

#ifdef __cplusplus
}
#endif
#endif
