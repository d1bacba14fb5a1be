// csrc/host/builder.h -- host-side mirror of the reference's builder interface for the bootstrap path.
//
// Same names, argument meaning and error variants as oaxaca_blinder's OaxacaBuilder (builder.rs:37-246,
// :711-757, :787-951), ReferenceCoefficients (decomposition.rs:5-20), OaxacaResults / ComponentResult
// (types.rs:10-47, :162-180), OaxacaError (error.rs:6-40) and Formula (formula.rs:12-60).  The frame is a
// minimal columnar table (f64 / string columns with validity) standing in for polars::DataFrame.
// Everything numeric is delegated to libobboot's C ABI (include/obboot.h): this layer only cleans, codes,
// names and assembles.
#pragma once
#include <cstdint>
#include <iosfwd>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../../include/obboot.h"

namespace ob {

struct Column {
    std::string name;
    bool is_str = false;
    std::vector<double> f64;
    std::vector<std::string> str;
    std::vector<uint8_t> valid;   // empty = no nulls
    bool is_valid(size_t i) const { return valid.empty() || valid[i]; }
};

class DataFrame {
public:
    void add_f64(const std::string& name, std::vector<double> data, std::vector<uint8_t> valid = {});
    void add_str(const std::string& name, std::vector<std::string> data, std::vector<uint8_t> valid = {});
    const Column* find(const std::string& name) const;
    size_t height() const { return height_; }
    const std::vector<Column>& columns() const { return cols_; }
    // header + rows; a column is f64 if every non-empty cell parses as a number (empty cell = null)
    static DataFrame read_csv(const std::string& path);
private:
    std::vector<Column> cols_;
    size_t height_ = 0;
};

// OaxacaError (error.rs:6-19); kind is the ob_status of the variant
class OaxacaError : public std::runtime_error {
public:
    OaxacaError(ob_status k, const std::string& msg) : std::runtime_error(msg), kind(k) {}
    ob_status kind;
    static std::string display(ob_status k, const std::string& detail);   // Display impl, error.rs:27-38
};

enum class ReferenceCoefficients { GroupA = 0, GroupB = 1, Pooled = 2, Weighted = 3, Cotton = 4, Neumark = 5 };

struct ComponentResult {   // types.rs:172-180
    std::string name;
    double estimate, std_err, t_stat, p_value, ci_lower, ci_upper;
};

struct OaxacaResults {     // types.rs:24-47
    double total_gap = 0;
    struct { std::vector<ComponentResult> aggregate, detailed_explained, detailed_unexplained, detailed_selection; } two_fold;
    struct { std::vector<ComponentResult> aggregate, detailed; } three_fold;
    size_t n_a = 0, n_b = 0;
    std::vector<double> residuals, xa_mean, xb_mean, beta_star;
    // not in the reference struct: bookkeeping of the replicate loop (builder.rs:841-847)
    int64_t bootstrap_reps = 0, successful_bootstraps = 0;
    std::vector<std::string> predictor_names;
    double ms_total = 0, ms_gram = 0;
    // cluster bootstrap (OaxacaBuilder::cluster): ob_cluster_strata and the units resampled per replicate (JOINT: a == b)
    int cluster_strata = OB_CLUSTER_NONE;
    int64_t cluster_units_a = 0, cluster_units_b = 0;
    bool bayesian = false;     // OaxacaBuilder::bayesian_bootstrap: Dirichlet-weighted replicates

    void summary(std::ostream& os) const;                          // display.rs:9-79
    std::string to_json(bool with_residuals, bool with_extra) const;   // display.rs to_json (serde layout) [+ extras]
    std::string to_markdown() const;
};

struct Formula {           // formula.rs:12-60
    std::string outcome;
    std::vector<std::string> predictors, categorical_predictors;
    static Formula parse(const std::string& s);
};

struct DataMatrices {      // get_data_matrices, builder.rs:252-291 (row-major)
    std::vector<double> x_a, y_a, x_b, y_b;
    size_t n_a = 0, n_b = 0, k = 0;
    std::vector<std::string> predictor_names;
};

class QuantileDecompositionBuilder;

class OaxacaBuilder {
    friend class QuantileDecompositionBuilder;   // shares the device ingest (cleaning, coding, pack)
public:
    OaxacaBuilder(DataFrame df, const std::string& outcome, const std::string& group, const std::string& reference_group);
    static OaxacaBuilder from_formula(DataFrame df, const std::string& formula, const std::string& group,
                                      const std::string& reference_group);
    OaxacaBuilder& reference_coefficients(ReferenceCoefficients r) { reference_coeffs_ = r; return *this; }
    OaxacaBuilder& predictors(std::vector<std::string> p) { predictors_ = std::move(p); return *this; }
    OaxacaBuilder& categorical_predictors(std::vector<std::string> p) { categorical_ = std::move(p); return *this; }
    OaxacaBuilder& bootstrap_reps(size_t reps) { bootstrap_reps_ = reps; return *this; }
    OaxacaBuilder& normalize(std::vector<std::string> v) { normalization_vars_ = std::move(v); return *this; }
    OaxacaBuilder& weights(const std::string& w) { weights_col_ = w; has_weights_ = true; return *this; }
    OaxacaBuilder& heckman_selection(const std::string& outcome, std::vector<std::string> preds) {
        selection_outcome_ = outcome; has_selection_ = true; selection_predictors_ = std::move(preds); return *this;
    }
    // additions of the GPU path (SURVEY.md 8b): resampling seed, device, test-only explicit index stream
    OaxacaBuilder& seed(uint64_t s) { seed_ = s; return *this; }
    OaxacaBuilder& device(int d) { device_ = d; return *this; }
    OaxacaBuilder& index_stream(const uint32_t* idx_a, const uint32_t* idx_b) { idx_a_ = idx_a; idx_b_ = idx_b; return *this; }
    // cluster bootstrap: resample whole clusters of `column` (string or numeric labels; codes follow their sorted order)
    // with ob_cluster_strata `strata` (OB_CLUSTER_NONE: back to rows).  The column joins the null filter.
    OaxacaBuilder& cluster(const std::string& column, int strata = OB_CLUSTER_BY_GROUP) {
        cluster_col_ = strata == OB_CLUSTER_NONE ? std::string() : column; cluster_strata_ = strata; return *this;
    }

    // Bayesian bootstrap (ob_bootstrap_run_bayes): every row keeps a Dirichlet weight in every replicate instead of a
    // multinomial count; run, run_outcomes and decompose_quantile honour it
    OaxacaBuilder& bayesian_bootstrap(bool on = true) { bayesian_ = on; return *this; }

    OaxacaResults run() const;                              // builder.rs:787-951
    // run() once per listed outcome column on one ingest: rows are cleaned over all of them, the first run fills a Gram
    // cache and the others only contract their outcome columns (ob_bootstrap_run_cached)
    std::vector<OaxacaResults> run_outcomes(const std::vector<std::string>& outcomes) const;
    OaxacaResults decompose_quantile(double quantile) const; // builder.rs:711-757
    DataMatrices get_data_matrices() const;                 // builder.rs:252-291
    std::string describe() const;                           // host-only JSON view of the prepared frame (tests)

private:
    struct Prepared;
    Prepared prepare() const;                                    // host-only restatement (describe(), CPU tests)
    void fill_norm_spec(Prepared& p) const;
    // production path; sweep (run_outcomes): the outcome columns, sweep[0] packed in place of outcome_
    ob_design* ingest_on_device(ob_ctx* ctx, Prepared& meta, bool with_weights, const std::vector<std::string>* sweep = nullptr) const;
    std::vector<OaxacaResults> run_impl(bool rif, double tau, const std::vector<std::string>* sweep = nullptr) const;

    DataFrame dataframe_;
    std::string outcome_, group_, reference_group_;
    std::vector<std::string> predictors_, categorical_, normalization_vars_, selection_predictors_;
    size_t bootstrap_reps_ = 20;                                           // builder.rs:122
    ReferenceCoefficients reference_coeffs_ = ReferenceCoefficients::GroupA; // builder.rs:123 (the code, not the doc comment)
    std::string weights_col_, selection_outcome_;
    bool has_weights_ = false, has_selection_ = false;
    std::string cluster_col_;
    int cluster_strata_ = OB_CLUSTER_NONE;
    bool bayesian_ = false;
    uint64_t seed_ = 0x0B5EEDull;
    int device_ = 0;
    const uint32_t* idx_a_ = nullptr;
    const uint32_t* idx_b_ = nullptr;
};

// ---- Machado-Mata quantile decomposition (quantile_decomposition.rs:21-522) ----
struct QuantileDecompositionDetail {      // quantile_decomposition.rs:512-522
    ComponentResult total_gap, characteristics_effect, coefficients_effect;
};

struct QuantileDecompositionResults {     // quantile_decomposition.rs:425-437
    std::map<std::string, QuantileDecompositionDetail> results_by_quantile;   // keys "q{(tau * 100) as u32}" (:277)
    size_t n_a = 0, n_b = 0;
    // bookkeeping of the GPU path (not in the reference struct)
    int64_t bootstrap_reps = 0, successful_bootstraps = 0;
    int64_t qr_total = 0, qr_vertex = 0, qr_approx = 0, qr_failed = 0;
    double ms_total = 0, ms_qr = 0;

    void summary(std::ostream& os) const;                     // quantile_decomposition.rs:441-505
    std::string to_json() const;
};

class QuantileDecompositionBuilder {      // quantile_decomposition.rs:21-100
public:
    QuantileDecompositionBuilder(DataFrame df, const std::string& outcome, const std::string& group, const std::string& reference_group);
    QuantileDecompositionBuilder& predictors(std::vector<std::string> p) { predictors_ = std::move(p); return *this; }
    QuantileDecompositionBuilder& categorical_predictors(std::vector<std::string> p) { categorical_ = std::move(p); return *this; }
    QuantileDecompositionBuilder& quantiles(std::vector<double> q) { quantiles_ = std::move(q); return *this; }
    QuantileDecompositionBuilder& simulations(size_t reps) { simulations_ = reps; return *this; }
    QuantileDecompositionBuilder& bootstrap_reps(size_t reps) { bootstrap_reps_ = reps; return *this; }
    // additions of the GPU path: seed of the native streams, device, test-only explicit streams (ob_mm_opts)
    QuantileDecompositionBuilder& seed(uint64_t s) { seed_ = s; return *this; }
    QuantileDecompositionBuilder& device(int d) { device_ = d; return *this; }
    QuantileDecompositionBuilder& streams(const uint32_t* idx_a, const uint32_t* idx_b, const double* taus, const uint32_t* draw_a,
                                          const uint32_t* draw_b) {
        idx_a_ = idx_a; idx_b_ = idx_b; taus_ = taus; draw_a_ = draw_a; draw_b_ = draw_b; return *this;
    }
    QuantileDecompositionResults run() const;                 // quantile_decomposition.rs:281-421
    static std::string quantile_key(double tau);              // format!("q{}", (tau * 100.0) as u32), :277

private:
    DataFrame dataframe_;
    std::string outcome_, group_, reference_group_;
    std::vector<std::string> predictors_, categorical_;
    std::vector<double> quantiles_ = {0.1, 0.25, 0.5, 0.75, 0.9};     // :57
    size_t simulations_ = 200, bootstrap_reps_ = 20;                 // :58-59
    uint64_t seed_ = 0x0B5EEDull;
    int device_ = 0;
    const uint32_t *idx_a_ = nullptr, *idx_b_ = nullptr, *draw_a_ = nullptr, *draw_b_ = nullptr;
    const double* taus_ = nullptr;
};

}  // namespace ob
