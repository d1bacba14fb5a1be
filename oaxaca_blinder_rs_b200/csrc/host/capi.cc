// csrc/host/capi.cc -- plain-C surface of the OaxacaBuilder mirror (include/obboot_builder.h).
#include "../../../include/obboot_builder.h"

#include <cstring>
#include <memory>
#include <sstream>

#include "builder.h"

struct ob_frame { ob::DataFrame df; };
struct ob_builder { std::unique_ptr<ob::OaxacaBuilder> b; std::string err, desc; ob_status last = OB_OK; };
struct ob_results { ob::OaxacaResults r; std::string json, summary, markdown; };
struct ob_qd_builder { std::unique_ptr<ob::QuantileDecompositionBuilder> b; std::string err; ob_status last = OB_OK; };
struct ob_qd_results { ob::QuantileDecompositionResults r; std::string json, summary; };

namespace {
std::vector<std::string> strs(const char* const* names, int32_t n) {
    std::vector<std::string> v;
    for (int32_t i = 0; i < n; ++i) v.emplace_back(names[i] ? names[i] : "");
    return v;
}
void put_err(char* err, size_t len, const std::string& m) {
    if (err && len) { std::strncpy(err, m.c_str(), len - 1); err[len - 1] = '\0'; }
}
template <typename B, typename F>
ob_status guarded(B* b, F&& f) {
    if (!b) return OB_ERR_INVALID_ARG;
    try { f(); return OB_OK; }
    catch (const ob::OaxacaError& e) { b->err = e.what(); b->last = e.kind; return e.kind; }
    catch (const std::exception& e) { b->err = e.what(); b->last = OB_ERR_INVALID_ARG; return OB_ERR_INVALID_ARG; }
}
}  // namespace

extern "C" {

ob_frame* ob_frame_new(void) { return new ob_frame; }
void ob_frame_free(ob_frame* f) { delete f; }

ob_status ob_frame_add_f64(ob_frame* f, const char* name, const double* data, const uint8_t* valid, int64_t n) {
    if (!f || !name || (n && !data) || n < 0) return OB_ERR_INVALID_ARG;
    try {
        f->df.add_f64(name, std::vector<double>(data, data + n), valid ? std::vector<uint8_t>(valid, valid + n) : std::vector<uint8_t>{});
        return OB_OK;
    } catch (const ob::OaxacaError& e) { return e.kind; }
}

ob_status ob_frame_add_str(ob_frame* f, const char* name, const char* const* values, int64_t n) {
    if (!f || !name || (n && !values) || n < 0) return OB_ERR_INVALID_ARG;
    try {
        std::vector<std::string> v((size_t)n);
        std::vector<uint8_t> valid((size_t)n, 1);
        bool nulls = false;
        for (int64_t i = 0; i < n; ++i) { if (values[i]) v[i] = values[i]; else { valid[i] = 0; nulls = true; } }
        if (!nulls) valid.clear();
        f->df.add_str(name, std::move(v), std::move(valid));
        return OB_OK;
    } catch (const ob::OaxacaError& e) { return e.kind; }
}

ob_status ob_frame_read_csv(const char* path, ob_frame** out, char* err, size_t err_len) {
    if (!path || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    try {
        auto f = std::make_unique<ob_frame>();
        f->df = ob::DataFrame::read_csv(path);
        *out = f.release();
        return OB_OK;
    } catch (const ob::OaxacaError& e) { put_err(err, err_len, e.what()); return e.kind; }
}

ob_builder* ob_builder_new(const ob_frame* f, const char* outcome, const char* group, const char* reference_group) {
    if (!f || !outcome || !group || !reference_group) return nullptr;
    auto b = new ob_builder;
    b->b = std::make_unique<ob::OaxacaBuilder>(f->df, outcome, group, reference_group);
    return b;
}

ob_status ob_builder_from_formula(const ob_frame* f, const char* formula, const char* group, const char* reference_group,
                                  ob_builder** out, char* err, size_t err_len) {
    if (!f || !formula || !group || !reference_group || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    try {
        auto b = std::make_unique<ob_builder>();
        b->b = std::make_unique<ob::OaxacaBuilder>(ob::OaxacaBuilder::from_formula(f->df, formula, group, reference_group));
        *out = b.release();
        return OB_OK;
    } catch (const ob::OaxacaError& e) { put_err(err, err_len, e.what()); return e.kind; }
}

void ob_builder_free(ob_builder* b) { delete b; }

ob_status ob_builder_predictors(ob_builder* b, const char* const* names, int32_t n) {
    return guarded(b, [&] { b->b->predictors(strs(names, n)); });
}
ob_status ob_builder_categorical_predictors(ob_builder* b, const char* const* names, int32_t n) {
    return guarded(b, [&] { b->b->categorical_predictors(strs(names, n)); });
}
ob_status ob_builder_normalize(ob_builder* b, const char* const* names, int32_t n) {
    return guarded(b, [&] { b->b->normalize(strs(names, n)); });
}
ob_status ob_builder_weights(ob_builder* b, const char* column) {
    return guarded(b, [&] { b->b->weights(column ? column : ""); });
}
ob_status ob_builder_bootstrap_reps(ob_builder* b, int64_t reps) {
    if (reps < 0) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->bootstrap_reps((size_t)reps); });
}
ob_status ob_builder_reference_coefficients(ob_builder* b, int32_t kind) {
    if (kind < 0 || kind > 5) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->reference_coefficients((ob::ReferenceCoefficients)kind); });
}
ob_status ob_builder_heckman_selection(ob_builder* b, const char* outcome, const char* const* predictors, int32_t n) {
    return guarded(b, [&] { b->b->heckman_selection(outcome ? outcome : "", strs(predictors, n)); });
}
ob_status ob_builder_cluster(ob_builder* b, const char* column, int32_t strata) {
    if (strata < OB_CLUSTER_NONE || strata > OB_CLUSTER_JOINT || (strata != OB_CLUSTER_NONE && !column)) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->cluster(column ? column : "", strata); });
}
ob_status ob_builder_bayesian(ob_builder* b, int32_t on) { return guarded(b, [&] { b->b->bayesian_bootstrap(on != 0); }); }
ob_status ob_builder_seed(ob_builder* b, uint64_t seed) { return guarded(b, [&] { b->b->seed(seed); }); }
ob_status ob_builder_device(ob_builder* b, int32_t device) { return guarded(b, [&] { b->b->device(device); }); }
ob_status ob_builder_index_stream(ob_builder* b, const uint32_t* idx_a, const uint32_t* idx_b) {
    return guarded(b, [&] { b->b->index_stream(idx_a, idx_b); });
}

ob_status ob_builder_run(ob_builder* b, ob_results** out) {
    if (!out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(b, [&] { auto r = std::make_unique<ob_results>(); r->r = b->b->run(); *out = r.release(); });
}
ob_status ob_builder_run_outcomes(ob_builder* b, const char* const* names, int32_t n, ob_results** outs) {
    if (!outs || n < 0 || (n > 0 && !names)) return OB_ERR_INVALID_ARG;
    for (int32_t k = 0; k < n; ++k) outs[k] = nullptr;
    return guarded(b, [&] {
        std::vector<std::string> cols;
        for (int32_t k = 0; k < n; ++k) {
            if (!names[k]) throw ob::OaxacaError(OB_ERR_INVALID_ARG, "null outcome column name");
            cols.emplace_back(names[k]);
        }
        std::vector<ob::OaxacaResults> rs = b->b->run_outcomes(cols);
        for (int32_t k = 0; k < n; ++k) { auto r = std::make_unique<ob_results>(); r->r = std::move(rs[(size_t)k]); outs[k] = r.release(); }
    });
}
ob_status ob_builder_decompose_quantile(ob_builder* b, double quantile, ob_results** out) {
    if (!out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(b, [&] { auto r = std::make_unique<ob_results>(); r->r = b->b->decompose_quantile(quantile); *out = r.release(); });
}
ob_status ob_builder_get_data_matrices(ob_builder* b, int64_t* n_a, int64_t* n_b, int32_t* k,
                                       double* x_a, double* y_a, double* x_b, double* y_b) {
    return guarded(b, [&] {
        const ob::DataMatrices m = b->b->get_data_matrices();
        if (n_a) *n_a = (int64_t)m.n_a;
        if (n_b) *n_b = (int64_t)m.n_b;
        if (k) *k = (int32_t)m.k;
        if (x_a) std::memcpy(x_a, m.x_a.data(), sizeof(double) * m.x_a.size());
        if (y_a) std::memcpy(y_a, m.y_a.data(), sizeof(double) * m.y_a.size());
        if (x_b) std::memcpy(x_b, m.x_b.data(), sizeof(double) * m.x_b.size());
        if (y_b) std::memcpy(y_b, m.y_b.data(), sizeof(double) * m.y_b.size());
    });
}
const char* ob_builder_describe(ob_builder* b) {
    if (!b) return "";
    if (guarded(b, [&] { b->desc = b->b->describe(); }) != OB_OK) return "";
    return b->desc.c_str();
}
ob_status ob_builder_last_status(const ob_builder* b) { return b ? b->last : OB_ERR_INVALID_ARG; }
const char* ob_builder_last_error(const ob_builder* b) { return b ? b->err.c_str() : "null builder"; }

void ob_results_free(ob_results* r) { delete r; }
const char* ob_results_json(ob_results* r, int32_t with_residuals, int32_t with_extra) {
    if (!r) return "";
    r->json = r->r.to_json(with_residuals != 0, with_extra != 0);
    return r->json.c_str();
}
const char* ob_results_summary(ob_results* r) {
    if (!r) return "";
    std::ostringstream os; r->r.summary(os); r->summary = os.str();
    return r->summary.c_str();
}
const char* ob_results_markdown(ob_results* r) {
    if (!r) return "";
    r->markdown = r->r.to_markdown();
    return r->markdown.c_str();
}
int64_t ob_results_residuals(const ob_results* r, double* out) {
    if (!r) return 0;
    if (out) std::memcpy(out, r->r.residuals.data(), sizeof(double) * r->r.residuals.size());
    return (int64_t)r->r.residuals.size();
}


/* ---- Machado-Mata: QuantileDecompositionBuilder (quantile_decomposition.rs:21-522) ---- */
ob_qd_builder* ob_qd_builder_new(const ob_frame* f, const char* outcome, const char* group, const char* reference_group) {
    if (!f || !outcome || !group || !reference_group) return nullptr;
    auto b = new ob_qd_builder;
    b->b = std::make_unique<ob::QuantileDecompositionBuilder>(f->df, outcome, group, reference_group);
    return b;
}
void ob_qd_builder_free(ob_qd_builder* b) { delete b; }
ob_status ob_qd_builder_predictors(ob_qd_builder* b, const char* const* names, int32_t n) {
    return guarded(b, [&] { b->b->predictors(strs(names, n)); });
}
ob_status ob_qd_builder_categorical_predictors(ob_qd_builder* b, const char* const* names, int32_t n) {
    return guarded(b, [&] { b->b->categorical_predictors(strs(names, n)); });
}
ob_status ob_qd_builder_quantiles(ob_qd_builder* b, const double* q, int32_t n) {
    if (n < 0 || (n && !q)) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->quantiles(std::vector<double>(q, q + n)); });
}
ob_status ob_qd_builder_simulations(ob_qd_builder* b, int64_t reps) {
    if (reps < 0) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->simulations((size_t)reps); });
}
ob_status ob_qd_builder_bootstrap_reps(ob_qd_builder* b, int64_t reps) {
    if (reps < 0) return OB_ERR_INVALID_ARG;
    return guarded(b, [&] { b->b->bootstrap_reps((size_t)reps); });
}
ob_status ob_qd_builder_seed(ob_qd_builder* b, uint64_t seed) { return guarded(b, [&] { b->b->seed(seed); }); }
ob_status ob_qd_builder_device(ob_qd_builder* b, int32_t device) { return guarded(b, [&] { b->b->device(device); }); }
ob_status ob_qd_builder_streams(ob_qd_builder* b, const uint32_t* idx_a, const uint32_t* idx_b, const double* taus,
                                const uint32_t* draw_a, const uint32_t* draw_b) {
    return guarded(b, [&] { b->b->streams(idx_a, idx_b, taus, draw_a, draw_b); });
}
ob_status ob_qd_builder_run(ob_qd_builder* b, ob_qd_results** out) {
    if (!out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(b, [&] { auto r = std::make_unique<ob_qd_results>(); r->r = b->b->run(); *out = r.release(); });
}
int32_t ob_qd_quantile_key(double tau, char* out, size_t out_len) {
    const std::string k = ob::QuantileDecompositionBuilder::quantile_key(tau);
    put_err(out, out_len, k);
    return (int32_t)k.size();
}
const char* ob_qd_builder_last_error(const ob_qd_builder* b) { return b ? b->err.c_str() : "null builder"; }
ob_status ob_qd_builder_last_status(const ob_qd_builder* b) { return b ? b->last : OB_ERR_INVALID_ARG; }
void ob_qd_results_free(ob_qd_results* r) { delete r; }
const char* ob_qd_results_json(ob_qd_results* r) {
    if (!r) return "";
    r->json = r->r.to_json();
    return r->json.c_str();
}
const char* ob_qd_results_summary(ob_qd_results* r) {
    if (!r) return "";
    std::ostringstream os; r->r.summary(os); r->summary = os.str();
    return r->summary.c_str();
}

}  // extern "C"
