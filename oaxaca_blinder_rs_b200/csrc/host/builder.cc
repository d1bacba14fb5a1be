// csrc/host/builder.cc -- see builder.h.  Citations: file:line under oaxaca_blinder/src/ of the reference.
#include "builder.h"

#include <unordered_map>
#include <cstring>
#include <charconv>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <set>
#include <sstream>

namespace ob {

// ------------------------------------------------------------------ frame
void DataFrame::add_f64(const std::string& name, std::vector<double> data, std::vector<uint8_t> valid) {
    if (!cols_.empty() && data.size() != height_) throw OaxacaError(OB_ERR_POLARS, "column length mismatch: " + name);
    height_ = data.size();
    Column c; c.name = name; c.is_str = false; c.f64 = std::move(data); c.valid = std::move(valid);
    cols_.push_back(std::move(c));
}
void DataFrame::add_str(const std::string& name, std::vector<std::string> data, std::vector<uint8_t> valid) {
    if (!cols_.empty() && data.size() != height_) throw OaxacaError(OB_ERR_POLARS, "column length mismatch: " + name);
    height_ = data.size();
    Column c; c.name = name; c.is_str = true; c.str = std::move(data); c.valid = std::move(valid);
    cols_.push_back(std::move(c));
}
const Column* DataFrame::find(const std::string& name) const {
    for (const auto& c : cols_) if (c.name == name) return &c;
    return nullptr;
}

static std::vector<std::string> split_csv_line(const std::string& line) {
    std::vector<std::string> out; std::string cur; bool q = false;
    for (size_t i = 0; i < line.size(); ++i) {
        const char ch = line[i];
        if (q) { if (ch == '"') { if (i + 1 < line.size() && line[i + 1] == '"') { cur += '"'; ++i; } else q = false; } else cur += ch; }
        else if (ch == '"') q = true;
        else if (ch == ',') { out.push_back(cur); cur.clear(); }
        else if (ch != '\r') cur += ch;
    }
    out.push_back(cur);
    return out;
}

// One cell of a CSV line starting at p (end = end of line, exclusive).  Unquoted cells are returned as a view into the
// buffer; quoted ones are unescaped into `tmp`.  Same grammar as split_csv_line: "" inside quotes is a quote, '\r' is dropped.
static inline const char* next_cell(const char* p, const char* end, std::string& tmp, const char*& cb, const char*& ce) {
    if (p < end && *p != '"') {                       // fast path: no quotes before the next comma
        const char* q = p;
        bool plain = true;
        while (q < end && *q != ',') { if (*q == '"' || *q == '\r') plain = false; ++q; }
        if (plain) { cb = p; ce = q; return q < end ? q + 1 : nullptr; }
    }
    tmp.clear();
    bool quoted = false;
    const char* q = p;
    for (; q < end; ++q) {
        const char ch = *q;
        if (quoted) { if (ch == '"') { if (q + 1 < end && q[1] == '"') { tmp += '"'; ++q; } else quoted = false; } else tmp += ch; }
        else if (ch == '"') quoted = true;
        else if (ch == ',') break;
        else if (ch != '\r') tmp += ch;
    }
    cb = tmp.data(); ce = tmp.data() + tmp.size();
    return q < end ? q + 1 : nullptr;
}

// full-cell numeric parse with strtod's acceptance (from_chars first: no allocation, no locale)
static inline bool parse_number(const char* b, const char* e, double& out) {
    auto r = std::from_chars(b, e, out);
    if (r.ec == std::errc() && r.ptr == e) return true;
    std::string z(b, e);                              // rare: leading '+' / blanks, "inf", hex floats ...
    char* endp = nullptr;
    out = std::strtod(z.c_str(), &endp);
    return endp != z.c_str() && *endp == '\0';
}

DataFrame DataFrame::read_csv(const std::string& path) {   // main.rs:161-165 (LazyCsvReader, has_header)
    // Single pass over the file held in memory; numeric columns are parsed straight into doubles (no per-cell
    // std::string), a column is f64 if every non-empty cell parses as a number (empty cell = null).
    std::string buf;
    {
        std::ifstream in(path, std::ios::binary);
        if (!in) throw OaxacaError(OB_ERR_POLARS, "No such file or directory: " + path);
        in.seekg(0, std::ios::end);
        const std::streamoff sz = in.tellg();
        in.seekg(0, std::ios::beg);
        buf.resize((size_t)std::max<std::streamoff>(sz, 0));
        if (sz > 0) in.read(&buf[0], sz);
    }
    const char* p = buf.data();
    const char* const fend = p + buf.size();
    auto line_end = [&](const char* q) { const void* nl = memchr(q, '\n', (size_t)(fend - q)); return nl ? (const char*)nl : fend; };
    if (p == fend) throw OaxacaError(OB_ERR_POLARS, "empty CSV: " + path);
    const char* le = line_end(p);
    const std::vector<std::string> header = split_csv_line(std::string(p, le));
    const char* const data_begin = le < fend ? le + 1 : fend;
    const size_t C = header.size();

    enum Kind { UNKNOWN, NUM, STR };
    struct ColState { Kind kind = UNKNOWN; std::vector<double> num; std::vector<std::string> str; std::vector<uint8_t> valid; bool has_null = false; };
    std::vector<ColState> cols(C);
    size_t rows = 0;
    std::string tmp;

    // a numeric column met a non-numeric cell at row `upto`: fetch its earlier cells as text again (rare)
    auto refill_as_strings = [&](size_t c, size_t upto) {
        ColState& cs = cols[c];
        cs.str.assign(upto, std::string());
        const char* q = data_begin; size_t r = 0; std::string t2;
        while (q < fend && r < upto) {
            const char* e = line_end(q);
            const bool blank = (e == q) || (e - q == 1 && *q == '\r');
            if (!blank) {
                const char* cur = q; size_t ci = 0;
                while (cur && ci <= c) {
                    const char *cb, *ce;
                    cur = next_cell(cur, e, t2, cb, ce);
                    if (ci == c) cs.str[r].assign(cb, ce);
                    ++ci;
                }
                ++r;
            }
            q = e < fend ? e + 1 : fend;
        }
        cs.num.clear(); cs.num.shrink_to_fit();
        cs.kind = STR;
    };

    for (const char* q = data_begin; q < fend;) {
        const char* e = line_end(q);
        const bool blank = (e == q) || (e - q == 1 && *q == '\r');
        if (!blank) {
            const char* cur = q;
            for (size_t c = 0; c < C; ++c) {
                const char* cb = nullptr; const char* ce = nullptr;
                if (cur) cur = next_cell(cur, e, tmp, cb, ce);            // short rows: missing cells are empty
                ColState& cs = cols[c];
                const bool empty = cb == ce;
                cs.valid.push_back(empty ? 0 : 1);
                cs.has_null |= empty;
                if (cs.kind == STR) { cs.str.emplace_back(cb ? std::string(cb, ce) : std::string()); continue; }
                double v = 0.0;
                if (empty) { if (cs.kind == NUM) cs.num.push_back(0.0); continue; }
                if (parse_number(cb, ce, v)) {
                    if (cs.kind == UNKNOWN) { cs.num.assign(rows, 0.0); cs.kind = NUM; }
                    cs.num.push_back(v);
                } else {
                    const std::string keep(cb, ce);                      // cb may point into tmp, which refill reuses? (it uses t2)
                    if (cs.kind == NUM) refill_as_strings(c, rows);
                    else { cs.str.assign(rows, std::string()); cs.kind = STR; }
                    cs.str.push_back(keep);
                }
            }
            ++rows;
        }
        q = e < fend ? e + 1 : fend;
    }
    DataFrame df;
    for (size_t c = 0; c < C; ++c) {
        ColState& cs = cols[c];
        if (!cs.has_null) cs.valid.clear();
        if (cs.kind == NUM) df.add_f64(header[c], std::move(cs.num), std::move(cs.valid));
        else {
            if (cs.kind == UNKNOWN) cs.str.assign(rows, std::string());   // all cells empty: a string column of nulls
            df.add_str(header[c], std::move(cs.str), std::move(cs.valid));
        }
    }
    return df;
}

// ------------------------------------------------------------------ errors, formula
std::string OaxacaError::display(ob_status k, const std::string& d) {   // error.rs:27-38
    switch (k) {
    case OB_ERR_POLARS: return "Polars error: " + d;
    case OB_ERR_COLUMN_NOT_FOUND: return "Column not found: " + d;
    case OB_ERR_INVALID_GROUP: return "Invalid group variable: " + d;
    case OB_ERR_NALGEBRA: return "Nalgebra error: " + d;
    case OB_ERR_DIAGNOSTIC: return "Diagnostic error: " + d;
    case OB_ERR_INSUFFICIENT_DATA: return "Insufficient data: " + d;
    default: return d;
    }
}

static std::string trim(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) ++a;
    while (b > a && std::isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

Formula Formula::parse(const std::string& s) {   // formula.rs:12-60
    std::vector<std::string> parts;
    { std::stringstream ss(s); std::string p; while (std::getline(ss, p, '~')) parts.push_back(p); if (!s.empty() && s.back() == '~') parts.push_back(""); }
    if (parts.size() != 2)
        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP,
                          "Invalid formula format. Expected 'outcome ~ predictors', got '" + s + "'"));
    Formula f;
    f.outcome = trim(parts[0]);
    if (f.outcome.empty())
        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Outcome variable is missing"));
    std::stringstream ss(parts[1]);
    std::string term;
    while (std::getline(ss, term, '+')) {
        term = trim(term);
        if (term.empty()) continue;
        if (term.rfind("C(", 0) == 0 && term.back() == ')') f.categorical_predictors.push_back(trim(term.substr(2, term.size() - 3)));
        else if (term.rfind("factor(", 0) == 0 && term.back() == ')') f.categorical_predictors.push_back(trim(term.substr(7, term.size() - 8)));
        else f.predictors.push_back(term);
    }
    if (f.predictors.empty() && f.categorical_predictors.empty())
        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "No predictors specified"));
    return f;
}

// ------------------------------------------------------------------ builder
OaxacaBuilder::OaxacaBuilder(DataFrame df, const std::string& outcome, const std::string& group,
                             const std::string& reference_group)
    : dataframe_(std::move(df)), outcome_(outcome), group_(group), reference_group_(reference_group) {}

OaxacaBuilder OaxacaBuilder::from_formula(DataFrame df, const std::string& formula, const std::string& group,
                                          const std::string& reference_group) {   // builder.rs:139-160
    const Formula f = Formula::parse(formula);
    OaxacaBuilder b(std::move(df), f.outcome, group, reference_group);
    b.predictors_ = f.predictors;
    b.categorical_ = f.categorical_predictors;
    return b;
}

// the cleaned, coded frame at builder.rs:808
struct OaxacaBuilder::Prepared {
    size_t n = 0;                                   // rows after drop_nulls
    std::vector<std::vector<double>> cont;          // predictors, compacted
    std::vector<std::vector<int32_t>> cat_codes;
    std::vector<int32_t> cat_levels;
    std::vector<double> y, w;
    std::vector<uint8_t> group;
    std::vector<std::string> names;                 // design column names (builder.rs:325-327)
    std::map<std::string, size_t> category_counts;  // builder.rs:799
    std::map<std::string, std::string> base_categories;   // builder.rs:800
    // .normalize spec (normalization.rs:14-38, builder.rs:636-647)
    std::vector<int32_t> norm_m, norm_off, norm_idx, norm_has_base;
    std::vector<std::string> base_names;
};

static void require_f64(const Column* c) {
    if (c->is_str) throw OaxacaError(OB_ERR_POLARS, OaxacaError::display(OB_ERR_POLARS,
                       "invalid series dtype: expected `Float64`, got `str` for series with name `" + c->name + "`"));
}
static void require_str(const Column* c) {
    if (!c->is_str) throw OaxacaError(OB_ERR_POLARS, OaxacaError::display(OB_ERR_POLARS,
                        "invalid series dtype: expected `String`, got `f64` for series with name `" + c->name + "`"));
}

// .normalize(): membership by name prefix "{var}_" over ALL predictor names (normalization.rs:14-20)
void OaxacaBuilder::fill_norm_spec(Prepared& p) const {
    p.norm_off.push_back(0);
    for (const auto& var : normalization_vars_) {
        const std::string prefix = var + "_";
        int cnt = 0;
        for (size_t i = 0; i < p.names.size(); ++i)
            if (p.names[i].rfind(prefix, 0) == 0) { p.norm_idx.push_back((int32_t)i); ++cnt; }
        p.norm_off.push_back((int32_t)p.norm_idx.size());
        auto cc = p.category_counts.find(var);
        p.norm_m.push_back(cc != p.category_counts.end() ? (int32_t)cc->second : cnt + 1);   // normalization.rs:31-34
        auto bc = p.base_categories.find(var);
        p.norm_has_base.push_back(bc != p.base_categories.end() ? 1 : 0);                     // builder.rs:636-640
        if (bc != p.base_categories.end()) p.base_names.push_back(bc->second);
    }
}

OaxacaBuilder::Prepared OaxacaBuilder::prepare() const {
    Prepared p;
    // clean_dataframe (builder.rs:760-784): existence check in this order, then drop rows with a null in any used column
    std::vector<std::string> cols = {outcome_, group_};
    cols.insert(cols.end(), predictors_.begin(), predictors_.end());
    cols.insert(cols.end(), categorical_.begin(), categorical_.end());
    if (has_weights_) cols.push_back(weights_col_);
    if (has_selection_) cols.push_back(selection_outcome_);
    cols.insert(cols.end(), selection_predictors_.begin(), selection_predictors_.end());
    if (cluster_strata_ != OB_CLUSTER_NONE) cols.push_back(cluster_col_);
    std::vector<const Column*> used;
    for (const auto& c : cols) {
        const Column* col = dataframe_.find(c);
        if (!col) throw OaxacaError(OB_ERR_COLUMN_NOT_FOUND, OaxacaError::display(OB_ERR_COLUMN_NOT_FOUND, c));
        used.push_back(col);
    }
    const size_t N = dataframe_.height();
    std::vector<size_t> keep;
    keep.reserve(N);
    for (size_t i = 0; i < N; ++i) {
        bool ok = true;
        for (const Column* c : used) if (!c->is_valid(i)) { ok = false; break; }
        if (ok) keep.push_back(i);
    }
    p.n = keep.size();

    // create_dummies_manual (builder.rs:380-418) on the FULL cleaned frame, before the split (:794-806)
    p.names.push_back("__ob_intercept__");
    for (const auto& pr : predictors_) p.names.push_back(pr);
    for (const auto& cat : categorical_) {
        const Column* c = dataframe_.find(cat);
        require_str(c);
        std::set<std::string> uniq;
        for (size_t i : keep) uniq.insert(c->str[i]);
        if (uniq.empty())
            throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Could not get reference category for " + cat));
        const std::vector<std::string> levels(uniq.begin(), uniq.end());   // sorted ascending (:384-388)
        std::map<std::string, int32_t> code;
        for (size_t l = 0; l < levels.size(); ++l) code[levels[l]] = (int32_t)l;
        std::vector<int32_t> codes(p.n);
        for (size_t r = 0; r < p.n; ++r) codes[r] = code[c->str[keep[r]]];
        p.cat_codes.push_back(std::move(codes));
        p.cat_levels.push_back((int32_t)levels.size());
        p.category_counts[cat] = levels.size();
        p.base_categories[cat] = cat + "_" + levels[0];                    // :400
        for (size_t l = 1; l < levels.size(); ++l) p.names.push_back(cat + "_" + levels[l]);   // :402-404
    }

    // numeric columns
    const Column* yc = dataframe_.find(outcome_);
    require_f64(yc);
    p.y.resize(p.n);
    for (size_t r = 0; r < p.n; ++r) p.y[r] = yc->f64[keep[r]];
    for (const auto& pr : predictors_) {
        const Column* c = dataframe_.find(pr);
        require_f64(c);
        std::vector<double> v(p.n);
        for (size_t r = 0; r < p.n; ++r) v[r] = c->f64[keep[r]];
        p.cont.push_back(std::move(v));
    }
    if (has_weights_) {
        const Column* c = dataframe_.find(weights_col_);
        require_f64(c);
        p.w.resize(p.n);
        for (size_t r = 0; r < p.n; ++r) p.w[r] = c->f64[keep[r]];
    }

    // split_groups (builder.rs:61-102)
    const Column* gc = dataframe_.find(group_);
    require_str(gc);
    std::set<std::string> ug;
    for (size_t i : keep) ug.insert(gc->str[i]);
    if (ug.size() < 2)
        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Not enough groups for comparison"));
    auto it = ug.begin();
    std::string a_name = *it;
    if (a_name == reference_group_) a_name = *(++it);                      // :79-83
    p.group.resize(p.n);
    for (size_t r = 0; r < p.n; ++r) {
        const std::string& g = gc->str[keep[r]];
        p.group[r] = g == a_name ? 0 : (g == reference_group_ ? 1 : 2);   // rows of any third group are ignored (:85-94)
    }

    fill_norm_spec(p);
    return p;
}

namespace {
struct CtxGuard {
    ob_ctx* ctx = nullptr; ob_design* des = nullptr;
    ~CtxGuard() { if (des) ob_design_destroy(des); if (ctx) ob_ctx_destroy(ctx); }
};
void check(ob_ctx* ctx, ob_status st) {
    if (st == OB_OK) return;
    std::string msg = ctx ? ob_last_error(ctx) : "";
    if (msg.empty()) msg = "libobboot error " + std::to_string((int)st);
    throw OaxacaError(st, msg);
}
}  // namespace


// The production path of run() / decompose_quantile() / get_data_matrices(): the same cleaning and coding as
// prepare(), but with the O(n) work on the device (ob_ingest_begin / ob_ingest_finish).  The host only
// dictionary-encodes the string columns (what a polars Categorical / Arrow dictionary column already is) and sorts
// the handful of values that occur.  Fills the metadata of `p` (names, levels, normalize spec, n); returns the design.
ob_design* OaxacaBuilder::ingest_on_device(ob_ctx* ctx, Prepared& p, bool with_weights, const std::vector<std::string>* sweep) const {
    const std::string& outcome = sweep ? sweep->front() : outcome_;
    std::vector<std::string> cols = {outcome, group_};
    if (sweep) cols.insert(cols.end(), sweep->begin() + 1, sweep->end());
    cols.insert(cols.end(), predictors_.begin(), predictors_.end());
    cols.insert(cols.end(), categorical_.begin(), categorical_.end());
    if (has_weights_) cols.push_back(weights_col_);
    if (has_selection_) cols.push_back(selection_outcome_);
    cols.insert(cols.end(), selection_predictors_.begin(), selection_predictors_.end());
    if (cluster_strata_ != OB_CLUSTER_NONE) cols.push_back(cluster_col_);
    for (const auto& c : cols)
        if (!dataframe_.find(c)) throw OaxacaError(OB_ERR_COLUMN_NOT_FOUND, OaxacaError::display(OB_ERR_COLUMN_NOT_FOUND, c));
    const int64_t n = (int64_t)dataframe_.height();

    struct Dict { std::vector<int32_t> codes; std::vector<std::string> values; };
    auto encode = [&](const Column* c) {                       // first-seen order, null -> -1
        Dict d; d.codes.resize((size_t)n);
        std::unordered_map<std::string, int32_t> idx;
        for (int64_t i = 0; i < n; ++i) {
            if (!c->is_valid((size_t)i)) { d.codes[(size_t)i] = -1; continue; }
            auto it = idx.find(c->str[(size_t)i]);
            if (it == idx.end()) { it = idx.emplace(c->str[(size_t)i], (int32_t)d.values.size()).first; d.values.push_back(c->str[(size_t)i]); }
            d.codes[(size_t)i] = it->second;
        }
        return d;
    };
    auto raw_f64 = [&](const Column* c) {
        ob_raw_f64 r{};
        r.data = c->f64.data();
        r.valid = c->valid.empty() ? nullptr : c->valid.data();
        return r;
    };
    std::vector<Dict> cat_dicts;
    for (const auto& cat : categorical_) { const Column* c = dataframe_.find(cat); require_str(c); cat_dicts.push_back(encode(c)); }
    const Column* yc = dataframe_.find(outcome);
    require_f64(yc);
    std::vector<ob_raw_f64> cont;
    for (const auto& pr : predictors_) { const Column* c = dataframe_.find(pr); require_f64(c); cont.push_back(raw_f64(c)); }
    ob_raw_frame fr{};
    fr.n = n;
    fr.outcome = raw_f64(yc);
    // columns that only take part in the null filter (clean_dataframe covers every configured column, builder.rs:760-784):
    // their validity is folded into the outcome's
    std::vector<const Column*> filter_only;
    if (has_weights_) {
        const Column* c = dataframe_.find(weights_col_);
        require_f64(c);
        if (with_weights) fr.weights = raw_f64(c); else filter_only.push_back(c);
    }
    if (has_selection_) filter_only.push_back(dataframe_.find(selection_outcome_));
    for (const auto& sp : selection_predictors_) filter_only.push_back(dataframe_.find(sp));
    if (cluster_strata_ != OB_CLUSTER_NONE) filter_only.push_back(dataframe_.find(cluster_col_));
    if (sweep)           // the other outcomes of the sweep: one cleaned frame for all of them
        for (size_t k = 1; k < sweep->size(); ++k) { const Column* c = dataframe_.find((*sweep)[k]); require_f64(c); filter_only.push_back(c); }
    std::vector<uint8_t> merged_valid;
    for (const Column* c : filter_only) {
        if (c->valid.empty()) continue;
        if (merged_valid.empty()) merged_valid = yc->valid.empty() ? std::vector<uint8_t>((size_t)n, 1) : yc->valid;
        for (int64_t i = 0; i < n; ++i) merged_valid[(size_t)i] &= c->valid[(size_t)i];
    }
    if (!merged_valid.empty()) fr.outcome.valid = merged_valid.data();
    const Column* gc = dataframe_.find(group_);
    require_str(gc);
    Dict gd = encode(gc);
    std::vector<ob_raw_dict> cats;
    for (auto& d : cat_dicts) cats.push_back(ob_raw_dict{d.codes.data(), (int32_t)d.values.size()});
    fr.n_cont = (int32_t)cont.size(); fr.cont = cont.data();
    fr.n_cat = (int32_t)cats.size(); fr.cat = cats.data();
    fr.group = ob_raw_dict{gd.codes.data(), (int32_t)gd.values.size()};

    ob_ingest* ing = nullptr;
    check(ctx, ob_ingest_begin(ctx, &fr, &ing));
    struct IngGuard { ob_ingest* i; ~IngGuard() { ob_ingest_destroy(i); } } guard{ing};
    int64_t kept = 0;
    ob_ingest_rows_kept(ing, &kept);
    p.n = (size_t)kept;

    // create_dummies_manual (builder.rs:380-418) on the cleaned frame: levels sorted ascending, first = base
    p.names.push_back("__ob_intercept__");
    for (const auto& pr : predictors_) p.names.push_back(pr);
    std::vector<std::vector<int32_t>> remaps;
    for (size_t q = 0; q < categorical_.size(); ++q) {
        const std::string& cat = categorical_[q];
        std::vector<uint8_t> present(std::max<size_t>(cat_dicts[q].values.size(), 1), 0);
        ob_ingest_presence(ing, (int32_t)q, present.data());
        std::vector<std::string> levels;
        for (size_t i = 0; i < cat_dicts[q].values.size(); ++i) if (present[i]) levels.push_back(cat_dicts[q].values[i]);
        std::sort(levels.begin(), levels.end());
        if (levels.empty())
            throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Could not get reference category for " + cat));
        std::vector<int32_t> remap(std::max<size_t>(cat_dicts[q].values.size(), 1), -1);
        for (size_t i = 0; i < cat_dicts[q].values.size(); ++i)
            if (present[i]) remap[i] = (int32_t)(std::lower_bound(levels.begin(), levels.end(), cat_dicts[q].values[i]) - levels.begin());
        remaps.push_back(std::move(remap));
        p.cat_levels.push_back((int32_t)levels.size());
        p.category_counts[cat] = levels.size();
        p.base_categories[cat] = cat + "_" + levels[0];
        for (size_t l = 1; l < levels.size(); ++l) p.names.push_back(cat + "_" + levels[l]);
    }
    // split_groups (builder.rs:61-102)
    std::vector<uint8_t> gpresent(std::max<size_t>(gd.values.size(), 1), 0);
    ob_ingest_presence(ing, -1, gpresent.data());
    std::set<std::string> ug;
    for (size_t i = 0; i < gd.values.size(); ++i) if (gpresent[i]) ug.insert(gd.values[i]);
    if (ug.size() < 2)
        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Not enough groups for comparison"));
    auto it = ug.begin();
    std::string a_name = *it;
    if (a_name == reference_group_) a_name = *(++it);
    std::vector<int32_t> gmap(std::max<size_t>(gd.values.size(), 1), 2);
    for (size_t i = 0; i < gd.values.size(); ++i) gmap[i] = gd.values[i] == a_name ? 0 : (gd.values[i] == reference_group_ ? 1 : 2);
    fill_norm_spec(p);

    std::vector<const int32_t*> remap_ptrs(std::max<size_t>(remaps.size(), 1), nullptr);
    for (size_t q = 0; q < remaps.size(); ++q) remap_ptrs[q] = remaps[q].data();
    ob_design* des = nullptr;
    check(ctx, ob_ingest_finish(ctx, ing, gmap.data(), remap_ptrs.data(), p.cat_levels.data(), &des));
    return des;
}

OaxacaResults OaxacaBuilder::run() const { return run_impl(false, 0.0).front(); }

std::vector<OaxacaResults> OaxacaBuilder::run_outcomes(const std::vector<std::string>& outcomes) const {
    if (outcomes.empty()) throw OaxacaError(OB_ERR_INVALID_ARG, "run_outcomes needs at least one outcome column");
    if (has_selection_) throw OaxacaError(OB_ERR_UNSUPPORTED, "run_outcomes with heckman_selection is not supported");
    if (idx_a_ || idx_b_) throw OaxacaError(OB_ERR_UNSUPPORTED, "run_outcomes needs the native resampling stream (no index_stream)");
    return run_impl(false, 0.0, &outcomes);
}

OaxacaResults OaxacaBuilder::decompose_quantile(double quantile) const {
    // builder.rs:711-757: RIF per group on the cleaned frame, then a fresh builder with the same predictors /
    // categoricals / reps / reference / normalize / weights (Heckman settings are NOT forwarded) -> run()
    OaxacaBuilder b = *this;
    b.has_selection_ = false; b.selection_outcome_.clear(); b.selection_predictors_.clear();
    return b.run_impl(true, quantile).front();
}

std::vector<OaxacaResults> OaxacaBuilder::run_impl(bool rif, double tau, const std::vector<std::string>* sweep) const {
    Prepared p;
    CtxGuard g;
    ob_status st = ob_ctx_create(device_, &g.ctx);
    if (st != OB_OK) throw OaxacaError(st, "no usable CUDA device (B200 / sm_100a required; there is no CPU fallback)");
    // HeckmanEstimator (estimation.rs:114-269) ignores the sample weights in both of its steps; the library refuses the
    // combination rather than guess what beta* = Weighted should weigh with
    if (has_selection_ && has_weights_)
        throw OaxacaError(OB_ERR_UNSUPPORTED, "heckman_selection together with weights is not supported on the B200 path");
    g.des = ingest_on_device(g.ctx, p, has_weights_, sweep);
    if (rif) check(g.ctx, ob_design_apply_rif(g.ctx, g.des, tau));
    int K1 = 0;
    if (has_selection_) {
        // heckman_selection (builder.rs:236-246): the selection columns were part of the null filter already; hand them
        // over in frame order (the design's frame-row map picks the kept rows)
        const Column* so = dataframe_.find(selection_outcome_);
        require_f64(so);
        std::vector<const double*> preds;
        for (const auto& sp : selection_predictors_) { const Column* c = dataframe_.find(sp); require_f64(c); preds.push_back(c->f64.data()); }
        ob_selection_view sv{(int32_t)preds.size(), preds.data(), so->f64.data()};
        check(g.ctx, ob_design_attach_selection(g.ctx, g.des, &sv, (int64_t)dataframe_.height()));
        K1 = 1 + (int)preds.size();
    }
    if (cluster_strata_ != OB_CLUSTER_NONE) {
        // cluster codes in the sorted order of the labels, one per frame row (the design's frame-row map picks the kept
        // rows; null rows were dropped by the filter and get any code)
        const Column* c = dataframe_.find(cluster_col_);
        const size_t n = dataframe_.height();
        std::vector<int32_t> codes(n, 0);
        size_t levels = 0;
        if (c->is_str) {
            std::set<std::string> uniq;
            for (size_t i = 0; i < n; ++i) if (c->is_valid(i)) uniq.insert(c->str[i]);
            const std::vector<std::string> sorted(uniq.begin(), uniq.end());
            for (size_t i = 0; i < n; ++i)
                if (c->is_valid(i)) codes[i] = (int32_t)(std::lower_bound(sorted.begin(), sorted.end(), c->str[i]) - sorted.begin());
            levels = sorted.size();
        } else {
            std::vector<double> sorted;
            for (size_t i = 0; i < n; ++i) if (c->is_valid(i) && c->f64[i] == c->f64[i]) sorted.push_back(c->f64[i]);
            std::sort(sorted.begin(), sorted.end());
            sorted.erase(std::unique(sorted.begin(), sorted.end()), sorted.end());
            for (size_t i = 0; i < n; ++i) {
                if (!c->is_valid(i)) continue;
                const double v = c->f64[i];      // a NaN label is a cluster of its own, after every number
                codes[i] = v == v ? (int32_t)(std::lower_bound(sorted.begin(), sorted.end(), v) - sorted.begin()) : (int32_t)sorted.size();
            }
            levels = sorted.size() + 1;
        }
        if (levels >= (size_t)INT32_MAX) throw OaxacaError(OB_ERR_UNSUPPORTED, "more than 2^31 - 1 cluster labels");
        check(g.ctx, ob_design_attach_clusters(g.ctx, g.des, codes.data(), (int64_t)n, (int32_t)std::max<size_t>(levels, 1), cluster_strata_));
    }
    int32_t cl_strata = OB_CLUSTER_NONE; int64_t cl_ua = 0, cl_ub = 0;
    ob_design_clusters(g.des, &cl_strata, &cl_ua, &cl_ub);

    int64_t na = 0, nb = 0; int32_t K = 0, nc = 0;
    ob_design_shape(g.des, &na, &nb, &K, &nc);
    const int n_norm = has_selection_ ? 0 : (int)normalization_vars_.size();        // no Yun rows under Heckman (builder.rs:634)
    const int Kc = has_selection_ ? K + 1 : K;                                      // coefficient vectors: IMR last (estimation.rs:139-151)
    const int S = has_selection_ ? ob_num_stats_heckman(K, K1) : ob_num_stats(K, n_norm, p.norm_has_base.data());
    const int D = has_selection_ ? Kc : (S - 5) / 2;

    struct CacheGuard { ob_gram_cache* c = nullptr; ~CacheGuard() { ob_gram_cache_destroy(c); } } cache;
    if (sweep && sweep->size() > 1) check(g.ctx, ob_gram_cache_create(g.ctx, &cache.c));
    std::vector<OaxacaResults> all;
    for (size_t k = 0; k < (sweep ? sweep->size() : 1); ++k) {
        if (k > 0) {     // the next outcome into the packed rows; X, weights and the group split stay in HBM
            const Column* c = dataframe_.find((*sweep)[k]);
            check(g.ctx, ob_design_update_outcome(g.ctx, g.des, c->f64.data(), (int64_t)dataframe_.height()));
        }
        ob_boot_opts o{};
        switch (reference_coeffs_) {
        case ReferenceCoefficients::GroupA: o.ref_kind = OB_REF_GROUP_A; break;
        case ReferenceCoefficients::GroupB: o.ref_kind = OB_REF_GROUP_B; break;
        case ReferenceCoefficients::Pooled: case ReferenceCoefficients::Neumark: o.ref_kind = OB_REF_POOLED; break;
        default: o.ref_kind = OB_REF_WEIGHTED; break;
        }
        o.n_norm = n_norm; o.norm_m = p.norm_m.data(); o.norm_off = p.norm_off.data();
        o.norm_idx = p.norm_idx.data(); o.norm_has_base = p.norm_has_base.data();
        o.reps = (int64_t)bootstrap_reps_; o.seed = seed_;
        o.idx_a = idx_a_; o.idx_b = idx_b_;

        OaxacaResults R;
        std::vector<double> point(S), se(S), pv(S), lo(S), hi(S), t(S);
        R.xa_mean.resize(Kc); R.xb_mean.resize(Kc); R.beta_star.resize(Kc); R.residuals.resize((size_t)nb);
        ob_result r{};
        r.point_stats = point.data(); r.xa_mean = R.xa_mean.data(); r.xb_mean = R.xb_mean.data(); r.beta_star = R.beta_star.data();
        r.residuals_b = R.residuals.data();
        r.std_err = se.data(); r.p_value = pv.data(); r.ci_lower = lo.data(); r.ci_upper = hi.data(); r.t_stat = t.data();
        if (bayesian_) check(g.ctx, ob_bootstrap_run_bayes(g.ctx, g.des, &o, nullptr, cache.c, &r));
        else check(g.ctx, cache.c ? ob_bootstrap_run_cached(g.ctx, g.des, &o, cache.c, &r) : ob_bootstrap_run(g.ctx, g.des, &o, &r));

        R.bootstrap_reps = (int64_t)bootstrap_reps_;
        R.successful_bootstraps = r.n_ok;
        if (r.n_ok < (int64_t)bootstrap_reps_)   // builder.rs:841-847
            std::cerr << "Warning: " << (bootstrap_reps_ - r.n_ok) << " out of " << bootstrap_reps_
                      << " bootstrap replications failed and were discarded. The analysis is based on " << r.n_ok
                      << " successful replications." << std::endl;
        auto comp = [&](const std::string& name, int j) {
            return ComponentResult{name, point[j], se[j], t[j], pv[j], lo[j], hi[j]};
        };
        R.total_gap = r.total_gap;
        R.two_fold.aggregate = {comp("explained", 0), comp("unexplained", 1)};                            // :867-884
        R.three_fold.aggregate = {comp("endowments", 2), comp("coefficients", 3), comp("interaction", 4)}; // :885-910
        std::vector<std::string> rows = p.names;
        if (has_selection_) rows.push_back("IMR");                                                        // estimation.rs:153-154
        else rows.insert(rows.end(), p.base_names.begin(), p.base_names.end());                           // :661-669
        for (int j = 0; j < D; ++j) {
            R.two_fold.detailed_explained.push_back(comp(rows[j], 5 + j));
            R.two_fold.detailed_unexplained.push_back(comp(rows[j], 5 + D + j));
        }
        if (has_selection_) {                                                                             // builder.rs:507-534, :925-930
            R.two_fold.detailed_selection.push_back(comp("__ob_intercept__", 5 + 2 * D));
            for (size_t j = 0; j < selection_predictors_.size(); ++j)
                R.two_fold.detailed_selection.push_back(comp(selection_predictors_[j], 5 + 2 * D + 1 + (int)j));
        }
        R.n_a = (size_t)na; R.n_b = (size_t)nb;
        R.predictor_names = has_selection_ ? rows : p.names;
        R.ms_total = r.ms_total; R.ms_gram = r.ms_gram;
        R.cluster_strata = cl_strata; R.cluster_units_a = cl_ua; R.cluster_units_b = cl_ub;
        R.bayesian = bayesian_;
        all.push_back(std::move(R));
    }
    return all;
}

DataMatrices OaxacaBuilder::get_data_matrices() const {   // builder.rs:252-291
    Prepared p;
    CtxGuard g;
    ob_status st = ob_ctx_create(device_, &g.ctx);
    if (st != OB_OK) throw OaxacaError(st, "no usable CUDA device (B200 / sm_100a required; there is no CPU fallback)");
    g.des = ingest_on_device(g.ctx, p, false);
    int64_t na = 0, nb = 0; int32_t K = 0, nc = 0;
    ob_design_shape(g.des, &na, &nb, &K, &nc);
    DataMatrices m;
    m.n_a = (size_t)na; m.n_b = (size_t)nb; m.k = (size_t)K; m.predictor_names = p.names;
    m.x_a.resize(m.n_a * m.k); m.y_a.resize(m.n_a); m.x_b.resize(m.n_b * m.k); m.y_b.resize(m.n_b);
    check(g.ctx, ob_design_download(g.ctx, g.des, m.x_a.data(), m.y_a.data(), nullptr, m.x_b.data(), m.y_b.data(), nullptr));
    return m;
}

std::string OaxacaBuilder::describe() const {
    const Prepared p = prepare();
    std::ostringstream os;
    size_t na = 0, nb = 0;
    for (uint8_t g : p.group) { na += g == 0; nb += g == 1; }
    auto ivec = [&](const std::vector<int32_t>& v) { os << '['; for (size_t i = 0; i < v.size(); ++i) { if (i) os << ','; os << v[i]; } os << ']'; };
    auto svec = [&](const std::vector<std::string>& v) {
        os << '[';
        for (size_t i = 0; i < v.size(); ++i) {
            if (i) os << ',';
            os << '"';
            for (char ch : v[i]) { if (ch == '"' || ch == '\\') os << '\\'; os << ch; }   // JSON string escaping
            os << '"';
        }
        os << ']';
    };
    os << "{\"rows\":" << p.n << ",\"n_a\":" << na << ",\"n_b\":" << nb << ",\"names\":"; svec(p.names);
    os << ",\"base_names\":"; svec(p.base_names);
    os << ",\"cat_levels\":"; ivec(p.cat_levels);
    os << ",\"norm_m\":"; ivec(p.norm_m); os << ",\"norm_off\":"; ivec(p.norm_off);
    os << ",\"norm_idx\":"; ivec(p.norm_idx); os << ",\"norm_has_base\":"; ivec(p.norm_has_base);
    os << ",\"group\":["; for (size_t i = 0; i < p.group.size(); ++i) { if (i) os << ','; os << (int)p.group[i]; } os << "]";
    // sums of the kept rows of the outcome and of every continuous predictor (CSV / cleaning checks on the host)
    os.precision(17);
    auto dsum = [](const std::vector<double>& v) { long double t = 0; for (double x : v) t += x; return (double)t; };
    os << ",\"outcome_sum\":" << dsum(p.y) << ",\"cont_sums\":[";
    for (size_t c = 0; c < p.cont.size(); ++c) { if (c) os << ','; os << dsum(p.cont[c]); }
    os << "]}";
    return os.str();
}

// ------------------------------------------------------------------ presentation
static std::string fmt(double v, int prec) {
    char b[64];
    if (std::isnan(v)) return "NaN";
    snprintf(b, sizeof b, "%.*f", prec, v);
    return b;
}

static void table(std::ostream& os, const char* first, const char* second, const std::vector<ComponentResult>& rows) {
    std::vector<std::vector<std::string>> cells;
    cells.push_back({first, second, "Std. Err.", "p-value", "95% CI"});
    for (const auto& c : rows)
        cells.push_back({c.name, fmt(c.estimate, 4), fmt(c.std_err, 4), fmt(c.p_value, 4),
                         "[" + fmt(c.ci_lower, 3) + ", " + fmt(c.ci_upper, 3) + "]"});
    std::vector<size_t> wdt(5, 0);
    for (const auto& r : cells) for (int i = 0; i < 5; ++i) wdt[i] = std::max(wdt[i], r[i].size());
    auto rule = [&] { os << '+'; for (int i = 0; i < 5; ++i) os << std::string(wdt[i] + 2, '-') << '+'; os << '\n'; };
    rule();
    for (size_t r = 0; r < cells.size(); ++r) {
        os << '|';
        for (int i = 0; i < 5; ++i) os << ' ' << cells[r][i] << std::string(wdt[i] - cells[r][i].size() + 1, ' ') << '|';
        os << '\n';
        if (r == 0) rule();
    }
    rule();
}

void OaxacaResults::summary(std::ostream& os) const {   // display.rs:9-79
    os << "Oaxaca-Blinder Decomposition Results\n";
    os << "========================================\n";
    os << "Group A (Advantaged): " << n_a << " observations\n";
    os << "Group B (Reference):  " << n_b << " observations\n";
    if (cluster_strata == OB_CLUSTER_BY_GROUP)
        os << "Cluster bootstrap (by group): " << cluster_units_a << " units in A, " << cluster_units_b << " in B\n";
    else if (cluster_strata == OB_CLUSTER_JOINT)
        os << "Cluster bootstrap (joint): " << cluster_units_a << " units\n";
    if (bayesian) os << "Bootstrap scheme: Bayesian (Dirichlet row weights)\n";
    os << "Total Gap: " << fmt(total_gap, 4) << "\n\n";
    os << "Two-Fold Decomposition\n";
    table(os, "Component", "Estimate", two_fold.aggregate);
    os << "\nDetailed Decomposition (Explained)\n";
    table(os, "Variable", "Contribution", two_fold.detailed_explained);
    os << "\nDetailed Decomposition (Unexplained)\n";
    table(os, "Variable", "Contribution", two_fold.detailed_unexplained);
}

static void jnum(std::ostream& os, double v) {   // serde_json: non-finite -> null
    if (!std::isfinite(v)) { os << "null"; return; }
    char b[40]; snprintf(b, sizeof b, "%.17g", v); os << b;
}
static void jstr(std::ostream& os, const std::string& s) {
    os << '"';
    for (char ch : s) { if (ch == '"' || ch == '\\') os << '\\'; os << ch; }
    os << '"';
}
static void jcomp(std::ostream& os, const ComponentResult& c) {
    os << "{\"name\":"; jstr(os, c.name);
    os << ",\"estimate\":"; jnum(os, c.estimate); os << ",\"std_err\":"; jnum(os, c.std_err);
    os << ",\"t_stat\":"; jnum(os, c.t_stat); os << ",\"p_value\":"; jnum(os, c.p_value);
    os << ",\"ci_lower\":"; jnum(os, c.ci_lower); os << ",\"ci_upper\":"; jnum(os, c.ci_upper); os << '}';
}
static void jcomps(std::ostream& os, const std::vector<ComponentResult>& v) {
    os << '[';
    for (size_t i = 0; i < v.size(); ++i) {
        if (i) os << ',';
        jcomp(os, v[i]);
    }
    os << ']';
}
static void jvec(std::ostream& os, const std::vector<double>& v) {
    os << '[';
    for (size_t i = 0; i < v.size(); ++i) { if (i) os << ','; jnum(os, v[i]); }
    os << ']';
}

std::string OaxacaResults::to_json(bool with_residuals, bool with_extra) const {   // serde layout of types.rs:10-47
    std::ostringstream os;
    os << "{\"total_gap\":"; jnum(os, total_gap);
    os << ",\"two_fold\":{\"aggregate\":"; jcomps(os, two_fold.aggregate);
    os << ",\"detailed_explained\":"; jcomps(os, two_fold.detailed_explained);
    os << ",\"detailed_unexplained\":"; jcomps(os, two_fold.detailed_unexplained);
    os << ",\"detailed_selection\":"; jcomps(os, two_fold.detailed_selection);
    os << "},\"three_fold\":{\"aggregate\":"; jcomps(os, three_fold.aggregate);
    os << ",\"detailed\":"; jcomps(os, three_fold.detailed);
    os << "},\"n_a\":" << n_a << ",\"n_b\":" << n_b;
    if (cluster_strata != OB_CLUSTER_NONE)
        os << ",\"clusters\":{\"strata\":\"" << (cluster_strata == OB_CLUSTER_JOINT ? "joint" : "group") << "\",\"units_a\":"
           << cluster_units_a << ",\"units_b\":" << cluster_units_b << '}';
    if (bayesian) os << ",\"bootstrap_scheme\":\"bayes\"";
    if (with_residuals) { os << ",\"residuals\":"; jvec(os, residuals); }
    if (with_extra) {   // #[serde(skip)] fields + replicate bookkeeping, for the Python mirror and tests
        os << ",\"xa_mean\":"; jvec(os, xa_mean); os << ",\"xb_mean\":"; jvec(os, xb_mean);
        os << ",\"beta_star\":"; jvec(os, beta_star);
        os << ",\"bootstrap_reps\":" << bootstrap_reps << ",\"successful_bootstraps\":" << successful_bootstraps;
        os << ",\"predictor_names\":[";
        for (size_t i = 0; i < predictor_names.size(); ++i) { if (i) os << ','; jstr(os, predictor_names[i]); }
        os << "],\"ms_total\":"; jnum(os, ms_total); os << ",\"ms_gram\":"; jnum(os, ms_gram);
    }
    os << '}';
    return os.str();
}

std::string OaxacaResults::to_markdown() const {
    std::ostringstream os;
    os << "# Oaxaca-Blinder Decomposition Results\n\n";
    os << "- Group A: " << n_a << " observations\n- Group B: " << n_b << " observations\n- Total Gap: " << fmt(total_gap, 4) << "\n\n";
    auto tab = [&](const char* title, const std::vector<ComponentResult>& rows) {
        os << "## " << title << "\n\n| Component | Estimate | Std. Err. | p-value | 95% CI |\n|---|---|---|---|---|\n";
        for (const auto& c : rows)
            os << "| " << c.name << " | " << fmt(c.estimate, 4) << " | " << fmt(c.std_err, 4) << " | " << fmt(c.p_value, 4)
               << " | [" << fmt(c.ci_lower, 3) << ", " << fmt(c.ci_upper, 3) << "] |\n";
        os << "\n";
    };
    tab("Two-Fold Decomposition", two_fold.aggregate);
    tab("Detailed Decomposition (Explained)", two_fold.detailed_explained);
    tab("Detailed Decomposition (Unexplained)", two_fold.detailed_unexplained);
    return os.str();
}

// ---------------------------------------------------------------------------------------------------------------------
// Machado-Mata quantile decomposition: QuantileDecompositionBuilder (quantile_decomposition.rs:21-522)
QuantileDecompositionBuilder::QuantileDecompositionBuilder(DataFrame df, const std::string& outcome, const std::string& group,
                                                           const std::string& reference_group)
    : dataframe_(std::move(df)), outcome_(outcome), group_(group), reference_group_(reference_group) {}

std::string QuantileDecompositionBuilder::quantile_key(double tau) {
    double v = tau * 100.0;                           // `as u32` saturates: negative / NaN -> 0
    uint32_t k = !(v > 0.0) ? 0u : (v >= 4294967295.0 ? 4294967295u : (uint32_t)v);
    return "q" + std::to_string(k);
}

QuantileDecompositionResults QuantileDecompositionBuilder::run() const {
    // The reference's run() does not clean the frame (quantile_decomposition.rs:286-287 only selects the columns): rows of
    // the two groups with a null outcome are an error in prepare_data (:111-118), nulls in predictors fail the
    // to_ndarray conversion (:141).  Rows whose group is null or a third group never reach a design (:195-206).
    {
        std::vector<const Column*> used;
        const Column* gc = dataframe_.find(group_);
        const Column* yc = dataframe_.find(outcome_);
        if (gc && gc->is_str && yc) {
            bool any_nulls = !yc->valid.empty();
            for (const auto& c : predictors_) { const Column* x = dataframe_.find(c); if (x) { used.push_back(x); any_nulls |= !x->valid.empty(); } }
            for (const auto& c : categorical_) { const Column* x = dataframe_.find(c); if (x) { used.push_back(x); any_nulls |= !x->valid.empty(); } }
            if (any_nulls) {
                std::set<std::string> ug;
                for (size_t i = 0; i < dataframe_.height(); ++i) if (gc->is_valid(i)) ug.insert(gc->str[i]);
                std::string a_name = ug.empty() ? reference_group_ : *ug.begin();
                if (a_name == reference_group_ && ug.size() > 1) a_name = *(++ug.begin());
                for (size_t i = 0; i < dataframe_.height(); ++i) {
                    if (!gc->is_valid(i) || (gc->str[i] != a_name && gc->str[i] != reference_group_)) continue;
                    if (!yc->is_valid(i))
                        throw OaxacaError(OB_ERR_INVALID_GROUP, OaxacaError::display(OB_ERR_INVALID_GROUP, "Null outcome encountered"));
                    for (const Column* x : used)
                        if (!x->is_valid(i))
                            throw OaxacaError(OB_ERR_POLARS, OaxacaError::display(OB_ERR_POLARS, "null value in predictor column '" + x->name + "'"));
                }
            }
        }
    }
    if (quantiles_.empty()) throw OaxacaError(OB_ERR_INVALID_ARG, "no target quantiles");
    OaxacaBuilder ingest(dataframe_, outcome_, group_, reference_group_);
    ingest.predictors(predictors_).categorical_predictors(categorical_).device(device_);
    OaxacaBuilder::Prepared p;
    CtxGuard g;
    ob_status st = ob_ctx_create(device_, &g.ctx);
    if (st != OB_OK) throw OaxacaError(st, "no usable CUDA device (B200 / sm_100a required; there is no CPU fallback)");
    g.des = ingest.ingest_on_device(g.ctx, p, false);
    int64_t na = 0, nb = 0; int32_t K = 0, nc = 0;
    ob_design_shape(g.des, &na, &nb, &K, &nc);

    const int nq = (int)quantiles_.size(), S = 3 * nq;
    ob_mm_opts o{};
    o.simulations = (int32_t)simulations_; o.n_quantiles = nq; o.quantiles = quantiles_.data();
    o.reps = (int64_t)bootstrap_reps_; o.seed = seed_;
    o.idx_a = idx_a_; o.idx_b = idx_b_; o.taus = taus_; o.draw_a = draw_a_; o.draw_b = draw_b_;
    std::vector<double> point(S), se(S), pv(S), lo(S), hi(S), t(S);
    ob_mm_result r{};
    r.point_stats = point.data(); r.std_err = se.data(); r.p_value = pv.data(); r.ci_lower = lo.data(); r.ci_upper = hi.data(); r.t_stat = t.data();
    check(g.ctx, ob_mm_run(g.ctx, g.des, &o, &r));

    QuantileDecompositionResults R;
    for (int q = 0; q < nq; ++q) {                     // a later quantile with the same key replaces an earlier one (HashMap insert, :277)
        auto comp = [&](const char* name, int j) { return ComponentResult{name, point[j], se[j], t[j], pv[j], lo[j], hi[j]}; };
        R.results_by_quantile[quantile_key(quantiles_[q])] =
            QuantileDecompositionDetail{comp("Total Gap", 3 * q), comp("Characteristics", 3 * q + 1), comp("Coefficients", 3 * q + 2)};   // :365-407
    }
    R.n_a = (size_t)na; R.n_b = (size_t)nb;
    R.bootstrap_reps = (int64_t)bootstrap_reps_; R.successful_bootstraps = r.n_ok;
    R.qr_total = r.qr_total; R.qr_vertex = r.qr_vertex; R.qr_approx = r.qr_approx; R.qr_failed = r.qr_failed;
    R.ms_total = r.ms_total; R.ms_qr = r.ms_qr;
    return R;
}

void QuantileDecompositionResults::summary(std::ostream& os) const {   // quantile_decomposition.rs:441-505
    os << "Machado-Mata Quantile Decomposition Results\n";
    os << "============================================\n";
    os << "Group A (Advantaged): " << n_a << " observations\n";
    os << "Group B (Reference):  " << n_b << " observations\n";
    for (const auto& kv : results_by_quantile) {       // sorted keys (:449-450)
        os << "\n--- Decomposition for Quantile: " << kv.first << " ---\n";
        os << "| Component       | Estimate | Std. Err. | p-value | 95% CI |\n";
        for (const ComponentResult* c : {&kv.second.total_gap, &kv.second.characteristics_effect, &kv.second.coefficients_effect}) {
            os << "| " << c->name << std::string(c->name.size() < 15 ? 15 - c->name.size() : 0, ' ') << " | " << fmt(c->estimate, 4) << " | "
               << fmt(c->std_err, 4) << " | " << fmt(c->p_value, 4) << " | [" << fmt(c->ci_lower, 3) << ", " << fmt(c->ci_upper, 3) << "] |\n";
        }
    }
}

std::string QuantileDecompositionResults::to_json() const {
    std::ostringstream os;
    os << "{\"results_by_quantile\":{";
    bool first = true;
    for (const auto& kv : results_by_quantile) {
        if (!first) os << ",";
        first = false;
        jstr(os, kv.first);
        os << ":{\"total_gap\":";
        jcomp(os, kv.second.total_gap);
        os << ",\"characteristics_effect\":";
        jcomp(os, kv.second.characteristics_effect);
        os << ",\"coefficients_effect\":";
        jcomp(os, kv.second.coefficients_effect);
        os << "}";
    }
    os << "},\"n_a\":" << n_a << ",\"n_b\":" << n_b << ",\"bootstrap_reps\":" << bootstrap_reps << ",\"successful_bootstraps\":" << successful_bootstraps
       << ",\"qr\":{\"total\":" << qr_total << ",\"vertex\":" << qr_vertex << ",\"approx\":" << qr_approx << ",\"failed\":" << qr_failed << "}"
       << ",\"ms_total\":";
    jnum(os, ms_total);
    os << "}";
    return os.str();
}

}  // namespace ob
