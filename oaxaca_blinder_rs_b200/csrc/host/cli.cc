// csrc/host/cli.cc -- `oaxaca-cli` front-end, same flags as the reference's clap RunArgs (main.rs:44-128) and the same
// dispatch as run_mean_analysis (main.rs:175-232) and run_quantile_analysis (Machado-Mata, main.rs:234-258).  The other
// analysis types (AKM, matching) are outside the B200 bootstrap path and are refused.
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <sstream>

#include "builder.h"

static std::vector<std::string> split_commas(const std::string& s) {
    std::vector<std::string> out; std::stringstream ss(s); std::string t;
    while (std::getline(ss, t, ',')) if (!t.empty()) out.push_back(t);
    return out;
}

// clap's typed arguments reject what does not parse (exit code 2, "error: invalid value ... for '--flag <X>'")
struct ArgError { std::string msg; };
static unsigned long long parse_u64(const std::string& flag, const std::string& v) {
    char* end = nullptr;
    errno = 0;
    const unsigned long long x = std::strtoull(v.c_str(), &end, 10);
    if (v.empty() || v[0] == '-' || *end != '\0' || errno == ERANGE)
        throw ArgError{"invalid value '" + v + "' for '--" + flag + "': not a non-negative integer"};
    return x;
}
static double parse_f64(const std::string& flag, const std::string& v) {
    char* end = nullptr;
    const double x = std::strtod(v.c_str(), &end);
    if (v.empty() || *end != '\0' || x != x) throw ArgError{"invalid value '" + v + "' for '--" + flag + "': not a number"};
    return x;
}

static void usage() {
    std::cerr <<
        "Usage: oaxaca-cli --data <DATA> --outcome <OUTCOME> --group <GROUP> --reference <REFERENCE> [OPTIONS]\n\n"
        "Options:\n"
        "  -d, --data <DATA>                  Path to the input CSV data file\n"
        "      --outcome <OUTCOME>            Outcome variable column\n"
        "      --group <GROUP>                Column that divides the data into two groups\n"
        "      --reference <REFERENCE>        Value of the group column identifying the reference group\n"
        "      --predictors <A,B,..>          Numerical predictor columns\n"
        "      --categorical <A,B,..>         Categorical predictor columns\n"
        "      --analysis-type <TYPE>         mean (default) | quantile (Machado-Mata) | akm | match  [mean and quantile run on the B200 path]\n"
        "      --quantiles <A,B,..>           Quantiles to analyse (quantile analysis) [default: 0.1,0.25,0.5,0.75,0.9]\n"
        "      --simulations <N>              Simulations of the Machado-Mata algorithm [default: 200]\n"
        "      --ref-coeffs <KIND>            group-a | group-b (default) | pooled | weighted\n"
        "      --bootstrap-reps <N>           Bootstrap replications [default: 50]\n"
        "      --formula <FORMULA>            R-style formula, e.g. \"wage ~ education + C(sector)\"\n"
        "      --weights <COLUMN>             Sample-weight column (WLS)\n"
        "      --normalize <A,B,..>           Categorical variables to Yun-normalise (builder.normalize)\n"
        "      --rif-quantile <TAU>           RIF-regression decomposition at quantile TAU (decompose_quantile)\n"
        "      --seed <N>                     Resampling seed\n"
        "      --cluster <COLUMN>             Cluster bootstrap: resample whole clusters of COLUMN instead of rows\n"
        "      --cluster-strata <MODE>        group (default: each group resamples its own clusters) | joint (one stratum)\n"
        "      --bootstrap-scheme <SCHEME>    multinomial (default: resample rows) | bayes (Bayesian bootstrap: Dirichlet row weights)\n"
        "      --output-json <PATH>           Export results as JSON\n"
        "      --output-markdown <PATH>       Export results as Markdown\n";
}

int main(int argc, char** argv) {
    std::map<std::string, std::string> a;
    a["analysis-type"] = "mean"; a["ref-coeffs"] = "group-b"; a["bootstrap-reps"] = "50";   // main.rs:70-83
    for (int i = 1; i < argc; ++i) {
        std::string k = argv[i];
        if (k == "-h" || k == "--help") { usage(); return 0; }
        if (k == "-d") k = "--data";
        if (k.rfind("--", 0) != 0 || i + 1 >= argc) { std::cerr << "Error: unexpected argument '" << k << "'\n\n"; usage(); return 2; }
        a[k.substr(2)] = argv[++i];
    }
    // typed flags, validated before any work (clap ValueEnum / typed args, main.rs:44-128): a typo must not silently
    // change which reference coefficients or how many replicates are used
    ob::ReferenceCoefficients ref_kind = ob::ReferenceCoefficients::GroupB;
    unsigned long long reps = 0, seed = 0, sims = 200;                                    // main.rs:86-87
    double tau = 0.0;
    std::vector<double> quantiles = {0.1, 0.25, 0.5, 0.75, 0.9};                          // main.rs:236-239
    int cluster_strata = OB_CLUSTER_BY_GROUP;
    bool bayesian = false;
    try {
        if (a.count("bootstrap-scheme")) {
            const std::string& bs = a["bootstrap-scheme"];
            if (bs == "bayes") bayesian = true;
            else if (bs != "multinomial")
                throw ArgError{"invalid value '" + bs + "' for '--bootstrap-scheme <SCHEME>'\n  [possible values: multinomial, bayes]"};
            if (bayesian && a["analysis-type"] == "quantile")
                throw ArgError{"'--bootstrap-scheme bayes' applies to the mean and RIF decompositions, not to '--analysis-type quantile'"};
        }
        if (a.count("cluster-strata")) {
            const std::string& cs = a["cluster-strata"];
            if (cs == "group") cluster_strata = OB_CLUSTER_BY_GROUP;
            else if (cs == "joint") cluster_strata = OB_CLUSTER_JOINT;
            else throw ArgError{"invalid value '" + cs + "' for '--cluster-strata <MODE>'\n  [possible values: group, joint]"};
            if (!a.count("cluster")) throw ArgError{"'--cluster-strata <MODE>' requires '--cluster <COLUMN>'"};
        }
        if (a.count("cluster") && a["analysis-type"] == "quantile")
            throw ArgError{"'--cluster <COLUMN>' applies to the mean and RIF decompositions, not to '--analysis-type quantile'"};
        const std::string& rc = a["ref-coeffs"];
        if (rc == "group-a") ref_kind = ob::ReferenceCoefficients::GroupA;
        else if (rc == "group-b") ref_kind = ob::ReferenceCoefficients::GroupB;
        else if (rc == "pooled") ref_kind = ob::ReferenceCoefficients::Pooled;
        else if (rc == "weighted") ref_kind = ob::ReferenceCoefficients::Weighted;
        else throw ArgError{"invalid value '" + rc + "' for '--ref-coeffs <KIND>'\n  [possible values: group-a, group-b, pooled, weighted]"};
        reps = parse_u64("bootstrap-reps", a["bootstrap-reps"]);
        if (a.count("seed")) seed = parse_u64("seed", a["seed"]);
        if (a.count("simulations")) sims = parse_u64("simulations", a["simulations"]);
        if (a.count("quantiles")) {
            quantiles.clear();
            for (const auto& q : split_commas(a["quantiles"])) quantiles.push_back(parse_f64("quantiles", q));
        }
        if (a.count("rif-quantile")) {
            tau = parse_f64("rif-quantile", a["rif-quantile"]);
            if (!(tau > 0.0 && tau < 1.0)) throw ArgError{"invalid value '" + a["rif-quantile"] + "' for '--rif-quantile <TAU>': must lie in (0, 1)"};
        }
    } catch (const ArgError& e) {
        std::cerr << "error: " << e.msg << "\n\nFor more information, try '--help'.\n";
        return 2;
    }
    try {
        for (const char* req : {"data", "outcome", "group", "reference"})
            if (!a.count(req) && !(std::string(req) == "outcome" && a.count("formula")))
                throw ob::OaxacaError(OB_ERR_INVALID_ARG, std::string("the following required argument was not provided: --") + req);
        if (a["analysis-type"] != "mean" && a["analysis-type"] != "quantile")
            throw ob::OaxacaError(OB_ERR_UNSUPPORTED, "analysis type '" + a["analysis-type"] +
                                  "' is outside the B200 bootstrap path (mean decomposition, RIF quantiles and Machado-Mata only)");
        ob::DataFrame df = ob::DataFrame::read_csv(a["data"]);
        if (a["analysis-type"] == "quantile") {                                           // run_quantile_analysis, main.rs:234-258
            ob::QuantileDecompositionBuilder qb(df, a["outcome"], a["group"], a["reference"]);
            qb.predictors(split_commas(a["predictors"])).categorical_predictors(split_commas(a["categorical"]))
              .quantiles(quantiles).bootstrap_reps((size_t)reps).simulations((size_t)sims);
            if (a.count("seed")) qb.seed(seed);
            const ob::QuantileDecompositionResults qr = qb.run();
            qr.summary(std::cout);
            if (a.count("output-json")) { std::ofstream(a["output-json"]) << qr.to_json(); }
            return 0;
        }
        ob::OaxacaBuilder b = a.count("formula")
            ? ob::OaxacaBuilder::from_formula(df, a["formula"], a["group"], a["reference"])
            : ob::OaxacaBuilder(df, a["outcome"], a["group"], a["reference"]);
        if (!a.count("formula")) {
            b.predictors(split_commas(a["predictors"]));
            b.categorical_predictors(split_commas(a["categorical"]));
        }
        b.reference_coefficients(ref_kind);
        b.bootstrap_reps((size_t)reps);
        if (a.count("weights")) b.weights(a["weights"]);
        if (a.count("normalize")) b.normalize(split_commas(a["normalize"]));
        if (a.count("seed")) b.seed(seed);
        if (a.count("cluster")) b.cluster(a["cluster"], cluster_strata);
        if (bayesian) b.bayesian_bootstrap(true);
        if (a.count("selection-outcome")) b.heckman_selection(a["selection-outcome"], split_commas(a["selection-predictors"]));
        const ob::OaxacaResults r = a.count("rif-quantile") ? b.decompose_quantile(tau) : b.run();
        r.summary(std::cout);
        if (a.count("output-json")) { std::ofstream(a["output-json"]) << r.to_json(true, false); }
        if (a.count("output-markdown")) { std::ofstream(a["output-markdown"]) << r.to_markdown(); }
        return 0;
    } catch (const std::exception& e) {
        std::cerr << "Error: " << e.what() << "\n\n";   // main.rs:379-384: error + help, exit 1
        usage();
        return 1;
    }
}
