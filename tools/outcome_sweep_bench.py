#!/usr/bin/env python
"""Outcome sweeps over fixed resamples: ob_bootstrap_run_cached against the uncached refresh, on one GPU.

The step a sweep repeats is ob_design_update_outcome + one bootstrap.  Uncached, every step contracts the whole Gram
again; with a GramCache (ob_gram_cache) an OUTCOME_ONLY step contracts the K T + 1 outcome columns, a SOLVE_ONLY step
(another ref_kind on the same outcome) nothing.  Uncached and cached steps alternate, each cached step is checked bit for
bit against its uncached twin (the script exits 1 on any difference), medians over --steps steps after --warmup.

Recorded: per kind of step the wall time (update_outcome + bootstrap, host clock around calls that end in a device
synchronise) and the device stage breakdown (counts, Gram launch, Gram kernel, solve, reduce: CUDA events), the narrow
launch's rate 2 n K T B / t against the measured FP64 DMMA peak (profiles/r01_fp64_peaks.json), the device name, SM
clocks (NVML, sampled during the timed region) and power limit.

  python tools/outcome_sweep_bench.py --out results/sweep [--workload config3_n10M_k50_wls_yun_B2000] [--steps 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KEYS = ("point_stats", "rep_stats", "rep_status", "rep_beta_a", "rep_beta_b", "std_err", "p_value", "ci_lower", "ci_upper",
        "t_stat", "residuals_b", "total_gap_multi", "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")


def identical(a, b):
    return all(np.array_equal(a[k], b[k], equal_nan=True) for k in KEYS) and a["total_gap"] == b["total_gap"]


def dmma_peak_tflops():
    with open(os.path.join(ROOT, "profiles", "r01_fp64_peaks.json")) as f:
        rows = json.load(f)["rows"]
    return max(r["tflops"] for r in rows if r["kind"].startswith("dmma"))


def device_info(index):
    info = {}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        name = pynvml.nvmlDeviceGetName(h)
        info["device"] = name.decode() if isinstance(name, bytes) else name
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:  # noqa: BLE001
        info["nvml_error"] = str(e)
    return info


def main():
    import bench
    import oaxaca_blinder_rs_b200 as ob
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workload", default="config3_n10M_k50_wls_yun_B2000", choices=list(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)

    d, norm_spec, reps, ref = bench.make_data(args.workload)
    norm = [ob.NormVar(m, i) for m, i in norm_spec]
    n = d["outcome"].shape[0]
    rng = np.random.default_rng(11)
    x0 = d["cont"][0]
    outcomes = [d["outcome"] + 0.05 * k * x0 + 0.1 * rng.standard_normal(n) for k in range(args.steps + args.warmup + 1)]
    ctx = ob.Context(args.device)
    des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
    K = des.K
    cache = ob.GramCache(ctx)
    seed0 = 20261020
    clocks = bench.ClockSampler(args.device)
    mismatches = []
    rec = {"outcome_only": [], "uncached": [], "filled": [], "uncached_filled": [], "solve_only": [], "uncached_solve": [],
           "rif3": [], "uncached_rif3": []}

    def timed(kind, y, **kw):
        clocks.step_begins()
        t0 = time.perf_counter()
        if y is not None:
            des.update_outcome(y)
        r = ob.bootstrap(des, reps, ref_kind=kw.pop("ref_kind", ref), norm=norm, want_rep=True, **kw)
        wall = (time.perf_counter() - t0) * 1e3
        return r, dict(kind=kind, wall_ms=wall, cache_use=ob.core.CACHE_USE_NAMES.get(r.get("cache_use", 0)), **r["timings_ms"])

    def check(a, b, what, expect_use):
        if not identical(a, b):
            mismatches.append(what)
        if a.get("cache_use") != expect_use:
            mismatches.append(f"{what}: cache use {a.get('cache_use')} != {expect_use}")

    clocks.start()
    # ---- outcome refresh: uncached vs OUTCOME_ONLY (the cache filled once at the sweep's seed) ----
    timed("fill", None, seed=seed0, cache=cache)
    for i in range(args.warmup + args.steps):
        y = outcomes[i]
        ru, su = timed("uncached", y, seed=seed0)
        rc, sc = timed("outcome_only", y, seed=seed0, cache=cache)
        check(rc, ru, f"outcome_only step {i}", ob.CACHE_OUTCOME_ONLY)
        if i >= args.warmup:
            rec["uncached"].append(su); rec["outcome_only"].append(sc)
    # ---- SOLVE_ONLY: a ref_kind sweep (four kinds) on the current outcome ----
    for i in range(args.warmup + args.steps):
        for rk in (0, 1, 2, 3):
            ru, su = timed("uncached_solve", None, seed=seed0, ref_kind=rk)
            rc, sc = timed("solve_only", None, seed=seed0, ref_kind=rk, cache=cache)
            check(rc, ru, f"solve_only step {i} ref_kind {rk}", ob.CACHE_SOLVE_ONLY)
            if i >= args.warmup:
                rec["uncached_solve"].append(su); rec["solve_only"].append(sc)
    # ---- FILLED: every step at a new seed, so the cache never applies; its twin runs uncached at that seed ----
    for i in range(args.warmup + args.steps):
        y = outcomes[i]
        ru, su = timed("uncached_filled", y, seed=seed0 + 1 + i)
        rc, sc = timed("filled", y, seed=seed0 + 1 + i, cache=cache)
        check(rc, ru, f"filled step {i}", ob.CACHE_FILLED)
        if i >= args.warmup:
            rec["uncached_filled"].append(su); rec["filled"].append(sc)
    # ---- T = 3 RIF step after a T = 1 fill ----
    taus = [0.1, 0.5, 0.9]
    for i in range(args.warmup + args.steps):
        des.update_outcome(outcomes[i])
        timed("fill_t1", None, seed=seed0 + 100, cache=cache)        # filled (first step) or outcome-only, T = 1
        des.apply_rif_multi(taus)
        rc, sc = timed("rif3", None, seed=seed0 + 100, cache=cache)
        ru, su = timed("uncached_rif3", None, seed=seed0 + 100)
        check(rc, ru, f"rif3 step {i}", ob.CACHE_OUTCOME_ONLY)
        if i >= args.warmup:
            rec["uncached_rif3"].append(su); rec["rif3"].append(sc)
    clocks.stop_flag.set(); clocks.step_begins(); clocks.join(timeout=5)

    def med(kind):
        rows = rec[kind]
        return {k: float(np.median([r[k] for r in rows])) for k in rows[0] if isinstance(rows[0][k], (int, float))}

    peak = dmma_peak_tflops()
    n_glob = des.n_a + des.n_b
    out = {"workload": args.workload, "n": n_glob, "K": K, "reps": reps, "steps": args.steps, "warmup": args.warmup,
           **device_info(args.device), "clocks": clocks.summary(), "cache_bytes": cache.bytes,
           "medians": {k: med(k) for k in rec}, "runs": rec, "mismatches": mismatches, "bit_identical": not mismatches}
    m = out["medians"]
    out["speedup_outcome_only_vs_uncached"] = m["uncached"]["wall_ms"] / m["outcome_only"]["wall_ms"]
    out["filled_vs_uncached"] = m["filled"]["wall_ms"] / m["uncached_filled"]["wall_ms"] - 1.0
    out["speedup_solve_only_vs_uncached"] = m["uncached_solve"]["wall_ms"] / m["solve_only"]["wall_ms"]
    out["speedup_rif3_vs_uncached"] = m["uncached_rif3"]["wall_ms"] / m["rif3"]["wall_ms"]
    for kind, T in (("outcome_only", 1), ("rif3", 3)):
        t = m[kind]["gram_main"] * 1e-3
        tf = 2.0 * n_glob * K * T * reps / t / 1e12
        out[f"narrow_launch_{kind}"] = {"tflops": tf, "of_dmma_peak": tf / peak, "gram_main_ms": m[kind]["gram_main"],
                                        "flop": "2 n K T B", "peak_tflops": peak}
    with open(os.path.join(args.out, "outcome_sweep.json"), "w") as f:
        json.dump(out, f, indent=1)
    summary = {k: out[k] for k in ("device", "power_limit_w", "speedup_outcome_only_vs_uncached", "filled_vs_uncached",
                                   "speedup_solve_only_vs_uncached", "speedup_rif3_vs_uncached", "bit_identical") if k in out}
    summary["narrow_of_peak"] = out["narrow_launch_outcome_only"]["of_dmma_peak"]
    summary["medians_wall_ms"] = {k: round(v["wall_ms"], 2) for k, v in m.items()}
    print(json.dumps(summary))
    des.close(); cache.close(); ctx.close()
    return 1 if mismatches else 0


if __name__ == "__main__":
    sys.exit(main())
