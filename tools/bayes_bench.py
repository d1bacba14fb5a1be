#!/usr/bin/env python
"""Bayesian bootstrap against the row bootstrap, on one GPU.

Per workload (config 3: n = 10M, K = 51, WLS + Yun, B = 2000; config 5: n = 100M, K = 17, B = 10000 unless --reps
overrides it) row-bootstrap steps and Bayesian steps of one design alternate in one process; medians over --steps steps
after --warmup.  Every step of a scheme must equal that scheme's first step bit for bit (the script exits 1 otherwise).

Recorded per workload and scheme: wall time (host clock around a call that ends in a device synchronise) and the device
stage breakdown (CUDA events inside the library): ms_counts (replicate generation: the multinomial kernels, or the
Bayesian weight kernel and the leaf sums of the weights) and ms_gram_kernel (the DMMA contraction alone).  Derived:
  * the generator's share of the HBM roofline from its algorithmic bytes: the weights written, 4 n_pad slots_pad bytes,
    over ms_counts, against 7.7 TB/s (the data sheet's HBM3e bandwidth of one B200 at 1000 W, not a measured figure);
  * the Gram kernel's DMMA fraction by the DESIGN section 8d formula: 2 (n_a + n_b) slots Pc flops (Pc = the columns the
    contraction computes) over ms_gram_kernel, against the measured FP64 DMMA issue peak of 37.09 TFLOP/s
    (profiles/r01_fp64_peaks.json).
Device name, power limit and SM clocks are read in the same run.

  python tools/bayes_bench.py --out results/bayes [--workloads config3_n10M_k50_wls_yun_B2000] [--steps 3] [--warmup 1]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_BYTES_PER_S = 7.7e12
DMMA_PEAK_FLOPS = 37.09e12
KEYS = ("point_stats", "rep_stats", "rep_status", "std_err", "p_value", "ci_lower", "ci_upper", "t_stat", "residuals_b",
        "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")


def identical(a, b):
    return all(np.array_equal(a[k], b[k], equal_nan=True) for k in KEYS) and a["total_gap"] == b["total_gap"]


def computed_columns(K, n_cont, cat_levels):
    from oaxaca_blinder_rs_b200 import _native
    L = _native.lib()
    L.ob_debug_gram_columns.restype = C.c_int64
    L.ob_debug_gram_columns.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                        C.POINTER(C.c_uint16), C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int32)]
    lv = np.asarray(list(cat_levels) + [0], dtype=np.int32)
    til = np.zeros(3, dtype=np.int32)
    L.ob_debug_gram_columns(K, 1, n_cont, lv.ctypes.data_as(C.POINTER(C.c_int32)), len(cat_levels), None, None, 0,
                            til.ctypes.data_as(C.POINTER(C.c_int32)))
    return int(til[0])


def main():
    import bench
    from outcome_sweep_bench import device_info
    import oaxaca_blinder_rs_b200 as ob
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="config3_n10M_k50_wls_yun_B2000,config5_n100M_k16_B10000")
    ap.add_argument("--reps", type=int, default=0, help="override the workload's replicate count (0: the workload's)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    ctx = ob.Context(args.device)
    clocks = bench.ClockSampler(args.device)
    seed = 20261021
    rows, mismatches = [], []
    clocks.start()
    for name in args.workloads.split(","):
        d, norm_spec, reps, ref = bench.make_data(name)
        reps = args.reps or reps
        norm = [ob.NormVar(m, i) for m, i in norm_spec]
        des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
        n, K = d["outcome"].shape[0], des.K
        slots = reps + 1
        slots_pad = (slots + 127) // 128 * 128
        n_pad = sum((m + 31) // 32 * 32 for m in (des.n_a, des.n_b))
        pc = computed_columns(K, len(d["cont"]), d["cat_levels"])
        first, rec = {}, {"multinomial": [], "bayes": []}

        def step(scheme):
            clocks.step_begins()
            t0 = time.perf_counter()
            r = ob.bootstrap(des, reps, ref_kind=ref, norm=norm, seed=seed, want_rep=True, scheme=scheme)
            return r, dict(wall_ms=(time.perf_counter() - t0) * 1e3, **r["timings_ms"])

        n_ok = {}
        for i in range(args.warmup + args.steps):
            for scheme in ("multinomial", "bayes"):
                r, s = step(scheme)
                n_ok[scheme] = r["n_ok"]
                if scheme not in first:
                    first[scheme] = r
                elif not identical(r, first[scheme]):
                    mismatches.append(f"{name}: {scheme} step {i} differs from its first step")
                if i >= args.warmup:
                    rec[scheme].append(s)
        med = {k: {f: float(np.median([r[f] for r in v])) for f in v[0]} for k, v in rec.items()}
        gen_bytes = 4.0 * n_pad * slots_pad
        flops = 2.0 * n * slots * pc
        derived = {}
        for k, m in med.items():
            derived[k] = {"dmma_fraction": flops / DMMA_PEAK_FLOPS / (m["gram_main"] * 1e-3) if m["gram_main"] > 0 else None}
        derived["bayes"]["weights_bytes"] = gen_bytes
        derived["bayes"]["counts_of_hbm_roofline"] = gen_bytes / HBM_BYTES_PER_S / (med["bayes"]["counts"] * 1e-3)
        row = dict(workload=name, n=n, K=K, reps=reps, slots_pad=slots_pad, Pc=pc, n_ok=n_ok, medians=med, derived=derived,
                   runs=rec, bayes_vs_rows_step=med["bayes"]["wall_ms"] / med["multinomial"]["wall_ms"] - 1.0,
                   gram_kernel_bayes_vs_rows=med["bayes"]["gram_main"] / med["multinomial"]["gram_main"] - 1.0,
                   counts_share_of_bayes_step=med["bayes"]["counts"] / med["bayes"]["wall_ms"])
        rows.append(row)
        print(json.dumps({k: row[k] for k in ("workload", "reps", "n_ok", "bayes_vs_rows_step", "gram_kernel_bayes_vs_rows",
                                              "counts_share_of_bayes_step")} |
                         {"wall_ms": {k: round(v["wall_ms"], 1) for k, v in med.items()},
                          "ms_counts": {k: round(v["counts"], 2) for k, v in med.items()},
                          "ms_gram_kernel": {k: round(v["gram_main"], 1) for k, v in med.items()},
                          "derived": derived}), flush=True)
        des.close()
    clocks.stop_flag.set(); clocks.step_begins(); clocks.join(timeout=5)
    out = {"steps": args.steps, "warmup": args.warmup, **device_info(args.device), "clocks": clocks.summary(),
           "hbm_roofline_bytes_per_s": HBM_BYTES_PER_S, "dmma_peak_flops": DMMA_PEAK_FLOPS, "workloads": rows,
           "mismatches": mismatches, "steps_bit_identical": not mismatches}
    with open(os.path.join(args.out, "bayes_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("device", "power_limit_w", "steps_bit_identical") if k in out}))
    ctx.close()
    return 1 if mismatches else 0


if __name__ == "__main__":
    sys.exit(main())
