#!/usr/bin/env python
"""Cluster bootstrap against the row bootstrap, on one GPU.

Config 3 (n = 10M, K = 51, WLS + Yun, B = 2000) with random cluster labels (clusters hold rows of both groups) for
M in {1e3, 1e5, 1e6} clusters, JOINT and BY_GROUP.  Per configuration, clustered steps (one design with the clusters
attached) and unclustered steps (a second design of the same frame) alternate; medians over --steps steps after --warmup.
Every unclustered step of the whole run must equal the first one bit for bit (the script exits 1 otherwise).

Recorded per configuration: wall time (host clock around a call that ends in a device synchronise) and the device stage
breakdown (CUDA events inside the library: counts, Gram, solve, reduce) of both kinds of step; then, in a separate
profiled step (torch.profiler, CUDA activities), the kernel time of counts_expand_kernel and of the unit-count kernels,
and the expansion's share of the HBM roofline from its algorithmic bytes: writes n * slots * count_bytes, reads 4 n per
panel (the unit map) plus the unit matrices, sum over them of M_g * slots * count_bytes.  Roofline: 7.7 TB/s, the data
sheet's HBM3e bandwidth of one B200 at 1000 W (a data-sheet figure, not a measured one).  Device name, power limit and
SM clocks are read in the same run.

  python tools/cluster_bench.py --out results/cluster [--steps 3] [--warmup 1]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_BYTES_PER_S = 7.7e12
KEYS = ("point_stats", "rep_stats", "rep_status", "std_err", "p_value", "ci_lower", "ci_upper", "t_stat", "residuals_b",
        "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")


def identical(a, b):
    return all(np.array_equal(a[k], b[k], equal_nan=True) for k in KEYS) and a["total_gap"] == b["total_gap"]


def kernel_ms(prof, needle):
    """Summed device time (ms) of the kernels whose name contains needle."""
    tot = 0.0
    for ev in prof.key_averages():
        if needle in ev.key:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0.0)
            tot += t / 1e3
    return tot


def main():
    import bench
    from outcome_sweep_bench import device_info
    import oaxaca_blinder_rs_b200 as ob
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workload", default="config3_n10M_k50_wls_yun_B2000", choices=list(bench.WORKLOADS))
    ap.add_argument("--clusters", default="1000,100000,1000000")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)

    d, norm_spec, reps, ref = bench.make_data(args.workload)
    norm = [ob.NormVar(m, i) for m, i in norm_spec]
    n = d["outcome"].shape[0]
    ctx = ob.Context(args.device)
    pack = lambda: ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])  # noqa: E731
    des_row, des_cl = pack(), pack()
    seed = 20261021
    clocks = bench.ClockSampler(args.device)
    slots = ((reps + 1 + 127) // 128) * 128
    first_row, mismatches, configs = None, [], []

    def step(des):
        clocks.step_begins()
        t0 = time.perf_counter()
        r = ob.bootstrap(des, reps, ref_kind=ref, norm=norm, seed=seed, want_rep=True)
        return r, dict(wall_ms=(time.perf_counter() - t0) * 1e3, **r["timings_ms"])

    clocks.start()
    for M in [int(x) for x in args.clusters.split(",")]:
        codes = np.random.default_rng(M).integers(0, M, n).astype(np.int32)
        for strata in ("joint", "group"):
            t0 = time.perf_counter()
            des_cl.attach_clusters(codes, n_codes=M, strata=strata)
            attach_ms = (time.perf_counter() - t0) * 1e3
            cl = des_cl.clusters
            rec = {"clustered": [], "rows": []}
            n_ok = None
            for i in range(args.warmup + args.steps):
                rc, sc = step(des_cl)
                rr, sr = step(des_row)
                n_ok = rc["n_ok"]
                if first_row is None:
                    first_row = rr
                elif not identical(rr, first_row):
                    mismatches.append(f"unclustered step differs (M={M}, {strata}, step {i})")
                if i >= args.warmup:
                    rec["clustered"].append(sc); rec["rows"].append(sr)
            med = {k: {f: float(np.median([r[f] for r in v])) for f in v[0]} for k, v in rec.items()}
            row = dict(M=M, strata=strata, units_a=cl["units_a"], units_b=cl["units_b"], attach_ms=attach_ms, n_ok=n_ok,
                       medians=med, runs=rec,
                       clustered_vs_rows=med["clustered"]["wall_ms"] / med["rows"]["wall_ms"] - 1.0)
            if not args.no_profile:
                import torch
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    step(des_cl)
                    torch.cuda.synchronize()
                cb = 1                                     # the native stream never saturates 8-bit counts at these sizes
                mats = [cl["units_a"]] if strata == "joint" else [cl["units_a"], cl["units_b"]]
                bytes_expand = n * slots * cb + 4 * n * (slots // 128) + sum(mats) * slots * cb
                t_exp = kernel_ms(prof, "counts_expand_kernel")
                row["kernels_ms"] = {"counts_expand_kernel": t_exp, "counts_philox_body": kernel_ms(prof, "counts_philox_body"),
                                     "counts_philox_fixup": kernel_ms(prof, "counts_philox_fixup"),
                                     "counts_lut_kernel": kernel_ms(prof, "counts_lut_kernel")}
                row["expand_bytes"] = bytes_expand
                if t_exp > 0:
                    row["expand_tb_per_s"] = bytes_expand / (t_exp * 1e-3) / 1e12
                    row["expand_of_hbm_roofline"] = bytes_expand / HBM_BYTES_PER_S / (t_exp * 1e-3)
            configs.append(row)
            print(json.dumps({k: row[k] for k in ("M", "strata", "units_a", "units_b", "clustered_vs_rows", "n_ok")} |
                             {"wall_ms": {k: round(v["wall_ms"], 1) for k, v in med.items()},
                              "counts_ms": {k: round(v["counts"], 2) for k, v in med.items()},
                              "expand_ms": row.get("kernels_ms", {}).get("counts_expand_kernel"),
                              "expand_of_hbm_roofline": row.get("expand_of_hbm_roofline")}), flush=True)
    clocks.stop_flag.set(); clocks.step_begins(); clocks.join(timeout=5)
    out = {"workload": args.workload, "n": n, "reps": reps, "slots": slots, "steps": args.steps, "warmup": args.warmup,
           **device_info(args.device), "clocks": clocks.summary(), "hbm_roofline_bytes_per_s": HBM_BYTES_PER_S,
           "configs": configs, "mismatches": mismatches, "unclustered_bit_identical": not mismatches}
    with open(os.path.join(args.out, "cluster_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("device", "power_limit_w", "unclustered_bit_identical") if k in out}))
    des_row.close(); des_cl.close(); ctx.close()
    return 1 if mismatches else 0


if __name__ == "__main__":
    sys.exit(main())
