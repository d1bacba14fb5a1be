#!/usr/bin/env python
"""bench.py -- bootstrap replicates/sec of the B200-native oaxaca_blinder bootstrap path.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): synthetic wage data,
n = 10M rows, k = 50 predictors (44 continuous + C(sector) + C(region), 4 levels each -> K = 51 design
columns), sample weights (WLS), Yun normalisation of both categoricals, B = 2000 bootstrap replicates.
A "step" is one full bootstrap (point estimate + 2000 replicates + SE/CI reduction).

  value  reps/s with the packed design already resident in HBM (ob_bootstrap_run only)
  e2e    reps/s through the C ABI from pinned HOST columns: H2D + pack + bootstrap + results D2H per step
  roofline     Gram contraction kernel: algorithmic 2*n*P*B flop / its CUDA-event time vs the FP64 DMMA peak
  cpu_baseline the oracle port (reference-shaped CPU restatement) on the box's host cores, bounded sample

--impl reference times that CPU restatement on all host threads (the Rust reference cannot be built here:
no cargo/rustc in the image, dependencies not vendored).  N > 1: one rank per GPU (torchrun), replicates
sharded inside the library (ob_boot_opts.shard_replicates): one NCCL all-gather of the statistics block, device to
device, reduction on every rank; total work fixed -> strong.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n, n_cont, cat_levels, weights, normalize, reps, ref_kind)   [BASELINE.json configs]
    "config3_n10M_k50_wls_yun_B2000": (10_000_000, 44, (4, 4), True, True, 2000, 0),   # configs[2]: the headline
    "config2_n1M_k20_B1000": (1_000_000, 20, (), False, False, 1000, 0),               # configs[1]
    "config1_n10k_wage_B500": (10_000, 2, (4,), False, False, 500, 0),                 # configs[0]: the CPU-runnable case
    "config4_n5M_k30_rif_B1000": (5_000_000, 30, (), False, False, 1000, 0),           # configs[3]: one tau per step (--rif-tau)
    "config5_n100M_k16_B10000": (100_000_000, 16, (), False, False, 10000, 0),         # configs[4]
    "smoke_n200k_k50_B256": (200_000, 44, (4, 4), True, True, 256, 0),
    "probe_n1M_k50_B255": (1_000_000, 44, (4, 4), True, True, 255, 0),   # ncu-sized: two full panels
    "probe5_n20M_k16_B2000": (20_000_000, 16, (), False, False, 2000, 0),  # config-5 column shape (1 full + 1 half tile)
}
# roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE Gram launch, measured by ncu on THIS build of
# the kernel: profiles/gram_traffic.json holds {workload, n_gpus, bytes, src_sha256, csv}; an entry counts only while the
# hash of the kernel sources it was taken on equals the current sources -- otherwise the key is null, never stale.
GRAM_SOURCES = ("oaxaca_blinder_rs_b200/csrc/gram.cu", "oaxaca_blinder_rs_b200/csrc/common.cuh")
GRAM_GEOMETRY = "oaxaca_blinder_rs_b200/csrc/internal.h"      # only the tile / leaf constants below shape the kernel
GRAM_GEOMETRY_NAMES = ("constexpr int BM ", "constexpr int BN ", "constexpr int KT ", "constexpr int GRAM_THREADS ", "constexpr int MAX_SEGS ")


def gram_source_hash():
    import hashlib
    h = hashlib.sha256()
    for f in GRAM_SOURCES:
        with open(os.path.join(ROOT, f), "rb") as fh:
            h.update(fh.read())
    with open(os.path.join(ROOT, GRAM_GEOMETRY)) as fh:
        h.update("".join(ln for ln in fh if ln.lstrip().startswith(GRAM_GEOMETRY_NAMES)).encode())
    return h.hexdigest()


def measured_gram_traffic(name, world):
    try:
        with open(os.path.join(ROOT, "profiles", "gram_traffic.json")) as fh:
            entries = json.load(fh)["entries"]
    except (OSError, ValueError, KeyError):
        return None, None
    sha = gram_source_hash()
    for e in entries:
        if e.get("workload") == name and e.get("n_gpus") == world and e.get("src_sha256") == sha:
            return int(e["bytes"]), e.get("csv")
    return None, None


def _measured_hbm_peak():
    """MEASURED_PEAKS.json (driver-written copy bandwidth on this pool); the value it held when this was written if the
    file is absent."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"])
    except (OSError, ValueError, KeyError, TypeError):
        return 6550.1


HBM_PEAK_GBS = _measured_hbm_peak()
FP64_DMMA_PEAK_TFLOPS = 37.1     # measured on this pool (profiles/r01_fp64_peaks.json): DMMA.8x8x4 issue peak
FP64_CUBLAS_DGEMM_TFLOPS = 35.4  # measured on this pool (profiles/r01_dgemm_peak.json): cuBLAS DGEMM 8192^3


def algorithmic_flops(n, K, reps):
    P = K * (K + 1) // 2 + K      # SURVEY.md 8d: F_rep = 2 n P, P = K(K+1)/2 + K
    return 2.0 * n * P * reps, P


def hbm_stage_rooflines(d, K, reps, world, shard_rows, out, pack_ms):
    """The HBM-bound stages (SURVEY.md 8d): algorithmic bytes / CUDA-event time against the measured copy bandwidth."""
    n_loc = d["n"]                                      # rows this rank holds
    slots = (reps + 1) if (world == 1 or shard_rows) else (-(-reps // world) + 1)
    gen_bytes = float(n_loc) * slots                    # uint8 multiplicity matrix written once
    t_gen = out["timings_ms"]["counts"] - out["timings_ms"].get("comm", 0.0)
    src = 8 * (len(d["cont"]) + 1 + (1 if d["weights"] is not None else 0)) + 4 * len(d["cat_codes"]) + 1
    dst = 8 * (K + 1) * (2 if d["weights"] is not None else 1) + (8 if d["weights"] is not None else 0)
    pack_bytes = float(n_loc) * (src + dst)
    def entry(b, ms):
        gbs = b / (ms * 1e-3) / 1e9 if ms > 0 else None
        return {"bytes": b, "ms": ms, "achieved": gbs, "peak": HBM_PEAK_GBS, "unit": "GB/s",
                "frac": None if gbs is None else gbs / HBM_PEAK_GBS}
    return {"replicate_generation": dict(entry(gen_bytes, t_gen), note="integer-ALU bound (Philox4x32-10 + table lookup per "
                                         "count), not HBM: bytes are the multiplicity matrix written"),
            "pack": entry(pack_bytes, pack_ms[1]),
            "h2d_copy": {"bytes": float(n_loc) * src, "ms": pack_ms[0]}}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML during the timed region.

    NVML queries take a driver lock that host-side CUDA calls need too: a call of the step that coincides with a query
    stalls 8-22 ms (measured).  So the sampler does not free-run: the timed loop announces every step (`step_begins`),
    and a sample is taken 40 ms into a step -- the host is then parked in the library's wait for the Gram contraction
    (>= 170 ms at every bench workload that matters), the GPU is under load, and nothing of the step is delayed -- at
    most once every 2 s.  Without announcements it falls back to one sample every 2 s."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.stop_flag = threading.Event()
        self.step_flag = threading.Event()
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def step_begins(self):
        self.step_flag.set()

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        def sample():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
        last = 0.0
        while not self.stop_flag.is_set():
            announced = self.step_flag.wait(2.0)
            self.step_flag.clear()
            if self.stop_flag.is_set():
                break
            if announced:
                if time.perf_counter() - last < 2.0 and self.samples:
                    continue
                if self.stop_flag.wait(0.04):          # 40 ms into the step: the host sits in the Gram wait
                    break
            sample()
            last = time.perf_counter()
        if not self.samples:                           # a timed region shorter than 40 ms: one sample right at its end
            sample()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def make_data(name):
    from oaxaca_blinder_rs_b200 import synth
    n, n_cont, cats, weights, normalize, reps, ref = WORKLOADS[name]
    d = synth.make_wage(n, n_cont, cat_levels=cats, weights=weights)
    norm = synth.norm_spec(d) if normalize else []
    return d, norm, reps, ref


def default_rif_tau(args, name):
    return args.rif_tau if args.rif_tau is not None else (0.5 if name.startswith("config4") else None)


def config_dict(name, world, shard_rows, rif_tau):
    """`config` of the JSON line: identical for both arms (the driver compares them)."""
    n, n_cont, cats, weights, normalize, reps, _ = WORKLOADS[name]
    K = 1 + n_cont + sum(m - 1 for m in cats)
    return {"workload": name, "n": n, "k": K - 1, "K": K, "P": K * (K + 1) // 2 + K, "reps": reps,
            "wls": bool(weights), "yun": bool(normalize and cats), "rif_tau": rif_tau,
            "parallelism": (f"row-shard x{world}" if shard_rows else f"replicate-shard x{world}"),
            "l2": "inputs larger than L2 (design %.2f GB, multiplicities %.1f GB per GPU per step)"
                  % (n * (K + 1) * 8 / 1e9 / (world if shard_rows else 1), n * (reps + 1) / world / 1e9)}


def rows_sharded(args, name, world):
    return world > 1 and (args.shard == "rows" or (args.shard == "auto" and name.startswith("config5")))


README_SHAPE = dict(n=100_000, p=10, reps=500, published_s=3.11, source="/root/reference README.md:310-317 "
                    "(\"100k rows x 10 predictors, 500 bootstrap reps: 3.11 s\"; hardware and core count not stated)")


def readme_calibration_cpu(threads):
    """The one shape the reference publishes a time for (n = 1e5, p = 10, B = 500: 3.11 s), run through the oracle port
    in its reference-shaped mode on `threads` host threads: calibrates the port against the Rust binary's own number."""
    from oracle import pyoracle as orc
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(README_SHAPE["n"], README_SHAPE["p"])
    Xa, ya, wa, Xb, yb, wb = synth.dense_design(d)
    spec = orc.Spec(K=Xa.shape[1], n_cont=README_SHAPE["p"], ref_kind=0, norm=[])
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        orc.run(spec, Xa, ya, wa, Xb, yb, wb, README_SHAPE["reps"], None, None, seed=1, nthreads=threads, precise=False,
                want_rep=False)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"shape": "n=1e5, p=10, B=500, OLS", "port_seconds": best, "threads": threads,
            "published_seconds": README_SHAPE["published_s"], "published_source": README_SHAPE["source"],
            "port_over_published": best / README_SHAPE["published_s"]}


def dense_for_cpu(d, rif_tau):
    """Dense per-group matrices for the oracle port, built ONCE per run (the reference clones its frame once, too)."""
    from oracle import pyoracle as orc
    from oaxaca_blinder_rs_b200 import synth
    Xa, ya, wa, Xb, yb, wb = synth.dense_design(d)
    if rif_tau is not None:             # decompose_quantile: RIF outcome computed once per group (builder.rs:721-737)
        ya, yb = orc.rif(ya, rif_tau), orc.rif(yb, rif_tau)
    return Xa, ya, wa, Xb, yb, wb


def cpu_baseline(dense, n_cont, norm, ref, threads, reps_cpu):
    """Times the oracle port (reference-shaped arithmetic) on `threads` host threads over reps_cpu replicates + the
    point pass (reps_cpu + 1 passes, run concurrently)."""
    from oracle import pyoracle as orc
    Xa, ya, wa, Xb, yb, wb = dense
    spec = orc.Spec(K=Xa.shape[1], n_cont=n_cont, ref_kind=ref, norm=[orc.NormVar(m, i) for m, i in norm])
    t0 = time.perf_counter()
    out = orc.run(spec, Xa, ya, wa, Xb, yb, wb, reps_cpu, None, None, seed=1, nthreads=threads, precise=False, want_rep=False)
    dt = time.perf_counter() - t0
    # the point pass is part of run(); per-replicate cost is independent of B -> reps/s over (reps_cpu + 1) passes
    return (reps_cpu + 1) / dt, dt, out["n_ok"]


def host_threads_and_sample(d, K):
    import psutil
    cores = os.cpu_count() or 1
    per_thread = d["n"] * K * 8 * (2.2 if d["weights"] is not None else 1.2)     # gathered copy (+ sqrt(w)-scaled copy)
    avail = psutil.virtual_memory().available
    dense = d["n"] * K * 8 * 1.3
    threads = int(max(1, min(cores, (0.7 * avail - dense) // per_thread)))
    return cores, threads


def run_reference(args, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    d, norm, reps, ref = make_data(name)
    K = 1 + len(d["cont"]) + sum(m - 1 for m in d["cat_levels"])
    cores, threads = host_threads_and_sample(d, K)
    reps_cpu = max(threads - 1, 1)          # + the point pass = `threads` passes, one per thread
    rif_tau = default_rif_tau(args, name)
    dense = dense_for_cpu(d, rif_tau)
    n_cont = len(d["cont"])
    del d
    vals = []
    frac, budget_s = 1.0, 300.0        # the whole --steps K --warmup W run must end within a few minutes
    for it in range(args.warmup + args.steps):
        v, dt, _ = cpu_baseline(dense, n_cont, norm, ref, threads, reps_cpu)
        if it == 0 and dt * (args.warmup + args.steps) > budget_s:
            # bounded sample: the first `frac` of each group's rows (per-replicate cost is linear in n; every thread stays
            # busy); reps/s at the full n = reps/s on the sample x frac
            frac = max(0.05, budget_s / (dt * (args.warmup + args.steps)))
            Xa, ya, wa, Xb, yb, wb = dense
            ka, kb = max(int(len(ya) * frac), Xa.shape[1] + 2), max(int(len(yb) * frac), Xb.shape[1] + 2)
            dense = (np.ascontiguousarray(Xa[:ka]), ya[:ka].copy(), None if wa is None else wa[:ka].copy(),
                     np.ascontiguousarray(Xb[:kb]), yb[:kb].copy(), None if wb is None else wb[:kb].copy())
            frac = (ka + kb) / float(len(ya) + len(yb))
            del Xa, Xb
            continue
        if it >= args.warmup:
            vals.append((v * frac, dt))
    if not vals:
        vals.append((v * frac, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    sample = f"{reps_cpu} replicates + point pass per step on {threads} OpenMP threads (of {cores} cores), " + \
        ("full n" if frac == 1.0 else f"the first {frac:.3f} of each group's rows, reps/s scaled by that fraction (cost is linear in n)")
    world = max(args.gpus, 1)
    line = {"impl": "reference", "metric": "bootstrap_reps_per_sec", "value": value, "unit": "reps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(name, world, rows_sharded(args, name, world), rif_tau),
            "cpu_baseline": {"value": value, "unit": "reps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "reps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "readme_shape": readme_calibration_cpu(min(cores, 64)),
            "note": "CPU restatement of the reference algorithm (oracle port: gather, sqrt(w) scaling, cache-blocked AVX2 "
                    "X'X, Cholesky, residuals, inverse per replicate; OpenMP over replicates), not the Rust binary"}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64_000_000      # --dump-outputs: every file together, .npy headers included
DUMP_SAMPLE_SEED = 2026


def dump_outputs(out, path):
    """Writes the arrays a caller of ob.bootstrap receives (the dict of one step) as <path>/<name>.npy in float64, so
    that two builds can be compared output for output; total_gap and n_ok become 0-d arrays.  An array that does not
    fit the share of DUMP_LIMIT_BYTES left to it is replaced by a seeded sample of its flattened elements (sorted
    indices, the same on every run of the same workload).  Returns {name: [elements written, elements]} of those."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in out.items()
              if isinstance(v, np.ndarray) or k in ("total_gap", "n_ok")}
    os.makedirs(path, exist_ok=True)
    left = DUMP_LIMIT_BYTES - 128 * len(arrays)        # 128 bytes of .npy header per file at these ranks
    names = sorted(arrays, key=lambda k: (arrays[k].size, k))
    sampled = {}
    for i, k in enumerate(names):
        a = arrays[k]
        cap = left // a.itemsize // (len(names) - i)   # the smaller arrays before it have left their unused share
        if a.size > cap:
            idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(a.size, cap, replace=False))
            sampled[k] = [int(cap), int(a.size)]
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, k + ".npy"), a)
        left -= a.nbytes
    return sampled


def readme_shape_gpu(ob, ctx):
    """Same README shape end to end on the GPU (host columns -> pack -> point + 500 replicates -> results), best of 3."""
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(README_SHAPE["n"], README_SHAPE["p"])
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
        ob.bootstrap(des, README_SHAPE["reps"], ref_kind=0, seed=1)
        des.close()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best


def nccl_selftest(ob, obd, ctx, rank, world, dist, torch):
    """Before any multi-GPU timing: both sharding modes over the library's NCCL communicator must reproduce a one-GPU
    run of the same frame BIT FOR BIT (statistics, SEs, CIs).  Small shape, a second of work.  Raises on mismatch."""
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(300_000, 6, cat_levels=(4,), weights=True, seed=5)
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    reps, kw = 200, dict(ref_kind=ob.REF_WEIGHTED, norm=norm, seed=5, want_rep=True)
    whole = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
    one = ob.bootstrap(whole, reps, **kw)
    mode_r = ob.bootstrap(whole, reps, shard_replicates=True, **kw)
    whole.close()
    keys = ("point_stats", "rep_stats", "std_err", "ci_lower", "ci_upper", "p_value")
    same = lambda a, b: bool(np.array_equal(np.nan_to_num(a, nan=-7.0), np.nan_to_num(b, nan=-7.0)))
    ok_r = all(same(mode_r[k], one[k]) for k in keys)
    ok_n = None
    if world & (world - 1) == 0:
        shard = obd.pack_row_shard_from_slice(ctx, d, rank, world)
        mode_n = ob.bootstrap(shard, reps, max_workspace_bytes=200_000_000, **kw)      # several panel batches
        shard.close()
        ok_n = all(same(mode_n[k], one[k]) for k in keys)
    # the Machado-Mata passes under mode R (ob_mm_opts.shard_replicates): pass rows gathered over the same communicator
    dm = synth.make_wage(20_000, 3, cat_levels=(3,), weights=False, seed=6)
    mdes = ob.Design.pack(ctx, dm["cont"], dm["cat_codes"], dm["cat_levels"], dm["outcome"], None, dm["group"])
    mkw = dict(quantiles=[0.1, 0.5, 0.9], simulations=32, reps=2 * world + 1, seed=3, want_rep=True)
    m_one = ob.machado_mata(mdes, **mkw)
    m_r = ob.machado_mata(mdes, shard_replicates=True, **mkw)
    mdes.close()
    ok_m = all(same(m_r[k], m_one[k]) for k in ("point_stats", "rep_stats", "std_err", "ci_lower", "ci_upper", "p_value"))
    flags = torch.tensor([int(ok_r), int(ok_n is not False), int(ok_m)], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok_r, ok_n_all, ok_m = bool(flags[0].item()), bool(flags[1].item()), bool(flags[2].item())
    if not (ok_r and ok_n_all and ok_m):
        raise SystemExit(f"NCCL self-test failed: mode R bit-identical = {ok_r}, mode N bit-identical = {ok_n_all}, "
                         f"Machado-Mata mode R bit-identical = {ok_m}")
    return {"mode_r_bit_identical_to_one_gpu": ok_r, "mode_n_bit_identical_to_one_gpu": None if ok_n is None else ok_n_all,
            "machado_mata_mode_r_bit_identical_to_one_gpu": ok_m,
            "shape": "n=300k, K=10, WLS + Yun, B=200 (Machado-Mata: n=20k, K=6, 32 simulations, 2 world + 1 passes), every rank "
                     "compared with its own unsharded run"}


def mm_roofline(r, rows_per_group):
    """mm_qr_kernel against the HBM roofline: algorithmic bytes = the iterate traffic of the interior-point sweeps, 21
    doubles per row and iteration (DESIGN 7c: sweep 1 reads 6 and writes 4 vectors, sweep 2 reads 4 and writes 1, sweep 3
    reads 5 and writes 1), summed over the iterations of all regressions of the launch; the design rows come from L2."""
    bytes_ = 168.0 * r["qr"]["iterations"] * rows_per_group
    ms = r["timings_ms"]["qr"]
    peak = HBM_PEAK_GBS
    ach = bytes_ / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "mm_qr_kernel (one block per quantile regression)", "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak, "traffic": None, "launch_ms": ms, "bytes_per_launch": bytes_,
            "note": "latency-bound in practice (profiles/r02_mm_qr_ncu.json: long-scoreboard stalls, issue slots 44 % busy); "
                    "ncu DRAM traffic of a smaller launch is within 15 % of this model"}


def measure_machado_mata_sharded(ob, ctx, torch, dist, world, n=200_000, n_cont=7, sims=200, reps=20, steps=2):
    """The Machado-Mata record at N > 1: the same workload as measure_machado_mata, the regressions of every pass split
    over the ranks inside the library (ob_mm_opts.shard_replicates), coefficients all-gathered over NCCL."""
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(n, n_cont, cat_levels=(3,), weights=False, seed=7)
    des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], None, d["group"])
    q = [0.1, 0.25, 0.5, 0.75, 0.9]
    ob.machado_mata(des, q, simulations=16, reps=1, seed=1, shard_replicates=True)
    best, r = None, None
    for it in range(steps):
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ob.machado_mata(des, q, simulations=sims, reps=reps, seed=10 + it, shard_replicates=True)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = t.item() if best is None else min(best, t.item())
    des.close()
    nprob = r["qr"]["total"]
    return {"workload": f"synthetic wage n={n}, K={des.K}, simulations={sims}, bootstrap_reps={reps}: {nprob} regressions per step, "
                        f"split evenly over {world} ranks inside the library",
            "seconds_per_step": best, "value": nprob / best, "unit": "regressions/s", "passes_per_s": (reps + 1) / best,
            "qr_status": {k: r["qr"][k] for k in ("vertex", "approx", "failed")}}


def measure_machado_mata(ob, ctx, threads, n=200_000, n_cont=7, sims=200, reps=20, steps=2):
    """SURVEY 8f-3 beside the headline: the Machado-Mata decomposition (ob_mm_run; QuantileDecompositionBuilder defaults:
    200 simulations, 20 bootstrap passes, 5 quantiles) on synthetic wage data, n = 2e5 rows, K = 1 + 7 + 2 columns:
    (reps + 1) x sims x 2 = 8400 quantile regressions per step, each solved to the LP's vertex.  CPU: the oracle port's
    solver on a bounded sample of the same regressions, one per host thread."""
    import concurrent.futures as cf
    from oaxaca_blinder_rs_b200 import synth
    from oracle import pyoracle as orc
    d = synth.make_wage(n, n_cont, cat_levels=(3,), weights=False, seed=7)
    des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], None, d["group"])
    q = [0.1, 0.25, 0.5, 0.75, 0.9]
    ob.machado_mata(des, q, simulations=16, reps=1, seed=1)              # warm-up
    runs = []
    for it in range(steps):
        t0 = time.perf_counter()
        r = ob.machado_mata(des, q, simulations=sims, reps=reps, seed=10 + it)
        runs.append((time.perf_counter() - t0, r))
    dt, r = min(runs, key=lambda x: x[0])
    K, na = des.K, des.n_a
    nprob = r["qr"]["total"]
    # end to end: host columns -> ob_design_pack (H2D + pack) -> ob_mm_run -> results on the host, per step
    e2e = []
    for it in range(steps):
        t0 = time.perf_counter()
        d2 = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], None, d["group"])
        ob.machado_mata(d2, q, simulations=sims, reps=reps, seed=10 + it)
        d2.close()
        e2e.append(time.perf_counter() - t0)
    h2d = 8 * n * (len(d["cont"]) + 1) + 4 * n * len(d["cat_codes"]) + n
    X = np.c_[np.ones(n), np.stack(d["cont"], 1), d["cat_codes"][0] == 1, d["cat_codes"][0] == 2].astype(np.float64)
    A = d["group"] == 0
    Xa, ya = np.ascontiguousarray(X[A]), np.ascontiguousarray(d["outcome"][A])
    des.close()
    taus = np.random.default_rng(0).uniform(0.01, 0.99, size=8 * max(threads, 1))
    orc.qr(Xa[:1000], ya[:1000], 0.5)
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(max(threads, 1)) as ex:                    # ctypes releases the GIL: one regression per host thread
        infos = list(ex.map(lambda t: orc.qr(Xa, ya, float(t))[1], taus))
    cdt = time.perf_counter() - t0
    return {"what": "ob_mm_run: Machado-Mata quantile decomposition (quantile_decomposition.rs:281-421), every quantile "
                    "regression solved on the device to the LP's vertex (interior point + polish)",
            "workload": f"synthetic wage n={n} (n_a={na}), K={K}, simulations={sims}, bootstrap_reps={reps}, 5 target quantiles",
            "regressions_per_step": nprob, "seconds_per_step": dt, "regressions_per_s": nprob / dt, "passes_per_s": (reps + 1) / dt,
            "e2e": {"value": nprob / min(e2e), "unit": "regressions/s", "seconds_per_step": min(e2e), "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(8 * 6 * 3 * len(q)), "path": "host columns -> ob_design_pack -> ob_mm_run -> host results"},
            "qr_kernel_ms": r["timings_ms"]["qr"], "mean_ip_iterations": r["qr"]["iterations"] / max(nprob, 1),
            "roofline": mm_roofline(r, n / 2.0),
            "qr_status": {k: r["qr"][k] for k in ("vertex", "approx", "failed")}, "gpu_launches": r["gpu_launches"],
            "cpu_baseline": {"value": len(taus) / cdt, "unit": "regressions/s", "cores": int(threads), "kind": "port",
                             "sample": f"{len(taus)} regressions of group A ({na} rows) at random quantiles, one per thread at a time, {cdt:.1f} s; "
                                       f"mean {np.mean([i['iters'] for i in infos]):.1f} interior-point iterations"}}


def measure_also(name, ob, obd, ctx, torch, dist, rank, world, local, shard_rows, rif_tau, steps=2):
    """A BASELINE config other than the headline one at the same N (the row-sharded config 5, the RIF config 4), so
    that the driver's multi-GPU record holds them too: resident reps/s over `steps` steps after one warm-up, Gram
    kernel fraction of the DMMA peak, and an end-to-end step from host columns."""
    from oaxaca_blinder_rs_b200 import synth
    n, n_cont, cats, wts, normalize, reps, ref = WORKLOADS[name]
    if shard_rows:
        d = synth.make_wage_rows(n, n_cont, cat_levels=cats, weights=wts, rank=rank, world=world)
    else:
        d = synth.make_wage(n, n_cont, cat_levels=cats, weights=wts)
    norm = [ob.NormVar(m, i) for m, i in (synth.norm_spec(d) if normalize else [])]
    K = 1 + n_cont + sum(m - 1 for m in cats)
    # the frame's columns page-locked in place (ob_host_register), as a caller holding its own buffers would do
    pinned_cols = ob.pin_in_place(list(d["cont"]) + list(d["cat_codes"]) + [d["outcome"], d["weights"], d["group"]])

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def pack(asynchronous=False):
        if shard_rows:
            des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"],
                                 asynchronous=asynchronous)
            des.set_row_shard(d["n_a_global"], d["n_b_global"], world, rank)
            return des
        if world > 1:
            des = obd.pack_replicated(ctx, d, rank, world)
        else:
            des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
        if rif_tau is not None:
            des.apply_rif(rif_tau)
        return des

    def step(des):
        return ob.bootstrap(des, reps, ref_kind=ref, norm=norm, seed=2026, want_residuals=False,
                            shard_replicates=(world > 1 and not shard_rows))
    des = pack()
    step(des)
    sync()
    t0 = time.perf_counter()
    gram_ms = []
    for _ in range(steps):
        out = step(des)
        gram_ms.append(out["timings_ms"]["gram_main"])
    sync()
    dt = time.perf_counter() - t0
    sweep = None
    if rif_tau is not None:        # BASELINE configs[3]: the tau = 0.1 / 0.5 / 0.9 sweep, as three runs and as one pass
        taus = (0.1, 0.5, 0.9)

        def run_sweep(multi):
            sync()
            t = time.perf_counter()
            if multi:
                des.apply_rif_multi(taus)
                step(des)
            else:
                for tau in taus:
                    des.apply_rif(tau)
                    step(des)
            sync()
            return time.perf_counter() - t
        run_sweep(False); run_sweep(True)
        t3 = min(run_sweep(False) for _ in range(2))
        t1s = min(run_sweep(True) for _ in range(2))
        tt = torch.tensor([t3, t1s], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t3, t1s = tt.tolist()
        sweep = {"taus": list(taus), "three_runs_s": t3, "one_pass_s": t1s, "speedup": t3 / t1s,
                 "fits_per_s_one_pass": 3 * reps / t1s, "fits_per_s_three_runs": 3 * reps / t3}
    des.close()

    def e2e_step():
        if world > 1 and not shard_rows and world & (world - 1) == 0:
            dsg = obd.pack_row_shard_async(ctx, d, rank, world)        # host frame -> row shards, overlapped (mode N)
            if rif_tau is not None:
                dsg.apply_rif(rif_tau)
            ob.bootstrap(dsg, reps, ref_kind=ref, norm=norm, seed=2026, want_residuals=False)
        else:
            dsg = pack(asynchronous=rif_tau is None)
            step(dsg)
        dsg.close()
    e2e_step()                                   # warm-up of the pools this path uses
    sync()
    t1 = time.perf_counter()
    e2e_step()
    sync()
    dt_e = time.perf_counter() - t1
    times = torch.tensor([dt, dt_e], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e = times.tolist()
    ob.unpin(pinned_cols)
    flops, P = algorithmic_flops(n, K, reps)
    g_ms = float(np.mean(gram_ms))
    ach = flops / world / (g_ms * 1e-3) / 1e12
    return {"config": config_dict(name, world, shard_rows, rif_tau), "value": reps * steps / dt, "unit": "reps/s", "steps": steps,
            "warmup": 1, "ms_per_step": dt / steps * 1e3, "e2e": {"value": reps / dt_e, "unit": "reps/s", "steps": 1},
            "roofline": {"bound": "tensor", "achieved": ach, "peak": FP64_DMMA_PEAK_TFLOPS, "unit": "TFLOP/s",
                         "frac": ach / FP64_DMMA_PEAK_TFLOPS, "launch_ms": g_ms},
            "stage_ms": {k: float(v) for k, v in out["timings_ms"].items()}, "n_ok": int(out["n_ok"]), "quantile_sweep": sweep}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config3_n10M_k50_wls_yun_B2000", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rif-tau", type=float, default=None, help="RIF-regression outcome at this quantile (config 4)")
    ap.add_argument("--shard", default="auto", choices=["auto", "reps", "rows"],
                    help="N > 1: shard replicates (mode R; every GPU holds the design) or rows (mode N; config 5)")
    ap.add_argument("--e2e-upload", default="auto", choices=["auto", "gather", "rowshard"],
                    help="N > 1, replicate-sharded workloads, end-to-end leg: every rank uploads 1/N of the frame, then either "
                         "the packed rows are all-gathered so that every GPU holds the design (gather: mode R) or re-cut into "
                         "row shards (rowshard: mode N, a rank never needs the other rows); auto = rowshard")
    ap.add_argument("--also", default="auto", choices=["auto", "on", "off"],
                    help="N > 1: also measure the row-sharded config 5 and the RIF config 4 at the same N (key `also`)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them returned (point statistics, SE / p / CI / t, "
                         "coefficients, means, residuals) as DIR/<name>.npy in float64, at most 64 MB in all: arrays "
                         "beyond that are a fixed seeded sample.  Rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    name = args.workload
    if args.impl == "reference":
        return run_reference(args, name)

    import torch
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import distributed as obd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU path. Use --impl reference for the CPU baseline.")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    shard_rows = rows_sharded(args, name, world)
    ctx = ob.Context(local)
    if shard_rows:
        # mode N: this rank generates and holds only its rows; the library exchanges column sums and per-rank Gram
        # sums over its own NCCL communicator (results are bit-identical to one GPU)
        from oaxaca_blinder_rs_b200 import synth
        n_, n_cont_, cats_, wts_, normalize_, reps, ref = WORKLOADS[name]
        d = synth.make_wage_rows(n_, n_cont_, cat_levels=cats_, weights=wts_, rank=rank, world=world)
        norm = synth.norm_spec(d) if normalize_ else []
        n = n_
        ctx.init_nccl(rank, world)
    else:
        d, norm, reps, ref = make_data(name)
        n = d["n"]
        if world > 1:
            ctx.init_nccl(rank, world)       # mode R: the statistics all-gather and the upload (frame slices over NVLink)
    K = 1 + len(d["cont"]) + sum(m - 1 for m in d["cat_levels"])
    normv = [ob.NormVar(m, i) for m, i in norm]
    # multi-GPU: no timing before both sharding modes have reproduced a one-GPU run bit for bit over NCCL
    selftest = nccl_selftest(ob, obd, ctx, rank, world, dist, torch) if world > 1 else None

    # pinned host columns for the end-to-end leg
    def pin(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a[:1]).dtype, pin_memory=True)
        t.numpy()[...] = a
        return t
    pinned = dict(cont=[pin(c) for c in d["cont"]], cat=[pin(c) for c in d["cat_codes"]], y=pin(d["outcome"]),
                  w=pin(d["weights"]) if d["weights"] is not None else None, g=pin(d["group"]))
    h2d = sum(t.numel() * t.element_size() for t in pinned["cont"] + pinned["cat"] + [pinned["y"], pinned["g"]]
              + ([pinned["w"]] if pinned["w"] is not None else []))
    if world > 1 and not shard_rows:
        h2d //= world                       # each rank uploads its frame slice only

    rif_tau = default_rif_tau(args, name)

    e2e_rowshard = (world > 1 and not shard_rows and world & (world - 1) == 0 and
                    args.e2e_upload in ("rowshard", "auto"))

    def pack(asynchronous=False, e2e=False):
        if world > 1 and not shard_rows:
            fr = dict(n=n, cont=[t.numpy() for t in pinned["cont"]], cat_codes=[t.numpy() for t in pinned["cat"]],
                      cat_levels=d["cat_levels"], outcome=pinned["y"].numpy(),
                      weights=None if pinned["w"] is None else pinned["w"].numpy(), group=pinned["g"].numpy())
            if e2e and e2e_rowshard:
                # host frame -> this rank uploads 1/world of it in chunks (ob_design_pack_row_shard_async): rows go straight
                # to their place in the rank's row shard, the few rows other ranks own are exchanged over NVLink, and the
                # row-sharded bootstrap (mode N: bit-identical to one GPU, like mode R) overlaps all of it with its
                # replicate generation and a first Gram launch.  No GPU ever needs the other ranks' rows.
                des = obd.pack_row_shard_async(ctx, fr, rank, world)
                if rif_tau is not None:          # RIF on the row shard: histograms / leaf sums all-reduced over NVLink
                    des.apply_rif(rif_tau)
                return des
            # mode R: this rank uploads 1/world of the frame; the packed rows are all-gathered over NVLink
            des = obd.pack_replicated(ctx, fr, rank, world)
            if rif_tau is not None:
                des.apply_rif(rif_tau)
            return des
        # ob_design_pack_async: the call returns once the group split is known; the chunked column upload and the pack
        # run on the library's copy stream under the replicate generation and the first Gram launch of step()
        des = ob.Design.pack(ctx, [t.numpy() for t in pinned["cont"]], [t.numpy() for t in pinned["cat"]],
                             d["cat_levels"], pinned["y"].numpy(), None if pinned["w"] is None else pinned["w"].numpy(),
                             pinned["g"].numpy(), asynchronous=asynchronous and rif_tau is None)
        if shard_rows:
            des.set_row_shard(d["n_a_global"], d["n_b_global"], world, rank)
        if rif_tau is not None:          # decompose_quantile: RIF pre-step on the device (builder.rs:721-737)
            des.apply_rif(rif_tau)
        return des

    res_buf = {}

    def step(design):
        # OaxacaResults.residuals goes into a caller-owned, page-locked buffer reused across steps (ob_host_alloc: what a
        # Rust caller would keep instead of a fresh Vec), so the 8 n_b byte D2H is one DMA on the library's side stream
        if design.n_b not in res_buf:
            res_buf[design.n_b] = ob.PinnedBuffer((design.n_b,))
        rb = res_buf[design.n_b].array
        if world == 1 or design.world > 1:       # one GPU, or a row shard (mode N: the library's collectives do the rest)
            return ob.bootstrap(design, reps, ref_kind=ref, norm=normv, seed=2026, residuals_out=rb)
        # mode R inside the library: replicate shard, NCCL all-gather of the statistics device to device, reduction on
        # every rank (ob_boot_opts.shard_replicates); residuals are fetched once, on rank 0
        return ob.bootstrap(design, reps, ref_kind=ref, norm=normv, seed=2026, shard_replicates=True,
                            want_residuals=rank == 0, residuals_out=rb if rank == 0 else None)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    design = pack()
    pack_ms = design.pack_timings()
    for _ in range(args.warmup):
        out = step(design)

    # ---- device-resident leg: K steps, CUDA events on the library's stream are summed inside (ms_total);
    #      the wall bracket below (barrier + synchronize on both sides) is what is reported ----
    sampler = ClockSampler(local)
    sampler.start()
    sync()
    t0 = time.perf_counter()
    gram_ms, total_ms, launches = [], [], 0
    for _ in range(args.steps):
        sampler.step_begins()
        out = step(design)
        gram_ms.append(out["timings_ms"]["gram_main"] if "gram_main" in out["timings_ms"] else out["timings_ms"]["gram"])
        total_ms.append(out["timings_ms"]["total"])
        launches += out["gpu_launches"]
    sync()
    dt = time.perf_counter() - t0
    sampler.stop_flag.set()
    sampler.step_flag.set()
    sampler.join()
    if args.dump_outputs and rank == 0:
        # here, before the legs below write into the same page-locked residuals buffer
        sampled = dump_outputs(out, args.dump_outputs)
        print(f"bench: outputs of timed step {args.steps} in {args.dump_outputs}"
              + (f"; sampled (written, of): {sampled}" if sampled else ""), file=sys.stderr, flush=True)
    design.close()

    # ---- end-to-end leg: pinned host columns -> H2D + pack + bootstrap + D2H, every step ----
    for _ in range(min(args.warmup, 2)):       # untimed: lets the allocator pools reach their steady state
        dsg = pack(True, e2e=True); step(dsg); dsg.close()
    sync()
    t1 = time.perf_counter()
    e2e_ms = []
    for _ in range(args.steps):
        ts = time.perf_counter()
        dsg = pack(True, e2e=True)
        out_e = step(dsg)
        dsg.close()
        e2e_ms.append((time.perf_counter() - ts) * 1e3)
    sync()
    dt_e = time.perf_counter() - t1
    if not (world > 1 and not shard_rows):
        dsg = pack(False)                         # one synchronous pack, untimed: the upload and the pack kernels alone,
        pack_ms = dsg.pack_timings()              # steady state (the very first pack pays for the memory pools)
        dsg.close()
    # ---- outcome-refresh leg (SURVEY 8f-2: callers re-running on the same X with another y): 8 n bytes H2D per step ----
    refresh = None
    if world == 1 and rif_tau is None:
        dsg = pack()
        y_pin = pinned["y"].numpy()
        dsg.update_outcome(y_pin)
        step(dsg)
        sync()
        t2 = time.perf_counter()
        for _ in range(args.steps):
            dsg.update_outcome(y_pin)
            step(dsg)
        sync()
        refresh = time.perf_counter() - t2
        dsg.close()
    S = out["S"]
    d2h = 8 * (S * 6 + 3 * K + 1) + 8 * (out["residuals_b"].size if "residuals_b" in out else 0)

    times = torch.tensor([dt, dt_e, refresh or 0.0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e, refresh = times.tolist()

    # config 4 (BASELINE configs[3]: tau = 0.1 / 0.5 / 0.9): the sweep as three runs on a design packed once, and as ONE
    # pass with three RIF outcome columns (ob_design_apply_rif_multi) -- both accountings of SURVEY 8d
    sweep = None
    if name.startswith("config4"):
        taus = (0.1, 0.5, 0.9)
        dsg = pack()

        def run_sweep(multi):
            sync()
            t = time.perf_counter()
            if multi:
                dsg.apply_rif_multi(taus)
                o = ob.bootstrap(dsg, reps, ref_kind=ref, norm=normv, seed=2026, want_residuals=False, shard_replicates=world > 1)
            else:
                for tau in taus:
                    dsg.apply_rif(tau)
                    o = ob.bootstrap(dsg, reps, ref_kind=ref, norm=normv, seed=2026, want_residuals=False, shard_replicates=world > 1)
            sync()
            return time.perf_counter() - t, o
        run_sweep(False); run_sweep(True)                    # warm-up of both shapes
        t3, o3 = min((run_sweep(False) for _ in range(3)), key=lambda r: r[0])
        t1, o1 = min((run_sweep(True) for _ in range(3)), key=lambda r: r[0])
        dsg.close()
        tt = torch.tensor([t3, t1], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t3, t1 = tt.tolist()
        Ksw = K
        sweep = {"taus": list(taus), "reps_per_tau": reps,
                 "three_runs": {"seconds": t3, "fits_per_s": 3 * reps / t3, "gram_columns": 3 * (Ksw * (Ksw + 1) // 2 + Ksw),
                                "what": "apply_rif(tau) + ob_bootstrap_run per quantile on a design packed once"},
                 "one_pass": {"seconds": t1, "fits_per_s": 3 * reps / t1, "gram_columns": Ksw * (Ksw + 1) // 2 + 3 * Ksw,
                              "gram_ms": o1["timings_ms"]["gram_main"],
                              "what": "apply_rif_multi(taus) + ONE ob_bootstrap_run: X'WX contracted once, three X'Wy column sets"},
                 "speedup": t3 / t1,
                 "identical": bool(np.array_equal(np.nan_to_num(o1["std_err"][2], nan=-7.0), np.nan_to_num(o3["std_err"], nan=-7.0)))}

    # the other multi-GPU configurations of BASELINE.json at the same N, so that the driver's record holds them
    also = None
    if world > 1 and args.also != "off" and name.startswith("config3"):
        del pinned
        d_keep = {k: d[k] for k in ("n", "cont", "cat_codes", "cat_levels", "weights")}     # hbm_stage_rooflines needs the shapes only
        d_keep["cont"] = [c[:1] for c in d_keep["cont"]]; d_keep["cat_codes"] = [c[:1] for c in d_keep["cat_codes"]]
        d_keep["weights"] = None if d_keep["weights"] is None else d_keep["weights"][:1]
        d = d_keep
        also = {}
        also["config4_n5M_k30_rif_B1000"] = measure_also("config4_n5M_k30_rif_B1000", ob, obd, ctx, torch, dist, rank, world, local,
                                                          shard_rows=False, rif_tau=0.5, steps=3)
        try:
            also["machado_mata"] = measure_machado_mata_sharded(ob, ctx, torch, dist, world)
        except Exception as e:                         # never lose the headline line to a side measurement
            also["machado_mata"] = {"error": f"{type(e).__name__}: {e}"}
        if world & (world - 1) == 0:
            also["config5_n100M_k16_B10000"] = measure_also("config5_n100M_k16_B10000", ob, obd, ctx, torch, dist, rank, world, local,
                                                             shard_rows=True, rif_tau=None, steps=2)

    if rank == 0:
        flops, P = algorithmic_flops(n, K, reps)
        flops_rank = flops / world                        # replicates are sharded: per-launch algorithmic work
        g_ms = float(np.mean(gram_ms))
        traffic, traffic_csv = measured_gram_traffic(name, world)
        achieved = flops_rank / (g_ms * 1e-3) / 1e12
        line = {"metric": "bootstrap_reps_per_sec", "value": reps * args.steps / dt, "unit": "reps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_dict(name, world, shard_rows, rif_tau),
                "e2e": {"value": reps * args.steps / dt_e, "unit": "reps/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h),
                        "path": ("ob_design_pack_async (chunked upload + pack on the copy stream, under the replicate generation and "
                                 "the first Gram launch) -> ob_bootstrap_run" if world == 1 and rif_tau is None else
                                 "per rank: ob_design_pack_row_shard_async (1/N of the frame uploaded in chunks, rows packed straight into "
                                 "the rank's row shard, boundary rows exchanged over NVLink) overlapped with the row-sharded "
                                 "ob_bootstrap_run (mode N)" if e2e_rowshard else
                                 "per rank: upload 1/N of the frame -> pack -> ob_design_allgather_rows (NVLink) -> replicate-sharded "
                                 "ob_bootstrap_run (mode R)" if world > 1 and not shard_rows else
                                 "ob_design_pack -> ob_bootstrap_run")},
                "nccl_selftest": selftest,
                "also": also,
                "quantile_sweep": sweep,
                "e2e_outcome_refresh": None if not (refresh and world == 1) else
                    {"value": reps * args.steps / refresh, "unit": "reps/s", "h2d_bytes_per_step": int(8 * n),
                     "what": "ob_design_update_outcome (new y from pinned host memory, X resident) + bootstrap per step"},
                "gpu_launches": int(launches),
                "device_ms_per_step": float(np.mean(total_ms)),
                "device_step_ms": [round(float(x), 1) for x in total_ms],       # every timed step: library events, whole call
                "gram_step_ms": [round(float(x), 1) for x in gram_ms],          # ... and its Gram launch
                "timing": "value: host clock between barrier + cuda synchronize brackets around exactly K steps, max over ranks "
                          "(the library runs on its own stream, so torch.cuda.Event would not see it); device_ms_per_step and "
                          "stage_ms: CUDA events recorded by the library on that stream",
                "roofline": {"bound": "tensor", "kernel": "gram_ws_kernel (FP64 DMMA.8x8x4, warp-specialised)", "achieved": achieved,
                             "peak": FP64_DMMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / FP64_DMMA_PEAK_TFLOPS,
                             "frac_of_cublas_dgemm": achieved / FP64_CUBLAS_DGEMM_TFLOPS,
                             "peak_source": "measured on this pool: FP64 DMMA issue peak, profiles/r01_fp64_peaks.json "
                                            "(MEASURED_PEAKS.json has no fp64 entry); cuBLAS DGEMM 35.4",
                             "launch_ms": g_ms, "flop_per_launch": flops_rank,
                             "traffic": traffic,
                             "traffic_source": None if traffic is None else
                                 f"ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch of this command on this "
                                 f"build of the kernel ({traffic_csv}; profiles/gram_traffic.json, keyed by the kernel-source hash)"},
                "stage_ms": dict({k: float(v) for k, v in out["timings_ms"].items()},
                                 other=float(out["timings_ms"]["total"] - sum(out["timings_ms"][k] for k in
                                                                             ("counts", "gram", "solve", "reduce")))),
                "hbm_stages": hbm_stage_rooflines(d, K, reps, world, shard_rows, out, pack_ms),
                "e2e_step_ms": [round(x, 1) for x in e2e_ms],
                "clocks": sampler.summary(),
                "n_ok": int(out["n_ok"])}
        if world == 1 and not args.no_cpu_baseline:
            cores, threads = host_threads_and_sample(d, K)
            reps_cpu = max(threads - 1, 1)
            dense = dense_for_cpu(d, rif_tau)
            cpu_baseline(dense, len(d["cont"]), norm, ref, threads, reps_cpu)        # untimed: first-touch of the thread buffers
            v, cdt, _ = cpu_baseline(dense, len(d["cont"]), norm, ref, threads, reps_cpu)
            line["cpu_baseline"] = {"value": v, "unit": "reps/s", "cores": threads, "kind": "port",
                                    "sample": f"{reps_cpu} replicates + point pass, full n, {cdt:.1f} s on {threads} of {cores} cores"}
            line["readme_shape"] = readme_calibration_cpu(min(cores, 64))
            line["readme_shape"]["gpu_seconds_e2e"] = readme_shape_gpu(ob, ctx)
            if name.startswith("config3"):
                try:
                    line["machado_mata"] = measure_machado_mata(ob, ctx, threads)
                except Exception as e:                     # never lose the headline line to the side measurement
                    line["machado_mata"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
