"""Bayesian bootstrap (ob_bootstrap_run_bayes): Dirichlet-weighted replicates on the FP64 Gram contraction.

Replicate b gives row i of group g the weight pi_i = n_g E_i / sum_g E with E_i ~ Exp(1), and is the reference's single
pass (builder.rs:420-699) with the multiplicity replaced by pi_i.  The oracle helper below states exactly that: per
replicate, pyoracle.single_pass in precise mode with per-row weights pi_i w_i (pi_i on an unweighted design), whose weighted
branch gives the WLS fits, the means sum(pi w x) / sum(pi w), the Cotton / Weighted omega from sum_g pi w (= n_g on an
unweighted design) and the Pooled stack of the two weighted groups.

CPU part: the helper with E = 1 is the point pass, and with E = a multinomial count vector it is the oracle's index-stream
replicate of that draw; the fp32 width limit restated from gram_ws_smem; the builder and CLI options.
GPU part: oracle parity under explicit fp32 streams; native equals explicit; the native stream's distribution; batching,
mode R and mode N invariance; the fp32 Gram variant cell by cell; the rare-level case the row bootstrap drops; the Gram
cache; the refusals; the builder and the CLI.
"""
import threading

import numpy as np
import pytest

from helpers import relerr, worst
import test_gram_exact as ge
from test_cluster_bootstrap import _builder_frame, _cli_path, _dense, _frame, _spec

TOL = 1e-10
KEYS = ("point_stats", "rep_stats", "rep_status", "rep_beta_a", "rep_beta_b", "std_err", "p_value", "ci_lower", "ci_upper",
        "t_stat", "residuals_b", "total_gap_multi", "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")
INVALID, UNSUPPORTED = 7, 11


def oracle_bayes_run(orc, spec, data, wt_a, wt_b):
    """The Bayesian bootstrap on the CPU oracle: the point pass, then per replicate the single pass with per-row weights
    pi_i w_i, pi = n_g E / sum_g E (E in float64 from the given stream), then the reduction."""
    Xa, ya, wa, Xb, yb, wb = data
    point = orc.single_pass(spec, Xa, ya, wa, Xb, yb, wb)
    reps, S, K = wt_a.shape[0], spec.n_stats, spec.K
    stats, status = np.full((reps, S), np.nan), np.zeros(reps, dtype=np.int32)
    ba, bb = np.full((reps, K), np.nan), np.full((reps, K), np.nan)
    na, nb = len(ya), len(yb)
    for b in range(reps):
        ea, eb = np.asarray(wt_a[b], np.float64), np.asarray(wt_b[b], np.float64)
        pa, pb = na * ea / ea.sum(), nb * eb / eb.sum()
        try:
            r = orc.single_pass(spec, Xa, ya, pa if wa is None else pa * wa, Xb, yb, pb if wb is None else pb * wb,
                                want_resid=False)
        except orc.OracleError as e:
            status[b] = e.code
            continue
        stats[b], ba[b], bb[b] = r["stats"], r["beta_a"], r["beta_b"]
    red = orc.reduce(stats, status, point["stats"])
    return dict(point=point, rep_stats=stats, rep_status=status, rep_beta_a=ba, rep_beta_b=bb, **red)


def _streams(seed, reps, na, nb):
    rng = np.random.default_rng(seed)
    f = lambda n: np.maximum(rng.exponential(size=(reps, n)), 1e-6).astype(np.float32)  # noqa: E731
    return f(na), f(nb)


# ------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ref_kind", [0, 2, 3])
def test_unit_weights_give_the_point_pass(orc, weighted, ref_kind):
    d = _frame(500, 3, weighted, cat_levels=(3, 4))
    data, A, B = _dense(d)
    spec = _spec(orc, d, ref_kind, yun=True)
    reps = 4
    got = oracle_bayes_run(orc, spec, data, np.ones((reps, int(A.sum())), np.float32), np.ones((reps, int(B.sum())), np.float32))
    for b in range(reps):
        assert relerr(got["rep_stats"][b], got["point"]["stats"]) <= 1e-12


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ref_kind", [0, 1, 2, 3])
def test_count_weights_give_the_index_stream_replicate(orc, weighted, ref_kind):
    """E = the multinomial counts of a draw: pi = n_g c / n_g = c, the row bootstrap's replicate of that draw."""
    d = _frame(400, 11, weighted, cat_levels=(3,))
    data, A, B = _dense(d)
    spec = _spec(orc, d, ref_kind, yun=True)
    reps, na, nb = 12, int(A.sum()), int(B.sum())
    ia, ib = orc.index_stream(5, reps, 0, na), orc.index_stream(5, reps, 1, nb)
    ca = np.stack([np.bincount(ia[b], minlength=na) for b in range(reps)]).astype(np.float32)
    cb = np.stack([np.bincount(ib[b], minlength=nb) for b in range(reps)]).astype(np.float32)
    got = oracle_bayes_run(orc, spec, data, ca, cb)
    want = orc.run(spec, *data, reps, idx_a=ia, idx_b=ib)
    np.testing.assert_array_equal(got["rep_status"], want["rep_status"])
    for k in ("rep_stats", "rep_beta_a", "rep_beta_b"):
        assert relerr(got[k], want[k]) <= 1e-12, (k, worst(got[k], want[k]))
    for k in ("se", "p", "ci_lo", "ci_hi"):
        assert relerr(got[k], want[k]) <= 1e-12, k


def test_fp32_width_limit():
    """gram_fits(ldx, 4) and the fp32 ring choice, restated from gram_ws_smem: ring 2 up to ldx 236 (K + outcomes <= 236),
    ring 3 up to ldx 84 (every specialised stride but 92)."""
    assert ge.ws_smem(236, 4, 2) == 231_472 <= ge.SMEM_MAX < ge.ws_smem(244, 4, 2)
    assert ge.fits(236, 4) and not ge.fits(244, 4)
    assert ge.ring_depth(84, 4) == 3 and ge.ring_depth(92, 4) == 2
    assert ge.design_ldx(236) == 236 and ge.design_ldx(237) == 244


def test_builder_and_cli_options():
    import subprocess
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import _native, builder
    _native.build()
    assert {"ob_bootstrap_run_bayes", "ob_debug_bayes_weights"} <= set(_native.SYMBOLS)
    assert "ob_builder_bayesian" in builder.BUILDER_SYMBOLS
    frame, *_ = _builder_frame(50, 1, 5)
    b = ob.OaxacaBuilder(frame, "wage", "gender", "F").predictors(["x1", "x2"])
    assert b.bayesian_bootstrap() is b and b.bayesian_bootstrap(False) is b
    for args in (["--bootstrap-scheme", "poisson"], ["--bootstrap-scheme", "Bayes"],
                 ["--bootstrap-scheme", "bayes", "--analysis-type", "quantile"]):
        r = subprocess.run([_cli_path(), "--data", "nope.csv", "--outcome", "y", "--group", "g", "--reference", "r", *args],
                           capture_output=True, text=True)
        assert r.returncode == 2 and "bootstrap-scheme" in r.stderr, (args, r.stderr)


# ------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def ctx():
    import oaxaca_blinder_rs_b200 as ob
    c = ob.Context(0)
    yield c
    c.close()


def _pack(ctx, d):
    import oaxaca_blinder_rs_b200 as ob
    return ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])


def _assert_equal(a, b, what=""):
    for k in KEYS:
        if k in a or k in b:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what} {k}")
    assert a["n_ok"] == b["n_ok"]


def _check_parity(gpu, want, what, t=None):
    sel = (lambda x: x) if t is None else (lambda x: x[t])
    rs = gpu["rep_stats"] if t is None else gpu["rep_stats"][:, t]
    np.testing.assert_array_equal(gpu["rep_status"], want["rep_status"], err_msg=what)
    assert relerr(sel(gpu["point_stats"]), want["point"]["stats"]) <= TOL, what
    assert relerr(rs, want["rep_stats"]) <= TOL, (what, worst(rs, want["rep_stats"]))
    for kg, kw in (("rep_beta_a", "rep_beta_a"), ("rep_beta_b", "rep_beta_b")):
        g = gpu[kg] if t is None else gpu[kg][:, t]
        assert relerr(g, want[kw]) <= TOL, (what, kg, worst(g, want[kw]))
    for kg, kw in (("std_err", "se"), ("p_value", "p"), ("ci_lower", "ci_lo"), ("ci_upper", "ci_hi")):
        assert relerr(sel(gpu[kg]), want[kw]) <= TOL, (what, kg, worst(sel(gpu[kg]), want[kw]))
    assert gpu["n_ok"] == want["n_ok"]


# ------------------------------------------------------------------------------------------- GPU: oracle parity
@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ref_kind", [0, 1, 2, 3])
def test_oracle_parity_under_explicit_streams(orc, ctx, weighted, ref_kind):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d = _frame(1500, 21 + ref_kind, weighted, n_cont=3, cat_levels=(3, 4))
    data, A, B = _dense(d)
    spec = _spec(orc, d, ref_kind, yun=True)
    reps = 40
    wa, wb = _streams(ref_kind, reps, int(A.sum()), int(B.sum()))
    des = _pack(ctx, d)
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    kw = dict(ref_kind=ref_kind, norm=norm, want_rep=True, scheme="bayes", wt_a=wa, wt_b=wb)
    gpu = ob.bootstrap(des, reps, **kw)
    want = oracle_bayes_run(orc, spec, data, wa, wb)
    _check_parity(gpu, want, f"ref {ref_kind} weighted {weighted}")
    # an explicit stream over three panels, one panel per batch: the same numbers bit for bit as one batch
    kw.update(wt_a=np.tile(wa, (8, 1))[:300], wt_b=np.tile(wb, (8, 1))[:300])
    _assert_equal(ob.bootstrap(des, 300, max_workspace_bytes=1, **kw), ob.bootstrap(des, 300, **kw), "batched")
    des.close()


@pytest.mark.gpu
def test_oracle_parity_three_rif_outcomes_multi_batch(orc, ctx):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    taus = (0.1, 0.5, 0.9)
    d = synth.make_wage(6000, 4, cat_levels=(3,), weights=True, seed=9)
    Xa, ya, wa_, Xb, yb, wb_ = synth.dense_design(d)
    reps = 140                                     # two panels; max_workspace_bytes = 1: one panel per batch
    wa, wb = _streams(2, reps, len(ya), len(yb))
    des = _pack(ctx, d)
    des.apply_rif_multi(taus)
    norm = synth.norm_spec(d)
    gpu = ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, norm=[ob.NormVar(m, i) for m, i in norm], want_rep=True,
                       scheme="bayes", wt_a=wa, wt_b=wb, max_workspace_bytes=1)
    des.close()
    spec = orc.Spec(K=Xa.shape[1], n_cont=4, ref_kind=orc.REF_POOLED, norm=[orc.NormVar(m, i) for m, i in norm])
    for t, tau in enumerate(taus):
        want = oracle_bayes_run(orc, spec, (Xa, orc.rif(ya, tau), wa_, Xb, orc.rif(yb, tau), wb_), wa, wb)
        _check_parity(gpu, want, f"tau {tau}", t)


@pytest.mark.gpu
@pytest.mark.parametrize("n_cont,weighted", [(16, True),     # K + 1 = 18 -> ldx 20: a specialised stride (ring 3)
                                             (2, False),     # K + 1 = 4 -> ldx 4: run-time stride, ring 3
                                             (234, True)])   # K + 1 = 236: run-time stride, ring 2, the fp32 width limit
def test_oracle_parity_across_kernel_variants(orc, ctx, n_cont, weighted):
    import oaxaca_blinder_rs_b200 as ob
    # the wide case with about 13 rows per column, as test_gpu_parity's wide designs: fewer rows leave the 235-column
    # systems too ill-conditioned for ten digits in any fp64 evaluation
    d = _frame(1300 if n_cont < 200 else 6000, 40 + n_cont, weighted, n_cont=n_cont, cat_levels=())
    data, A, B = _dense(d)
    spec = _spec(orc, d, 2, yun=False)
    reps = 30 if n_cont < 200 else 8
    wa, wb = _streams(n_cont, reps, int(A.sum()), int(B.sum()))
    des = _pack(ctx, d)
    gpu = ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, want_rep=True, scheme="bayes", wt_a=wa, wt_b=wb)
    des.close()
    _check_parity(gpu, oracle_bayes_run(orc, spec, data, wa, wb), f"n_cont {n_cont}")


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_native_equals_explicit_readback(ctx, weighted):
    import oaxaca_blinder_rs_b200 as ob
    d = _frame(5000, 31, weighted, n_cont=3, cat_levels=(4,))
    des = _pack(ctx, d)
    reps, seed = 150, 99
    wa = np.stack([des.debug_bayes_weights(seed, r, 0) for r in range(reps)])
    wb = np.stack([des.debug_bayes_weights(seed, r, 1) for r in range(reps)])
    kw = dict(ref_kind=ob.REF_WEIGHTED, want_rep=True, scheme="bayes")
    _assert_equal(ob.bootstrap(des, reps, seed=seed, **kw), ob.bootstrap(des, reps, wt_a=wa, wt_b=wb, **kw), "native vs explicit")
    des.close()


@pytest.mark.gpu
def test_native_stream_is_exp1_and_independent(ctx):
    from scipy import stats
    d = _frame(40_000, 5, False, n_cont=2, cat_levels=())
    des = _pack(ctx, d)
    n = min(des.n_a, des.n_b)
    e = {(r, g): des.debug_bayes_weights(17, r, g).astype(np.float64) for r in range(4) for g in (0, 1)}
    for (r, g), v in e.items():
        assert v.dtype == np.float64 and np.all(v > 0) and np.all(np.isfinite(v))
        m = len(v)
        assert abs(v.mean() - 1.0) < 5 / np.sqrt(m), (r, g, v.mean())
        assert abs(v.var() - 1.0) < 0.1, (r, g, v.var())
        assert stats.kstest(v, "expon").pvalue > 1e-4, (r, g)
    pairs = [((0, 0), (1, 0)), ((2, 1), (3, 1)), ((0, 0), (0, 1)), ((1, 0), (1, 1))]
    for x, y in pairs:
        c = np.corrcoef(e[x][:n], e[y][:n])[0, 1]
        assert abs(c) < 5 / np.sqrt(n), (x, y, c)
    assert not np.array_equal(des.debug_bayes_weights(18, 0, 0), e[(0, 0)])       # another seed, another stream
    des.close()


# ------------------------------------------------------------------------------------------- GPU: invariance
def _in_process(world, make, call):
    from oaxaca_blinder_rs_b200 import core
    import oaxaca_blinder_rs_b200 as ob
    grp = core.LocalGroup(world)
    outs, errs = [None] * world, [None] * world

    def work(r):
        try:
            c = ob.Context(0)
            c.init_local(grp, r)
            dd = make(c, r)
            outs[r] = call(dd)
            dd.close(); c.close()
        except Exception as e:  # noqa: BLE001
            errs[r] = e
    ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=600)
    assert all(e is None for e in errs), errs
    return outs


@pytest.mark.gpu
def test_batching_and_replicate_sharding_invariance(ctx):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d = _frame(30_000, 61, True, n_cont=4, cat_levels=(4,))
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    reps = 300
    kw = dict(seed=5, want_rep=True, ref_kind=ob.REF_POOLED, norm=norm, scheme="bayes")
    des = _pack(ctx, d)
    ref = ob.bootstrap(des, reps, **kw)
    assert ref["n_ok"] == reps
    _assert_equal(ob.bootstrap(des, reps, max_workspace_bytes=1, **kw), ref, "batched")
    des.close()
    for world in (2, 3):
        for o in _in_process(world, lambda c, r: _pack(c, d), lambda dd: ob.bootstrap(dd, reps, shard_replicates=True, **kw)):
            _assert_equal(o, ref, f"mode R x{world}")


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_row_sharding_invariance_weighted(ctx, world):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import distributed as obd, synth
    d = synth.make_wage(60_000, 4, cat_levels=(4,), weights=True, seed=11)
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    reps = 300
    kw = dict(seed=77, want_rep=True, ref_kind=ob.REF_WEIGHTED, norm=norm, scheme="bayes")
    des = _pack(ctx, d)
    one = ob.bootstrap(des, reps, **kw)
    pooled = ob.bootstrap(des, reps, **{**kw, "ref_kind": ob.REF_POOLED})
    des.close()
    for k, ref in ((ob.REF_WEIGHTED, one), (ob.REF_POOLED, pooled)):
        outs = _in_process(world, lambda c, r: obd.pack_row_shard(c, d, r, world),
                           lambda dd: ob.bootstrap(dd, reps, max_workspace_bytes=16_000_000, **{**kw, "ref_kind": k}))
        for o in outs:
            for key in ("point_stats", "rep_stats", "rep_status", "rep_beta_a", "rep_beta_b", "std_err", "ci_lower", "ci_upper", "p_value"):
                np.testing.assert_array_equal(o[key], ref[key], err_msg=f"mode N x{world} ref {k} {key}")


# ------------------------------------------------------------------------------------------- GPU: fp32 Gram cells
CELL_CASES = [c for c in ge.CASES if c.kind == "plain" and ge.fits(ge.design_ldx(c.K + c.T), 4) and
              (c.name.startswith("ldx") or c.name.startswith("tail"))]


def test_cell_cases_cover_the_fp32_variants():
    seen = {(ge.design_ldx(c.K + c.T), ge.ring_depth(ge.design_ldx(c.K + c.T), 4)) for c in CELL_CASES}
    assert {ldx for ldx, _ in seen} >= set(ge.SPECIALISED)
    assert any(ring == 3 and ldx not in ge.SPECIALISED for ldx, ring in seen)
    assert any(ring == 2 and ldx not in ge.SPECIALISED for ldx, ring in seen)
    assert {c.name for c in CELL_CASES} >= {"tail1", "tail2", "tail3"}


def _cell_reference(X, Y, w, E):
    """Per slot: the cells in the cache layout as a long-double sum (64-bit significand: its own error is below 2^-11
    of the bound checked against) and the bound depth 2^-53 sum |terms| of any fp64 summation order, depth = n + 2.
    Every term is exact in fp64: fp32 E times a quarter-integer weight times integer products."""
    K = X.shape[1]
    iu = np.triu_indices(K)
    V = np.concatenate([X, Y], axis=1)
    cw = (E * (1.0 if w is None else w)).astype(np.longdouble)
    Vl = V.astype(np.longdouble)
    Z = np.concatenate([(Vl[:, :K, None] * Vl[:, None, :K])[:, iu[0], iu[1]],
                        (Vl[:, :K, None] * Vl[:, None, K:]).reshape(len(V), -1), (Vl[:, K] * Vl[:, K])[:, None]], axis=1)
    ref = cw @ Z
    bound = (len(V) + 2) * 2.0 ** -53 * (np.abs(cw) @ np.abs(Z))
    nx = iu[0].size
    return ref[:, :nx], ref[:, nx:], bound[:, :nx], bound[:, nx:]


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c.name for c in CELL_CASES])
def test_fp32_cells_within_the_rounding_bound(name, ctx):
    import oaxaca_blinder_rs_b200 as ob
    case = ge.BY_NAME[name]
    d = ge.frame(case)
    des = _pack(ctx, d)
    host = ge.host_design(d)
    seed = 4243
    reps_list = (20, 50, 80, 110) if name.startswith("tail") else (20,)
    maxreps = max(reps_list)
    E = [np.concatenate([np.ones((1, n), np.float32), np.stack([des.debug_bayes_weights(seed, r, g) for r in range(maxreps)])])
         for g, n in enumerate((des.n_a, des.n_b))]
    for reps in reps_list:
        cache = ob.GramCache(ctx)
        r = ob.bootstrap(des, reps, seed=seed, want_residuals=False, cache=cache, scheme="bayes")
        assert r["cache_use"] == ob.CACHE_FILLED
        cells = cache.debug_cells()
        assert cells["count_bytes"] == 4 and cells["slots"] == reps + 1
        for g, (X, Y, w) in enumerate(host):
            xx, yy, bx, by = _cell_reference(X, Y, w, E[g][:reps + 1].astype(np.float64))
            for got, want, bd, what in ((cells["xx"][g], xx, bx, "X'WX"), (cells["yy"][g], yy, by, "X'Wy")):
                err = np.abs(got.astype(np.longdouble) - want)
                bad = np.argwhere(err > bd)
                assert bad.size == 0, f"{name} reps {reps} {what} group {g}: {len(bad)} cells outside the bound, first {bad[:4].tolist()}"
        cache.close()
    des.close()


# ------------------------------------------------------------------------------------------- GPU: rare level, cache, refusals
@pytest.mark.gpu
def test_rare_level_is_never_lost(ctx):
    import oaxaca_blinder_rs_b200 as ob
    rng = np.random.default_rng(8)
    n = 3000
    group = (rng.random(n) < 0.5).astype(np.uint8)
    lvl = rng.integers(0, 3, n).astype(np.int32)
    a_rows, b_rows = np.flatnonzero(group == 0), np.flatnonzero(group == 1)
    lvl[a_rows[:2]] = 3                             # level 3 has two rows in group A (and many in group B)
    lvl[b_rows[:300]] = 3
    x = rng.standard_normal(n)
    y = 1.0 + 0.5 * x + 0.2 * lvl + 0.3 * group + 0.4 * rng.standard_normal(n)
    des = ob.Design.pack(ctx, [x], [lvl], [4], y, None, group)
    reps = 300
    row = ob.bootstrap(des, reps, seed=3, want_rep=True)
    bay = ob.bootstrap(des, reps, seed=3, want_rep=True, scheme="bayes")
    des.close()
    assert row["n_ok"] < reps                        # about e^-2 of the row replicates miss the level
    assert bay["n_ok"] == reps and np.all(bay["rep_status"] == 0)
    assert np.all(np.isfinite(bay["std_err"]))


@pytest.mark.gpu
def test_gram_cache_uses_and_scheme_switch(ctx):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d = _frame(20_000, 71, True, n_cont=4, cat_levels=(3,))
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    reps = 200
    des = _pack(ctx, d)
    kw = dict(seed=12, want_rep=True, norm=norm, scheme="bayes")
    cache = ob.GramCache(ctx)
    filled = ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, cache=cache, **kw)
    assert filled["cache_use"] == ob.CACHE_FILLED
    _assert_equal(filled, ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, **kw), "filled")
    solve = ob.bootstrap(des, reps, ref_kind=ob.REF_WEIGHTED, cache=cache, **kw)
    assert solve["cache_use"] == ob.CACHE_SOLVE_ONLY
    _assert_equal(solve, ob.bootstrap(des, reps, ref_kind=ob.REF_WEIGHTED, **kw), "solve only")
    des.update_outcome(d["outcome"] * 0.5 + d["cont"][0])
    outc = ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, cache=cache, **kw)
    assert outc["cache_use"] == ob.CACHE_OUTCOME_ONLY
    _assert_equal(outc, ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, **kw), "outcome only")
    # a row-bootstrap run on the same cache refills, and so does the Bayesian run after it
    rows = ob.bootstrap(des, reps, seed=12, want_rep=True, norm=norm, ref_kind=ob.REF_POOLED, cache=cache)
    assert rows["cache_use"] == ob.CACHE_FILLED
    assert ob.bootstrap(des, reps, ref_kind=ob.REF_POOLED, cache=cache, **kw)["cache_use"] == ob.CACHE_FILLED
    cache.close()
    des.close()


@pytest.mark.gpu
def test_refusals(ctx):
    import oaxaca_blinder_rs_b200 as ob
    d = _frame(2000, 91)
    des = _pack(ctx, d)
    na, nb, reps = des.n_a, des.n_b, 4
    wa, wb = _streams(0, reps, na, nb)

    def refused(code, text, **kw):
        with pytest.raises(ob.OaxacaError) as e:
            ob.bootstrap(des, reps, scheme="bayes", **kw)
        assert e.value.code == code and text in str(e.value), (e.value.code, str(e.value))
    ia = np.zeros((reps, na), np.uint32)
    ib = np.zeros((reps, nb), np.uint32)
    refused(INVALID, "index stream", idx_a=ia, idx_b=ib)
    refused(INVALID, "count_bits", count_bits=8)
    bad = wa.copy(); bad[1, 3] = 0.0
    refused(INVALID, "positive normal", wt_a=bad, wt_b=wb)
    refused(UNSUPPORTED, "cannot be keyed", wt_a=wa, wt_b=wb, cache=ob.GramCache(ctx))
    des.attach_clusters(np.arange(na + nb, dtype=np.int32) % 50, strata="group")
    refused(UNSUPPORTED, "clustered")
    des.attach_clusters(None, strata=None)
    des.attach_selection((np.asarray(d["cont"][1]) > 0).astype(float), [d["cont"][0]])
    refused(UNSUPPORTED, "selection equation")
    des.close()
    wide = _frame(1200, 5, False, n_cont=236, cat_levels=())       # K + outcome = 238 > 236
    des = _pack(ctx, wide)
    refused(UNSUPPORTED, "236")
    assert ob.bootstrap(des, 2, seed=1)["n_ok"] >= 0                # the row bootstrap still takes it
    des.close()


# ------------------------------------------------------------------------------------------- GPU: builders and CLI
@pytest.mark.gpu
def test_builder_and_cli_end_to_end(ctx, tmp_path):
    import json
    import subprocess
    import oaxaca_blinder_rs_b200 as ob
    n = 3000
    frame, _, _, _ = _builder_frame(n, 23, 150)

    def builder():
        return (ob.OaxacaBuilder(frame, "wage", "gender", "F").predictors(["x1", "x2"]).categorical_predictors(["sector"])
                .bootstrap_reps(200).seed(77).bayesian_bootstrap())
    r = builder().run()
    assert r.bootstrap_scheme == "bayes" and "Bayesian" in r.summary()
    plain = builder().bayesian_bootstrap(False).run()
    assert plain.bootstrap_scheme == "multinomial" and "Bayesian" not in plain.summary()
    assert r.total_gap == plain.total_gap and r.two_fold.aggregate[0].estimate == plain.two_fold.aggregate[0].estimate
    # the core call on the same design: group A = "M", the sector dummies s1, s2 in sorted order
    sector = np.array([int(s[1:]) for s in frame["sector"]], np.int32)
    group = (np.array(frame["gender"]) == "F").astype(np.uint8)
    des = ob.Design.pack(ctx, [frame["x1"], frame["x2"]], [sector], [3], frame["wage"], None, group)
    core = ob.bootstrap(des, 200, ref_kind=ob.REF_GROUP_A, seed=77, scheme="bayes")
    des.close()
    got = [c.std_err for c in r.two_fold.aggregate + r.three_fold.aggregate]
    assert relerr(got, core["std_err"][:5]) <= 1e-12
    assert [c.std_err for c in builder().run_outcomes(["wage", "x1"])[0].two_fold.aggregate] == \
           [c.std_err for c in r.two_fold.aggregate]
    assert builder().decompose_quantile(0.5).bootstrap_scheme == "bayes"
    path = tmp_path / "f.csv"
    with open(path, "w") as fh:
        fh.write("wage,x1,x2,sector,gender\n")
        for i in range(n):
            fh.write(f"{float(frame['wage'][i])!r},{float(frame['x1'][i])!r},{float(frame['x2'][i])!r},{frame['sector'][i]},"
                     f"{frame['gender'][i]}\n")
    out = tmp_path / "o.json"
    cmd = [_cli_path(), "--data", str(path), "--outcome", "wage", "--group", "gender", "--reference", "F", "--predictors", "x1,x2",
           "--categorical", "sector", "--bootstrap-reps", "200", "--seed", "77", "--ref-coeffs", "group-a", "--output-json", str(out)]
    p = subprocess.run(cmd + ["--bootstrap-scheme", "bayes"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "Bootstrap scheme: Bayesian" in p.stdout
    j = json.load(open(out))
    assert j["bootstrap_scheme"] == "bayes"
    assert relerr([c["std_err"] for c in j["two_fold"]["aggregate"]], [c.std_err for c in r.two_fold.aggregate]) <= 1e-15
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "Bootstrap scheme" not in p.stdout and "bootstrap_scheme" not in json.load(open(out))
