"""Cluster bootstrap (ob_design_attach_clusters): resample whole clusters instead of rows.

A clustered replicate is the reference's single pass (builder.rs:420-699) on the frame made of the drawn units' rows.  The
oracle helper below builds exactly that frame per replicate -- units in draw order, a unit's rows in frame order -- and
runs pyoracle.single_pass on it; a pass that fails is that replicate's status, as in the reference's bootstrap loop.

CPU part: the helper is the row bootstrap when every cluster is a single row.
GPU part: oracle parity under explicit unit streams; bit-identity with the row bootstrap for singleton clusters; the
native unit stream (constant counts within a unit, exact totals, batching / widening / replicate-sharding invariance, the
Binomial(M, 1/M) marginal); the Gram cache; the inflation of the SE under intra-cluster correlation; the refusals.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from helpers import relerr, worst

TOL = 1e-10
KEYS = ("point_stats", "rep_stats", "rep_status", "rep_beta_a", "rep_beta_b", "std_err", "p_value", "ci_lower", "ci_upper",
        "t_stat", "residuals_b", "total_gap_multi", "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")


# ------------------------------------------------------------------------------------------- data + oracle helper
def _frame(n, seed, weighted=False, n_cont=3, cat_levels=(3,)):
    from oaxaca_blinder_rs_b200 import synth
    return synth.make_wage(n, n_cont, cat_levels=cat_levels, weights=weighted, seed=seed)


def _dense(d):
    """The packed design restated on the host: intercept, continuous columns, dummies of levels 1.. of each categorical;
    group 0 = A, 1 = B, rows in frame order."""
    n = d["outcome"].shape[0]
    cols = [np.ones(n)] + [np.asarray(c, float) for c in d["cont"]]
    for codes, m in zip(d["cat_codes"], d["cat_levels"]):
        cols += [(np.asarray(codes) == lv).astype(float) for lv in range(1, m)]
    X = np.stack(cols, 1)
    y, w, g = d["outcome"], d["weights"], d["group"]
    A, B = g == 0, g == 1
    return (X[A], y[A], None if w is None else w[A], X[B], y[B], None if w is None else w[B]), A, B


def _spec(orc, d, ref_kind, yun):
    from oaxaca_blinder_rs_b200 import synth
    K = 1 + len(d["cont"]) + sum(m - 1 for m in d["cat_levels"])
    norm = [orc.NormVar(m, i) for m, i in synth.norm_spec(d)] if yun else []
    return orc.Spec(K=K, n_cont=len(d["cont"]), ref_kind=ref_kind, norm=norm)


def unit_rows(ca, cb, strata):
    """Rows (positions within the group, frame order) of every unit, units by ascending cluster code: (rows_a, rows_b),
    one list per stratum ("group": a unit is a (cluster, group) pair; "joint": one list of units over both groups)."""
    if strata == "group":
        return [np.flatnonzero(ca == u) for u in np.unique(ca)], [np.flatnonzero(cb == u) for u in np.unique(cb)]
    units = np.unique(np.concatenate([ca, cb]))
    return [np.flatnonzero(ca == u) for u in units], [np.flatnonzero(cb == u) for u in units]


def oracle_cluster_run(orc, spec, data, ca, cb, strata, idx_a, idx_b=None):
    """The clustered bootstrap on the CPU oracle: point pass on the full sample, then per replicate b the single pass on
    the drawn units' rows (units in draw order, a unit's rows in frame order; "joint": idx_a draws units for both groups),
    then the reduction."""
    Xa, ya, wa, Xb, yb, wb = data
    rows_a, rows_b = unit_rows(ca, cb, strata)
    if strata == "joint":
        assert idx_b is None
        idx_b = idx_a
    point = orc.single_pass(spec, Xa, ya, wa, Xb, yb, wb)
    reps, S, K = idx_a.shape[0], spec.n_stats, spec.K
    stats, status = np.full((reps, S), np.nan), np.zeros(reps, dtype=np.int32)
    ba, bb = np.full((reps, K), np.nan), np.full((reps, K), np.nan)

    def gather(rows, draws):
        parts = [rows[u] for u in draws]
        return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
    for b in range(reps):
        ia, ib = gather(rows_a, idx_a[b]), gather(rows_b, idx_b[b])
        try:
            r = orc.single_pass(spec, Xa[ia], ya[ia], None if wa is None else wa[ia], Xb[ib], yb[ib], None if wb is None else wb[ib],
                                want_resid=False)
        except orc.OracleError as e:
            status[b] = e.code
            continue
        stats[b], ba[b], bb[b] = r["stats"], r["beta_a"], r["beta_b"]
    red = orc.reduce(stats, status, point["stats"])
    return dict(point=point, rep_stats=stats, rep_status=status, rep_beta_a=ba, rep_beta_b=bb, **red)


# ------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ref_kind", [0, 2, 3])
def test_helper_with_singleton_clusters_is_the_row_bootstrap(orc, weighted, ref_kind):
    d = _frame(400, 11, weighted)
    data, A, B = _dense(d)
    spec = _spec(orc, d, ref_kind, yun=True)
    reps = 25
    rng = np.random.default_rng(3)
    na, nb = int(A.sum()), int(B.sum())
    ia = rng.integers(0, na, (reps, na)).astype(np.uint32)
    ib = rng.integers(0, nb, (reps, nb)).astype(np.uint32)
    codes = np.arange(na + nb)
    got = oracle_cluster_run(orc, spec, data, codes[:na], codes[na:], "group", ia, ib)
    want = orc.run(spec, *data, reps, idx_a=ia, idx_b=ib)
    np.testing.assert_array_equal(got["rep_status"], want["rep_status"])
    for k in ("rep_stats", "rep_beta_a", "rep_beta_b"):
        assert relerr(got[k], want[k]) <= 1e-12, k
    for k in ("se", "p", "ci_lo", "ci_hi", "t"):
        assert relerr(got[k], want[k]) <= 1e-12, k
    assert got["n_ok"] == want["n_ok"]


def test_unit_numbering_follows_ascending_codes():
    ca, cb = np.array([7, 2, 7, 5]), np.array([5, 9, 2])
    ra, rb = unit_rows(ca, cb, "group")
    assert [r.tolist() for r in ra] == [[1], [3], [0, 2]] and [r.tolist() for r in rb] == [[2], [0], [1]]
    ra, rb = unit_rows(ca, cb, "joint")              # units 2, 5, 7, 9
    assert [r.tolist() for r in ra] == [[1], [3], [0, 2], []] and [r.tolist() for r in rb] == [[2], [0], [], [1]]


# ------------------------------------------------------------------------------------------- GPU helpers
def _pack(ctx, d):
    import oaxaca_blinder_rs_b200 as ob
    return ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])


def _assert_equal(a, b):
    for k in KEYS:
        if k in a or k in b:
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["total_gap"] == b["total_gap"] and a["n_ok"] == b["n_ok"]


def _clustered_codes(n, n_clusters, seed):
    """Cluster codes drawn at random over the frame (clusters hold rows of both groups), with unused codes in between."""
    rng = np.random.default_rng(seed)
    return (3 * rng.integers(0, n_clusters, n) + 1).astype(np.int32)


def _compare(got, want, label):
    np.testing.assert_array_equal(got["rep_status"], want["rep_status"], err_msg=label)
    for k in ("rep_stats", "rep_beta_a", "rep_beta_b"):
        e = relerr(got[k], want[k])
        assert e <= TOL, (label, k, worst(got[k], want[k]))
    for gk, ok in (("std_err", "se"), ("p_value", "p"), ("ci_lower", "ci_lo"), ("ci_upper", "ci_hi"), ("t_stat", "t")):
        e = relerr(got[gk], want[ok])
        assert e <= TOL, (label, gk, worst(got[gk], want[ok]))
    assert relerr(got["point_stats"], want["point"]["stats"]) <= TOL
    assert got["n_ok"] == want["n_ok"], label


# ------------------------------------------------------------------------------------------- GPU: oracle parity
@pytest.mark.gpu
@pytest.mark.parametrize("strata", ["group", "joint"])
@pytest.mark.parametrize("weighted", [False, True])
def test_oracle_parity_under_unit_streams(orc, strata, weighted):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    n, reps = 3000, 60
    d = _frame(n, 21 + weighted, weighted)
    data, A, B = _dense(d)
    codes = _clustered_codes(n, 150, 5)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    des.attach_clusters(codes, strata=strata)
    cl = des.clusters
    rows_a, rows_b = unit_rows(codes[A], codes[B], strata)
    assert cl["strata"] == strata and cl["units_a"] == len(rows_a) and cl["units_b"] == len(rows_b)
    rng = np.random.default_rng(8)
    ia = rng.integers(0, cl["units_a"], (reps, cl["units_a"])).astype(np.uint32)
    ib = None if strata == "joint" else rng.integers(0, cl["units_b"], (reps, cl["units_b"])).astype(np.uint32)
    for ref_kind in (0, 1, 2, 3):
        for yun in (False, True):
            spec = _spec(orc, d, ref_kind, yun)
            norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)] if yun else []
            got = ob.bootstrap(des, reps, ref_kind=ref_kind, norm=norm, idx_a=ia, idx_b=ib, want_rep=True)
            want = oracle_cluster_run(orc, spec, data, codes[A], codes[B], strata, ia, ib)
            _compare(got, want, (strata, weighted, ref_kind, yun))
    des.close(); ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_joint_replicates_without_group_a_are_dropped_as_the_oracle_drops_them(orc, weighted):
    """Six clusters, group A lives in two of them: about one replicate in eleven draws no group-A row."""
    import oaxaca_blinder_rs_b200 as ob
    n, reps = 600, 120
    d = _frame(n, 31, weighted)
    rng = np.random.default_rng(4)
    g = d["group"]
    codes = np.where(g == 0, rng.integers(0, 2, n), rng.integers(0, 6, n)).astype(np.int32)
    data, A, B = _dense(d)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    des.attach_clusters(codes, strata="joint")
    M = des.clusters["units_a"]
    assert M == 6
    ia = rng.integers(0, M, (reps, M)).astype(np.uint32)
    for ref_kind in (0, 2, 3):
        spec = _spec(orc, d, ref_kind, yun=False)
        got = ob.bootstrap(des, reps, ref_kind=ref_kind, idx_a=ia, want_rep=True)
        want = oracle_cluster_run(orc, spec, data, codes[A], codes[B], "joint", ia)
        _compare(got, want, ("joint-small", weighted, ref_kind))
        assert (got["rep_status"] != 0).sum() >= 3 and got["n_ok"] < reps
    des.close(); ctx.close()


# ------------------------------------------------------------------------------------------- GPU: bit-identity
@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_singleton_clusters_in_frame_order_are_the_row_bootstrap(weighted):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    n, reps = 20_000, 300
    d = _frame(n, 41, weighted, n_cont=4, cat_levels=(4, 3))
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    kw = dict(seed=99, want_rep=True, norm=norm, ref_kind=ob.REF_WEIGHTED)
    row = [ob.bootstrap(des, reps, **kw), ob.bootstrap(des, reps, max_workspace_bytes=1, **kw)]
    des.attach_clusters(np.arange(n, dtype=np.int32), strata="group")
    assert des.clusters == dict(strata="group", units_a=des.n_a, units_b=des.n_b)
    _assert_equal(ob.bootstrap(des, reps, **kw), row[0])
    _assert_equal(ob.bootstrap(des, reps, max_workspace_bytes=1, **kw), row[1])
    _assert_equal(row[0], row[1])
    a = des.debug_counts(99, 5, 0)
    des.attach_clusters(None, strata=None)
    assert des.clusters is None
    np.testing.assert_array_equal(a, des.debug_counts(99, 5, 0))
    _assert_equal(ob.bootstrap(des, reps, **kw), row[0])
    des.close(); ctx.close()


# ------------------------------------------------------------------------------------------- GPU: native unit stream
@pytest.mark.gpu
@pytest.mark.parametrize("strata", ["group", "joint"])
def test_native_unit_counts(strata):
    import oaxaca_blinder_rs_b200 as ob
    n = 8000
    d = _frame(n, 51)
    codes = _clustered_codes(n, 400, 6)
    A, B = d["group"] == 0, d["group"] == 1
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    des.attach_clusters(codes, strata=strata)
    cl = des.clusters
    for rep in (0, 1, 77, 300):
        ca, cb = des.debug_counts(7, rep, 0).astype(np.int64), des.debug_counts(7, rep, 1).astype(np.int64)
        units = {}
        for cnt, cod in ((ca, codes[A]), (cb, codes[B])):
            for u in np.unique(cod):
                vals = np.unique(cnt[cod == u])
                assert len(vals) == 1, "rows of one unit carry different counts"
                key = (u, cnt is cb) if strata == "group" else u
                assert units.setdefault(key, int(vals[0])) == int(vals[0])
        if strata == "group":
            assert sum(v for (u, isb), v in units.items() if not isb) == cl["units_a"]
            assert sum(v for (u, isb), v in units.items() if isb) == cl["units_b"]
        else:
            assert sum(units.values()) == cl["units_a"] == cl["units_b"]
    des.close(); ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("strata", ["group", "joint"])
def test_native_results_do_not_depend_on_batching_width_or_sharding(strata):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core
    n, reps = 30_000, 300
    d = _frame(n, 61, True, n_cont=4, cat_levels=(4,))
    codes = _clustered_codes(n, 900, 7)
    kw = dict(seed=5, want_rep=True, ref_kind=ob.REF_POOLED)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    des.attach_clusters(codes, strata=strata)
    ref = ob.bootstrap(des, reps, **kw)
    assert ref["n_ok"] > reps // 2
    _assert_equal(ob.bootstrap(des, reps, max_workspace_bytes=1, **kw), ref)
    _assert_equal(ob.bootstrap(des, reps, count_bits=16, **kw), ref)
    des.close(); ctx.close()
    for world in (2, 3):
        grp = core.LocalGroup(world)
        outs, errs = [None] * world, [None] * world

        def work(r):
            try:
                c = ob.Context(0)
                c.init_local(grp, r)
                dd = _pack(c, d)
                dd.attach_clusters(codes, strata=strata)
                outs[r] = ob.bootstrap(dd, reps, shard_replicates=True, **kw)
                dd.close(); c.close()
            except Exception as e:  # noqa: BLE001
                errs[r] = e
        ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert all(e is None for e in errs), errs
        for o in outs:
            _assert_equal(o, ref)


@pytest.mark.gpu
def test_pooled_unit_counts_follow_binomial_m_1_over_m():
    import oaxaca_blinder_rs_b200 as ob
    from scipy import stats
    n = 6000
    d = _frame(n, 71)
    codes = np.arange(n, dtype=np.int32) // 12             # 500 clusters of 12 rows, both groups
    A, B = d["group"] == 0, d["group"] == 1
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    des.attach_clusters(codes, strata="joint")
    M = des.clusters["units_a"]
    assert M == 500
    hist = np.zeros(7)
    for rep in range(200):
        ca, cb = des.debug_counts(2024, rep, 0), des.debug_counts(2024, rep, 1)
        per_unit = np.zeros(M, dtype=np.int64)
        per_unit[codes[A]] = ca
        per_unit[codes[B]] = cb
        assert per_unit.sum() == M
        hist += np.bincount(np.minimum(per_unit, 6), minlength=7)
    p = stats.binom.pmf(np.arange(6), M, 1.0 / M)
    p = np.append(p, 1.0 - p.sum())
    chi = stats.chisquare(hist, hist.sum() * p)
    assert chi.pvalue > 1e-3, (hist, chi)
    des.close(); ctx.close()


# ------------------------------------------------------------------------------------------- GPU: Gram cache
@pytest.mark.gpu
def test_gram_cache_on_a_clustered_joint_design():
    import oaxaca_blinder_rs_b200 as ob
    n, reps = 20_000, 300
    d = _frame(n, 81, True, n_cont=4, cat_levels=(4, 3))
    codes = _clustered_codes(n, 500, 9)
    y1 = 0.6 * d["outcome"] + 0.2 * d["cont"][0]
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    run = lambda c=None, **kw: ob.bootstrap(des, reps, seed=3, want_rep=True, cache=c, **kw)  # noqa: E731
    assert run(cache)["cache_use"] == ob.CACHE_FILLED
    assert run(cache)["cache_use"] == ob.CACHE_SOLVE_ONLY
    des.attach_clusters(codes, strata="joint")             # new resamples: the cache refills
    r = run(cache)
    assert r["cache_use"] == ob.CACHE_FILLED
    _assert_equal(r, run())
    des.update_outcome(y1)
    r = run(cache, ref_kind=ob.REF_WEIGHTED)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY
    _assert_equal(r, run(ref_kind=ob.REF_WEIGHTED))
    for rk in (0, 1, 2):
        r = run(cache, ref_kind=rk, max_workspace_bytes=1)
        assert r["cache_use"] == ob.CACHE_SOLVE_ONLY
        _assert_equal(r, run(ref_kind=rk))
    des.close(); cache.close(); ctx.close()


# ------------------------------------------------------------------------------------------- GPU: statistics
@pytest.mark.gpu
def test_cluster_bootstrap_widens_the_se_under_intra_cluster_correlation():
    """Clusters of 20 rows nested in the groups, ICC about 0.3: design effect sqrt(1 + 19 * 0.3) = 2.6 on the SE of
    the group-mean difference, which carries the unexplained part."""
    import oaxaca_blinder_rs_b200 as ob
    rng = np.random.default_rng(2026)
    n_cl, m = 1000, 20
    n = n_cl * m
    code = np.repeat(np.arange(n_cl), m).astype(np.int32)
    group = np.repeat((np.arange(n_cl) % 2).astype(np.uint8), m)
    x = rng.standard_normal(n)
    u = np.sqrt(0.3) * rng.standard_normal(n_cl)[code]
    y = 1.0 + 0.2 * (group == 0) + 0.5 * x + u + np.sqrt(0.7) * rng.standard_normal(n)
    ctx = ob.Context(0)
    des = ob.Design.pack(ctx, [x], [], [], y, None, group)
    row = ob.bootstrap(des, 400, seed=1)
    des.attach_clusters(code, strata="group")
    assert des.clusters == dict(strata="group", units_a=n_cl // 2, units_b=n_cl // 2)
    cl = ob.bootstrap(des, 400, seed=1)
    np.testing.assert_array_equal(cl["point_stats"], row["point_stats"])     # the point estimate does not change
    ratio = cl["std_err"][1] / row["std_err"][1]
    assert ratio > 1.5, ratio
    des.close(); ctx.close()


# ------------------------------------------------------------------------------------------- GPU: refusals
def _raw_boot(des, reps, idx_a, idx_b):
    """ob_bootstrap_run through the C ABI (the Python layer checks stream shapes before the library sees them)."""
    from oaxaca_blinder_rs_b200 import _native as N
    o = N.BootOpts()
    o.reps = reps
    keep = [np.ascontiguousarray(idx_a, dtype=np.uint32), np.ascontiguousarray(idx_b, dtype=np.uint32)]
    o.idx_a, o.idx_b = keep[0].ctypes.data_as(N._U32P), keep[1].ctypes.data_as(N._U32P)
    r = N.Result()
    bufs = [np.empty(64) for _ in range(5)]
    r.point_stats, r.xa_mean, r.xb_mean, r.beta_star, r.std_err = [b.ctypes.data_as(N._DP) for b in bufs]
    return N.lib().ob_bootstrap_run(des.ctx._h, des._h, C.byref(o), C.byref(r))


@pytest.mark.gpu
def test_refusals():
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core
    INVALID, UNSUPPORTED = 7, 11
    n = 2000
    d = _frame(n, 91)
    codes = _clustered_codes(n, 50, 10)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    for bad in (np.full(n, 1000, dtype=np.int32), np.full(n, -1, dtype=np.int32)):
        with pytest.raises(ob.OaxacaError) as e:
            des.attach_clusters(bad, n_codes=160, strata="group")
        assert e.value.code == INVALID
    assert des.clusters is None                              # a refused attach leaves the design as it was
    with pytest.raises(ob.OaxacaError) as e:
        des.attach_clusters(codes[:-1], strata="group")     # n_frame differs from the packed frame
    assert e.value.code == INVALID
    with pytest.raises(ValueError):
        des.attach_clusters(codes, strata="rows")
    # Machado-Mata
    des.attach_clusters(codes, strata="joint")
    with pytest.raises(ob.OaxacaError) as e:
        ob.machado_mata(des, simulations=20, reps=2)
    assert e.value.code == UNSUPPORTED
    # JOINT takes one unit stream
    M = des.clusters["units_a"]
    assert _raw_boot(des, 2, np.zeros((2, M)), np.zeros((2, M))) == INVALID
    # Heckman, either order
    sel = (np.arange(n) % 3 != 0).astype(float)
    with pytest.raises(ob.OaxacaError) as e:
        des.attach_selection(sel, [d["cont"][0]])
    assert e.value.code == UNSUPPORTED
    des.attach_clusters(None, strata=None)
    des.attach_selection(sel, [d["cont"][0]])
    with pytest.raises(ob.OaxacaError) as e:
        des.attach_clusters(codes, strata="group")
    assert e.value.code == UNSUPPORTED
    des.close()
    # row shards (mode N): refused at attach, and by the run when the design is marked a shard afterwards
    data, A, B = _dense(d)
    Xa, ya, _, Xb, yb, _ = data
    (a0, a1), (b0, b1) = core.row_shard_plan(len(ya), 2, 0), core.row_shard_plan(len(yb), 2, 0)
    shard = ob.Design.from_dense(ctx, Xa[a0:a1], ya[a0:a1], None, Xb[b0:b1], yb[b0:b1], None, n_cont=3)
    shard.set_row_shard(len(ya), len(yb), 2, 0)
    with pytest.raises(ob.OaxacaError) as e:
        shard.attach_clusters(np.zeros(shard.n_a + shard.n_b, dtype=np.int32), strata="group")
    assert e.value.code == UNSUPPORTED
    shard.close()
    whole = ob.Design.from_dense(ctx, Xa[a0:a1], ya[a0:a1], None, Xb[b0:b1], yb[b0:b1], None, n_cont=3)
    whole.attach_clusters(np.arange(whole.n_a + whole.n_b, dtype=np.int32) // 4, strata="group")
    whole.set_row_shard(len(ya), len(yb), 2, 0)
    with pytest.raises(ob.OaxacaError) as e:
        ob.bootstrap(whole, 4)
    assert e.value.code == UNSUPPORTED
    whole.close(); ctx.close()


# ------------------------------------------------------------------------------------------- builders and CLI
def _cli_path():
    import os
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    return os.path.join(os.path.dirname(_native.LIB_PATH), "oaxaca-cli")


@pytest.mark.parametrize("args", [["--cluster", "firm", "--cluster-strata", "rows"],
                                  ["--cluster", "firm", "--cluster-strata", "Joint"],
                                  ["--cluster-strata", "joint"],
                                  ["--cluster", "firm", "--analysis-type", "quantile"]])
def test_cli_rejects_bad_cluster_arguments(args):
    """Exit code 2 before any file is read or any device is touched (the data path does not exist)."""
    import subprocess
    r = subprocess.run([_cli_path(), "--data", "nope.csv", "--outcome", "y", "--group", "g", "--reference", "r", *args],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "error:" in r.stderr and "cluster" in r.stderr, r.stderr


def _builder_frame(n, seed, n_firms):
    rng = np.random.default_rng(seed)
    firm = rng.integers(0, n_firms, n)
    gender = np.where(rng.random(n) < 0.5, "M", "F")
    x1, x2 = rng.standard_normal(n), rng.standard_normal(n)
    sector = rng.integers(0, 3, n)
    u = 0.5 * rng.standard_normal(n_firms)[firm]
    wage = 2.0 + 0.3 * (gender == "M") + 0.4 * x1 - 0.2 * x2 + 0.1 * sector + u + 0.5 * rng.standard_normal(n)
    frame = dict(wage=wage, x1=x1, x2=x2, sector=[f"s{s}" for s in sector], gender=list(gender),
                 firm=[f"f{f:04d}" for f in firm], firm_id=firm.astype(float))
    A, B = gender == "M", gender == "F"
    X = np.stack([np.ones(n), x1, x2, (sector == 1).astype(float), (sector == 2).astype(float)], 1)
    return frame, (X[A], wage[A], None, X[B], wage[B], None), firm[A], firm[B]


@pytest.mark.gpu
@pytest.mark.parametrize("strata", ["group", "joint"])
def test_builder_against_the_oracle_under_a_unit_stream(orc, strata):
    import oaxaca_blinder_rs_b200 as ob
    n, reps = 2500, 50
    frame, data, fa, fb = _builder_frame(n, 17, 120)
    rows_a, rows_b = unit_rows(fa, fb, strata)
    rng = np.random.default_rng(1)
    ia = rng.integers(0, len(rows_a), (reps, len(rows_a))).astype(np.uint32)
    ib = None if strata == "joint" else rng.integers(0, len(rows_b), (reps, len(rows_b))).astype(np.uint32)
    for rc, kind in ((ob.ReferenceCoefficients.GroupB, 1), (ob.ReferenceCoefficients.Pooled, 2), (ob.ReferenceCoefficients.Weighted, 3)):
        b = (ob.OaxacaBuilder(frame, "wage", "gender", "F").predictors(["x1", "x2"]).categorical_predictors(["sector"])
             .bootstrap_reps(reps).reference_coefficients(rc))
        b.cluster("firm", strata)
        b.index_stream(ia, ib)
        r = b.run()
        assert r.clusters == dict(strata=strata, units_a=len(rows_a), units_b=len(rows_b))
        want = oracle_cluster_run(orc, orc.Spec(K=5, n_cont=2, ref_kind=kind), data, fa, fb, strata, ia, ib)
        comps = r.two_fold.aggregate + r.three_fold.aggregate + r.two_fold.detailed_explained + r.two_fold.detailed_unexplained
        for field, key in (("std_err", "se"), ("p_value", "p"), ("ci_lower", "ci_lo"), ("ci_upper", "ci_hi")):
            got = np.array([getattr(c, field) for c in comps])
            assert relerr(got, want[key]) <= TOL, (strata, kind, field, worst(got, want[key]))
        assert r.successful_bootstraps == want["n_ok"]
        assert "Cluster bootstrap" in r.summary()


@pytest.mark.gpu
def test_builder_paths_and_cli_honour_the_cluster_column(tmp_path):
    import json
    import subprocess
    import oaxaca_blinder_rs_b200 as ob
    n = 3000
    frame, _, fa, fb = _builder_frame(n, 23, 150)

    def builder(col="firm", strata="group"):
        b = (ob.OaxacaBuilder(frame, "wage", "gender", "F").predictors(["x1", "x2"]).categorical_predictors(["sector"])
             .bootstrap_reps(200).seed(77))
        b.cluster(col, strata)
        return b
    plain = builder(None, None).run()
    assert plain.clusters is None
    by_label = builder().run()
    by_number = builder("firm_id").run()                     # numeric labels: the same clusters in the same order
    assert by_label.clusters == by_number.clusters == dict(strata="group", units_a=len(np.unique(fa)), units_b=len(np.unique(fb)))
    for x, y in zip(by_label.two_fold.aggregate, by_number.two_fold.aggregate):
        assert (x.estimate, x.std_err, x.p_value) == (y.estimate, y.std_err, y.p_value)
    assert by_label.two_fold.aggregate[1].std_err != plain.two_fold.aggregate[1].std_err
    assert by_label.total_gap == plain.total_gap
    sweep = builder(strata="joint").run_outcomes(["wage", "x1"])
    joint = builder(strata="joint").run()
    assert sweep[0].clusters == joint.clusters and joint.clusters["strata"] == "joint"
    assert [c.std_err for c in sweep[0].two_fold.aggregate] == [c.std_err for c in joint.two_fold.aggregate]
    rif = builder().decompose_quantile(0.5)
    assert rif.clusters == by_label.clusters
    # CLI on the same data from a CSV file: numeric cluster ids, same seed -> the builder's numbers
    path = tmp_path / "f.csv"
    with open(path, "w") as fh:
        fh.write("wage,x1,x2,sector,gender,firm_id\n")
        for i in range(n):
            fh.write(f"{float(frame['wage'][i])!r},{float(frame['x1'][i])!r},{float(frame['x2'][i])!r},{frame['sector'][i]},"
                     f"{frame['gender'][i]},{int(frame['firm_id'][i])}\n")
    out = tmp_path / "o.json"
    p = subprocess.run([_cli_path(), "--data", str(path), "--outcome", "wage", "--group", "gender", "--reference", "F",
                        "--predictors", "x1,x2", "--categorical", "sector", "--bootstrap-reps", "200", "--seed", "77",
                        "--ref-coeffs", "group-a", "--cluster", "firm_id", "--cluster-strata", "group", "--output-json", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "Cluster bootstrap (by group)" in p.stdout
    d = json.load(open(out))
    assert d["clusters"] == by_label.clusters
    got = [c["std_err"] for c in d["two_fold"]["aggregate"]]
    want = [c.std_err for c in by_label.two_fold.aggregate]
    assert relerr(got, want) <= 1e-15
