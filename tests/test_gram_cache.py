"""Per-replicate Gram cache (ob_gram_cache, ob_bootstrap_run_cached): outcome sweeps over fixed resamples.

CPU part: the outcome-only column table (ob_debug_gram_outcome_columns) is exactly the outcome part of the full table.

GPU part: every cached run equals an uncached ob_bootstrap_run on the same design state bit for bit -- whether the cache
was (re)filled, only the outcome columns were contracted, or only the solves ran -- for every reference kind, weights,
Yun normalisation, several outcomes (RIF), batching, and replicate (mode R) or row (mode N) sharding.
"""
import ctypes as C
import threading

import numpy as np
import pytest

N_ROWS, REPS, SEED = 80_000, 300, 1234      # >= 256 leaves per group; 301 slots = three panels, the last one partial


# ------------------------------------------------------------------------------------------- CPU
def _table(fn, *args):
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    L = _native.lib()
    til = np.zeros(3, dtype=np.int32)
    n = fn(L)(*args, None, None, 0, til.ctypes.data_as(C.POINTER(C.c_int32)))
    assert n > 0
    pairs, cmap = np.zeros((n, 2), dtype=np.uint16), np.zeros(n, dtype=np.int32)
    assert fn(L)(*args, pairs.ctypes.data_as(C.POINTER(C.c_uint16)), cmap.ctypes.data_as(C.POINTER(C.c_int32)), n, None) == n
    return pairs, cmap, til


def _full(L):
    L.ob_debug_gram_columns.restype = C.c_int64
    L.ob_debug_gram_columns.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_uint16),
                                        C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int32)]
    return L.ob_debug_gram_columns


def _outcome(L):
    return L.ob_debug_gram_outcome_columns


@pytest.mark.parametrize("K,T,n_cont,levels", [
    (51, 1, 44, (4, 4)),          # config 3: 52 outcome columns = one tail tile of 2 quanta (the full table: 43 quanta)
    (51, 3, 44, (4, 4)),          # config 3 with three RIF outcomes
    (31, 1, 30, ()), (31, 8, 30, ()), (17, 1, 16, ()), (12, 2, 3, (3, 2, 6)), (2, 1, 1, ()), (127, 1, 126, ()),
    (200, 2, 199, ()),            # 401 columns: three full tiles + a tail tile
])
def test_outcome_columns_are_the_outcome_part_of_the_full_table(K, T, n_cont, levels):
    lv = np.asarray(levels, dtype=np.int32)
    lvp = lv.ctypes.data_as(C.POINTER(C.c_int32)) if len(lv) else None
    fp, fc, _ = _table(_full, K, T, n_cont, lvp, len(lv))
    op, oc, til = _table(_outcome, K, T)
    full_y = [(tuple(p), c) for p, c in zip(fp.tolist(), fc.tolist()) if c >= 0 and p[1] >= K]
    got = [(tuple(p), c) for p, c in zip(op.tolist(), oc.tolist()) if c >= 0]
    assert got == full_y                                   # every outcome column once, same (j, l), target and order
    assert len(got) == K * T + 1
    assert all(p[1] >= K for p, _ in got)                  # no column of X'WX
    assert all(c == -1 for c in oc[len(got):]) and len(oc) % 128 == 0
    quanta = (K * T + 1 + 31) // 32
    assert til[0] == K * T + 1 and til[1] * 4 + til[2] == quanta and len(oc) == 128 * (til[1] + (til[2] > 0))


def test_outcome_columns_reject_bad_shapes():
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    L = _native.lib()
    for K, T in ((0, 1), (5, 0), (65535, 1)):
        assert L.ob_debug_gram_outcome_columns(K, T, None, None, 0, None) == -1


# ------------------------------------------------------------------------------------------- GPU
KEYS = ("point_stats", "rep_stats", "rep_status", "rep_beta_a", "rep_beta_b", "std_err", "p_value", "ci_lower", "ci_upper",
        "t_stat", "residuals_b", "total_gap_multi", "xa_mean", "xb_mean", "beta_star", "beta_a", "beta_b")


def _assert_equal(a, b):
    for k in KEYS:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["total_gap"] == b["total_gap"] and a["n_ok"] == b["n_ok"]


def _data(weighted, seed=7, n=N_ROWS):
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(n, 4, cat_levels=(4, 3), weights=weighted, seed=seed)       # two categoricals: structural zeros
    rng = np.random.default_rng(seed + 1)
    y1 = 0.7 * d["outcome"] + 0.3 * rng.standard_normal(n) + 0.1 * d["cont"][0]
    return d, y1


def _pack(ctx, d):
    import oaxaca_blinder_rs_b200 as ob
    return ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])


def _run(des, cache=None, reps=REPS, seed=SEED, **kw):
    import oaxaca_blinder_rs_b200 as ob
    return ob.bootstrap(des, reps, seed=seed, want_rep=True, cache=cache, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ref_kind", [0, 1, 2, 3])
@pytest.mark.parametrize("yun", [False, True])
def test_outcome_refresh_contracts_only_the_outcome_columns(weighted, ref_kind, yun):
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d, y1 = _data(weighted)
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)] if yun else []
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    r = _run(des, cache, ref_kind=ref_kind, norm=norm)
    assert r["cache_use"] == ob.CACHE_FILLED and cache.last_use == ob.CACHE_FILLED
    K, slots = des.K, REPS + 1
    assert cache.bytes == 2 * 8 * slots * (K * (K + 1) // 2 + K + 1)
    _assert_equal(r, _run(des, ref_kind=ref_kind, norm=norm))
    assert "cache_use" not in _run(des, ref_kind=ref_kind, norm=norm)
    des.update_outcome(y1)
    r = _run(des, cache, ref_kind=ref_kind, norm=norm)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY
    _assert_equal(r, _run(des, ref_kind=ref_kind, norm=norm))
    des.close(); cache.close(); ctx.close()


@pytest.mark.gpu
def test_reference_and_normalisation_sweep_only_solves():
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d, _ = _data(True)
    norm = [ob.NormVar(m, i) for m, i in synth.norm_spec(d)]
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    assert _run(des, cache)["cache_use"] == ob.CACHE_FILLED
    for rk in (1, 2, 3, 0):
        for nv in ([], norm):
            r = _run(des, cache, ref_kind=rk, norm=nv)
            assert r["cache_use"] == ob.CACHE_SOLVE_ONLY
            _assert_equal(r, _run(des, ref_kind=rk, norm=nv))
    r = _run(des, cache, skip_reduce=True)              # skip_reduce and count_bits are not part of the key either
    assert r["cache_use"] == ob.CACHE_SOLVE_ONLY
    np.testing.assert_array_equal(r["rep_stats"], _run(des, skip_reduce=True)["rep_stats"])
    des.close(); cache.close(); ctx.close()


@pytest.mark.gpu
def test_quantile_sweep_after_a_single_outcome_fill():
    import oaxaca_blinder_rs_b200 as ob
    d, y1 = _data(True)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    assert _run(des, cache)["cache_use"] == ob.CACHE_FILLED
    des.apply_rif_multi([0.1, 0.5, 0.9])
    r = _run(des, cache, ref_kind=ob.REF_POOLED)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY and r["n_outcomes"] == 3
    _assert_equal(r, _run(des, ref_kind=ob.REF_POOLED))
    K = des.K
    assert cache.bytes == 2 * 8 * (REPS + 1) * (K * (K + 1) // 2 + 3 * K + 1)
    r = _run(des, cache)
    assert r["cache_use"] == ob.CACHE_SOLVE_ONLY
    _assert_equal(r, _run(des))
    des.update_outcome(y1)                               # back to T = 1
    r = _run(des, cache)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY and r["n_outcomes"] == 1
    _assert_equal(r, _run(des))
    des.close(); cache.close(); ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fill_ws,hit_ws", [(1, 0), (0, 1)])
def test_batching_of_fill_and_hit_is_value_neutral(fill_ws, hit_ws):
    """max_workspace_bytes = 1: one panel per batch (three batches); 0: all panels in one batch."""
    import oaxaca_blinder_rs_b200 as ob
    d, y1 = _data(False)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    r = _run(des, cache, max_workspace_bytes=fill_ws)
    assert r["cache_use"] == ob.CACHE_FILLED
    _assert_equal(r, _run(des))
    des.update_outcome(y1)
    r = _run(des, cache, max_workspace_bytes=hit_ws)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY
    _assert_equal(r, _run(des))
    r = _run(des, cache, max_workspace_bytes=fill_ws, ref_kind=ob.REF_GROUP_B)
    assert r["cache_use"] == ob.CACHE_SOLVE_ONLY
    _assert_equal(r, _run(des, ref_kind=ob.REF_GROUP_B))
    des.close(); cache.close(); ctx.close()


@pytest.mark.gpu
def test_what_invalidates_the_cache():
    import oaxaca_blinder_rs_b200 as ob
    d, y1 = _data(True)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)

    def step(expect, **kw):
        r = _run(des, cache, **kw)
        assert r["cache_use"] == expect, kw
        _assert_equal(r, _run(des, **kw))

    step(ob.CACHE_FILLED)
    step(ob.CACHE_FILLED, seed=SEED + 1)                 # another resampling stream
    step(ob.CACHE_SOLVE_ONLY, seed=SEED + 1)
    step(ob.CACHE_FILLED, seed=SEED + 1, reps=REPS - 40)
    r = _run(des, cache, seed=SEED + 1, reps=REPS - 40, rep_begin=10, rep_end=200, skip_reduce=True)
    assert r["cache_use"] == ob.CACHE_FILLED             # another replicate range
    np.testing.assert_array_equal(r["rep_stats"], _run(des, seed=SEED + 1, reps=REPS - 40, rep_begin=10, rep_end=200,
                                                       skip_reduce=True)["rep_stats"])
    step(ob.CACHE_FILLED)
    des.set_row_shard(des.n_a, des.n_b, 1, 0)            # the row-shard marking changed (here: to the trivial one)
    step(ob.CACHE_FILLED)
    # a failing call leaves the cache empty
    with pytest.raises(ob.OaxacaError):
        _run(des, cache, ref_kind=9)
    assert cache.last_use == ob.CACHE_NONE and cache.bytes == 0
    step(ob.CACHE_FILLED)
    # a destroyed design and a fresh pack of the same frame (possibly at the same address) is another design
    des.close()
    des = _pack(ctx, d)
    step(ob.CACHE_FILLED)
    des.update_outcome(y1)
    step(ob.CACHE_OUTCOME_ONLY)
    des.close(); cache.close(); ctx.close()


@pytest.mark.gpu
def test_refusals_and_lifetime():
    import oaxaca_blinder_rs_b200 as ob
    d, _ = _data(False, n=20_000)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    ia = np.zeros((8, des.n_a), dtype=np.uint32)
    ib = np.zeros((8, des.n_b), dtype=np.uint32)
    with pytest.raises(ob.OaxacaError) as e:
        ob.bootstrap(des, 8, idx_a=ia, idx_b=ib, cache=cache)
    assert e.value.kind == "Unsupported"
    other = ob.Context(0)
    foreign = ob.GramCache(other)
    with pytest.raises(ob.OaxacaError) as e:
        ob.bootstrap(des, 8, cache=foreign)
    assert e.value.kind == "InvalidArgument"
    assert _run(des, cache, reps=8)["cache_use"] == ob.CACHE_FILLED
    rng = np.random.default_rng(3)
    des.attach_selection((rng.random(d["outcome"].shape[0]) < 0.7).astype(np.float64), [rng.standard_normal(d["outcome"].shape[0])])
    with pytest.raises(ob.OaxacaError) as e:
        _run(des, cache, reps=8)
    assert e.value.kind == "Unsupported"
    # caches outliving their context: the context releases their memory, destroy only frees the host struct
    other.close()
    assert foreign.bytes == 0
    foreign.close()
    assert _run(_pack(ctx, d), cache, reps=8)["cache_use"] == ob.CACHE_FILLED
    assert cache.bytes > 0
    des.close(); ctx.close()
    assert cache.bytes == 0
    cache.close()


def _threads(world, work):
    ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert not any(t.is_alive() for t in ts), "a rank did not finish"


@pytest.mark.gpu
def test_replicate_sharded_fill_and_hit():
    """Mode R: both ranks fill, then reuse; a rank whose cache cannot be reused makes all ranks refill."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core
    d, y1 = _data(True)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    one = [_run(des, ref_kind=ob.REF_WEIGHTED)]
    des.update_outcome(y1)
    one.append(_run(des, ref_kind=ob.REF_WEIGHTED))
    des.close(); ctx.close()
    world = 2
    grp = core.LocalGroup(world)
    outs, errs = [None] * world, [None] * world

    def work(r):
        try:
            c = ob.Context(0)
            c.init_local(grp, r)
            dd = _pack(c, d)
            cache = ob.GramCache(c)
            kw = dict(ref_kind=ob.REF_WEIGHTED, shard_replicates=True)
            res = [_run(dd, cache, **kw)]
            dd.update_outcome(y1)
            res.append(_run(dd, cache, **kw))
            if r == 0:                               # rank 0 starts over with an empty cache: everybody refills
                cache.close()
                cache = ob.GramCache(c)
            res.append(_run(dd, cache, **kw))
            res.append(_run(dd, cache, **kw))
            outs[r] = res
            dd.close(); cache.close(); c.close()
        except Exception as e:  # noqa: BLE001
            errs[r] = e
    _threads(world, work)
    assert all(e is None for e in errs), errs
    for res in outs:
        assert [x["cache_use"] for x in res] == [ob.CACHE_FILLED, ob.CACHE_OUTCOME_ONLY, ob.CACHE_FILLED, ob.CACHE_SOLVE_ONLY]
        for x, ref in zip(res, [one[0], one[1], one[1], one[1]]):
            _assert_equal(x, ref)


@pytest.mark.gpu
def test_row_sharded_fill_and_hit():
    """Mode N: row shards fill and reuse; results equal the unsharded uncached runs (residuals_b: the local rows)."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core, distributed as obd
    d, y1 = _data(True)
    ctx = ob.Context(0)
    des = _pack(ctx, d)
    one = [_run(des, ref_kind=ob.REF_POOLED)]
    des.update_outcome(y1)
    one.append(_run(des, ref_kind=ob.REF_POOLED))
    one.append(_run(des, ref_kind=ob.REF_GROUP_B))
    des.close(); ctx.close()
    world = 2
    grp = core.LocalGroup(world)
    outs, errs = [None] * world, [None] * world

    def work(r):
        try:
            c = ob.Context(0)
            c.init_local(grp, r)
            dd = obd.pack_row_shard(c, d, r, world)
            cache = ob.GramCache(c)
            res = [_run(dd, cache, ref_kind=ob.REF_POOLED, max_workspace_bytes=1)]
            dd.update_outcome(obd.shard_frame({**d, "outcome": y1}, r, world)["outcome"])
            res.append(_run(dd, cache, ref_kind=ob.REF_POOLED))
            res.append(_run(dd, cache, ref_kind=ob.REF_GROUP_B))
            outs[r] = res
            dd.close(); cache.close(); c.close()
        except Exception as e:  # noqa: BLE001
            errs[r] = e
    _threads(world, work)
    assert all(e is None for e in errs), errs
    for res in outs:
        assert [x["cache_use"] for x in res] == [ob.CACHE_FILLED, ob.CACHE_OUTCOME_ONLY, ob.CACHE_SOLVE_ONLY]
    for i in range(3):
        for res in outs:
            for k in KEYS:
                if k != "residuals_b":
                    np.testing.assert_array_equal(res[i][k], one[i][k], err_msg=k)
        np.testing.assert_array_equal(np.concatenate([res[i]["residuals_b"] for res in outs]), one[i]["residuals_b"])


# ------------------------------------------------------------------------------------------- builder
def _frame(n=30_000, seed=5, nulls=()):
    rng = np.random.default_rng(seed)
    x1, x2 = rng.normal(size=n), rng.normal(size=n)
    sector = rng.choice(["a", "b", "c", "d"], size=n)
    grp = np.where(rng.random(n) < 0.5, "M", "F")
    y = 1.0 + 0.5 * x1 - 0.2 * x2 + (grp == "M") * 0.3 + 0.4 * rng.normal(size=n)
    y2 = 0.3 + 0.2 * x1 + 0.6 * x2 + (sector == "b") * 0.2 + 0.3 * rng.normal(size=n)
    y3 = np.exp(0.1 * y)
    f = {"y": y, "y2": y2, "y3": y3, "x1": x1, "x2": x2, "w": 0.5 + rng.random(n), "sector": sector.tolist(),
         "gender": grp.tolist()}
    if nulls:
        f["y3"] = [None if i in set(nulls) else float(v) for i, v in enumerate(y3)]
    return f


def _builder(ob, frame, outcome="y"):
    return (ob.OaxacaBuilder(frame, outcome, "gender", "F").predictors(["x1", "x2"]).categorical_predictors(["sector"])
            .normalize(["sector"]).weights("w").bootstrap_reps(150).seed(9))


def _same_results(a, b):
    assert a.total_gap == b.total_gap and (a.n_a, a.n_b) == (b.n_a, b.n_b)
    for part in ("aggregate", "detailed_explained", "detailed_unexplained"):
        assert getattr(a.two_fold, part) == getattr(b.two_fold, part), part
    assert a.three_fold.aggregate == b.three_fold.aggregate
    for k in ("residuals", "xa_mean", "xb_mean", "beta_star"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k), err_msg=k)


@pytest.mark.gpu
def test_builder_run_outcomes_equals_run_per_outcome():
    import oaxaca_blinder_rs_b200 as ob
    f = _frame()
    rs = _builder(ob, f).run_outcomes(["y", "y2", "y3"])
    assert len(rs) == 3
    for name, r in zip(["y", "y2", "y3"], rs):
        _same_results(r, _builder(ob, f, name).run())


@pytest.mark.gpu
def test_builder_run_outcomes_cleans_over_every_outcome():
    import oaxaca_blinder_rs_b200 as ob
    drop = (3, 500, 20_001)
    f = _frame(nulls=drop)
    rs = _builder(ob, f).run_outcomes(["y", "y3"])
    keep = np.ones(len(f["y"]), bool); keep[list(drop)] = False
    g = {k: (np.asarray(v)[keep] if isinstance(v, np.ndarray) else [v[i] for i in np.flatnonzero(keep)]) for k, v in f.items()}
    g["y3"] = np.asarray(g["y3"], dtype=float)
    for name, r in zip(["y", "y3"], rs):
        _same_results(r, _builder(ob, g, name).run())


@pytest.mark.gpu
def test_builder_run_outcomes_refusals():
    import oaxaca_blinder_rs_b200 as ob
    f = _frame(n=5_000)
    with pytest.raises(ob.OaxacaError) as e:
        _builder(ob, f).run_outcomes(["y", "nope"])
    assert e.value.kind == "ColumnNotFound"
    with pytest.raises(ob.OaxacaError) as e:
        _builder(ob, f).run_outcomes(["y", "sector"])
    assert e.value.kind == "PolarsError"
    with pytest.raises(ob.OaxacaError) as e:
        _builder(ob, f).run_outcomes([])
    assert e.value.kind == "InvalidArgument"
    b = ob.OaxacaBuilder(f, "y", "gender", "F").predictors(["x1"]).heckman_selection("y2", ["x2"])
    with pytest.raises(ob.OaxacaError) as e:
        b.run_outcomes(["y", "y2"])
    assert e.value.kind == "Unsupported"
    ia = np.zeros((4, 10), dtype=np.uint32)
    with pytest.raises(ob.OaxacaError) as e:
        _builder(ob, f).bootstrap_reps(4).index_stream(ia, ia).run_outcomes(["y", "y2"])
    assert e.value.kind == "Unsupported"
