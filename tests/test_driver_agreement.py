"""Failures inside the replicate-batch drivers: under mode R (shard_replicates) a rank that fails must not leave its peers
waiting in a collective -- every rank returns, the failing one with its own error, the others with the agreed status.
Two contexts of one process (threads) joined by the in-process communicator, as in test_replicate_sharding_lib.py.
Also the host-side checks that refuse bad input before any kernel reads a design row."""
import threading

import numpy as np
import pytest

from test_gpu_heckman import make_selection_frame
from test_gpu_mm import make_frame

pytestmark = pytest.mark.gpu
PEER_MSG = "another rank of the replicate-sharded run failed"


def _run_world(world, call):
    """call(rank, ctx) on `world` contexts joined by a LocalGroup; returns the exceptions, None where a rank succeeded."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core
    grp = core.LocalGroup(world)
    errs = ["no result"] * world

    def work(r):
        try:
            ctx = ob.Context(0)
            ctx.init_local(grp, r)
            call(r, ctx)
            ctx.close()
            errs[r] = None
        except Exception as e:  # noqa: BLE001
            errs[r] = e
    ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
    assert not any(t.is_alive() for t in ts), "a rank did not return (waiting for its peers)"
    return errs


def _bad_streams(n_a, n_b, reps, bad_rep, seed=3):
    rng = np.random.default_rng(seed)
    ia = rng.integers(0, n_a, size=(reps, n_a)).astype(np.uint32)
    ib = rng.integers(0, n_b, size=(reps, n_b)).astype(np.uint32)
    ia[bad_rep, n_a // 2] = n_a
    return ia, ib


def _assert_errors(errs, failed):
    """Ranks in `failed` raise their own error, the others the agreed status of their peers."""
    for r, e in enumerate(errs):
        assert e is not None and getattr(e, "kind", None) == "InvalidArgument", (r, e)
        assert ("resample index out of range" if r in failed else PEER_MSG) in str(e), (r, e)


def test_ols_mode_r_rank_failure_is_agreed():
    """A bad index in a replicate of rank 1's shard: rank 1 fails on it, rank 0 leaves with the agreed status."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import synth
    d = synth.make_wage(3_000, 2, cat_levels=(3,), weights=False, seed=4)
    n_a, n_b = int(np.sum(d["group"] == 0)), int(np.sum(d["group"] == 1))
    reps = 20                                              # rank 0: replicates [0, 10), rank 1: [10, 20)
    ia, ib = _bad_streams(n_a, n_b, reps, bad_rep=15)

    def call(r, ctx):
        des = ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"])
        try:
            ob.bootstrap(des, reps, idx_a=ia, idx_b=ib, shard_replicates=True)
        finally:
            des.close()
    _assert_errors(_run_world(2, call), failed=(1,))


def test_heckman_mode_r_rank_failure_is_agreed():
    import oaxaca_blinder_rs_b200 as ob
    fr = make_selection_frame(4_000, 2, seed=8)
    n_a, n_b = int(np.sum(fr["group"] == 0)), int(np.sum(fr["group"] == 1))
    reps = 20
    ia, ib = _bad_streams(n_a, n_b, reps, bad_rep=15)

    def call(r, ctx):
        des = ob.Design.pack(ctx, fr["cont"], [fr["cat"]], [3], fr["y"], None, fr["group"])
        try:
            des.attach_selection(fr["s"], fr["z"])
            ob.bootstrap(des, reps, ref_kind=1, idx_a=ia, idx_b=ib, shard_replicates=True)
        finally:
            des.close()
    _assert_errors(_run_world(2, call), failed=(1,))


def test_mm_mode_r_bad_index_fails_on_every_rank():
    """Machado-Mata mode R shards the regressions: every rank builds every pass's multiplicities, so every rank finds the
    bad index itself (native simulated rows: no draw_* stream)."""
    import oaxaca_blinder_rs_b200 as ob
    fr = make_frame(2_000, 2, seed=6)
    n_a, n_b = int(np.sum(fr["group"] == 0)), int(np.sum(fr["group"] == 1))
    reps = 6
    ia, ib = _bad_streams(n_a, n_b, reps, bad_rep=4)

    def call(r, ctx):
        des = ob.Design.pack(ctx, fr["cont"], [fr["cat"]], [3], fr["y"], None, fr["group"])
        try:
            ob.machado_mata(des, [0.25, 0.5, 0.75], simulations=16, reps=reps, idx_a=ia, idx_b=ib, shard_replicates=True)
        finally:
            des.close()
    _assert_errors(_run_world(2, call), failed=(0, 1))


def test_mm_explicit_draws_check_the_resample_index():
    """A simulated row is mapped through the caller's index stream on the host: an index outside the group is refused
    there, before any kernel reads that design row."""
    import oaxaca_blinder_rs_b200 as ob
    fr = make_frame(1_500, 2, seed=7)
    n_a, n_b = int(np.sum(fr["group"] == 0)), int(np.sum(fr["group"] == 1))
    reps, sims = 3, 12
    rng = np.random.default_rng(2)
    st = dict(taus=rng.uniform(0.01, 0.99, size=(reps + 1, sims)),
              draw_a=rng.integers(0, n_a, size=(reps + 1, sims)).astype(np.uint32),
              draw_b=rng.integers(0, n_b, size=(reps + 1, sims)).astype(np.uint32),
              idx_a=rng.integers(0, n_a, size=(reps, n_a)).astype(np.uint32),
              idx_b=rng.integers(0, n_b, size=(reps, n_b)).astype(np.uint32))
    st["idx_a"][1, st["draw_a"][2, 5]] = n_a + 1000          # replicate 1 = pass 2: its 6th simulated row of group A
    ctx = ob.Context(0)
    des = ob.Design.pack(ctx, fr["cont"], [fr["cat"]], [3], fr["y"], None, fr["group"])
    with pytest.raises(ob.OaxacaError) as e:
        ob.machado_mata(des, [0.5], simulations=sims, reps=reps, **st)
    assert e.value.kind == "InvalidArgument" and "resample index out of range" in str(e.value)
    des.close(); ctx.close()


def test_heckman_refuses_a_row_sharded_design():
    """ob_design_attach_selection refuses a row shard; marking the design as one afterwards must not let the Heckman
    bootstrap run on one shard as if it were the whole frame."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core
    fr = make_selection_frame(3_000, 2, seed=9)
    n_a, n_b = int(np.sum(fr["group"] == 0)), int(np.sum(fr["group"] == 1))
    keep = []
    for g, n_g in ((0, n_a), (1, n_b)):
        b, e = core.row_shard_plan(n_g, 2, 0)
        keep.append(np.flatnonzero(fr["group"] == g)[b:e])
    rows = np.sort(np.concatenate(keep))                    # rank 0's rows of each group, in frame order
    ctx = ob.Context(0)
    des = ob.Design.pack(ctx, [x[rows] for x in fr["cont"]], [fr["cat"][rows]], [3], fr["y"][rows], None, fr["group"][rows])
    des.attach_selection(fr["s"][rows], [z[rows] for z in fr["z"]])
    des.set_row_shard(n_a, n_b, 2, 0)
    with pytest.raises(ob.OaxacaError) as e:
        ob.bootstrap(des, 4, ref_kind=1, seed=1)
    assert e.value.kind == "Unsupported" and "row-sharded" in str(e.value)
    des.close(); ctx.close()
