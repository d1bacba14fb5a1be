"""Every compiled variant of the Gram contraction, read back cell by cell and compared with exact sums.

A cached bootstrap leaves each slot's reduced Gram cells in its cache (ob_debug_gram_cache_read): the cells the solves
read, produced by the production batch loop -- multiplicities, gram_ws_kernel, the leaf-tree reduction or the mode-N
combine, and the cache extraction.  The test data keep every product and every partial sum an exact binary fraction
below 2^50:
  * continuous predictors are integers in [-8, 8], categoricals have 2-6 levels, outcomes are integers in [-50, 50];
  * weights come from {0.25, 1, 4, 9, 16}, so sqrt(w) and sqrt(w) * sqrt(w) = w are exact at pack time.
Any summation order (DMMA chains, leaf tree, mode-N combine) then gives the exact value, and the device must equal the
float64 reference bit for bit.  RIF outcomes (T = 3) are not integers; their cells are held to a rounding bound instead.

CPU part: the case list reaches every kernel variant (tiling from ob_debug_gram_columns, row stride and ring depth
restated below), the exactness bound holds for every case's data, and the read-back entry point is exported.
GPU part: every case's cells against the reference, plus the 16-bit width limit.
"""
import ctypes as C
import threading
import zlib
from dataclasses import dataclass

import numpy as np
import pytest

# ---- restated from csrc/internal.h (design_ldx), csrc/gram.cu (gram_ws_smem, the ring choice of gram_make_plan,
# gram_fits, the specialised strides of gram_launch_leaves) and csrc/api.cu (Batch::tail_mi)
BM, KT = 128, 32
A_TILE = KT * 148                           # the widened fp64 count tile of one ring stage
SMEM_MAX = 227 * 1024
SPECIALISED = tuple(range(12, 93, 8))       # row strides compiled with immediate shared-memory offsets


def design_ldx(V):
    ldx = V
    while ldx % 8 != 4:
        ldx += 1
    return ldx


def ws_smem(ldx, count_bytes, ring):
    return 8 * (ring * A_TILE + 256 + ring * KT * ldx) + ring * KT * BM * count_bytes + 8 * 3 * ring


def ring_depth(ldx, count_bytes):
    return 3 if ws_smem(ldx, count_bytes, 3) <= SMEM_MAX else 2


def fits(ldx, count_bytes):
    return ws_smem(ldx, count_bytes, 2) <= SMEM_MAX


def tail_mi(slots_last_panel):
    return min(16, ((slots_last_panel + 7) // 8 + 3) // 4 * 4)


WEIGHTS = (0.25, 1.0, 4.0, 9.0, 16.0)
EXACT_LIMIT = 2.0 ** 50      # quarter-integer sums are exact below 2^51; the largest multiplicity a run can hold is 2^16 - 1
MAX_COUNT = 65535
TAUS = (0.1, 0.5, 0.9)
SEED = 4242


@dataclass(frozen=True)
class Case:
    name: str
    n: tuple                        # (n_a, n_b)
    n_cont: int
    levels: tuple = ()
    weighted: bool = False
    runs: tuple = ((20, 8, 0),)     # (reps, count_bits, max_workspace_bytes): one filled cache each
    kind: str = "plain"             # plain | async | cluster | outcome | rif | mode_r | mode_n
    world: int = 1
    strata: str = None

    @property
    def K(self):
        return 1 + self.n_cont + sum(m - 1 for m in self.levels)

    @property
    def T(self):
        return len(TAUS) if self.kind == "rif" else 1


def _runs(*rb):
    return tuple((r, b, 0) for r, b in rb)


MI_SWEEP = _runs((20, 8), (50, 16), (80, 8), (110, 16))     # last-panel slots 21 / 51 / 81 / 111: MI 4 / 8 / 12 / 16

CASES = [
    # every specialised row stride, both count widths (K + 1 = ldx, or just below it)
    Case("ldx12", (700, 513), 10, weighted=True, runs=_runs((20, 8), (50, 16))),
    Case("ldx20", (901, 650), 18, runs=_runs((80, 8), (110, 16))),
    Case("ldx28", (800, 777), 19, (4, 5), weighted=True, runs=_runs((50, 8), (80, 16))),
    Case("ldx36", (850, 700), 34, runs=_runs((110, 8), (20, 16))),
    Case("ldx44", (900, 731), 40, (3,), weighted=True, runs=_runs((20, 8), (50, 16))),
    Case("ldx52", (1000, 850), 44, (4, 4), runs=_runs((80, 8), (110, 16))),
    Case("ldx60", (1003, 900), 58, weighted=True, runs=_runs((50, 8), (20, 16))),
    Case("ldx68", (1100, 950), 66, runs=_runs((110, 8), (80, 16))),
    Case("ldx76", (1150, 1001), 69, (6,), weighted=True, runs=_runs((20, 8), (50, 16))),
    Case("ldx84", (1200, 1050), 82, runs=_runs((80, 8), (110, 16))),
    Case("ldx92", (1250, 1100), 90, weighted=True, runs=_runs((50, 8), (20, 16))),
    # run-time row stride: ring of 3 (ldx 4 for K <= 3; 100 ... 132 at 8 bits, 100 ... 116 at 16), ring of 2 (124 / 132 at
    # 16 bits, the widest strides 268 at 16 bits and 284 at 8)
    Case("ldx4_K2", (1001, 777), 1, weighted=True, runs=_runs((20, 8), (110, 16))),
    Case("ldx4_K3", (640, 999), 0, (3,), runs=_runs((50, 8), (80, 16))),
    Case("ldx100", (700, 650), 98, weighted=True, runs=_runs((20, 8), (50, 16))),
    Case("ldx116", (700, 680), 109, runs=_runs((50, 8), (20, 16))),
    Case("ldx124", (600, 550), 122, weighted=True, runs=_runs((20, 8), (20, 16))),
    Case("ldx132", (620, 590), 125, (3, 4), runs=_runs((20, 8), (20, 16))),
    Case("ldx268", (420, 401), 266, weighted=True, runs=_runs((20, 16), (20, 8))),
    Case("ldx276", (430, 410), 273, runs=_runs((20, 8))),             # K + T = 275: 8 bits only (16 is refused)
    Case("ldx284", (400, 385), 278, weighted=True, runs=_runs((20, 8))),
    # tail tiles of 0 / 1 / 2 / 3 quanta (structural zeros shift the tiling), each with MI 4 / 8 / 12 / 16
    Case("tail0", (1500, 1300), 7, (4, 3), weighted=True, runs=MI_SWEEP),
    Case("tail1", (1400, 1250), 9, (4, 3), runs=MI_SWEEP),
    Case("tail2", (1300, 1200), 11, (2, 6), weighted=True, runs=MI_SWEEP),
    Case("tail3", (1200, 1100), 6, (6,), runs=MI_SWEEP),
    # three panels, one panel per batch (max_workspace_bytes = 1) and all in one; >= 256 leaves in both groups
    Case("panels_batches", (40_000, 33_000), 4, (5,), weighted=True, runs=((300, 8, 1), (300, 16, 0))),
    # group sizes: n_a >> n_b, n_b < 32; both groups below one pipeline stage
    Case("huge_vs_tiny", (100_000, 17), 3, runs=_runs((50, 8), (120, 16))),
    Case("tiny", (29, 23), 2, weighted=True, runs=_runs((80, 8))),
    # the leaf sub-range launches of a design whose upload is still in flight (>= 2^18 frame rows: two chunks)
    Case("async", (150_011, 149_989), 3, (3, 3), weighted=True, runs=_runs((40, 8)), kind="async"),
    Case("cluster_group", (3000, 2500), 4, (3,), weighted=True, runs=_runs((80, 8), (20, 16)), kind="cluster", strata="group"),
    Case("cluster_joint", (2600, 3100), 5, runs=_runs((50, 16)), kind="cluster", strata="joint"),
    # OUTCOME_ONLY: the narrow outcome table (52 columns: a tail tile of 2 quanta) after a fill
    Case("outcome_only", (3000, 2500), 44, (4, 4), weighted=True, runs=_runs((130, 8), (130, 16)), kind="outcome"),
    # three RIF outcomes: filled with T = 3, and an outcome-only run from a T = 1 fill
    Case("rif", (2000, 1800), 6, (4,), weighted=True, runs=_runs((60, 8)), kind="rif"),
    Case("mode_r2", (6000, 5000), 6, (4,), weighted=True, runs=_runs((300, 8)), kind="mode_r", world=2),
    Case("mode_r3", (5000, 4400), 8, runs=_runs((200, 16)), kind="mode_r", world=3),
    Case("mode_n2", (40_000, 36_000), 5, (3,), weighted=True, runs=_runs((130, 8)), kind="mode_n", world=2),
    Case("mode_n4", (40_000, 500), 4, runs=_runs((60, 16)), kind="mode_n", world=4),   # group B: rank 0 holds every leaf
]
BY_NAME = {c.name: c for c in CASES}


def frame(case):
    """Host columns for Design.pack (the synth.make_wage layout) plus the cluster codes and a second outcome."""
    rng = np.random.default_rng(zlib.crc32(case.name.encode()))
    n_a, n_b = case.n
    n = n_a + n_b
    group = np.zeros(n, np.uint8)
    group[rng.permutation(n)[:n_b]] = 1
    cont = [rng.integers(-8, 9, n).astype(np.float64) for _ in range(case.n_cont)]
    cats = []
    for m in case.levels:           # every level in both groups: the point estimate's X'WX must be regular
        code = np.empty(n, np.int32)
        for g in (0, 1):
            rows = np.flatnonzero(group == g)
            code[rows] = rng.permutation(np.arange(rows.size) % m)
        cats.append(code)
    y = rng.integers(-50, 51, n).astype(np.float64)
    w = rng.choice(WEIGHTS, n) if case.weighted else None
    return dict(n=n, cont=cont, cat_codes=cats, cat_levels=list(case.levels), outcome=y, weights=w, group=group,
                outcome2=rng.integers(-50, 51, n).astype(np.float64), clusters=rng.integers(0, max(n // 5, 1), n).astype(np.int32))


def host_design(d, y_key="outcome"):
    """Per group: X [n_g, K], Y [n_g, 1] and w [n_g] (or None), in packed row order."""
    from oaxaca_blinder_rs_b200 import synth
    Xa, _, wa, Xb, _, wb = synth.dense_design(d)
    y = d[y_key]
    return [(Xa, y[d["group"] == 0][:, None], wa), (Xb, y[d["group"] == 1][:, None], wb)]


def reference(X, Y, w, counts):
    """Cells of every slot in the cache layout (gram_cache_map): X'WX upper triangle row-major; (j, y_t) j-major, then
    (y_0, y_0).  counts [slots, n]: slot 0 is the point estimate (all ones).  Exact for integer X, Y and counts and
    quarter-integer w: every float64 partial sum is then exact whatever the order."""
    K = X.shape[1]
    cw = counts * (1.0 if w is None else w)
    iu = np.triu_indices(K)
    xx = np.empty((counts.shape[0], iu[0].size))
    for b in range(counts.shape[0]):
        xx[b] = ((X * cw[b][:, None]).T @ X)[iu]
    Z = (X[:, :, None] * Y[:, None, :]).reshape(X.shape[0], -1)
    yy = np.concatenate([cw @ Z, (cw @ (Y[:, 0] * Y[:, 0]))[:, None]], axis=1)
    return xx, yy


def exactness_bound(X, Y, w, counts):
    """max over cells of sum_i c_i w_i |v_ij v_il| (Cauchy-Schwarz: at most the largest column's sum_i c_i w_i v_i^2)."""
    V = np.concatenate([X, Y], axis=1)
    cw = counts * (1.0 if w is None else w)
    return float((cw @ (V * V)).max())


# ------------------------------------------------------------------------------------------- CPU
def _columns(K, T, n_cont, levels, outcome_only):
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    L = _native.lib()
    til = np.zeros(3, dtype=np.int32)
    tp = til.ctypes.data_as(C.POINTER(C.c_int32))
    if outcome_only:
        assert L.ob_debug_gram_outcome_columns(K, T, None, None, 0, tp) > 0
    else:
        L.ob_debug_gram_columns.restype = C.c_int64
        L.ob_debug_gram_columns.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                            C.POINTER(C.c_uint16), C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int32)]
        lv = np.asarray(list(levels) + [0], dtype=np.int32)
        assert L.ob_debug_gram_columns(K, T, n_cont, lv.ctypes.data_as(C.POINTER(C.c_int32)), len(levels), None, None, 0, tp) > 0
    return int(til[1]), int(til[2])          # full tiles, quanta of the tail tile


def variants(case):
    """One record per contraction of the case: the kernel it runs and the shapes it sees."""
    out = []
    K, T = case.K, case.T
    ldx = design_ldx(K + T)
    contractions = [(r, False) for r in case.runs]
    if case.kind == "outcome":                 # the fill, then an outcome-only run at the second width
        contractions = [(case.runs[0], False), (case.runs[1], True)]
    if case.kind == "rif":                     # T = 3 filled, and T = 1 filled then T = 3 outcome-only
        contractions = [(case.runs[0], False), (case.runs[0], True)]
    for (reps, bits, ws), outcome_only in contractions:
        slots = 1 + reps
        if case.kind == "mode_r":              # the first rank's share (the largest)
            slots = 1 + -(-reps // case.world)
        panels = -(-slots // BM)
        nfull, tail_q = _columns(K, T, case.n_cont, case.levels, outcome_only)
        mis = {tail_mi(slots - (panels - 1) * BM)} | ({16} if panels > 1 else set())
        cb = bits // 8
        out.append(dict(ldx=ldx, cb=cb, ring=ring_depth(ldx, cb), specialised=ldx in SPECIALISED, tail_q=tail_q,
                        nfull=nfull, mis=mis, panels=panels, batches=panels if ws == 1 else 1, outcome_only=outcome_only,
                        weighted=case.weighted, kind=case.kind, world=case.world, strata=case.strata, n=case.n))
    return out


def test_ring_choice_and_width_limits():
    """The restated shared-memory arithmetic gives the limits gram.cu documents."""
    assert ring_depth(132, 1) == 3 and ring_depth(140, 1) == 2
    assert ring_depth(116, 2) == 3 and ring_depth(124, 2) == 2 and ring_depth(132, 2) == 2
    assert fits(284, 1) and fits(268, 2) and not fits(276, 2)
    assert ws_smem(268, 2, 2) == 231_472 and ws_smem(276, 2, 2) == 235_568 and ws_smem(284, 2, 2) == 239_664
    assert design_ldx(280) == 284 and design_ldx(275) == 276 and design_ldx(268) == 268 and design_ldx(4) == 4


def test_cases_cover_every_kernel_variant():
    vs = [v for c in CASES for v in variants(c)]
    seen = {(v["ldx"], v["cb"]) for v in vs}
    for ldx in SPECIALISED:                                    # every specialised stride at both widths
        assert (ldx, 1) in seen and (ldx, 2) in seen, ldx
    rt = [v for v in vs if not v["specialised"]]
    assert {(4, 1), (4, 2)} <= {(v["ldx"], v["cb"]) for v in rt}                            # K <= 3: run-time stride
    assert any(100 <= v["ldx"] <= 132 and v["cb"] == 1 and v["ring"] == 3 for v in rt)
    assert any(100 <= v["ldx"] <= 116 and v["cb"] == 2 and v["ring"] == 3 for v in rt)
    ring2 = {(v["ldx"], v["cb"]) for v in rt if v["ring"] == 2}
    assert {(124, 2), (132, 2), (268, 2), (284, 1)} <= ring2
    assert {(124, 1), (132, 1)} <= {(v["ldx"], v["cb"]) for v in rt if v["ring"] == 3}
    # tail tiles of none / 1 / 2 / 3 quanta, each under MI = 4 / 8 / 12 / 16 slot groups
    combos = {(v["tail_q"], mi) for v in vs for mi in v["mis"]}
    assert {(q, mi) for q in range(4) for mi in (4, 8, 12, 16)} <= combos
    assert any(v["tail_q"] and v["nfull"] == 0 for v in vs) and any(v["tail_q"] and v["nfull"] > 0 for v in vs)
    assert any(v["panels"] > 1 and v["batches"] > 1 for v in vs) and any(v["panels"] > 1 and v["batches"] == 1 for v in vs)
    ns = [n for v in vs for n in v["n"]]
    assert min(ns) < KT and any(n % KT for n in ns) and any(n >= 4 * KT * 256 for n in ns)   # >= 256 leaves
    assert any(v["n"][0] >= 1000 * v["n"][1] for v in vs)
    assert {True, False} == {v["weighted"] for v in vs}
    kinds = {(v["kind"], v["world"], v["strata"]) for v in vs}
    assert {("async", 1, None), ("cluster", 1, "group"), ("cluster", 1, "joint"), ("mode_r", 2, None), ("mode_r", 3, None),
            ("mode_n", 2, None), ("mode_n", 4, None)} <= kinds
    assert any(v["outcome_only"] and v["kind"] == "outcome" for v in vs) and any(v["outcome_only"] and v["kind"] == "rif" for v in vs)


@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_case_data_keep_every_sum_exact(name):
    """With the widest multiplicity a run can hold, every cell's sum of |terms| stays below 2^50."""
    case = BY_NAME[name]
    d = frame(case)
    for X, Y, w in host_design(d) + host_design(d, "outcome2"):
        assert X.shape[1] == case.K
        assert np.all(X == np.round(X)) and np.abs(X).max() <= 8 and np.abs(Y).max() <= 50
        assert exactness_bound(X, Y, w, np.full((1, X.shape[0]), float(MAX_COUNT))) < EXACT_LIMIT


def test_cache_read_back_is_exported():
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    L = _native.lib()
    assert "ob_debug_gram_cache_read" in _native.SYMBOLS and hasattr(L, "ob_debug_gram_cache_read")
    assert len(L.ob_debug_gram_cache_read.argtypes) == 6
    assert L.ob_debug_gram_cache_read(None, None, None, None, None, None) == 7        # OB_ERR_INVALID_ARG, no device needed


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    import oaxaca_blinder_rs_b200 as ob
    c = ob.Context(0)
    yield c
    c.close()


def _pack(ctx, d, asynchronous=False):
    import oaxaca_blinder_rs_b200 as ob
    return ob.Design.pack(ctx, d["cont"], d["cat_codes"], d["cat_levels"], d["outcome"], d["weights"], d["group"],
                          asynchronous=asynchronous)


def _fill(des, reps, bits, ws, seed, cache=None, **kw):
    import oaxaca_blinder_rs_b200 as ob
    cache = cache or ob.GramCache(des.ctx)
    r = ob.bootstrap(des, reps, seed=seed, count_bits=bits, max_workspace_bytes=ws, want_residuals=False, cache=cache, **kw)
    return r, cache


def _counts(des, seed, reps):
    """[group] -> [1 + reps, n_g]: the point slot's ones, then the native stream's replicates 0 .. reps - 1."""
    out = []
    for g, n in enumerate((des.n_a, des.n_b)):
        c = np.ones((1 + reps, n))
        for r in range(reps):
            c[1 + r] = des.debug_counts(seed, r, g)
        out.append(c)
    return out


def _exact(got, want, what):
    bad = np.argwhere(got != want)
    assert bad.size == 0, (f"{what}: {len(bad)} of {got.size} cells differ; first (slot, cell): {bad[:6].tolist()}, "
                           f"got {got[tuple(bad[:6].T)].tolist()}, want {want[tuple(bad[:6].T)].tolist()}")


def _check_exact(cells, host, counts, slots_sel, what):
    for g, (X, Y, w) in enumerate(host):
        cg = counts[g][slots_sel]
        assert exactness_bound(X, Y, w, cg) < EXACT_LIMIT
        xx, yy = reference(X, Y, w, cg)
        _exact(cells["xx"][g], xx, f"{what}: X'WX, group {g}")
        _exact(cells["yy"][g], yy, f"{what}: X'Wy, group {g}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c.name for c in CASES if c.kind in ("plain", "async", "cluster")])
def test_cells_equal_exact_sums(name, ctx):
    import oaxaca_blinder_rs_b200 as ob
    case = BY_NAME[name]
    d = frame(case)
    des = _pack(ctx, d, asynchronous=case.kind == "async")
    if case.kind == "cluster":
        des.attach_clusters(d["clusters"], strata=case.strata)
    seed = SEED + len(name)
    got = []
    for reps, bits, ws in case.runs:
        r, cache = _fill(des, reps, bits, ws, seed)
        assert r["cache_use"] == ob.CACHE_FILLED
        got.append((reps, bits, r, cache.debug_cells()))
        cache.close()
    # the replicates' counts only now: reading them completes an asynchronous pack, which the runs above must find in flight
    counts = _counts(des, seed, max(r[0] for r in case.runs))
    host = host_design(d)
    packed = des.download()
    for g, (X, Y, w) in enumerate(host):           # the pack itself (wide designs stage their rows in column passes)
        np.testing.assert_array_equal(packed[3 * g], X)
        np.testing.assert_array_equal(packed[3 * g + 1], Y[:, 0])
    for reps, bits, r, cells in got:
        what = f"{name} reps={reps} count_bits={bits}"
        assert (cells["slots"], cells["K"], cells["T"], cells["count_bytes"]) == (1 + reps, case.K, 1, bits // 8), what
        _check_exact(cells, host, counts, slice(0, 1 + reps), what)
        if case.kind == "cluster":
            for g in (0, 1):
                np.testing.assert_array_equal(cells["rows"][g], counts[g][:1 + reps].sum(axis=1), err_msg=f"{what}: rows, group {g}")
        else:
            assert cells["rows"] is None
    if case.kind == "async":       # the same run on a resident design: one Gram launch fewer
        sync = _pack(ctx, d)
        reps, bits, ws = case.runs[0]
        r_sync, cache = _fill(sync, reps, bits, ws, seed)
        assert got[0][2]["gpu_launches"] > r_sync["gpu_launches"]
        np.testing.assert_array_equal(cache.debug_cells()["xx"], got[0][3]["xx"])
        cache.close(); sync.close()
    des.close()


@pytest.mark.gpu
def test_outcome_only_cells(ctx):
    import oaxaca_blinder_rs_b200 as ob
    case = BY_NAME["outcome_only"]
    d = frame(case)
    des = _pack(ctx, d)
    (reps, bits, ws), (_, bits2, ws2) = case.runs
    r, cache = _fill(des, reps, bits, ws, SEED)
    assert r["cache_use"] == ob.CACHE_FILLED and cache.last_use == ob.CACHE_FILLED
    filled = cache.debug_cells()
    des.update_outcome(d["outcome2"])
    r, _ = _fill(des, reps, bits2, ws2, SEED, cache=cache)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY and cache.last_use == ob.CACHE_OUTCOME_ONLY
    hit = cache.debug_cells()
    counts = _counts(des, SEED, reps)
    _check_exact(filled, host_design(d), counts, slice(None), "fill")
    _check_exact(hit, host_design(d, "outcome2"), counts, slice(None), "outcome-only")
    cache.close(); des.close()


@pytest.mark.gpu
def test_three_rif_outcomes(ctx):
    """T = 3: X'WX exact; the (j, y_t) and (y_0, y_0) cells of the non-integer RIF columns within the rounding bound
    |d| <= (n_g + 2) 2^-53 sum |c w x_j r| against a long-double reference."""
    import oaxaca_blinder_rs_b200 as ob
    case = BY_NAME["rif"]
    d = frame(case)
    des = _pack(ctx, d)
    reps, bits, ws = case.runs[0]
    r, cache_a = _fill(des, reps, bits, ws, SEED)            # T = 1, integer outcome
    assert r["cache_use"] == ob.CACHE_FILLED
    des.apply_rif_multi(TAUS)
    r, _ = _fill(des, reps, bits, ws, SEED, cache=cache_a)
    assert r["cache_use"] == ob.CACHE_OUTCOME_ONLY and r["n_outcomes"] == 3
    r, cache_b = _fill(des, reps, bits, ws, SEED)
    assert r["cache_use"] == ob.CACHE_FILLED
    cells = {"outcome-only": cache_a.debug_cells(), "filled": cache_b.debug_cells()}
    cache_a.close(); cache_b.close()
    rif = [[], []]                                           # each quantile's RIF column: single-quantile transforms
    for tau in TAUS:
        des.apply_rif(tau)
        _, ya, _, _, yb, _ = des.download()
        rif[0].append(ya); rif[1].append(yb)
    counts = _counts(des, SEED, reps)
    K, T = case.K, len(TAUS)
    for what, cl in cells.items():
        assert (cl["K"], cl["T"], cl["slots"]) == (K, T, 1 + reps)
        for g, (X, _, w) in enumerate(host_design(d)):
            R = np.stack(rif[g], axis=1)
            cw = counts[g] * (1.0 if w is None else w)
            xx, _ = reference(X, R[:, :1], w, counts[g])
            _exact(cl["xx"][g], xx, f"{what}: X'WX, group {g}")
            Z = (X[:, :, None] * R[:, None, :]).reshape(X.shape[0], -1)
            Z = np.concatenate([Z, (R[:, 0] * R[:, 0])[:, None]], axis=1)
            want = cw.astype(np.longdouble) @ Z.astype(np.longdouble)
            bound = (X.shape[0] + 2) * 2.0 ** -53 * (np.abs(cw) @ np.abs(Z))
            err = np.abs(cl["yy"][g].astype(np.longdouble) - want)
            worst = np.unravel_index(int(np.argmax(err / bound)), err.shape)
            assert np.all(err <= bound), f"{what}: X'Wy group {g}, slot/cell {worst}: |d| = {float(err[worst])} > {bound[worst]}"
    des.close()


def _threads(world, work):
    ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert not any(t.is_alive() for t in ts), "a rank did not finish"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mode_r2", "mode_r3", "mode_n2", "mode_n4"])
def test_sharded_cells(name, ctx):
    """Mode R: each rank's cache holds the point slot and its replicate shard; mode N: every rank holds the combined sums
    of all slots.  Either way each rank's cells equal the exact sums of its slots (counts read on the unsharded design)."""
    import oaxaca_blinder_rs_b200 as ob
    from oaxaca_blinder_rs_b200 import core, distributed as obd
    case = BY_NAME[name]
    d = frame(case)
    reps, bits, ws = case.runs[0]
    twin = _pack(ctx, d)
    counts = _counts(twin, SEED, reps)
    twin.close()
    world = case.world
    grp = core.LocalGroup(world)
    cells, errs = [None] * world, [None] * world

    def work(r):
        try:
            c = ob.Context(0)
            c.init_local(grp, r)
            dd = obd.pack_row_shard(c, d, r, world) if case.kind == "mode_n" else _pack(c, d)
            res, cache = _fill(dd, reps, bits, ws, SEED, shard_replicates=case.kind == "mode_r")
            assert res["cache_use"] == ob.CACHE_FILLED
            cells[r] = cache.debug_cells()
            cache.close(); dd.close(); c.close()
        except Exception as e:  # noqa: BLE001
            errs[r] = e
    _threads(world, work)
    assert all(e is None for e in errs), errs
    host = host_design(d)
    for r in range(world):
        sel = list(range(1 + reps))
        if case.kind == "mode_r":
            rb, re = ob.replicate_shard(reps, world, r)
            sel = [0] + list(range(1 + rb, 1 + re))
        assert cells[r]["slots"] == len(sel)
        _check_exact(cells[r], host, counts, sel, f"{name} rank {r}")


@pytest.mark.gpu
def test_16bit_width_limit(ctx):
    """K + T = 275: 16-bit multiplicities are refused before any device work, and a run whose 8-bit counts saturate fails
    instead of widening; at K + T = 268 the same saturating stream widens to 16 bits and runs."""
    import oaxaca_blinder_rs_b200 as ob
    wide = BY_NAME["ldx276"]
    d = frame(wide)
    des = _pack(ctx, d)
    cache = ob.GramCache(ctx)
    with pytest.raises(ob.OaxacaError) as e:
        _fill(des, 20, 16, 0, SEED, cache=cache)
    assert e.value.kind == "Unsupported" and "16-bit multiplicities need K + outcomes <= 268" in str(e.value)
    assert cache.last_use == ob.CACHE_NONE and cache.bytes == 0
    with pytest.raises(ob.OaxacaError) as e:
        cache.debug_cells()                                  # an empty cache
    assert e.value.kind == "InvalidArgument"
    cache.close()
    reps = 3

    def saturating(des):           # replicate 1 draws row 0 of each group n_g > 255 times
        ia, ib = np.tile(np.arange(des.n_a, dtype=np.uint32), (reps, 1)), np.tile(np.arange(des.n_b, dtype=np.uint32), (reps, 1))
        ia[1], ib[1] = 0, 0
        return ob.bootstrap(des, reps, idx_a=ia, idx_b=ib, want_rep=True, want_residuals=False)
    with pytest.raises(ob.OaxacaError) as e:
        saturating(des)
    assert e.value.kind == "Unsupported" and "row multiplicity overflows the count width" in str(e.value)
    des.close()
    des = _pack(ctx, frame(BY_NAME["ldx268"]))
    r = saturating(des)
    assert r["rep_status"][0] == 0 and r["rep_status"][2] == 0
    des.close()
