"""The native random streams, bit for bit against a host restatement.

Every result computed without an explicit stream depends on the native Philox streams: the multinomial counts of the row
and cluster bootstraps (resample.cu, cluster.cu), the Bayesian bootstrap's Exp(1) weights (resample.cu) and the
Machado-Mata random quantiles and simulated rows (mm.cu).  DESIGN 4.2 says the counts are exactly the 64-bit inverse CDF
of a Poisson(lambda) body plus uniform fix-up draws, i.e. exactly Multinomial(n); DESIGN 7c says a simulated row is
original row i with probability c_i / n.  This file restates those definitions in plain numpy (Philox4x32-10 from the
published round function, the Poisson thresholds exactly in decimal arithmetic, the counter layouts of each stream) and
requires the device to produce the same bits.  A lane, octet, counter-word or comparison slip gives plausible random
numbers that statistical tests cannot see; it fails here.

CPU part: Philox known answers, the threshold table against the Poisson pmf, an exhaustive check that the lazy 14-bit /
16-bit / 64-bit resolve of the counts kernel is the 64-bit inverse CDF, and the law of the simulated-row draw.
GPU part: ob_debug_counts (row and clustered designs) and ob_debug_bayes_weights against the restatement, and a native
Machado-Mata run against the same run rebuilt from restated streams passed explicitly.
"""
import decimal
import math
from fractions import Fraction

import numpy as np
import pytest

M32 = 0xFFFFFFFF
U64 = np.uint64

# stream tags (resample.cu, mm.cu)
STREAM_BODY, STREAM_REFINE, STREAM_FIXUP, STREAM_BAYES = 0x0B0D1, 0x0F19E, 0x0F1C, 0x0BA7E5
MM_STREAM_TAU, MM_STREAM_ROW = 0x4D4D5441, 0x4D4D524F
KMAX, LUT_BITS = 24, 14


# ------------------------------------------------------------------------------------------- host restatement
def philox(c0, c1, c2, c3, key):
    """Philox4x32-10 (Salmon et al., SC'11) as common.cuh writes it, vectorised: counter words are integers or uint64
    arrays of 32-bit values (broadcast together), key = (k0, k1) Python ints, bumped after every round."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=U64) & U64(M32) for c in np.broadcast_arrays(c0, c1, c2, c3))
    k0, k1 = key
    for _ in range(10):
        p0 = U64(0xD2511F53) * c0
        p1 = U64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> U64(32)) ^ c1 ^ U64(k0), p1 & U64(M32), (p0 >> U64(32)) ^ c3 ^ U64(k1), p0 & U64(M32)
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


def seed_key(seed):
    return seed & M32, seed >> 32


def umulhi(u, n):
    """High 64 bits of u * n for uint64 u and n < 2^32 (__umul64hi)."""
    hi, lo = u >> U64(32), u & U64(M32)
    return (hi * U64(n) + ((lo * U64(n)) >> U64(32))) >> U64(32)


def poisson_table(n):
    """T[k] = floor(P(X <= k) 2^64) for X ~ Poisson(lambda), lambda = (n - ceil(8 sqrt n)) / n, in exact decimal
    arithmetic; None when ceil(8 sqrt n) >= n (lambda_zero: the body draws nothing and every count comes from the fix-up)."""
    delta = math.isqrt(64 * n - 1) + 1          # ceil(sqrt(64 n))
    if delta >= n:
        return None
    with decimal.localcontext() as dc:
        dc.prec = 80
        lam = decimal.Decimal(n - delta) / n
        p, cdf, T = (-lam).exp(), decimal.Decimal(0), []
        for k in range(KMAX):
            cdf += p
            T.append(min(int((cdf * 2 ** 64).to_integral_value(rounding=decimal.ROUND_FLOOR)), 2 ** 64 - 1))
            p = p * lam / (k + 1)
    return T


def bucket_ambiguous(T):
    """counts_lut_kernel's marking: bucket b (the top 14 bits of U) is ambiguous when its lowest and highest U give
    different counts."""
    Ta = np.array(T, dtype=U64)
    lo = np.arange(1 << LUT_BITS, dtype=U64) << U64(64 - LUT_BITS)
    hi = lo | U64((1 << (64 - LUT_BITS)) - 1)
    return np.searchsorted(Ta, lo, side="right") != np.searchsorted(Ta, hi, side="right")


def restate_counts(n, seed, rep, group, T="auto"):
    """The counts of global replicate `rep` over n rows (or units) of stream group `group` (0 = A, 1 = B, 2 = JOINT units),
    as DESIGN 4.2 defines them.  Body: stream id sid = rep + 1; the Philox call keyed by the octet sid >> 3 at counter
    (row, group << 8 | row >> 32, octet, STREAM_BODY ^ octet >> 32) gives u16 = 16-bit lane sid & 7 of its four words
    (odd lane = high half); the 48 low bits of U come from the refinement call (row, ..., rep, STREAM_REFINE ^ rep >> 32);
    the count is #{k : U >= T[k]}.  Fix-up: n - sum(body) uniform draws j at counter (j, group << 8 | j >> 32, rep,
    STREAM_FIXUP ^ rep >> 32), row umulhi(x:y, n).
    Returns (counts int64 [n], rows whose 14-bit bucket is ambiguous, rows whose u16 ties a threshold's top 16 bits)."""
    T = poisson_table(n) if isinstance(T, str) else T
    key = seed_key(seed)
    c = np.zeros(n, dtype=np.int64)
    n_ambig = n_tie = 0
    if T is not None:
        rows = np.arange(n, dtype=U64)
        c1 = (U64(group) << U64(8)) | (rows >> U64(32))
        sid = rep + 1
        oc, lane = sid >> 3, sid & 7
        w = philox(rows, c1, oc & M32, STREAM_BODY ^ (oc >> 32), key)[lane >> 1]
        u16 = (w >> U64(16)) if lane & 1 else (w & U64(0xFFFF))
        r = philox(rows, c1, rep & M32, STREAM_REFINE ^ (rep >> 32), key)
        U = (u16 << U64(48)) | (r[0] << U64(16)) | (r[1] >> U64(16))
        Ta = np.array(T, dtype=U64)
        c = np.searchsorted(Ta, U, side="right").astype(np.int64)
        n_ambig = int(bucket_ambiguous(T)[(u16 >> U64(2)).astype(np.int64)].sum())
        n_tie = int(np.isin(u16, Ta >> U64(48)).sum())
    need = n - int(c.sum())
    assert need >= 0
    j = np.arange(need, dtype=U64)
    r = philox(j, (U64(group) << U64(8)) | (j >> U64(32)), rep & M32, STREAM_FIXUP ^ (rep >> 32), key)
    c += np.bincount(umulhi((r[0] << U64(32)) | r[1], n).astype(np.int64), minlength=n)
    return c, n_ambig, n_tie


def restate_bayes(n, seed, rep, group):
    """The Bayesian bootstrap's E of replicate `rep`: word sid & 3 of the Philox call keyed by the quad sid >> 2 at counter
    (row, group << 8 | row >> 32, quad, STREAM_BAYES ^ quad >> 32); E = -log(((u >> 9) + 1/2) 2^-23), log in float64
    rounded to fp32."""
    rows = np.arange(n, dtype=U64)
    sid = rep + 1
    qd = sid >> 2
    u = philox(rows, (U64(group) << U64(8)) | (rows >> U64(32)), qd & M32, STREAM_BAYES ^ (qd >> 32), seed_key(seed))[sid & 3]
    return (-np.log(((u >> U64(9)).astype(np.float64) + 0.5) * 2.0 ** -23)).astype(np.float32)


# tau = 0.01 + (0.99 - 0.01) u.  The SASS of mm_streams_kernel (cuobjdump -sass, sm_100a, nvcc 12.9) is DMUL (u = m 2^-53,
# exact) then one DFMA: nvcc contracts the multiply-add, so tau is the product plus 0.01 rounded once.
MM_TAU_SCALE = Fraction(float(np.float64(0.99) - np.float64(0.01)))


def restate_mm_taus(seed, passes, sims):
    """Random quantiles [len(passes), sims] of the global passes (0 = point pass, r + 1 = replicate r)."""
    p = np.asarray(passes, dtype=U64)[:, None]
    s = np.arange(sims, dtype=U64)[None, :]
    x, y, _, _ = philox(p, p >> U64(32), s, MM_STREAM_TAU, seed_key(seed))
    u53 = ((x << U64(21)) ^ (y >> U64(11))).ravel()
    t = [float(Fraction(0.01) + MM_TAU_SCALE * Fraction(int(m), 2 ** 53)) for m in u53]
    return np.array(t).reshape(len(passes), sims)


def restate_mm_rows(seed, passes, sims, g, counts):
    """Simulated original rows [len(passes), sims] of group g: try t = 0, 1, ..: the Philox call (pass, pass >> 32 ^ t << 8,
    s | g << 31, MM_STREAM_ROW) proposes row umulhi(x:y, n) and accepts it when (z & 63) < min(c_row, 64).
    counts[i] = the multiplicity column of passes[i]."""
    counts = np.asarray(counts, dtype=np.int64)
    P, n = counts.shape
    p = np.repeat(np.asarray(passes, dtype=U64), sims)
    s = np.tile(np.arange(sims, dtype=U64), P) | U64(g << 31)
    which = np.repeat(np.arange(P), sims)
    out = np.zeros(P * sims, dtype=np.int64)
    todo = np.arange(P * sims)
    t = 0
    while todo.size:
        assert t <= 100000
        x, y, z, _ = philox(p[todo], (p[todo] >> U64(32)) ^ U64(t << 8), s[todo], MM_STREAM_ROW, seed_key(seed))
        row = umulhi((x << U64(32)) | y, n).astype(np.int64)
        ok = (z & U64(63)).astype(np.int64) < np.minimum(counts[which[todo], row], 64)
        out[todo[ok]] = row[ok]
        todo = todo[~ok]
        t += 1
    return out.reshape(P, sims)


def mm_row_law(c):
    """The law of one simulated row under the rejection rule above: a proposal is uniform over the rows and is accepted
    with probability min(c_i, 64) / 64."""
    a = np.minimum(np.asarray(c, dtype=np.float64), 64.0)
    return a / a.sum()


# ------------------------------------------------------------------------------------------- CPU
def test_philox_known_answers():
    """The published Random123 known-answer vectors of Philox4x32-10."""
    def hexwords(*a):
        return ["%08x" % int(v) for v in philox(*a[:4], a[4:])]
    assert hexwords(0, 0, 0, 0, 0, 0) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    assert hexwords(M32, M32, M32, M32, M32, M32) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert hexwords(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]
    # vectorised over arrays: the same words element by element
    ctr = np.array([0, M32, 0x243F6A88], dtype=U64)
    assert int(philox(ctr, 0, 0, 0, (0, 0))[0][0]) == 0x6627E8D5


@pytest.mark.parametrize("n", [66, 1000, 20_000, 5_000_000, 10 ** 8])
def test_threshold_table_is_the_poisson_pmf(n):
    """Consecutive thresholds differ by the Poisson pmf (computed directly as e^-lambda lambda^k / k!) to within 2^-62, and
    the table reaches 2^64 - 1 (P(X > 23) < 2^-64)."""
    T = poisson_table(n)
    assert T is not None and T == sorted(T) and T[-1] == 2 ** 64 - 1
    delta = math.isqrt(64 * n - 1) + 1
    assert delta == math.ceil(8 * math.sqrt(n))
    with decimal.localcontext() as dc:
        dc.prec = 80
        lam = decimal.Decimal(n - delta) / n
        prev = 0
        for k in range(KMAX):
            pmf = (-lam).exp() * lam ** k / math.factorial(k)
            assert abs(decimal.Decimal(T[k] - prev) / 2 ** 64 - pmf) <= decimal.Decimal(2) ** -62, (n, k)
            prev = T[k]


def test_lambda_zero_edge():
    """ceil(8 sqrt n) >= n up to n = 65: the body draws nothing there; n = 66 is the first size with a body."""
    assert poisson_table(64) is None and poisson_table(65) is None and poisson_table(66) is not None
    c, amb, tie = restate_counts(65, 3, 4, 0)
    assert c.sum() == 65 and amb == tie == 0


@pytest.mark.parametrize("n", [66, 1000, 20_000, 10 ** 8])
def test_lazy_resolve_is_the_64bit_inverse_cdf(n):
    """counts_lut_kernel + the body's table lookup + poisson_resolve, restated over every 16-bit draw: a 14-bit bucket is
    ambiguous exactly when a threshold falls inside it; for every u16 that ties no threshold's top 16 bits the 16-bit
    decision equals the 64-bit inverse CDF of every U with those top bits; for ties the 64-bit compare does, at the low
    bits 0, 2^48 - 1 and T[k] +- 1."""
    T = poisson_table(n)
    Ta = np.array(T, dtype=U64)
    T16 = Ta >> U64(48)
    amb = bucket_ambiguous(T)
    lo = np.arange(1 << LUT_BITS, dtype=object) << (64 - LUT_BITS)
    inside = np.array([any(int(b) < t <= int(b) + (1 << (64 - LUT_BITS)) - 1 for t in T) for b in lo])
    assert np.array_equal(amb, inside) and 0 < amb.sum() < 64
    lut = np.where(amb, 255, np.searchsorted(Ta, lo.astype(U64), side="right"))

    def cdf(U):
        return np.searchsorted(Ta, np.asarray(U, dtype=U64), side="right")

    u16 = np.arange(1 << 16, dtype=U64)
    tie = np.isin(u16, T16)
    c16 = np.searchsorted(T16, u16, side="left")                 # #{k : u16 > T16[k]}
    decided = np.where(lut[(u16 >> U64(2)).astype(np.int64)] != 255, lut[(u16 >> U64(2)).astype(np.int64)], c16)
    free = ~tie
    for low in (0, (1 << 48) - 1):
        assert np.array_equal(decided[free], cdf((u16[free] << U64(48)) | U64(low))), low
    # a tie is always in an ambiguous bucket, so it always reaches the 64-bit compare
    assert amb[(u16[tie] >> U64(2)).astype(np.int64)].all() and tie.sum() > 0
    for t in T:
        u = t >> 48
        for low in {0, (1 << 48) - 1, max((t & ((1 << 48) - 1)) - 1, 0), t & ((1 << 48) - 1),
                    min((t & ((1 << 48) - 1)) + 1, (1 << 48) - 1)}:
            U = (u << 48) | low
            assert int(cdf(U)) == sum(U >= x for x in T)


def test_restated_counts_sum_to_n():
    """Sanity of the restatement itself: counts sum to n, replicates differ, and ambiguous buckets occur at n = 20 000."""
    c, amb, tie = restate_counts(20_000, 7, 3, 1)
    assert c.sum() == 20_000 and c.min() >= 0 and amb > 0
    c2, _, _ = restate_counts(20_000, 7, 4, 1)
    assert not np.array_equal(c, c2)


def test_mm_row_law():
    """The simulated row is original row i with probability c_i / n while every multiplicity is <= 64 (DESIGN 7c); above
    64 the rejection rule caps the acceptance, which is why ob_mm_run refuses explicit index streams with such counts
    unless the draws are explicit too.  The restated sampler follows the law it is derived from."""
    rng = np.random.default_rng(4)
    for n in (5, 300, 2000):
        c = rng.multinomial(n, np.full(n, 1.0 / n))
        assert c.max() <= 64
        np.testing.assert_allclose(mm_row_law(c), c / n, rtol=1e-15, atol=0)
    c = np.zeros(300, dtype=np.int64)
    c[0], c[1:101] = 200, 1          # 300 draws: row 0 drawn 200 times
    assert c.sum() == 300
    assert abs(c[0] / 300 - 2 / 3) < 1e-15 and abs(mm_row_law(c)[0] - 64 / 164) < 1e-15
    # the restated sampler, 200 000 draws against the law (seeded: deterministic)
    c = np.zeros(40, dtype=np.int64)
    c[:20] = rng.integers(0, 65, 20)
    c[20] = 64
    rows = restate_mm_rows(11, np.arange(1, 201), 1000, 0, np.tile(c, (200, 1))).ravel()
    f = np.bincount(rows, minlength=40)
    p = mm_row_law(c)
    assert (f[p == 0] == 0).all()
    e = p[p > 0] * rows.size
    chi2 = float((((f[p > 0] - e) ** 2) / e).sum())
    from scipy.stats import chi2 as chi2_dist
    assert chi2_dist.sf(chi2, (p > 0).sum() - 1) > 1e-4, chi2


# ------------------------------------------------------------------------------------------- GPU
SEEDS = (0, 7, 2 ** 64 - 1, 0x9E3779B97F4A7C15)
REPS = tuple(range(16)) + (2 ** 32 + 3, 2 ** 35 + 5)     # every octet phase SH; the high words of the counters


def _pack(ctx, na, nb, seed, codes=None):
    """A design with exactly na rows in group A and nb in group B, interleaved in the frame."""
    import oaxaca_blinder_rs_b200 as ob
    rng = np.random.default_rng(seed)
    grp = np.r_[np.zeros(na), np.ones(nb)].astype(np.uint8)
    rng.shuffle(grp)
    n = na + nb
    x = rng.normal(size=n)
    cat = rng.integers(0, 3, n).astype(np.int32)
    y = 1.0 + 0.2 * x + 0.3 * (grp == 0) + 0.1 * (cat == 1) + rng.standard_t(4, n)
    return ob.Design.pack(ctx, [x, rng.uniform(0, 10, n)], [cat], [3], y, None, grp), grp


@pytest.mark.gpu
def test_debug_counts_equal_the_restatement():
    import oaxaca_blinder_rs_b200 as ob
    ctx = ob.Context(0)
    tally, bad = [0, 0], []
    for n in (64, 65, 66, 1000, 20_001, 200_003):
        des, _ = _pack(ctx, n, n, seed=n)
        T = poisson_table(n)
        for g in (0, 1):
            for seed in SEEDS:
                for rep in REPS:
                    got = des.debug_counts(seed, rep, g).astype(np.int64)
                    want, amb, tie = restate_counts(n, seed, rep, g, T)
                    tally[0] += amb
                    tally[1] += tie
                    if not np.array_equal(got, want):
                        bad.append((n, g, seed, rep, int((got != want).sum())))
        des.close()
    ctx.close()
    assert not bad, f"(n, group, seed, rep, rows differing): {bad[:12]} ({len(bad)} cases)"
    # both lazy paths were exercised: the 16-bit resolve of ambiguous buckets and the 48 refinement bits of exact ties
    assert tally[0] >= 500 and tally[1] >= 100, tally


@pytest.mark.gpu
@pytest.mark.parametrize("strata", ["group", "joint"])
def test_clustered_debug_counts_equal_the_restated_unit_counts(strata):
    """A clustered replicate draws counts over units (stream group 0 / 1, or 2 for JOINT) and gives every row its unit's
    count; a unit is the rank of its code among the stratum's present codes."""
    import oaxaca_blinder_rs_b200 as ob
    ctx = ob.Context(0)
    rng = np.random.default_rng(8)
    n = 9000
    des, grp = _pack(ctx, 4000, 5000, seed=3)
    cases = {"gapped": (rng.integers(0, 700, n) * 7 + 3).astype(np.int32),       # codes with gaps, units in [~650, 700]
             "few": rng.choice(np.array([5, 90, 91, 4000, 4001, 77777], np.int32), n),   # M <= 65: lambda_zero units
             "one_per_row": rng.permutation(n).astype(np.int32)}                 # a unit per row, codes out of frame order
    bad = []
    for name, codes in cases.items():
        des.attach_clusters(codes, strata=strata)
        cg = [codes[grp == 0], codes[grp == 1]]
        if strata == "group":
            units = [np.unique(cg[0]), np.unique(cg[1])]
        else:
            units = [np.unique(codes)] * 2
        cl = des.clusters
        assert (cl["units_a"], cl["units_b"]) == (len(units[0]), len(units[1]))
        for seed in (0, 2 ** 64 - 1, 12345678901234):
            for rep in (0, 1, 5, 2 ** 35 + 5):
                if strata == "joint":
                    uc = restate_counts(len(units[0]), seed, rep, 2)[0]
                for g in (0, 1):
                    if strata == "group":
                        uc = restate_counts(len(units[g]), seed, rep, g)[0]
                    want = uc[np.searchsorted(units[g], cg[g])]
                    got = des.debug_counts(seed, rep, g).astype(np.int64)
                    if not np.array_equal(got, want):
                        bad.append((name, seed, rep, g, int((got != want).sum())))
    des.close(); ctx.close()
    assert not bad, bad[:12]


@pytest.mark.gpu
def test_debug_bayes_weights_equal_the_restatement():
    """Every weight within 1 fp32 ulp of the restatement (CUDA's logf is accurate to 1 ulp)."""
    import oaxaca_blinder_rs_b200 as ob
    ctx = ob.Context(0)
    bad, worst = [], 0
    for n in (64, 66, 1000, 20_001, 200_003):
        des, _ = _pack(ctx, n, n, seed=n + 1)
        for g in (0, 1):
            for seed in (0, 2 ** 64 - 1, 0x9E3779B97F4A7C15):
                for rep in (0, 1, 2, 3, 6, 2 ** 32 + 3, 2 ** 35 + 5):
                    got = des.debug_bayes_weights(seed, rep, g)
                    want = restate_bayes(n, seed, rep, g)
                    ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
                    worst = max(worst, int(ulps.max()))
                    if ulps.max() > 1 or not (got > 0).all():
                        bad.append((n, g, seed, rep, int((ulps > 1).sum())))
        des.close()
    ctx.close()
    assert not bad, f"(n, group, seed, rep, weights off by > 1 ulp): {bad[:12]}; worst {worst} ulp"


def _mm_frame(n, seed):
    rng = np.random.default_rng(seed)
    grp = rng.integers(0, 2, n).astype(np.uint8)
    x = rng.normal(12, 2, n) + 0.5 * (grp == 0)
    x2 = rng.uniform(0, 30, n)
    cat = rng.integers(0, 3, n).astype(np.int32)
    y = 1.0 + 0.3 * (grp == 0) + 0.08 * x + 0.01 * x2 + 0.1 * (cat == 1) + rng.standard_t(4, n) * 0.3
    return [x, x2], cat, y, grp


@pytest.mark.gpu
def test_mm_native_run_equals_the_run_rebuilt_from_restated_streams():
    """A native Machado-Mata run, and the same run with every stream restated on the host and passed explicitly: the
    resamples as index streams (np.repeat of the restated counts), the restated quantiles, and as draws the first position
    of each restated simulated row in its pass's resampled frame.  Point statistics, replicate statistics, the point
    pass's coefficients and the reduction must be the same bits, under two batch splits and a replicate shard."""
    import oaxaca_blinder_rs_b200 as ob
    cont, cat, y, grp = _mm_frame(1500, 3)
    na, nb = int((grp == 0).sum()), int((grp == 1).sum())
    seed, reps, sims = 0xC0FFEE12345, 300, 8
    ctx = ob.Context(0)
    des = ob.Design.pack(ctx, cont, [cat], [3], y, None, grp)
    kw = dict(quantiles=[0.25, 0.5, 0.75], simulations=sims, reps=reps, want_rep=True, want_betas=True)
    native = ob.machado_mata(des, seed=seed, **kw)
    native_small = ob.machado_mata(des, seed=seed, max_workspace_bytes=1_000_000, **kw)     # one 128-slot panel per batch
    native_part = ob.machado_mata(des, seed=seed, rep_begin=130, rep_end=260, skip_reduce=True, **kw)

    passes = np.arange(reps + 1)                      # 0 = point pass, r + 1 = replicate r
    st = dict(taus=restate_mm_taus(seed, passes, sims))
    for g, n in ((0, na), (1, nb)):
        cnt = np.stack([np.ones(n, np.int64)] + [restate_counts(n, seed, r, g)[0] for r in range(reps)])
        assert cnt.max() <= 64
        rows = restate_mm_rows(seed, passes, sims, g, cnt)
        first = np.cumsum(cnt, axis=1) - cnt          # position of a row's first copy in np.repeat(arange(n), c)
        st["idx_a" if g == 0 else "idx_b"] = np.stack([np.repeat(np.arange(n), c) for c in cnt[1:]]).astype(np.uint32)
        st["draw_a" if g == 0 else "draw_b"] = np.take_along_axis(first, rows, axis=1).astype(np.uint32)
    explicit = ob.machado_mata(des, **st, **kw)
    explicit_small = ob.machado_mata(des, max_workspace_bytes=1_000_000, **st, **kw)
    explicit_part = ob.machado_mata(des, rep_begin=130, rep_end=260, skip_reduce=True, **st, **kw)
    des.close(); ctx.close()

    assert native["qr"]["failed"] == 0 and native["n_ok"] == reps
    assert native_small["gpu_launches"] > native["gpu_launches"]
    keys = ("point_stats", "rep_stats", "rep_status", "point_betas_a", "point_betas_b", "std_err", "p_value", "ci_lower",
            "ci_upper", "t_stat")
    for a, b in ((native, explicit), (native_small, explicit), (native, explicit_small)):
        for k in keys:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
        assert a["qr"] == b["qr"]
    for k in ("point_stats", "rep_stats", "rep_status", "point_betas_a", "point_betas_b"):
        assert np.array_equal(native_part[k], explicit_part[k], equal_nan=True), k
    assert np.array_equal(native_part["rep_stats"], native["rep_stats"][130:260])


@pytest.mark.gpu
def test_mm_refuses_explicit_resamples_it_cannot_draw_rows_from():
    """With an explicit index stream and no explicit draws, the simulated rows are drawn natively against the explicit
    multiplicities, by a rejection rule whose law is c_i / n only for c_i <= 64.  A multiplicity above 64 is refused
    (draws passed explicitly are still accepted); 64 itself is not."""
    import oaxaca_blinder_rs_b200 as ob
    cont, cat, y, grp = _mm_frame(600, 5)
    na, nb = int((grp == 0).sum()), int((grp == 1).sum())
    rng = np.random.default_rng(9)
    reps, sims = 3, 8
    ia = rng.integers(0, na, size=(reps, na)).astype(np.uint32)
    ib = rng.integers(0, nb, size=(reps, nb)).astype(np.uint32)
    ctx = ob.Context(0)
    des = ob.Design.pack(ctx, cont, [cat], [3], y, None, grp)
    kw = dict(quantiles=[0.5], simulations=sims, reps=reps)
    ok = ob.machado_mata(des, idx_a=ia, idx_b=ib, **kw)
    assert ok["n_ok"] == reps
    at64 = ib.copy()
    at64[1, 64:][at64[1, 64:] == 7] = 8
    at64[1, :64] = 7                                  # row 7 drawn exactly 64 times
    ob.machado_mata(des, idx_a=ia, idx_b=at64, **kw)
    over = ia.copy()
    over[2, :200] = 0                                 # row 0 drawn at least 200 times in replicate 2
    taus = rng.uniform(0.01, 0.99, size=(reps + 1, sims))
    for extra in ({}, dict(taus=taus), dict(rep_begin=2, rep_end=3)):
        with pytest.raises(ob.OaxacaError) as e:
            ob.machado_mata(des, idx_a=over, idx_b=ib, **extra, **kw)
        assert e.value.kind == "Unsupported" and "draw_a" in str(e.value), str(e.value)
    # a shard without the offending replicate is not refused
    ob.machado_mata(des, idx_a=over, idx_b=ib, rep_begin=0, rep_end=2, skip_reduce=True, **kw)
    draws = dict(taus=taus, draw_a=rng.integers(0, na, size=(reps + 1, sims)).astype(np.uint32),
                 draw_b=rng.integers(0, nb, size=(reps + 1, sims)).astype(np.uint32))
    assert ob.machado_mata(des, idx_a=over, idx_b=ib, **draws, **kw)["point_stats"].shape == (1, 3)
    des.close(); ctx.close()
