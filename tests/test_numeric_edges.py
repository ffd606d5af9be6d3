"""The exact top-k across the fp32 range, at k = MAX_K and through every merge mode (DESIGN.md section 4).

The exactness claim rests on the prefilter margin being an upper bound of the prefilter error.  Its inputs (norm
and error bounds of rows and queries) are sums of squares, which an fp32 sum flushes to zero below 2^-149 and
overflows above FLT_MAX.  These tests need no tolerance of their own: scaling rows by 2^a and queries by 2^b is
exact, and so are the reported scores (fp64 products, fixed order, one rounding), so an exact engine returns the
same ids and the scores times exactly 2^(a+b) as long as they are normal fp32 numbers.

CPU part: a numpy restatement of the bound arithmetic (kernels_util.cuh, pass_init_kernel), checked against the
fp64 truth on rows and queries scaled 2^-149 ... 2^127.
GPU part: power-of-two rescaling with a planted near-tie cluster (A), mixed magnitudes in one batch and one shard
(B), k at its limits (C) and every merge mode (D), on every scoring engine.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)

# ------------------------------------------------------------------------------------------------ CPU restatement


def ru32(x):
    """Smallest float32 >= x (x exact: Fraction or float); +inf above FLT_MAX."""
    x = Fraction(x)
    if x > FLT_MAX:
        return math.inf
    with np.errstate(over="ignore"):
        f = F32(float(x))
    if math.isinf(f):
        return FLT_MAX
    if Fraction(float(f)) < x:
        f = np.nextafter(f, F32(np.inf))
    return float(f)


def mul_ru(a, b):
    return math.inf if math.isinf(a) or math.isinf(b) else ru32(Fraction(a) * Fraction(b))


def add_ru(a, b):
    return math.inf if math.isinf(a) or math.isinf(b) else ru32(Fraction(a) + Fraction(b))


def sqrt_ru(a):
    if math.isinf(a):
        return math.inf
    r = F32(math.sqrt(a))
    while Fraction(float(r)) ** 2 < Fraction(a):
        r = np.nextafter(r, F32(np.inf))
    return float(r)


def bound_mul(a, b):
    return 0.0 if a == 0.0 or b == 0.0 else mul_ru(a, b)


def sumsq_upper(s):
    """sumsq_upper(): the fp64 sum times (1 + 2^-40) rounded up, then rounded up to fp32."""
    t = Fraction(s) * (1 + Fraction(1, 2**40))
    d = float(t)
    if Fraction(d) < t:
        d = math.nextafter(d, math.inf)
    return ru32(d)


def lane_sumsq(x):
    """Per row, the fp64 sum of squares in the kernels' order: lane l sums components 4(l + 32 i) + j (i outer, j
    inner), then the five butterfly steps of the warp; lane 0's value.  x: float32 [n, 768]."""
    sq = x.astype(np.float64) ** 2                       # exact: the square of an fp32 value fits fp64
    sq = sq.reshape(len(x), 6, 32, 4)
    acc = np.zeros((len(x), 32))
    for i in range(6):
        for j in range(4):
            acc = acc + sq[:, i, :, j]
    lanes = np.arange(32)
    for s in (16, 8, 4, 2, 1):
        acc = acc + acc[:, lanes ^ s]
    return acc[:, 0]


K_SUBNORMAL_NORM = 2.0**-145
K_SUBNORMAL_ABS = 2.0**-115


def shadow_err_upper(s, cn, rel_round):
    e = sqrt_ru(sumsq_upper(s))
    if rel_round:
        e = add_ru(mul_ru(e, float(F32(1.0000001))), K_SUBNORMAL_NORM)
    return add_ru(add_ru(e, mul_ru(cn, float(F32(6.0e-8)))), K_SUBNORMAL_NORM)


def centred_norm2_upper(cn):
    c = add_ru(mul_ru(cn, float(F32(1.0000001))), K_SUBNORMAL_NORM)
    return mul_ru(c, c)


def bf16_rn(x):
    """Round-to-nearest-even float32 -> bfloat16 (as float32); values past the bf16 range round to inf."""
    u = np.ascontiguousarray(x, dtype=F32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(F32)


def fma32(a, b, c):
    """fl32(a * b + c) for float32 arrays (the fp64 value is exact here: a 24-bit by 8-bit product plus a value of
    the same scale), rounded once."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


def quant8(x, amax):
    amax = F32(amax)
    with np.errstate(over="ignore", divide="ignore", invalid="ignore"):
        inv = F32(127.0) / amax if amax > 0 else F32(0.0)
        v = np.nan_to_num((x.astype(F32) * inv).astype(F32), nan=0.0)
    return np.clip(np.rint(v), -127, 127).astype(F32)


def row_bounds(X, mu):
    """The three per-shard slots of convert_rows_kernel (bf16) and slot [1] of convert_rows_i8_kernel, as the
    square roots the margin uses: (P_uncentred, E_bf16, P_centred, E_int8) and the shadows themselves."""
    d = (X - mu).astype(F32)
    cn = [sqrt_ru(sumsq_upper(s)) for s in lane_sumsq(d)]
    w = max(sumsq_upper(s) for s in lane_sumsq(X))
    p16 = bf16_rn(d)
    e16 = max(mul_ru(e, e) for e in (shadow_err_upper(s, c, False) for s, c in zip(lane_sumsq(d - p16), cn)))
    c = max(centred_norm2_upper(v) for v in cn)
    st = np.zeros(len(X), dtype=F32)
    p8 = np.zeros_like(d)
    for t in range(0, len(X), 32):
        amax = np.abs(d[t:t + 32]).max()
        st[t:t + 32] = F32(amax) / F32(127.0)
        p8[t:t + 32] = quant8(d[t:t + 32], amax)
    r8 = fma32(-st[:, None], p8, d)
    e8 = max(mul_ru(e, e) for e in (shadow_err_upper(s, c_, True) for s, c_ in zip(lane_sumsq(r8), cn)))
    return (sqrt_ru(w), sqrt_ru(e16), sqrt_ru(c), sqrt_ru(e8)), p16, st, p8


def query_bounds(q):
    """prep_queries_kernel (bf16) and prep_queries_i8_kernel: ||q||, ||q - bf16(q)||, sq, q8, ||q - sq q8||."""
    qn = sqrt_ru(sumsq_upper(lane_sumsq(q[None])[0]))
    qe = sqrt_ru(sumsq_upper(lane_sumsq((q - bf16_rn(q))[None])[0]))
    amax = np.abs(q).max()
    sq = F32(amax) / F32(127.0)
    q8 = quant8(q, amax)
    r = fma32(np.full_like(q, -sq), q8, q)
    qe8 = add_ru(mul_ru(sqrt_ru(sumsq_upper(lane_sumsq(r[None])[0])), float(F32(1.0000001))), K_SUBNORMAL_NORM)
    if amax == 0:
        qe8 = 0.0                        # a zero query is coded exactly
    return qn, qe, sq, q8, qe8


def eps_bf16(qn, qe, E, P):
    """pass_init_kernel mode 2 (before the factor 2 of the margin); None: the query takes the exact fallback."""
    a = bound_mul(bound_mul(qn, E), 1.00390625)
    b = bound_mul(qe, P)
    c = bound_mul(bound_mul(qn, P), float(F32(1.1e-4)))
    eps = add_ru(add_ru(add_ru(a, b), c), K_SUBNORMAL_ABS)
    return eps if math.isfinite(eps) and math.isfinite(mul_ru(eps, 2.0)) else None


def eps_int8(qn, qe, E8, P):
    """pass_init_kernel mode 4."""
    qh = add_ru(qn, qe)
    a = bound_mul(qh, E8)
    b = bound_mul(qe, P)
    c = bound_mul(bound_mul(qh, add_ru(P, E8)), 2.0**-21)
    eps = add_ru(add_ru(add_ru(a, b), c), K_SUBNORMAL_ABS)
    return eps if math.isfinite(eps) and math.isfinite(mul_ru(eps, 2.0)) else None


def _base_rows(rng, n=64):
    X = rng.standard_normal((n, 768)).astype(F32)
    X /= np.linalg.norm(X, axis=1, keepdims=True).astype(F32)
    X[5] = 0.0                           # a zero row
    X[9, 100] = 0.9                      # one large component
    X[40:] *= F32(2.0**-10)              # a tile of short rows: its int8 scale is its own
    return X.astype(F32)


def _norm(v):
    """fp64 norm of an exactly-known fp64 vector, with the squares summed exactly."""
    return math.sqrt(math.fsum((v.astype(np.float64) ** 2).tolist()))


SCALES = [-149, -140, -130, -126, -100, -75, -70, -62, -55, -20, 0, 20, 40, 60, 63, 64, 100, 120, 127]


@pytest.mark.parametrize("a", SCALES)
def test_norm_and_error_bounds_hold_over_the_fp32_range(a):
    """Every bound kept at ingest and computed per query is >= the fp64 truth, is never 0 for a nonzero vector, and
    is +inf (not a wrong finite value) where the truth exceeds FLT_MAX."""
    rng = np.random.default_rng(a & 0xffff)
    with np.errstate(under="ignore", over="ignore"):
        X = (_base_rows(rng) * np.float64(2.0**a)).astype(F32)
        for mu in (X[:16].mean(0, dtype=np.float64).astype(F32), np.zeros(768, F32)):
            (P0, E16, Pc, E8), p16, st, p8 = row_bounds(X, mu)
            exact_pc = X.astype(np.float64) - mu.astype(np.float64)   # exact: same-scale fp32 operands
            assert P0 >= max(_norm(x) for x in X)
            assert Pc >= max(_norm(x) for x in exact_pc)
            assert E16 >= max(_norm(x - y) for x, y in zip(exact_pc, p16.astype(np.float64)))
            ph8 = p8.astype(np.float64) * st[:, None].astype(np.float64)
            assert E8 >= max(_norm(x - y) for x, y in zip(exact_pc, ph8))
            if np.any(X != 0):
                assert P0 > 0
            if np.any(X != mu):
                assert Pc > 0
        for q in X[[0, 5, 9, 50]]:
            qn, qe, sq, q8, qe8 = query_bounds(q)
            assert qn >= _norm(q) and (qn > 0) == bool(np.any(q != 0))
            assert qe >= _norm(q.astype(np.float64) - bf16_rn(q).astype(np.float64))
            assert qe8 >= _norm(q.astype(np.float64) - q8.astype(np.float64) * np.float64(sq))


MARGIN_PAIRS = [(0, 0), (20, -20), (-20, 20), (40, 40), (-58, 58), (-75, 70), (70, -75), (64, -62), (-62, 64),
                (-55, -60), (-149, 120), (127, -127), (-100, -20)]


@pytest.mark.parametrize("a,b", MARGIN_PAIRS)
def test_margin_covers_the_prefilter_error_or_sends_the_query_to_the_exact_engine(a, b):
    """eps of the bf16 and int8 modes, from the restated bounds, is >= |s~ - s| for every row (s~ the prefilter score
    in exact arithmetic, s the exact centred score), or not finite, which flags the query for the exact engine.  It
    is never NaN, also for a zero query against rows whose norm bound is +inf."""
    rng = np.random.default_rng(7)
    with np.errstate(under="ignore", over="ignore"):
        X = (_base_rows(rng, 64) * np.float64(2.0**a)).astype(F32)
        Q = (_base_rows(np.random.default_rng(8), 16)[[0, 5, 9, 12]] * np.float64(2.0**b)).astype(F32)   # [1] = 0
        mu = X[:16].mean(0, dtype=np.float64).astype(F32)
        (_, E16, Pc, E8), p16, st, p8 = row_bounds(X, mu)
        ph8 = p8.astype(np.float64) * st[:, None].astype(np.float64)
        for q in Q:
            qn, qe, sq, q8, qe8 = query_bounds(q)
            e2, e4 = eps_bf16(qn, qe, E16, Pc), eps_int8(qn, qe8, E8, Pc)
            assert not (e2 is not None and math.isnan(e2)) and not (e4 is not None and math.isnan(e4))
            if not np.any(q):
                assert e2 is not None and e4 is not None, "a zero query has a finite margin"
            qh16 = bf16_rn(q).astype(np.float64)
            qh8 = q8.astype(np.float64) * np.float64(sq)
            q64 = q.astype(np.float64)
            for i in range(len(X)):
                exact = [*(q64 * X[i]).tolist(), *(-q64 * mu).tolist()]   # q.(x - mu), exact products
                if e2 is not None:
                    err = abs(math.fsum([*(qh16 * p16[i]).tolist(), *[-t for t in exact]]))
                    assert e2 >= err, (i, e2, err)
                if e4 is not None:
                    err = abs(math.fsum([*(qh8 * ph8[i]).tolist(), *[-t for t in exact]]))
                    assert e4 >= err, (i, e4, err)


def test_restated_bounds_detect_the_fp32_sum_failures():
    """The two failures of fp32 sums of squares that the fp64 sums remove: a row at 2^-75 has a zero fp32 norm
    bound, a row at 2^64 an infinite one although its norm is finite."""
    x = _base_rows(np.random.default_rng(3), 16)[0]
    with np.errstate(under="ignore", over="ignore"):
        tiny, huge = (x * F32(2.0**-75)).astype(F32), (x * F32(2.0**64)).astype(F32)
        assert float(np.sum(tiny * tiny, dtype=F32)) == 0.0
        assert math.isinf(float(np.sum(huge * huge, dtype=F32)))
    assert 0 < _norm(tiny) <= sqrt_ru(sumsq_upper(lane_sumsq(tiny[None])[0]))
    assert math.isinf(sqrt_ru(sumsq_upper(lane_sumsq(huge[None])[0]))) and math.isfinite(_norm(huge))


# ------------------------------------------------------------------------------------------------ GPU

# (path, umma_variant, shadow, center): every scoring engine, forced, plus AUTO and one uncentred tensor shard
ENGINES = {
    "scan_exact": ("scan_exact", 0, 1, 1), "scan_f32": ("scan_f32", 0, 1, 1),
    "qs_bf16": ("umma_bf16", 3, 1, 1), "qs_i8": ("umma_bf16", 3, 2, 1),
    "ts_bf16": ("umma_bf16", 2, 1, 1), "ts_i8": ("umma_bf16", 2, 2, 1),
    "auto": None, "qs_i8_uncentred": ("umma_bf16", 3, 2, 0),
}


def make_index(engine, P=None):
    from convdr_b200 import FlatIPIndex
    idx = FlatIPIndex(768)
    if ENGINES[engine] is not None:
        path, variant, shadow, center = ENGINES[engine]
        idx.set_option("path", path)
        idx.set_option("umma_variant", variant)
        idx.set_option("shadow", shadow)
        idx.set_option("center", center)
    if P is not None:
        idx.add(P)
    return idx


def search(engine, P, Q, k):
    """(D, I, fallback_queries) of one search on a fresh index."""
    idx = make_index(engine, P)
    D, I = idx.search(Q, k)
    f = idx.stat("fallback_queries")
    idx.close()
    return D, I, f


def scale(x, e):
    """x * 2^e for float32 arrays, exact as long as the results stay normal."""
    return np.ldexp(x, e).astype(F32)


def check_truth(D, I, P, Q, k, what):
    from oracle import flat_ip
    Dt, It = flat_ip.truth_fp64(Q, P, k)
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    r = flat_ip.compare(D, I, Dt, It, score_of, rtol=1e-5)
    assert r["violations"] == 0, (what, r)
    return Dt, It


N_A, K_A, CLUSTER_Q = 20000, 64, 0


@pytest.fixture(scope="module")
def scaled_data():
    """20k rows and 40 queries: 36 synthetic, a zero query, a bf16-exact one, an int8-exact one (small integers
    times 2^-7) and a copy of a stored row.  Query 0 gets a near-tie cluster: 64 rows whose exact scores are
    distinct in fp32 but spaced ~2^-21 apart, far below the bf16 and int8 prefilter resolution, straddling
    position K_A."""
    from oracle import c_oracle, flat_ip
    P = c_oracle.synth_block(0, N_A, seed=61)
    Q = c_oracle.synth_block(0, 40, seed=61, stream=1)
    Q[36] = 0.0
    Q[37] = bf16_rn(Q[37])
    ints = np.random.default_rng(4).integers(-127, 128, 768)
    ints[3] = 127
    Q[38] = (ints * 2.0**-7).astype(F32)
    Q[39] = P[1234]
    q = Q[CLUSTER_Q].astype(np.float64)
    _, It = flat_ip.truth_fp64(Q[CLUSTER_Q:CLUSTER_Q + 1], P, K_A)
    base = P[It[0, K_A // 2 - 1]].copy()     # the cluster takes ranks K_A/2 ... 3 K_A/2 - 1
    c = int(np.argmax(np.abs(q)))
    rows = np.random.default_rng(5).choice(np.setdiff1d(np.arange(N_A), It[0]), 64, replace=False)
    for j, r in enumerate(rows):
        P[r] = base
        P[r, c] = F32(base[c] + np.sign(q[c]) * (j - 32) * 2.0**-18)
    s = P[rows].astype(np.float64) @ q
    assert len(set(s.astype(F32).tolist())) == 64, "cluster scores must be distinct in fp32"
    return P, Q, rows


@pytest.fixture(scope="module")
def base_results(scaled_data):
    P, Q, rows = scaled_data
    out = {}
    for e in ENGINES:
        out[e] = search(e, P, Q, K_A)
    D0, I0, _ = out["scan_exact"]
    Dt, It = check_truth(D0, I0, P, Q, K_A, "scan_exact")
    assert np.array_equal(I0[CLUSTER_Q], It[CLUSTER_Q]), "near-tie cluster: the exact order is the fp64 order"
    assert len(np.intersect1d(I0[CLUSTER_Q], rows)) == 32, "the cluster straddles position k"
    for e, (D, I, _) in out.items():
        assert np.array_equal(I, I0) and D.tobytes() == D0.tobytes(), e
    return out


NORMAL_PAIRS = [(0, 0), (20, -20), (-20, 20), (20, 20), (-20, -20), (40, 40)]
EXTREME_PAIRS = [(-58, 58), (-62, 60), (-75, 70), (70, -75), (64, -62), (-62, 64), (-55, -60)]


@pytest.mark.gpu
@pytest.mark.parametrize("a,b", NORMAL_PAIRS + EXTREME_PAIRS)
def test_power_of_two_rescaling_is_exact_on_every_engine(a, b, scaled_data, base_results):
    """Rows x 2^a, queries x 2^b: every engine returns the base ids and the base scores times exactly 2^(a+b).
    Where every intermediate stays normal, the fallback count is the base run's as well."""
    P, Q, _ = scaled_data
    Ps, Qs = scale(P, a), scale(Q, b)
    Dx, Ix, _ = search("scan_exact", Ps, Qs, K_A)
    D0, I0, _ = base_results["scan_exact"]
    want = scale(D0, a + b)
    assert np.all(np.isfinite(want)) and np.all((np.abs(want) >= np.finfo(F32).tiny) | (want == 0))
    report = {}
    for e in ENGINES:
        D, I, f = search(e, Ps, Qs, K_A) if e != "scan_exact" else (Dx, Ix, 0.0)
        report[e] = f
        bad = np.nonzero(np.any(I != I0, axis=1) | np.any(D.view(np.uint32) != want.view(np.uint32), axis=1))[0]
        assert len(bad) == 0, f"{e} at (2^{a}, 2^{b}): queries {bad.tolist()} differ, fallback_queries={f}"
        assert np.array_equal(I, Ix) and D.tobytes() == Dx.tobytes(), e
        if (a, b) in NORMAL_PAIRS:
            assert f == base_results[e][2], f"{e}: fallback_queries {f} != base {base_results[e][2]}"
    print(f"fallback_queries at (2^{a}, 2^{b}):", report)


@pytest.mark.gpu
def test_a_batch_of_queries_from_2m40_to_2p40_equals_each_query_alone():
    """173 queries with scales 2^-40 ... 2^40 in one batch (QS chunks of 16 queries share a threshold snapshot,
    int8 queries have one scale each): row i of the batch is the unscaled batch's row times 2^b_i, and a query
    searched alone returns the same row."""
    from oracle import c_oracle
    P = c_oracle.synth_block(0, 30000, seed=62)
    Q = c_oracle.synth_block(0, 173, seed=62, stream=1)
    e = np.array([-40 + (80 * i) // 172 for i in range(173)])
    Qs = np.stack([scale(q, int(x)) for q, x in zip(Q, e)])
    D0, I0, _ = search("scan_exact", P, Q, 50)
    check_truth(D0, I0, P, Q, 50, "scan_exact")
    want = np.stack([scale(d, int(x)) for d, x in zip(D0, e)])
    for eng in ENGINES:
        idx = make_index(eng, P)
        D, I = idx.search(Qs, 50)
        assert np.array_equal(I, I0) and D.tobytes() == want.tobytes(), eng
        for i in (0, 1, 15, 16, 86, 171, 172):
            Da, Ia = idx.search(Qs[i:i + 1], 50)
            assert np.array_equal(Ia[0], I[i]) and Da[0].tobytes() == D[i].tobytes(), (eng, i)
        idx.close()


@pytest.mark.gpu
def test_a_shard_with_tiles_at_2m30_20_and_2p20():
    """32-row tiles at 2^-30 and 2^0 (different int8 tile scales) and one tile at 2^20 whose rows inflate the
    shard-wide margin: exact on every engine (fallbacks allowed) and bit-identical across engines."""
    from oracle import c_oracle
    P = c_oracle.synth_block(0, 20000, seed=63)
    Q = c_oracle.synth_block(0, 64, seed=63, stream=1)
    t = np.arange(len(P)) // 32
    ex = np.where(t % 2 == 1, -30, 0)
    ex[t == 100] = 20
    P = np.ldexp(P, ex[:, None]).astype(F32)
    D0, I0, _ = search("scan_exact", P, Q, 100)
    check_truth(D0, I0, P, Q, 100, "scan_exact")
    assert np.isin(np.arange(3200, 3232), I0).all(), "the 2^20 tile is in every top-100"
    for eng in ENGINES:
        D, I, f = search(eng, P, Q, 100)
        assert np.array_equal(I, I0) and D.tobytes() == D0.tobytes(), (eng, f)


K_VALUES = [1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2047, 2048]
N_BIG = 20000


@pytest.fixture(scope="module")
def k_data():
    """Rows in runs of three identical rows (exact ties at every rank, so across position k for most queries) and
    209 queries: one more than the largest batch AUTO runs on the QS kernel."""
    from oracle import c_oracle
    B = c_oracle.synth_block(0, N_BIG // 3 + 1, seed=64)
    return np.repeat(B, 3, axis=0)[:N_BIG].copy(), c_oracle.synth_block(0, 209, seed=64, stream=1)


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_VALUES)
def test_k_at_its_limits_on_every_engine(k, k_data):
    """n in {k-1, k, k+1, 20000}, 208 and 209 queries: every engine equals the exact engine bit for bit, the
    exact engine agrees with the fp64 truth, ties keep the insertion order, and padding is -1 / -FLT_MAX."""
    P_all, Q = k_data
    idx = {e: make_index(e) for e in ENGINES}
    for n in sorted({max(1, k - 1), k, k + 1, N_BIG}):
        P = P_all[:n]
        ref = {}
        for e, ix in idx.items():
            ix.reset()
            ix.add(P)
            for nq in (208, 209):
                D, I = ix.search(Q[:nq], k)
                if e == "scan_exact":
                    ref[nq] = (D, I)
                    if nq == 209:
                        check_truth(D, I, P, Q, k, f"scan_exact n={n} k={k}")
                        tie = D[:, 1:] == D[:, :-1]
                        valid = I[:, 1:] >= 0
                        assert np.all(I[:, 1:][tie & valid] > I[:, :-1][tie & valid]), "ties in insertion order"
                        if n < k:
                            assert (I[:, n:] == -1).all() and (D[:, n:] == -F32(FLT_MAX)).all()
                        assert np.array_equal(ref[208][1], I[:208]) and ref[208][0].tobytes() == D[:208].tobytes()
                D0, I0 = ref[nq]
                assert np.array_equal(I, I0) and D.tobytes() == D0.tobytes(), f"{e} n={n} k={k} nq={nq}"
    for ix in idx.values():
        ix.close()


@pytest.mark.gpu
def test_k_beyond_max_k_is_rejected_and_rank_dedup_takes_top_max_k(k_data):
    import torch
    import convdr_b200.faiss_compat as faiss
    from convdr_b200.index import MAX_K
    from oracle import flat_ip
    assert MAX_K == 2048
    P, Q = k_data
    idx = make_index("auto", P)
    qd = torch.from_numpy(Q[:7]).cuda()
    with pytest.raises(RuntimeError):
        idx.search(Q[:7], MAX_K + 1)
    with pytest.raises(RuntimeError):
        idx.search_device(qd, MAX_K + 1)
    with pytest.raises(RuntimeError):
        idx.search(Q[:7], MAX_K + 1, params=faiss.SearchParameters(sel=faiss.IDSelectorRange(0, 5000)))
    D, I = idx.search_device(qd, MAX_K)
    offset2pid = (np.arange(N_BIG, dtype=np.int64) // 3)         # the three copies of a row share a passage id
    want = flat_ip.eval_rank_dedup(D.cpu().numpy(), I.cpu().numpy(), MAX_K, offset2pid)
    got = idx.rank_dedup(I, D, MAX_K, torch.from_numpy(offset2pid).cuda())
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.cpu().numpy(), w)
    idx.close()


def _merge_mode(G, k):
    """kernels_select.cuh merge_mode(): 2 = sort in shared memory, 1 = rank-by-counting over staged lists, 0 = out
    of L2."""
    p2 = 32
    while p2 < G * k:
        p2 <<= 1
    if G >= 4 and p2 * 8 <= 96 * 1024:
        return 2
    return 1 if G * k * 12 <= 96 * 1024 else 0


MERGES = [(2, 2048), (3, 2048), (4, 2048), (5, 2048), (8, 2048), (16, 2048), (16, 100), (40, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("G,k", MERGES)
def test_every_merge_mode_equals_the_search_of_the_whole_index(G, k):
    """G parts, the first ones holding fewer than k rows (padded with -1), every row present twice (exact ties
    across parts): merge_device and the packed merge equal the whole index's search; an overflow marker in one part
    is reported by the packed merge."""
    import torch
    from oracle import c_oracle
    assert {_merge_mode(G, k) for G, k in MERGES} == {0, 1, 2}
    n = 30000
    B = c_oracle.synth_block(0, n // 2, seed=65)
    P = np.concatenate([B, B])
    Q = c_oracle.synth_block(0, 9, seed=65, stream=1)
    nq = len(Q)
    small = [7, k - 1][:G - 1]
    rest = n - sum(small)
    sizes = small + [rest // (G - len(small))] * (G - len(small))
    sizes[-1] += n - sum(sizes)
    edges = np.concatenate([[0], np.cumsum(sizes)])
    whole = make_index("auto", P)
    Dw, Iw = whole.search(Q, k)
    qd = torch.from_numpy(Q).cuda()
    Dp, Ip = [], []
    for a, b in zip(edges[:-1], edges[1:]):
        sub = make_index("auto")
        sub.add_with_ids(P[a:b], np.arange(a, b, dtype=np.int64))
        D, I = sub.search_device(qd, k)
        Dp.append(D)
        Ip.append(I)
        sub.close()
    assert (Ip[0][:, 7:] == -1).all(), "the first part pads"
    Dm, Im = whole.merge_device(torch.stack(Dp).contiguous(), torch.stack(Ip).contiguous())
    np.testing.assert_array_equal(Im.cpu().numpy(), Iw)
    assert Dm.cpu().numpy().tobytes() == Dw.tobytes()
    assert (Dw[:, 1:] == Dw[:, :-1]).any(), "the planted ties are in the results"
    i_off = (nq * k * 4 + 15) // 16 * 16
    part = i_off + nq * k * 8
    recv = torch.zeros((G, part), dtype=torch.uint8, device="cuda")
    for g in range(G):
        recv[g, :nq * k * 4].view(torch.float32).view(nq, k).copy_(Dp[g])
        recv[g, i_off:].view(torch.int64).view(nq, k).copy_(Ip[g])
    Dk = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    Ik = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    whole.merge_packed_device_async(recv, G, part, i_off, nq, k, Dk, Ik)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(Ik.cpu().numpy(), Iw)
    assert Dk.cpu().numpy().tobytes() == Dw.tobytes()
    assert whole.stat("merge_saw_overflow") == 0
    recv[G - 1, i_off:].view(torch.int64)[0] = -2
    whole.merge_packed_device_async(recv, G, part, i_off, nq, k, Dk, Ik)
    torch.cuda.synchronize()
    assert whole.stat("merge_saw_overflow") == 1
    assert whole.stat("merge_saw_overflow") == 0
    whole.close()
