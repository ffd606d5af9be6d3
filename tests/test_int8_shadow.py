"""The int8 prefilter shadow (DESIGN.md section 4).

CPU part: a numpy restatement of the int8 quantisation (per-32-row-tile row scales, per-query scales), of the
integer threshold and of the margin eps = (||q|| + e_q) E8 + e_q P + 2^-21 (||q|| + e_q)(P + E8), checked on
adversarial rows: |s~ - s| <= eps, and no row whose int8 score reaches tau is filtered out by the integer test.

GPU part: forced int8 and forced bf16 shadows return bit-identical results (they only differ in the prefilter; the
reported scores come from the exact rescoring), int8 agrees with the oracle, and AUTO picks the format per shard.
"""
import numpy as np
import pytest

F32 = np.float32


def quant8(x, amax):
    """Symmetric int8 codes of x for the group maximum amax (0 codes for an all-zero group)."""
    amax = F32(amax)
    inv = F32(127.0) / amax if amax > 0 else F32(0.0)
    return np.clip(np.rint((x.astype(F32) * inv).astype(F32)), -127, 127).astype(np.int32)


def int8_rows(pc):
    """Per-32-row-tile scales and codes, as convert_rows_i8_kernel makes them."""
    st = np.zeros((pc.shape[0] + 31) // 32, dtype=F32)
    p8 = np.zeros(pc.shape, dtype=np.int32)
    for t in range(len(st)):
        blk = pc[32 * t:32 * t + 32]
        amax = np.abs(blk).max()
        st[t] = F32(amax) / F32(127.0)
        p8[32 * t:32 * t + 32] = quant8(blk, amax)
    return st, p8


def i8_threshold(tau, sq, st):
    """Largest integer T with T <= tau / (sq * st), evaluated with directed roundings (restated in fp64 with the
    same outcome: the fp64 quotient of fp32 operands is within 2^-53 of the real one, floor() then rounds down)."""
    if not tau > -np.inf:
        return -2**31
    c = float(sq) * float(st)
    if c == 0.0:
        return 2**31 - 1 if tau > 0 else -2**31
    x = float(tau) / c
    x = np.nextafter(x, -np.inf)       # never above the real quotient
    if x >= 2147483520.0:
        return 2**31 - 1
    if x < -2147483520.0:
        return -2**31
    return int(np.floor(x))


def eps_int8(qn, qe, E8, P):
    qh = qn + qe
    return qh * E8 + qe * P + qh * (P + E8) * 2.0**-21


def _rows(rng):
    P = rng.standard_normal((256, 768)).astype(F32)
    P[3, 17] = 900.0                     # one huge component: its tile's scale is coarse for every other row
    P[40:72] = 0.0                       # an all-zero tile
    P[100] = -P[100] * 50                # a long row
    P[200:232] = 1e-30                   # tiny values (subnormal products)
    return P


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_int8_margin_bounds_the_prefilter_error_on_adversarial_rows(seed):
    rng = np.random.default_rng(seed)
    P = _rows(rng)
    mu = P[:128].mean(0).astype(F32)
    pc = (P - mu).astype(F32)
    st, p8 = int8_rows(pc)
    ph = p8.astype(np.float64) * np.repeat(st, 32)[:len(pc), None].astype(np.float64)
    exact_pc = P.astype(np.float64) - mu.astype(np.float64)
    E8 = np.linalg.norm(exact_pc - ph, axis=1).max()
    Pn = np.linalg.norm(exact_pc, axis=1).max()
    Q = rng.standard_normal((8, 768)).astype(F32)
    Q[0, 5] = -300.0                     # a query dominated by one component
    Q[1] = 0.0                           # a zero query
    for q in Q:
        amax = np.abs(q).max()
        sq = F32(amax) / F32(127.0)
        q8 = quant8(q, amax)
        qe = np.linalg.norm(q.astype(np.float64) - q8 * float(sq))
        qn = np.linalg.norm(q.astype(np.float64))
        eps = eps_int8(qn, qe, E8, Pn)
        acc = p8 @ q8                    # exact int32 accumulation
        assert np.abs(acc).max() < 2**24
        tiles = np.arange(len(pc)) // 32
        s_real = acc * (float(sq) * st[tiles].astype(np.float64))
        s_rec = (acc.astype(F32) * (sq * st[tiles]).astype(F32)).astype(F32).astype(np.float64)
        s = exact_pc @ q.astype(np.float64)
        assert (np.abs(s_real - s) <= eps).all()
        assert (np.abs(s_rec - s) <= eps).all()
        # the integer filter never drops a row whose int8 score reaches tau (including tau <= 0 and -inf)
        for tau in [-np.inf, -abs(s).max(), -1e-3, 0.0, float(np.median(s_real)), float(s_real.max()), 1e9]:
            for t in range(len(st)):
                T = i8_threshold(tau, sq, st[t])
                rows = tiles == t
                assert not np.any((s_real[rows] >= tau) & (acc[rows] < T)), (tau, t)


def test_integer_threshold_edge_cases():
    assert i8_threshold(-np.inf, 0.1, 0.2) == -2**31
    assert i8_threshold(float("nan"), 0.1, 0.2) == -2**31
    assert i8_threshold(0.5, 0.0, 0.2) == 2**31 - 1       # every score is 0 < tau
    assert i8_threshold(0.0, 0.0, 0.2) == -2**31          # 0 >= 0 passes
    assert i8_threshold(-0.5, 0.0, 0.2) == -2**31
    assert i8_threshold(1e30, 1e-3, 1e-3) == 2**31 - 1
    assert i8_threshold(-1e30, 1e-3, 1e-3) == -2**31
    # an exact quotient is never rounded up past the integer that reaches it
    assert i8_threshold(3.0, 1.0, 1.0) <= 3
    assert i8_threshold(-3.0, 1.0, 1.0) <= -3


# ------------------------------------------------------------------------------------------------ GPU


def _index(shadow, P=None, **opts):
    from convdr_b200 import FlatIPIndex
    idx = FlatIPIndex(768)
    idx.set_option("shadow", shadow)
    for k, v in opts.items():
        idx.set_option(k, v)
    if P is not None:
        idx.add(P)
    return idx


def _search_both(P, Q, k, **opts):
    out = []
    for shadow in (1, 2):
        idx = _index(shadow, P, **opts)
        assert idx.stat("shadow_format") == shadow
        D, I = idx.search(Q, k)
        out.append((D, I, idx.stat("fallback_queries")))
        idx.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2, 3])      # AUTO per pass, TS, QS
@pytest.mark.parametrize("nq,k", [(173, 100), (256, 100), (64, 1000), (300, 10)])
def test_int8_and_bf16_shadows_return_identical_results(variant, nq, k):
    from oracle import c_oracle
    P = c_oracle.synth_block(0, 100000)
    Q = c_oracle.synth_block(0, nq, stream=1)
    (D1, I1, f1), (D2, I2, f2) = _search_both(P, Q, k, umma_variant=variant)
    assert f1 == 0 and f2 == 0
    assert np.array_equal(D1, D2) and np.array_equal(I1, I2)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 4095, 70001])
def test_int8_ragged_sizes_and_incremental_adds_match_the_oracle(n):
    from oracle import c_oracle, flat_ip
    P = c_oracle.synth_block(0, n, seed=7)
    Q = c_oracle.synth_block(0, 40, seed=7, stream=1)
    k = min(50, n)
    idx = _index(2)
    for lo in range(0, n, 9000 if n > 9000 else max(1, n // 3)):   # adds that end inside a 32-row tile
        idx.add(P[lo:lo + (9000 if n > 9000 else max(1, n // 3))])
    assert idx.ntotal == n
    D, I = idx.search(Q, k)
    Dt, It = flat_ip.truth_fp64(Q, P, k)
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    assert flat_ip.compare(D, I, Dt, It, score_of, rtol=1e-5)["violations"] == 0
    ref = _index(1, P)
    Db, Ib = ref.search(Q, k)
    assert np.array_equal(D, Db) and np.array_equal(I, Ib)


@pytest.mark.gpu
def test_int8_planted_ties_and_overflow_marker():
    from oracle import c_oracle
    P = c_oracle.synth_block(0, 50000, seed=3)
    P[1000:1300] = P[77]                 # 301 identical rows: ties across the k-th score
    Q = np.concatenate([P[77:78], c_oracle.synth_block(0, 7, seed=3, stream=1)])
    (D1, I1, _), (D2, I2, _) = _search_both(P, Q, 100)
    assert np.array_equal(D1, D2) and np.array_equal(I1, I2)


@pytest.mark.gpu
def test_forced_int8_on_common_mean_rows_is_still_exact():
    from oracle import c_oracle, flat_ip
    P = c_oracle.synth_block(0, 60000, seed=51, norm=28.0, mean_shift=443)
    Q = c_oracle.synth_block(0, 32, seed=51, stream=1, norm=28.0, mean_shift=443)
    idx = _index(2, P)
    D, I = idx.search(Q, 100)            # fallbacks allowed: the margin is wide on these rows
    Dt, It = flat_ip.truth_fp64(Q, P, 100)
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    assert flat_ip.compare(D, I, Dt, It, score_of, rtol=1e-5)["violations"] == 0


@pytest.mark.gpu
def test_auto_picks_the_format_from_the_rows():
    from oracle import c_oracle
    iso = _index(3, c_oracle.synth_block(0, 20000, seed=13))
    assert iso.stat("shadow_format") == 2 and 0 < iso.stat("shadow_rho") <= 1.2
    aniso = _index(3, c_oracle.synth_block(0, 20000, seed=51, norm=28.0, mean_shift=443))
    assert aniso.stat("shadow_format") == 1 and aniso.stat("shadow_rho") > 1.2
    same = _index(3, np.ones((20000, 768), dtype=np.float32))
    assert same.stat("shadow_format") == 1
    small = _index(3, c_oracle.synth_block(0, 1000, seed=13))
    assert small.stat("shadow_format") == 1
    for idx in (iso, aniso, same, small):
        idx.close()
