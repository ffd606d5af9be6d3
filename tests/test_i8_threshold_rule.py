"""The integer threshold rule of the int8 tensor engine (kernels_util.cuh, i8_threshold; DESIGN.md section 4).

A prefilter score is s~ = acc * sq * st with acc the exact int32 dot product of the codes.  The kernels compare acc with
an integer threshold T formed from two factors, so that the step done per (query, tile) needs no division:

    u    = RD(tau / sq)                      per query, when tau changes
    r_lo = RD(1 / st),  r_hi = RU(1 / st)    per 32-row tile, at ingest
    x    = RD(u * (u >= 0 ? r_lo : r_hi)),   T = floor(x), saturated to int32, NaN -> INT_MIN

This file restates the rule with exact rational arithmetic and fp32 directed rounding, and checks that it is valid
(no integer acc with acc * sq * st >= tau lies below T) on random and adversarial inputs, and that it is nearly as
tight as the former single-division rule x = RD(tau / c), c = sq * st rounded towards the smaller quotient.
"""
from fractions import Fraction

import numpy as np
import pytest

F32 = np.float32
INF = float("inf")
NAN = float("nan")
FLT_MAX = float(np.finfo(F32).max)
DENORM_MIN = float(np.finfo(F32).smallest_subnormal)
INT_MIN, INT_MAX = -2**31, 2**31 - 1
ACC_MAX = 768 * 127 * 127          # |acc| of 768 products of codes in [-127, 127]


def _f32(x):
    return float(F32(x))


def _up(f):
    with np.errstate(over="ignore"):
        return float(np.nextafter(F32(f), F32(INF)))


def _down(f):
    with np.errstate(over="ignore"):
        return float(np.nextafter(F32(f), F32(-INF)))


def _round32(q, down):
    """fp32 rounding of the exact rational q towards -inf (down) or +inf, with IEEE overflow to +-inf."""
    if q == 0:
        return 0.0
    try:
        f = float(q)
    except OverflowError:
        f = INF if q > 0 else -INF
    with np.errstate(over="ignore"):
        f = _f32(f)
    f = min(max(f, -FLT_MAX), FLT_MAX)
    while Fraction(f) > q:
        f = _down(f)
        if f == -INF:
            return f if down else -FLT_MAX
    while Fraction(f) < q:
        f = _up(f)
        if f == INF:
            return FLT_MAX if down else f
    if Fraction(f) != q and down:
        f = _down(f)
    return f


def _is_special(*xs):
    return any(np.isnan(x) or np.isinf(x) for x in xs)


def div32(a, b, down):
    if np.isnan(a) or np.isnan(b) or (np.isinf(a) and np.isinf(b)) or (a == 0 and b == 0):
        return NAN
    sign = -1.0 if (np.signbit(a) != np.signbit(b)) else 1.0
    if np.isinf(a) or b == 0:
        return sign * INF
    if np.isinf(b) or a == 0:
        return sign * 0.0
    return _round32(Fraction(a) / Fraction(b), down)


def mul32(a, b, down):
    if np.isnan(a) or np.isnan(b) or ((np.isinf(a) or np.isinf(b)) and (a == 0 or b == 0)):
        return NAN
    sign = -1.0 if (np.signbit(a) != np.signbit(b)) else 1.0
    if np.isinf(a) or np.isinf(b):
        return sign * INF
    if a == 0 or b == 0:
        return sign * 0.0
    return _round32(Fraction(a) * Fraction(b), down)


def to_int(x):
    if x >= 2147483520.0:
        return INT_MAX
    if not x >= -2147483520.0:
        return INT_MIN
    return int(np.floor(x))


def tile_factors(st):
    """{RD(1/st), RU(1/st)}: what i8_tile_scale stores next to st."""
    return div32(1.0, st, True), div32(1.0, st, False)


def threshold(tau, sq, st):
    """The kernels' rule: T from u = RD(tau/sq) and the tile factors."""
    u = div32(tau, sq, True)
    r_lo, r_hi = tile_factors(st)
    return to_int(mul32(u, r_lo if u >= 0 else r_hi, True))


def threshold_single_division(tau, sq, st):
    """The former rule: c = sq * st rounded up (tau >= 0) or down, x = RD(tau / c)."""
    if not tau > -INF:
        return INT_MIN
    c = mul32(sq, st, tau < 0)
    if c == 0:
        return INT_MAX if tau > 0 else INT_MIN
    return to_int(div32(tau, c, True))


def least_passing_acc(tau, sq, st):
    """Smallest integer acc in [-ACC_MAX, ACC_MAX] with acc * sq * st >= tau (real arithmetic), or None."""
    if np.isnan(tau):
        return None
    if tau == -INF:
        return -ACC_MAX
    if tau == INF:
        return None
    c = Fraction(sq) * Fraction(st)
    t = Fraction(tau)
    if c == 0:
        return -ACC_MAX if 0 >= t else None
    a = -((-t) // c)       # ceil(t / c)
    a = max(a, -ACC_MAX)
    return a if a <= ACC_MAX else None


def assert_valid(tau, sq, st):
    T = threshold(tau, sq, st)
    a = least_passing_acc(tau, sq, st)
    assert a is None or T <= a, (tau, sq, st, T, a)
    return T


def _random_cases(rng, n):
    def f32s(lo, hi, size):
        mant = rng.uniform(1.0, 2.0, size)
        return (mant * 2.0 ** rng.integers(lo, hi, size)).astype(F32).astype(np.float64)
    taus = f32s(-140, 120, n) * rng.choice([-1.0, 1.0], n)
    sqs = f32s(-149, 30, n)
    sts = f32s(-149, 30, n)
    return zip(taus.tolist(), sqs.tolist(), sts.tolist())


def test_rule_is_valid_on_random_scales_of_every_magnitude():
    rng = np.random.default_rng(0)
    for tau, sq, st in _random_cases(rng, 4000):
        assert_valid(tau, sq, st)


@pytest.mark.parametrize("q", [2.0**24, 2.0**31, -2.0**31, 2147483520.0, -2147483520.0, ACC_MAX, -ACC_MAX, 0.5, -0.5])
def test_rule_is_valid_for_quotients_near_the_integer_edges(q):
    rng = np.random.default_rng(abs(int(q)) % 1000)
    for _ in range(150):
        sq = _f32(rng.uniform(1e-4, 1e-1))
        st = _f32(rng.uniform(1e-4, 1e-1))
        tau0 = _f32(q * sq * st)
        for tau in (tau0, _up(tau0), _down(tau0), _up(_up(tau0)), _down(_down(tau0))):
            assert_valid(tau, sq, st)


def test_rule_is_valid_on_zero_infinite_nan_and_subnormal_inputs():
    specials = [0.0, -0.0, DENORM_MIN, -DENORM_MIN, 1e-40, -1e-40, 1.17e-38, 1e-3, -1e-3, 1.0, -1.0, 3.0, -3.0,
                1e30, -1e30, FLT_MAX, -FLT_MAX, INF, -INF, NAN]
    scales = [0.0, DENORM_MIN, 2 * DENORM_MIN, 1e-40, 2.0**-127, 1.17e-38, 1e-20, 1e-3, 1.0 / 127, 0.5, 1.0, 1e20, FLT_MAX]
    for tau in specials:
        for sq in scales:
            for st in scales:
                assert_valid(_f32(tau) if not np.isnan(tau) else tau, _f32(sq), _f32(st))


def test_rule_edge_values():
    # tau = -inf and NaN pass everything; a padded query column (tau = +inf, sq = 0) passes nothing
    assert threshold(-INF, 0.1, 0.2) == INT_MIN
    assert threshold(-INF, 0.0, 0.0) == INT_MIN
    assert threshold(NAN, 0.1, 0.2) == INT_MIN
    assert threshold(INF, 0.0, 0.2) == INT_MAX
    assert threshold(INF, 0.0, 0.0) == INT_MAX
    # a zero query or a zero tile scores 0: nothing reaches tau > 0, everything reaches tau <= 0
    assert threshold(0.5, 0.0, 0.2) == INT_MAX
    assert threshold(0.5, 0.2, 0.0) == INT_MAX
    for tau in (0.0, -0.0, -0.5):
        assert threshold(tau, 0.0, 0.2) == INT_MIN
        assert threshold(tau, 0.2, 0.0) == INT_MIN
    # a subnormal tile scale whose reciprocal overflows: r_lo = FLT_MAX, r_hi = +inf
    assert tile_factors(DENORM_MIN) == (FLT_MAX, INF)
    assert tile_factors(0.0) == (INF, INF)
    # saturation
    assert threshold(1e30, 1e-3, 1e-3) == INT_MAX
    assert threshold(-1e30, 1e-3, 1e-3) == INT_MIN
    # an exact quotient is never rounded up past the integer that reaches it
    assert threshold(3.0, 1.0, 1.0) == 3
    assert threshold(-3.0, 1.0, 1.0) == -3


def normal(q):
    return q == 0 or 2.0**-126 <= abs(q) <= FLT_MAX


def test_rule_loses_at_most_a_few_units_against_the_single_division_rule():
    # Where the factors u and 1/st are normal fp32 numbers, each of the three roundings costs at most one ulp, so for
    # quotients below 2^24 T drops by at most a few units.  Outside that range the rule stays valid but may be loose
    # (a subnormal st whose reciprocal overflows lets every row with tau < 0 pass); DESIGN.md section 4 states the
    # domain of the exactness claim, and the margin already covers subnormal arithmetic.
    rng = np.random.default_rng(1)
    worst = 0
    n = 0
    for tau, sq, st in _random_cases(rng, 20000):
        if _is_special(tau, sq, st) or sq == 0 or st == 0:
            continue
        qt = Fraction(tau) / (Fraction(sq) * Fraction(st))
        if not abs(qt) < 2**24 or not normal(Fraction(tau) / Fraction(sq)) or not normal(1 / Fraction(st)):
            continue
        loss = threshold_single_division(tau, sq, st) - threshold(tau, sq, st)
        worst = max(worst, loss)
        n += 1
    # scale products of bench-like magnitude: quotients up to ACC_MAX
    for _ in range(5000):
        sq = _f32(rng.uniform(1e-3, 1e-2))
        st = _f32(rng.uniform(1e-4, 1e-2))
        tau = _f32(rng.uniform(-1.0, 1.0) * (2.0**24 - 1) * sq * st)
        worst = max(worst, threshold_single_division(tau, sq, st) - threshold(tau, sq, st))
        n += 1
    assert n > 5000
    assert worst <= 3, worst
