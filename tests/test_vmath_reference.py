"""not-gpu: the parts of the vmath.cuh tests that need no device.  The probe (tests/vmath_probe.cu) compiles for sm_100a
against the current vmath.cuh; the operand generators of tests/vmath_cases.py produce what they claim, checked with
exact rational arithmetic; the ulp measure agrees with mpmath, also for results next to a power of two."""
import ctypes as C
import math
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import vmath_cases as vc


def test_probe_compiles_for_sm_100a_and_exports_its_entry_points(tmp_path):
    out = tmp_path / "libvmath_probe.so"
    subprocess.run(vc.probe_command(out), check=True)
    lib = C.CDLL(str(out))          # loads without a device: nothing runs until an entry point is called
    for sym in ("vp_run", "vp_sweep", "vp_sweep_keep"):
        assert hasattr(lib, sym), sym
    assert lib.vp_sweep_keep() == 8


def _midpoint_distance(q):
    """relative distance of the positive rational q from the nearest midpoint of two adjacent doubles"""
    e = math.frexp(float(q))[1] - 1                   # floor(log2 q): q is not next to a power of two here
    u = q * Fraction(2) ** (52 - e)                   # in [2^52, 2^53): doubles are the integers, midpoints the halves
    assert 2 ** 52 <= u < 2 ** 53
    h = math.floor(u) + Fraction(1, 2)
    return abs(u - h) / u


def test_hard_quotients_lie_within_2_pow_minus_60_of_a_midpoint():
    a, b = vc.div_hard()
    assert len(a) == 1_000_000
    assert vc.in_range(a).all() and vc.in_range(b).all()
    assert (a < 0).any() and (b < 0).any()
    for i in np.random.default_rng(1).choice(len(a), 3000, replace=False):
        assert _midpoint_distance(abs(Fraction(float(a[i])) / Fraction(float(b[i])))) < Fraction(1, 2 ** 60), (a[i], b[i])


def test_hard_square_roots_lie_within_2_pow_minus_60_of_a_midpoint():
    x = vc.sqrt_hard()
    assert vc.in_range(x).all() and (x > 0).all()
    e = np.frexp(x)[1]
    assert (e % 2 == 0).any() and (e % 2 == 1).any(), "both exponent parities"
    for i in np.random.default_rng(2).choice(len(x), 3000, replace=False):
        xf = Fraction(float(x[i]))
        ey = math.frexp(math.sqrt(float(x[i])))[1] - 1          # floor(log2 sqrt x)
        q = xf * Fraction(2) ** (104 - 2 * ey)                  # (sqrt(x) 2^(52-ey))^2: doubles are the integers
        z = math.isqrt(math.floor(q))                           # floor(sqrt(q)) = isqrt(floor(q))
        w = (z + Fraction(1, 2)) ** 2                           # the nearest midpoint, squared
        # |sqrt(q) - m| / m = |q - m^2| / (m (sqrt(q) + m)) < |q - m^2| / (2 m^2 (1 - 2^-40)) for q this close to m^2
        assert abs(q - w) / w < Fraction(1, 2 ** 59), x[i]


def test_perfect_squares_are_exact():
    x, s = vc.sqrt_squares()
    assert vc.in_range(x).all()
    for i in range(0, len(x), 997):
        assert Fraction(float(s[i])) ** 2 == Fraction(float(x[i]))


def test_log_windows_hit_the_intended_high_mantissa_words():
    sets = vc.log_sets()
    for name, xs in sets.items():
        assert vc.in_range(xs).all() and (xs > 0).all(), name
        e = np.frexp(xs)[1] - 1
        assert e.min() == -500 and e.max() == 499, name
    hm = lambda v: vc.high_word(v) & 0xFFFFF
    mid = hm(sets["mid"])
    assert mid.min() == vc.LOG_MID[0] and mid.max() == vc.LOG_MID[1]
    halving = hm(sets["halving"])
    # fdlibm halves the mantissa from high word 0x6a09c on ((hm + 0x95f64) & 0x100000): both sides are present
    assert (halving < 0x6A09C).sum() > 100_000 and (halving >= 0x6A09C).sum() > 100_000
    assert halving.min() >= vc.LOG_HALVING[0] and halving.max() <= vc.LOG_HALVING[1]
    tiny = hm(sets["tiny"])
    assert set(np.unique(tiny).tolist()) == set(vc.LOG_TINY)
    # every low word is reached: the windows are not confined to round mantissas
    assert len(np.unique(sets["mid"].view(np.uint64) & np.uint64(0xFFFFFFFF))) > 400_000
    assert (sets["powers of two"] == np.ldexp(1.0, np.arange(-500, 500))).all()


def test_exp_sets_straddle_the_reduction_boundaries():
    sets = vc.exp_sets()
    b = sets["reduction boundaries"]
    assert (np.abs(b) < vc.EXP_MAX).all() and np.abs(b).max() > 699.0
    # for every k, operands lie on both sides of (k + 1/2) ln2 (long double ln2: 2^-64 relative)
    t = b.astype(np.longdouble) / np.log(np.longdouble(2)) - np.longdouble(0.5)
    k = np.rint(t)
    assert set(np.unique(k).astype(int).tolist()) == set(range(-1009, 1010))
    for kk in (-1009, -1, 0, 1, 1009):
        d = t[k == kk] - kk
        assert (d < 0).sum() >= 8 and (d > 0).sum() >= 8, kk
    one = sets["exactly 1"]
    assert (np.abs(one) < 2.0 ** -54).all() and (one == 0).sum() == 2 and (np.abs(one) < 2.0 ** -1022).sum() > 8000


def test_generators_are_reproducible():
    a1, b1 = vc.div_hard(1000)
    a2, b2 = vc.div_hard(1000)
    assert (a1 == a2).all() and (b1 == b2).all()
    assert (vc.sqrt_hard(1000) == vc.sqrt_hard(1000)).all()
    assert all((vc.log_sets()[k] == v).all() for k, v in vc.log_sets().items())


def test_documented_ranges():
    lo, hi = vc.LO, vc.HI
    below, above = np.nextafter(lo, 0.0), np.nextafter(hi, 0.0)
    x = np.array([0.0, -0.0, below, lo, above, hi, -lo, -above, np.inf, np.nan, 1.0])
    one = np.ones_like(x)
    assert vc.documented("div", x, one).tolist() == [True, False, False, True, True, False, True, True, False, False, True]
    assert vc.documented("div", one, x).tolist() == [False, False, False, True, True, False, True, True, False, False, True]
    assert vc.documented("sqrt", x).tolist() == [True, False, False, True, True, False, False, False, False, False, True]
    assert vc.documented("log", x).tolist() == [False, False, False, True, True, False, False, False, False, False, True]
    assert (vc.documented("powc", x) == vc.documented("log", x)).all()
    e = np.array([699.9999999999999, 700.0, -700.0, -699.9999999999999, np.nan, -np.inf, 0.0])
    assert vc.documented("exp", e).tolist() == [True, False, False, True, False, False, True]


def _ld(v):
    """the long double nearest to the mpf v (exact when v has at most 64 significant bits)"""
    import mpmath
    return np.longdouble(mpmath.nstr(v, 40, strip_zeros=False, min_fixed=1, max_fixed=0))


def _p2(e):
    import mpmath
    return mpmath.ldexp(1, e)


@pytest.mark.parametrize("y,exact", [
    (1.0, lambda m: 1 - _p2(-60)),                       # just below a power of two: the ulp is 2^-53
    (1.0, lambda m: 1 + _p2(-60)),                       # just above: 2^-52
    (np.nextafter(1.0, 0.0), lambda m: 1 - _p2(-54)),
    (2.0 ** 600, lambda m: _p2(600) * (1 - _p2(-62))),
    (2.0 ** -600, lambda m: _p2(-600) * (1 + 3 * _p2(-56))),
    (3.0, lambda m: 3 + _p2(-52)),
    (np.exp(1.0), lambda m: m.exp(1)),
    (np.log(10.0), lambda m: m.log(10)),
    (5e-324, lambda m: _p2(-1074) * m.mpf(1.25)),        # subnormal: the spacing is 2^-1074
    (2.0 ** -1030, lambda m: _p2(-1030) + _p2(-1076)),
    (0.0, lambda m: _p2(-1076)),
], ids=["below 1", "above 1", "below 1 by 2^-54", "below 2^600", "above 2^-600", "3", "e", "ln 10", "subnormal",
        "subnormal 2^-1030", "zero for 2^-1076"])
def test_ulp_error_agrees_with_mpmath(y, exact):
    import mpmath
    with mpmath.workdps(40):
        ex = exact(mpmath)
        ref = vc.ulp_error_mp(y, ex)
    got = float(vc.ulp_error(np.array([y]), np.array([_ld(ex)]))[0])
    assert abs(got - ref) <= 2e-3 * max(ref, 1.0), (got, ref)
    assert ref > 0


def test_ulp_error_uses_the_binade_of_the_exact_value():
    import mpmath
    with mpmath.workdps(40):
        below = mpmath.mpf(1) - mpmath.mpf(2) ** -60
        above = mpmath.mpf(1) + mpmath.mpf(2) ** -60
        assert vc.ulp_error_mp(1.0, below) == 2.0 ** -7
        assert vc.ulp_error_mp(1.0, above) == 2.0 ** -8
    assert float(vc.ulp_error(np.array([1.0]), np.array([_ld(below)]))[0]) == 2.0 ** -7
    assert float(vc.ulp_error(np.array([1.0]), np.array([_ld(above)]))[0]) == 2.0 ** -8
