"""Seeded operand sets, documented ranges and the ulp measure for the tests of csrc/vmath.cuh
(tests/test_gpu_vmath.py on the GPU, tests/test_vmath_reference.py without one).

The ranges below are the ones the header promises; `bad()` must be raised exactly outside them.  The operand sets
reach the ends of those ranges and the places where the fast sequences can go wrong: quotients and square roots
within 2^-60 of a rounding boundary, exp's reduction boundaries, and each branch of fdlibm's log."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "components", "flux_calculator_b200", "csrc")
PROBE_SRC = os.path.join(ROOT, "tests", "vmath_probe.cu")

C_EXNER = 287.05 / 1005.0          # R_d/c_p as make_consts (formulas.cuh) computes it
LO, HI = 2.0 ** -500, 2.0 ** 500   # FastVec's proven operand range [LO, HI) in magnitude
EXP_MAX = 700.0                    # FastVec::exp is proven for |x| < EXP_MAX

OPS = {"div": 0, "sqrt": 1, "exp": 2, "log": 3, "powc": 4}
POLICIES = {"fast1": 0, "fast2": 1, "exactvec2": 2, "exactscalar": 3}


def probe_command(out):
    """nvcc command line that builds tests/vmath_probe.cu into the shared library `out` (csrc/Makefile's flags)"""
    return [os.environ.get("NVCC", "nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
            "-shared", "-Xcompiler", "-fPIC", "-I", CSRC, PROBE_SRC, "-o", str(out)]


# ---------------------------------------------------------------------------------------------
# the ulp measure
def ulp_error(y, exact):
    """|y - exact| / 2^(floor(log2|exact|) - 52), with the subnormal spacing 2^-1074 below 2^-1022; y float64,
    exact long double (64-bit significand: 2^-11 of a double's ulp)"""
    exact = np.asarray(exact, dtype=np.longdouble)
    _, e = np.frexp(exact)                               # |exact| = m 2^e, m in [0.5, 1): floor(log2|exact|) = e - 1
    e = np.where(exact == 0, -1022, np.maximum(e.astype(np.int64) - 1, -1022))
    return np.abs(np.asarray(y, dtype=np.float64).astype(np.longdouble) - exact) / np.ldexp(np.longdouble(1), (e - 52).astype(np.int32))


def ulp_error_mp(y, exact):
    """the same measure in mpmath (exact: an mpf)"""
    import mpmath
    with mpmath.workdps(max(40, mpmath.mp.dps)):
        e = -1022
        if exact != 0:
            # floor(log2|exact|), settled against the power of two itself: log2 of a value a hair below 2^k may round to k
            e = int(mpmath.floor(mpmath.log(abs(exact), 2)))
            if mpmath.ldexp(1, e) > abs(exact):
                e -= 1
            elif mpmath.ldexp(1, e + 1) <= abs(exact):
                e += 1
            e = max(e, -1022)
        return float(abs(mpmath.mpf(float(y)) - exact) / mpmath.ldexp(1, e - 52))


def reference(op, x, c=C_EXNER):
    """exp / log / x**c of float64 operands in long double"""
    xl = np.asarray(x, dtype=np.float64).astype(np.longdouble)
    with np.errstate(all="ignore"):
        if op == "exp":
            return np.exp(xl)
        if op == "log":
            return np.log(xl)
        return np.power(xl, np.longdouble(c))


def reference_mp(op, x, c=C_EXNER, dps=40):
    import mpmath
    with mpmath.workdps(dps):
        xm = mpmath.mpf(float(x))
        if op == "exp":
            return mpmath.exp(xm)
        if op == "log":
            return mpmath.log(xm)
        return mpmath.power(xm, mpmath.mpf(float(c)))


# ---------------------------------------------------------------------------------------------
# documented ranges
def is_pos_zero(x):
    return np.asarray(x, dtype=np.float64).view(np.uint64) == 0


def in_range(x):
    ax = np.abs(np.asarray(x, dtype=np.float64))
    return (ax >= LO) & (ax < HI)


def documented(op, x, y=None, c=C_EXNER):
    """True where FastVec's fast sequence is proven: bad() must be clear exactly there"""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(all="ignore"):
        if op == "div":
            return (in_range(x) | is_pos_zero(x)) & in_range(y)
        if op == "sqrt":
            return ((x > 0) & in_range(x)) | is_pos_zero(x)
        if op == "exp":
            return np.abs(x) < EXP_MAX
        pos = (x > 0) & in_range(x)
        if op == "log":
            return pos
        y = np.where(pos, np.log(np.where(pos, x, 1.0).astype(np.longdouble)) * np.longdouble(c), 0)
        return pos & (np.abs(y) < EXP_MAX)


# ---------------------------------------------------------------------------------------------
# operand sets
def from_bits(bits):
    return np.asarray(bits, dtype=np.uint64).view(np.float64)


def _bits(sign, biased_exp, mant):
    return from_bits((np.uint64(sign) << np.uint64(63)) | (np.asarray(biased_exp, np.uint64) << np.uint64(52)) | np.asarray(mant, np.uint64))


def edge_values():
    """±0, subnormal and normal limits, both ends of [2^-500, 2^500) with their neighbours, 1 and 2 with theirs,
    all-ones and single-bit mantissas, the largest double, ±Inf, NaN; every finite value with both signs"""
    pos = [0.0, 5e-324, np.nextafter(2.0 ** -1022, 0.0), 2.0 ** -1022, 1.0, np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0),
           np.nextafter(2.0, 0.0), 2.0, np.finfo(np.float64).max]
    for p in (LO, HI):
        pos += [np.nextafter(p, 0.0), p, np.nextafter(p, np.inf)]
    for e in (-1000, -501, -500, -499, -1, 0, 1, 499, 500, 1000):
        pos += [float(_bits(0, e + 1023, (1 << 52) - 1)), float(_bits(0, e + 1023, 1)), float(_bits(0, e + 1023, 1 << 51))]
    pos = np.unique(np.array(pos, dtype=np.float64))
    return np.concatenate([pos, -pos, [np.inf, -np.inf, np.nan]])


def exp_edge_values():
    extra = []
    for v in (EXP_MAX, 709.78, 745.0, 709.782712893384, 745.1332191019412):
        extra += [np.nextafter(v, 0.0), v, np.nextafter(v, np.inf)]
    extra = np.array(extra, dtype=np.float64)
    return np.concatenate([edge_values(), extra, -extra])


def div_edge_pairs():
    v = edge_values()
    a, b = np.meshgrid(v, v, indexing="ij")
    return a.ravel(), b.ravel()


def random_doubles(rng, n, emin, emax, signed):
    """random mantissa, exponent uniform in [emin, emax], random sign if `signed`"""
    sign = rng.integers(0, 2, n, dtype=np.uint64) if signed else np.zeros(n, np.uint64)
    e = rng.integers(emin + 1023, emax + 1024, n).astype(np.uint64)
    mant = rng.integers(0, 1 << 52, n, dtype=np.uint64)
    return from_bits((sign << np.uint64(63)) | (e << np.uint64(52)) | mant)


def div_random(n=4_000_000, seed=101):
    rng = np.random.default_rng(seed)
    return random_doubles(rng, n, -500, 499, True), random_doubles(rng, n, -500, 499, True)


def _inverse_mod_2_64(b):
    """b^-1 mod 2^64 for odd b (Newton: each step doubles the correct low bits, b*b = 1 mod 8 to start)"""
    x = b.copy()
    with np.errstate(over="ignore"):
        for _ in range(5):
            x = x * (np.uint64(2) - b * x)
    return x


def div_hard(n=1_000_000, seed=102):
    """pairs (a, b) in the proven range whose exact quotient lies within 2^-60 (relative) of the midpoint of two
    adjacent doubles.  With B odd in [2^52, 2^53) and a small odd r, M = r B^-1 mod 2^54 gives B M = A 2^54 + r:
    A/B = M/2^54 - r/(B 2^54), and M/2^54 (M odd in [2^53, 2^54)) is a midpoint of [0.5, 1)."""
    rng = np.random.default_rng(seed)
    m54 = np.uint64((1 << 54) - 1)
    B = rng.integers(1 << 52, 1 << 53, 2 * n, dtype=np.uint64) | np.uint64(1)
    r = (rng.integers(1, 1 << 43, 2 * n, dtype=np.int64) * 2 + 1) * rng.choice(np.array([-1, 1], np.int64), 2 * n)
    with np.errstate(over="ignore"):
        M = (r.view(np.uint64) * _inverse_mod_2_64(B)) & m54
    keep = M >= np.uint64(1 << 53)
    B, M, r = B[keep][:n], M[keep][:n], r[keep][:n]
    # A = (B M - r) / 2^54 < 2^53: the long double product is within 2^-11 of B M / 2^54, which is within 2^-10 of A
    A = np.rint(B.astype(np.longdouble) * M.astype(np.longdouble) / np.longdouble(2.0 ** 54)).astype(np.uint64)
    with np.errstate(over="ignore"):
        assert np.array_equal(B * M - (A << np.uint64(54)), r.view(np.uint64)), "div_hard: B M != A 2^54 + r"
    m = len(B)
    ea = rng.integers(-499, 499, m)            # a = A 2^(ea-52), A in [2^51, 2^53): a in [2^-500, 2^499)
    eb = rng.integers(-499, 499, m)
    a = np.ldexp(A.astype(np.float64), (ea - 52).astype(np.int32))
    b = np.ldexp(B.astype(np.float64), (eb - 52).astype(np.int32))
    sa = rng.choice(np.array([-1.0, 1.0]), m)
    sb = rng.choice(np.array([-1.0, 1.0]), m)
    return a * sa, b * sb


def sqrt_random(n=1_000_000, seed=103):
    return random_doubles(np.random.default_rng(seed), n, -500, 499, False)


def sqrt_squares(n=200_000, seed=104):
    """s^2 with a 26-bit mantissa s, so s^2 is a double: sqrt must return s exactly.  Returns (x, s)."""
    rng = np.random.default_rng(seed)
    s = np.ldexp(rng.integers(1 << 25, 1 << 26, n).astype(np.float64), rng.integers(-274, 224, n).astype(np.int32))
    return s * s, s


def sqrt_hard(n=500_000, seed=105):
    """x in the proven range with sqrt(x) within 2^-60 (relative) of a midpoint: T odd in [2^53, 2^54) with
    T^2 = X 2^55 + r for a small r = 1 mod 8 (T is a square root of r mod 2^55, by Hensel lifting); then
    x = X 2^(2j-53) and sqrt(x) = T 2^(j-54) sqrt(1 - r/T^2).  X in [2^51, 2^53) covers both exponent parities."""
    rng = np.random.default_rng(seed)
    r = rng.integers(-(1 << 40), 1 << 40, n, dtype=np.int64) * 8 + 1
    ru = r.view(np.uint64)
    t = np.ones(n, np.uint64)
    with np.errstate(over="ignore"):
        for k in range(3, 55):                  # t^2 = r mod 2^k  ->  mod 2^(k+1)
            flip = ((t * t - ru) >> np.uint64(k)) & np.uint64(1)
            t = t + (flip << np.uint64(k - 1))
        t &= np.uint64((1 << 54) - 1)
        T = np.where(t >= np.uint64(1 << 53), t, np.uint64(1 << 54) - t)
        X = np.rint(T.astype(np.longdouble) ** 2 / np.longdouble(2.0 ** 55)).astype(np.uint64)
        assert np.array_equal(T * T - (X << np.uint64(55)), ru), "sqrt_hard: T^2 != X 2^55 + r"
    j = rng.integers(-249, 251, n)
    return np.ldexp(X.astype(np.float64), (2 * j - 53).astype(np.int32))


def exp_sets(seed=106):
    """name -> operands: uniform over (-700, 700); (k + 1/2) ln2 and 8 ulp either side for k in [-1009, 1009]
    (the reduction's rounding boundaries); [690, 700) and its negative densely (where the cold path's own switch
    between the fast sequence and libdevice lies); ±0, subnormals and |x| < 2^-54, where exp(x) is exactly 1"""
    rng = np.random.default_rng(seed)
    ks = np.arange(-1009, 1010).astype(np.longdouble)
    mid = ((ks + np.longdouble(0.5)) * np.log(np.longdouble(2))).astype(np.float64)
    near = [mid]
    lo_, hi_ = mid.copy(), mid.copy()
    for _ in range(8):
        lo_, hi_ = np.nextafter(lo_, -np.inf), np.nextafter(hi_, np.inf)
        near += [lo_, hi_]
    top = rng.uniform(690.0, 700.0, 200_000)
    sub = from_bits(rng.integers(1, 1 << 52, 4_000, dtype=np.uint64))
    tiny = np.concatenate([[0.0, -0.0, 5e-324, -5e-324, 2.0 ** -1022, -(2.0 ** -1022), 2.0 ** -55, -(2.0 ** -55)],
                           random_doubles(rng, 20_000, -1022, -55, True), sub, -sub])
    return {"uniform": rng.uniform(-700.0, 700.0, 1_000_000), "reduction boundaries": np.concatenate(near),
            "near 700": np.concatenate([top, -top]), "exactly 1": tiny}


def _log_operands(rng, n, hm_lo, hm_hi):
    """2^e (1 + hm/2^20 + lo/2^52): e uniform in [-500, 499] for half the cells and in {-1, 0} for the other half
    (there log's result is not dominated by e ln2, so its relative error is largest); high mantissa word uniform
    in [hm_lo, hm_hi], low word uniform"""
    e = np.where(rng.random(n) < 0.5, rng.integers(-500, 500, n), rng.integers(-1, 1, n))
    hm = rng.integers(hm_lo, hm_hi + 1, n).astype(np.uint64)
    lo = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    return _bits(0, (e + 1023).astype(np.uint64), (hm << np.uint64(32)) | lo)


# high mantissa words (the top 20 bits of the mantissa) of log's windows
LOG_MID = (0x6147A, 0x6B851)               # fdlibm's "mid" formula, inclusive
LOG_HALVING = (0x6A097, 0x6A0A0)           # halving (mantissa > sqrt 2) starts at 0x6a09c: both sides
LOG_TINY = (0xFFFFE, 0xFFFFF, 0x0, 0x1, 0x2)   # |f| < 2^-20 branch, after halving for 0xffffe/0xfffff


def log_sets(seed=107):
    rng = np.random.default_rng(seed)
    tiny = np.concatenate([_log_operands(rng, 100_000, h, h) for h in LOG_TINY])
    return {"[1, 2)": _log_operands(rng, 1_000_000, 0, 0xFFFFF), "mid": _log_operands(rng, 500_000, *LOG_MID),
            "halving": _log_operands(rng, 500_000, *LOG_HALVING), "tiny": tiny,
            "powers of two": np.ldexp(1.0, np.arange(-500, 500, dtype=np.int32))}


def pow_sets(seed=108):
    """x**(R_d/c_p): the Exner window |c log x| <= 0.1, the physical ratio p_s/p_a, the whole proven range"""
    rng = np.random.default_rng(seed)
    return {"Exner": rng.uniform(np.exp(-0.35), np.exp(0.35), 1_000_000), "physical": rng.uniform(1.0009, 1.016, 500_000),
            "proven range": random_doubles(rng, 500_000, -500, 499, False)}


def high_word(x):
    return (np.asarray(x, dtype=np.float64).view(np.uint64) >> np.uint64(32)).astype(np.uint32)
