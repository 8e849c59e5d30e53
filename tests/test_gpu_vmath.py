"""-m gpu: the arithmetic policies of csrc/vmath.cuh against references that are not the kernel.

FastVec<2> (the policy both production kernels evaluate every cell with) promises: division and square root
correctly rounded for operands in [2^-500, 2^500); exp within 1 ulp for |x| < 700; log within 1 ulp on
[2^-500, 2^500); x**(R_d/c_p) within 1 ulp where |c log x| <= 0.1; bad() raised exactly when an operand leaves those
ranges; and, where it is not raised, ExactVec<2> (the cold path) returning the same bits.  tests/vmath_probe.cu runs
one operation under one policy; the references are numpy's IEEE float64 division and square root, long double
exp/log/pow (the worst cells re-checked with mpmath at 40 digits), and C99 Annex F for special values.  The operand
sets are in tests/vmath_cases.py."""
import ctypes as C
import functools
import subprocess

import numpy as np
import pytest

import vmath_cases as vc

pytestmark = pytest.mark.gpu

# Largest error measured on a B200 over this module's seeded operand sets, in ulp (vmath_cases.ulp_error), rounded up
# by at most 0.01.  The kernels and the operands are deterministic, so any change of these maxima means vmath.cuh
# computes different bits; each ceiling sits below what the slip named beside it measures.
CEILINGS = {
    # exp_core over every exp window (max 0.8655 near a reduction boundary); a degree-12 polynomial measures 2.3 ulp
    ("exp", "all"): 0.87,
    # log_core over every log window (max 0.8645 in [0.5, 2), where log x is not dominated by k ln2)
    ("log", "all"): 0.87,
    # fdlibm's "mid" formula for high mantissa words 0x6147a..0x6b851 (max 0.8306).  Always taking the other formula
    # measures 0.94 here and stays below 1 ulp, so only this ceiling pins fdlibm's branch selection
    ("log", "mid"): 0.84,
    # both sides of the mantissa-halving threshold at high word 0x6a09c (max 0.8414; inside the mid window, 0.95
    # with the other formula)
    ("log", "halving"): 0.85,
    # the |f| < 2^-20 branch, high words 0xffffe..0x2 (max 0.5016: log(1+f) ~ f - f^2/2 is nearly exact there)
    ("log", "tiny"): 0.51,
    # exp(c log x) with |c log x| <= 0.1 (max 0.6618): c log x is small, so its rounding adds little to exp's error
    ("powc", "Exner"): 0.67,
}
DOCUMENTED_ULP = {"exp": 1.0, "log": 1.0, "powc": 1.0}   # vmath.cuh's header (powc: where |c log x| <= 0.1)
LIBDEVICE_ULP = {"exp": 1.0, "powc": 2.0}                # CUDA Math API documentation, exp and pow


class Probe:
    def __init__(self, path):
        lib = C.CDLL(path)
        dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        lib.vp_run.argtypes = [C.c_int, C.c_int, dp, dp, C.c_double, dp, u8p, C.c_int64]
        lib.vp_run.restype = C.c_int
        lib.vp_sweep.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.POINTER(C.c_ulonglong), dp]
        lib.vp_sweep.restype = C.c_int
        lib.vp_sweep_keep.restype = C.c_int
        self.lib = lib
        self.cache = {}

    def run(self, op, policy, x, y=None, c=vc.C_EXNER):
        """(results, per-cell bad() flag) of `op` under `policy` over x (and y)"""
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ones_like(x) if y is None else np.ascontiguousarray(y, dtype=np.float64)
        out = np.empty_like(x)
        bad = np.empty(len(x), np.uint8)
        dp = C.POINTER(C.c_double)
        rc = self.lib.vp_run(vc.OPS[op], vc.POLICIES[policy], x.ctypes.data_as(dp), y.ctypes.data_as(dp), c,
                             out.ctypes.data_as(dp), bad.ctypes.data_as(C.POINTER(C.c_uint8)), len(x))
        if rc != 0:
            raise RuntimeError("vp_run(%s, %s): CUDA error %d" % (op, policy, rc))
        return out, bad.astype(bool)

    def sweep(self, op, seed, count):
        mism = C.c_ulonglong(0)
        keep = np.zeros(2 * self.lib.vp_sweep_keep(), np.float64)
        rc = self.lib.vp_sweep(vc.OPS[op], seed, count, C.byref(mism), keep.ctypes.data_as(C.POINTER(C.c_double)))
        if rc != 0:
            raise RuntimeError("vp_sweep(%s): CUDA error %d" % (op, rc))
        return mism.value, keep.reshape(-1, 2)[:min(mism.value, len(keep) // 2)]


@pytest.fixture(scope="session")
def probe(tmp_path_factory):
    out = tmp_path_factory.mktemp("vmath_probe") / "libvmath_probe.so"
    subprocess.run(vc.probe_command(out), check=True)
    return Probe(str(out))


# ---------------------------------------------------------------------------------------------
# operand sets: op -> {window: (x, y)}
@functools.lru_cache(maxsize=None)
def operands(op):
    e = vc.edge_values()
    if op == "div":
        rng = np.random.default_rng(201)
        sub = (vc.random_doubles(rng, 100_000, -1022, -990, True), vc.random_doubles(rng, 100_000, 1, 60, True))
        return {"edge pairs": vc.div_edge_pairs(), "random": vc.div_random(), "hard": vc.div_hard(),
                "subnormal quotients": sub}
    if op == "sqrt":
        rng = np.random.default_rng(202)
        sub = vc.from_bits(rng.integers(1, 1 << 52, 100_000, dtype=np.uint64))
        return {"edges": (e, None), "random": (vc.sqrt_random(), None), "squares": (vc.sqrt_squares()[0], None),
                "hard": (vc.sqrt_hard(), None), "subnormals": (sub, None)}
    if op == "exp":
        rng = np.random.default_rng(203)
        beyond = np.concatenate([rng.uniform(700.0, 709.8, 100_000), rng.uniform(-745.2, -700.0, 100_000)])
        sets = {"edges": (vc.exp_edge_values(), None)}
        sets.update((k, (v, None)) for k, v in vc.exp_sets().items())
        sets["beyond 700"] = (beyond, None)
        return sets
    if op == "log":
        sets = {"edges": (e, None)}
        sets.update((k, (v, None)) for k, v in vc.log_sets().items())
        return sets
    rng = np.random.default_rng(204)
    sets = {"edges": (e, None)}
    sets.update((k, (v, None)) for k, v in vc.pow_sets().items())
    whole = np.concatenate([vc.random_doubles(rng, 200_000, -1022, 1023, False),
                            vc.from_bits(rng.integers(1, 1 << 52, 20_000, dtype=np.uint64))])
    sets["whole double range"] = (whole, None)
    return sets


def result(probe, op, policy, window):
    key = (op, policy, window)
    if key not in probe.cache:
        x, y = operands(op)[window]
        probe.cache[key] = probe.run(op, policy, x, y)
    return probe.cache[key]


def bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64)


def same_ieee(got, want):
    """bit-identical, any NaN matching any NaN"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return (bits(got) == bits(want)) | (np.isnan(got) & np.isnan(want))


def numpy_ref(op, x, y):
    with np.errstate(all="ignore"):
        return x / y if op == "div" else np.sqrt(x)


def show(capsys, text):
    with capsys.disabled():
        print("\n" + text)


# ---------------------------------------------------------------------------------------------
# 1. the flag guards exactly the documented range
@pytest.mark.parametrize("op,role", [("div", "numerator"), ("div", "denominator"), ("sqrt", None), ("exp", None),
                                     ("log", None), ("powc", None)])
def test_flag_guards_exactly_the_documented_range(probe, op, role):
    """each edge operand in lane 0 and in lane 1 with 1.0 in the other lane: bad() == (operand outside the range);
    the other lane's result is the one it has alone"""
    v = vc.exp_edge_values() if op == "exp" else vc.edge_values()
    n = len(v)
    lanes = np.ones(4 * n)
    lanes[0::4] = v          # pair (v, 1.0)
    lanes[3::4] = v          # pair (1.0, v)
    x, y = (lanes, None) if role != "denominator" else (np.ones(4 * n), lanes)
    want_ok = vc.documented(op, v, np.ones(n)) if role != "denominator" else vc.documented(op, np.ones(n), v)
    alone1, _ = probe.run(op, "fast1", np.ones(1), None)
    for pol in ("fast2", "fast1"):
        r, bad = probe.run(op, pol, x, y)
        for lane in (0, 3):
            wrong = np.flatnonzero(bad[lane::4] == want_ok)
            assert len(wrong) == 0, "%s %s lane %d: bad() wrong for %s" % (pol, op, lane & 1, v[wrong][:8])
        if pol == "fast2":
            assert (bad[1::4] == bad[0::4]).all() and (bad[2::4] == bad[3::4]).all()
        for lane in (1, 2):
            assert (bits(r[lane::4]) == bits(alone1)[0]).all(), "%s %s: the 1.0 lane depends on its neighbour" % (pol, op)


@pytest.mark.parametrize("op", ["div", "sqrt", "exp", "log", "powc"])
def test_flag_matches_the_range_on_every_set(probe, op):
    """FastVec<1>: bad() == outside the range, cell by cell; FastVec<2>: a thread is flagged iff one of its two cells is"""
    for window, (x, y) in operands(op).items():
        ok = vc.documented(op, x, np.ones_like(x) if y is None else y)
        _, bad1 = result(probe, op, "fast1", window)
        assert (bad1 == ~ok).all(), "%s/%s: FastVec<1> flag differs from the range at %s" % (op, window, x[bad1 == ok][:8])
        _, bad2 = result(probe, op, "fast2", window)
        okp = np.ones(len(x) + (len(x) & 1), bool)
        okp[:len(x)] = ok
        pair_ok = np.repeat(okp[0::2] & okp[1::2], 2)[:len(x)]
        assert (bad2 == ~pair_ok).all(), "%s/%s: FastVec<2> flag" % (op, window)


# ---------------------------------------------------------------------------------------------
# 2. unflagged means correct
@pytest.mark.parametrize("op", ["div", "sqrt"])
def test_div_sqrt_unflagged_are_correctly_rounded(probe, op, capsys):
    rows = []
    for window, (x, y) in operands(op).items():
        r, bad = result(probe, op, "fast2", window)
        if window in ("random", "hard", "squares"):
            assert not bad.any(), "%s/%s: operands in the proven range were flagged" % (op, window)
        ok = ~bad
        want = numpy_ref(op, x, y)
        wrong = np.flatnonzero(ok & ~same_ieee(r, want))
        assert len(wrong) == 0, "%s/%s: FastVec<2> not correctly rounded at %s" % (
            op, window, [(x[i], None if y is None else y[i], r[i], want[i]) for i in wrong[:4]])
        rows.append("  %-6s %-20s %9d cells, %9d unflagged, all bit-identical to IEEE" % (op, window, len(x), ok.sum()))
    if op == "sqrt":
        s = vc.sqrt_squares()[1]
        r, _ = result(probe, "sqrt", "fast2", "squares")
        assert (bits(r) == bits(s)).all(), "sqrt of a perfect square is not exact"
        r, bad = probe.run("sqrt", "fast2", np.array([0.0, 1.0]))
        assert bits(r)[0] == 0 and not bad.any(), "sqrt(+0) must be +0, unflagged"
    show(capsys, "\n".join(rows))


@pytest.mark.parametrize("op", ["div", "sqrt"])
def test_device_sweep_matches_ieee(probe, op):
    """2^32 operands (pairs for div) from a counter hash, exponents uniform in [-500, 499]: FastVec<2> against
    __ddiv_rn / __dsqrt_rn on the device, unflagged and bit-identical everywhere"""
    mism, first = probe.sweep(op, 0x5EEDF1C5 + vc.OPS[op], 1 << 32)
    assert mism == 0, "%s: %d mismatches, first operands %s" % (op, mism, first.tolist())


def _worst_confirmed(op, x, r, err, n):
    """the largest error, after re-measuring the n largest long double errors with mpmath at 40 digits"""
    idx = np.argsort(err)[-n:]
    mp = np.array([vc.ulp_error_mp(r[i], vc.reference_mp(op, x[i])) for i in idx])
    assert np.abs(mp - err[idx]).max() < 2e-3, "%s: the long double reference disagrees with mpmath" % op
    return max(err.max(), mp.max())


# windows with operands outside the proven range (the others must come through unflagged)
MIXED_WINDOWS = ("edges", "beyond 700", "whole double range")


@pytest.mark.parametrize("op", ["exp", "log", "powc"])
def test_fast_transcendentals_are_within_their_bounds(probe, op, capsys):
    """unflagged FastVec<2> results against long double: exp and log < 1 ulp everywhere, powc < 1 ulp for the
    Exner function, and every window at or below its ceiling; prints the maximum per window"""
    rows, over, pooled = [], [], []
    for window, (x, _) in operands(op).items():
        r, bad = result(probe, op, "fast2", window)
        if window not in MIXED_WINDOWS:
            assert not bad.any(), "%s/%s: operands in the proven range were flagged" % (op, window)
        xo, ro = x[~bad], r[~bad]
        if len(xo) == 0:
            continue
        err =vc.ulp_error(ro, vc.reference(op, xo)).astype(np.float64)
        worst = _worst_confirmed(op, xo, ro, err, n=200)
        limit = CEILINGS.get((op, window), DOCUMENTED_ULP[op] if op != "powc" or window == "physical" else None)
        rows.append("  %-5s %-22s %9d cells  max %.4f ulp  (bound %s)  at x = %r" % (
            op, window, len(err), worst, limit, xo[np.argmax(err)]))
        if limit is not None and worst > limit:
            over.append("%s/%s: %.4f ulp > %.2f" % (op, window, worst, limit))
        pooled.append((xo, ro, err))
    x, r, err = (np.concatenate(a) for a in zip(*pooled))
    worst = _worst_confirmed(op, x, r, err, n=1000)
    limit = min(CEILINGS[(op, "all")], DOCUMENTED_ULP[op]) if op != "powc" else None
    rows.append("  %-5s %-22s %9d cells  max %.4f ulp  (bound %s)" % (op, "all", len(err), worst, limit))
    if limit is not None and worst > limit:
        over.append("%s: %.4f ulp > %.2f" % (op, worst, limit))
    show(capsys, "\n".join(rows))
    assert not over, over
    if op == "exp":
        r, bad = result(probe, "exp", "fast2", "exactly 1")
        assert (r == 1.0).all() and not bad.any(), "exp(x) for |x| < 2^-54 must be exactly 1"
    if op == "log":
        r, bad = probe.run("log", "fast2", np.array([1.0, 1.0]))
        assert (bits(r) == 0).all() and not bad.any(), "log(1) must be +0"


# ---------------------------------------------------------------------------------------------
# 3. lane independence
@pytest.mark.parametrize("op", ["div", "sqrt", "exp", "log", "powc"])
def test_fastvec2_lanes_equal_fastvec1(probe, op):
    """bit for bit wherever the operand is in range.  Outside it only the sign and payload of a NaN may differ: the two
    widths compile to different instruction sequences, which may propagate a NaN with another sign (on a B200, NaN/-Inf
    of the division's edge pairs gives -NaN in one width and +NaN in the other), and a flagged cell's fast result is
    discarded anyway"""
    for window, (x, _) in operands(op).items():
        r2, _ = result(probe, op, "fast2", window)
        r1, bad1 = result(probe, op, "fast1", window)
        diff = np.flatnonzero(np.where(bad1, ~same_ieee(r2, r1), bits(r2) != bits(r1)))
        assert len(diff) == 0, "%s/%s: FastVec<2> differs from FastVec<1> at x = %s" % (op, window, x[diff][:8])


# ---------------------------------------------------------------------------------------------
# 4. the cold path keeps the hot path's bits (ExactVec has no log: powc carries log_core there)
@pytest.mark.parametrize("op", ["div", "sqrt", "exp", "powc"])
def test_cold_path_keeps_the_hot_path_bits(probe, op):
    for window, (x, _) in operands(op).items():
        rf, bad = result(probe, op, "fast2", window)
        rc, _ = result(probe, op, "exactvec2", window)
        diff = np.flatnonzero(~bad & (bits(rf) != bits(rc)))
        assert len(diff) == 0, "%s/%s: ExactVec<2> differs from unflagged FastVec<2> at x = %s" % (op, window, x[diff][:8])


# ---------------------------------------------------------------------------------------------
# 5. outside the range the cold path is IEEE and libm-grade
@pytest.mark.parametrize("policy", ["exactvec2", "exactscalar"])
@pytest.mark.parametrize("op", ["div", "sqrt"])
def test_cold_div_sqrt_are_ieee_everywhere(probe, op, policy):
    for window, (x, y) in operands(op).items():
        r, bad = result(probe, op, policy, window)
        assert not bad.any()
        want = numpy_ref(op, x, y)
        wrong = np.flatnonzero(~same_ieee(r, want))
        assert len(wrong) == 0, "%s %s/%s: not IEEE at %s" % (policy, op, window,
                                                              [(x[i], None if y is None else y[i], r[i], want[i]) for i in wrong[:4]])
    r, _ = probe.run("sqrt", policy, np.array([-0.0, -1.0, -np.inf]))
    assert bits(r)[0] == bits(np.array([-0.0]))[0] and np.isnan(r[1:]).all()


ANNEX_F = {
    # exp: C99 F.9.3.1 and overflow / underflow
    "exp": [(np.inf, np.inf), (-np.inf, 0.0), (np.nan, np.nan), (0.0, 1.0), (-0.0, 1.0), (709.79, np.inf), (710.0, np.inf),
            (1e308, np.inf), (np.finfo(np.float64).max, np.inf), (-745.2, 0.0), (-746.0, 0.0), (-1e308, 0.0)],
    # pow(x, c), c = R_d/c_p > 0 and not an integer: C99 F.9.4.4
    "powc": [(0.0, 0.0), (-0.0, 0.0), (-1.0, np.nan), (-2.0 ** -600, np.nan), (-1e300, np.nan), (np.inf, np.inf),
             (-np.inf, np.inf), (np.nan, np.nan), (1.0, 1.0)],
}


@pytest.mark.parametrize("policy", ["exactvec2", "exactscalar"])
@pytest.mark.parametrize("op", ["exp", "powc"])
def test_cold_exp_pow_special_values(probe, op, policy):
    x = np.array([a for a, _ in ANNEX_F[op]])
    want = np.array([b for _, b in ANNEX_F[op]])
    r, _ = probe.run(op, policy, x)
    wrong = np.flatnonzero(~same_ieee(r, want))
    assert len(wrong) == 0, "%s %s: %s" % (policy, op, [(x[i], r[i], want[i]) for i in wrong])


@pytest.mark.parametrize("policy", ["exactvec2", "exactscalar"])
@pytest.mark.parametrize("op", ["exp", "powc"])
def test_cold_exp_pow_are_within_libdevice_bounds(probe, op, policy, capsys):
    """finite results within libdevice's documented 1 ulp (exp) and 2 ulp (pow), subnormal results measured in
    the subnormal spacing"""
    rows = []
    for window, (x, _) in operands(op).items():
        r, bad = result(probe, op, policy, window)
        ref = vc.reference(op, x)
        fin = np.isfinite(ref) & (np.abs(ref) <= np.longdouble(np.finfo(np.float64).max))
        if policy == "exactvec2":
            fin &= ~vc.documented(op, x)         # inside, ExactVec runs FastVec's sequences (asserted above)
        err = vc.ulp_error(r[fin], ref[fin]).astype(np.float64)
        if len(err):
            rows.append("  %-11s %-5s %-22s max %.4f ulp" % (policy, op, window, err.max()))
            assert err.max() <= LIBDEVICE_ULP[op], "%s %s/%s: %.4f ulp at x = %r" % (
                policy, op, window, err.max(), x[fin][np.argmax(err)])
    show(capsys, "\n".join(rows))
