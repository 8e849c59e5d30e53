"""-m gpu: the fused / generic per-step path through the C ABI against the CPU oracle on seeded fields."""
import numpy as np
import pytest

from oracle_py import Oracle, ulp_diff
from tolerances import check_field, check_scenario

pytestmark = pytest.mark.gpu


def run_both(fcmod, sc, mode="host", t=0, force_generic=False, phases="all", chunks=None, diagnostics=0, staged=None):
    from components.flux_calculator_b200 import DeviceArray
    # oracle
    o_in, o_out = sc.clone()
    orc = Oracle(sc.n, sc.S)
    sc.apply(orc, o_in, o_out)
    if phases == "all":
        orc.step_all(t)
    else:
        orc.step_early(t)
        orc.step_normal(t)
    # CUDA
    g_in, g_out = sc.clone()
    fc = fcmod.FluxCalculator(sc.n, sc.S)
    if force_generic:
        fc.set_option("force_generic", 1)
    if chunks:
        fc.set_option("h2d_chunks", chunks)
    if staged is not None:      # 0: direct-load kernel only, 2: staged (cp.async.bulk + mbarrier) kernel whenever possible
        fc.set_option("staged", staged)
    if mode == "host":
        sc.apply(fc, g_in, g_out)
        wrapped = None
    else:
        wrapped = sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a))
    if diagnostics:
        for g in (1, 2, 3):
            fc.set_area(g, sc.area[g])
        fc.set_option("diagnostics", int(diagnostics))
    fc.prepare()
    if phases == "all":
        fc.step_all(t)
    else:
        fc.step_early(t)
        fc.step_normal(t)
    fc.synchronize()
    if wrapped is not None:
        for d in (g_in, g_out):
            for k, a in d.items():
                wrapped[id(a)].download(a)
    return fc, o_out, g_out, o_in, g_in


def compare(sc, o_out, g_out):
    return check_scenario(sc, g_out, o_out)


@pytest.mark.parametrize("fset", ["CCLM", "MOM5", "RCO"])
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("staged", [0, 2])
def test_step_all_s1(fcmod, fset, mode, staged):
    from synthetic import Scenario
    sc = Scenario(fset, n=(20000, 20000, 20000), S=1, bias=(fset == "MOM5"))
    fc, o_out, g_out, o_in, g_in = run_both(fcmod, sc, mode, staged=staged)
    assert fc.info("fused") == 1
    compare(sc, o_out, g_out)
    for k in o_in:      # inputs untouched
        assert np.array_equal(o_in[k], g_in[k], equal_nan=True)


@pytest.mark.parametrize("fset", ["CCLM", "MOM5", "RCO"])
def test_generic_path_matches(fcmod, fset):
    from synthetic import Scenario
    sc = Scenario(fset, n=(5003, 4999, 5001), S=2, bias=True, averaging=True)
    fc, o_out, g_out, _, _ = run_both(fcmod, sc, "host", force_generic=True)
    assert fc.info("fused") == 0
    compare(sc, o_out, g_out)
    fc2, _, f_out, _, _ = run_both(fcmod, sc, "device")
    assert fc2.info("fused") == 1
    # fused (lock-step exp / exp(c*log x)) and generic (libdevice exp / pow) kernels: identical wherever no
    # transcendental is upstream, within the stated tolerance elsewhere
    check_scenario(sc, f_out, g_out)


@pytest.mark.parametrize("S", [2, 3, 5])
def test_surface_types_and_averaging(fcmod, S):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(7001, 7003, 6999), S=S, bias=True, averaging=True)
    for mode in ("host", "device"):
        fc, o_out, g_out, _, _ = run_both(fcmod, sc, mode, t=40 * 86400)
        assert fc.info("fused") == 1
        compare(sc, o_out, g_out)
    # averaging itself is exact arithmetic on the per-type values
    for (i, g, name) in sc.send:
        acc = np.zeros(sc.n[g - 1])
        for t in range(1, S + 1):
            acc = acc + g_out[(t, g, name)] * sc.inputs[(t, g, "FARE")]
        assert np.array_equal(acc, g_out[(0, g, name)])


def test_split_phases_equal_fused_all(fcmod):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(4096, 4096, 4096), S=2, bias=True, averaging=True, passthrough_avg=True)
    _, o_out, a_out, _, _ = run_both(fcmod, sc, "device", phases="all")
    _, _, s_out, _, _ = run_both(fcmod, sc, "device", phases="split")
    compare(sc, o_out, a_out)
    for k in a_out:
        assert np.array_equal(a_out[k], s_out[k], equal_nan=True), k


@pytest.mark.parametrize("n", [(0, 0, 0), (1, 1, 1), (3, 2, 1), (511, 513, 1025), (33, 0, 7), (5121, 1024, 2047)])
@pytest.mark.parametrize("staged", [0, 2])
def test_ragged_and_tiny_grids(fcmod, n, staged):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=n, S=1, bias=True)
    for mode in ("host", "device"):
        _, o_out, g_out, _, _ = run_both(fcmod, sc, mode, staged=staged)
        compare(sc, o_out, g_out)


def test_staged_and_direct_kernels_agree_bitwise(fcmod):
    """same formula templates, same arithmetic policy: the shared-memory staged kernel and the direct-load kernel
    must produce identical bits (incl. a persistent grid that wraps: 700 tiles > 2 x 148 CTAs)"""
    from synthetic import Scenario
    for fset in ("CCLM", "RCO"):
        sc = Scenario(fset, n=(358400, 358400 + 77, 358400 - 513), S=1, bias=True)
        _, o_out, d_out, _, _ = run_both(fcmod, sc, "device", staged=0)
        _, _, s_out, _, _ = run_both(fcmod, sc, "device", staged=2)
        compare(sc, o_out, d_out)
        for k in d_out:
            assert np.array_equal(d_out[k], s_out[k], equal_nan=True), k


def test_extreme_operands_take_the_exact_path(fcmod):
    """operands outside [2^-500, 2^500] (or -0 / Inf where it matters) leave the lock-step fast path: the thread
    recomputes its cells with the IEEE routines, results stay bit-exact where no transcendental is involved"""
    from synthetic import Scenario
    sc = Scenario("RCO", n=(4096, 4096, 4096), S=1)
    before = None
    for staged in (0, 2):
        sc.inputs[(0, 2, "UATM")][5] = 1e200      # u*u overflows -> sqrt(inf)
        sc.inputs[(0, 2, "UATM")][6] = 1e-200     # u*u underflows to a tiny sqrt argument
        sc.inputs[(0, 3, "VATM")][9] = -0.0
        fc, o_out, g_out, _, _ = run_both(fcmod, sc, "device", staged=staged)
        calls = fc.info("exact_path_calls")
        assert calls > (before or 0)
        before = calls
        for k in ((1, 2, "UMOM"), (1, 3, "VMOM")):
            a, b = g_out[k], o_out[k]
            assert np.array_equal(a, b, equal_nan=True), k


def test_month_rollover_bias(fcmod):
    from synthetic import Scenario
    sc = Scenario("MOM5", n=(3000, 3000, 3000), S=1, bias=True, init_date=19611231)
    outs = []
    for t in (0, 86399, 86400, 31 * 86400 + 86400):     # Dec, Dec, Jan, Feb
        _, o_out, g_out, _, _ = run_both(fcmod, sc, "host", t=t)
        compare(sc, o_out, g_out)
        outs.append(g_out[(1, 1, "MEVA")].copy())
    assert np.array_equal(outs[0], outs[1])
    assert not np.array_equal(outs[1], outs[2])
    assert not np.array_equal(outs[2], outs[3])


def test_chunked_host_pipeline(fcmod):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(300001, 299999, 300003), S=1, bias=True)
    _, o_out, g1, _, _ = run_both(fcmod, sc, "host", chunks=1)
    _, _, g7, _, _ = run_both(fcmod, sc, "host", chunks=7)
    compare(sc, o_out, g1)
    for k in g1:
        assert np.array_equal(g1[k], g7[k], equal_nan=True), k


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("staged", [0, 2])
@pytest.mark.parametrize("S,n", [(2, (10007, 10009, 10011)), (1, (200000, 150001, 99999)), (1, (3, 700, 0))])
def test_diagnostics(fcmod, level, S, n, staged):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=n, S=S, bias=True, averaging=True)
    for mode in ("device", "host"):
        fc, o_out, g_out, _, _ = run_both(fcmod, sc, mode, diagnostics=level, staged=staged)
        compare(sc, o_out, g_out)
        for (i, g, name), arr in g_out.items():
            if arr.size == 0:
                continue
            s, mn, mx = fc.diagnostics(i, g, name)
            if level == 2:      # reproduces the reference's debug "range =" lines (flux_calculator.F90:1013)
                assert mn == arr.min() and mx == arr.max(), (i, g, name)
            else:
                assert np.isnan(mn) and np.isnan(mx)
            ref = float(np.sum(sc.area[g] * arr))
            assert abs(s - ref) <= 1e-11 * float(np.sum(np.abs(sc.area[g] * arr))), (i, g, name)


def _diag_check(fc, sc, g_out, level):
    for (i, g, name), arr in g_out.items():
        if arr.size == 0:
            continue
        s, mn, mx = fc.diagnostics(i, g, name)
        if level == 2:
            assert mn == arr.min() and mx == arr.max(), (i, g, name)
        ref = float(np.sum(sc.area[g] * arr))
        assert abs(s - ref) <= 1e-11 * float(np.sum(np.abs(sc.area[g] * arr))), (i, g, name)


@pytest.mark.parametrize("fset", ["CCLM", "MOM5", "RCO"])
@pytest.mark.parametrize("level", [0, 1, 2])
def test_spec_kernel_cold_epilogue(fcmod, fset, level):
    """specialised persistent kernel: tiles with operands outside the proven range are recomputed by the cold
    epilogue (IEEE routines, from global memory) and the warp's diagnostics are rebuilt from the stored outputs;
    every other cell keeps the bits of the lock-step path (same results as the direct-load kernel)"""
    from synthetic import Scenario
    sc = Scenario(fset, n=(300000 + 37, 200000, 250000 + 511), S=1, bias=True)
    a_t = {"CCLM": "AMOI", "MOM5": "CMOI", "RCO": "QATM"}[fset]
    t_key = [k for k in sc.inputs if k[1] == 1 and k[2] == a_t][0]
    sc.inputs[t_key][3] = 1e-310                     # denormal operand (t grid, first tile)
    sc.inputs[t_key][123457] = 1e-310                # ... and a tile deep inside another CTA's schedule
    for idx in (5, 199999):                          # u*u + v*v denormal: sqrt argument outside the proven range
        sc.inputs[(0, 2, "UATM")][idx] = 1e-160
        sc.inputs[(0, 2, "VATM")][idx] = 1e-160
    sc.inputs[(0, 3, "UATM")][77777] = 1e-160
    sc.inputs[(0, 3, "VATM")][77777] = -1e-160
    outs = {}
    for staged in (0, 2):
        fc, o_out, g_out, _, _ = run_both(fcmod, sc, "device", diagnostics=level, staged=staged)
        compare(sc, o_out, g_out)
        if level:
            _diag_check(fc, sc, g_out, level)
        outs[staged] = g_out
    assert fc.info("exact_path_calls") > 0
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[2][k], equal_nan=True), k


def test_spec_kernel_flag_overflow(fcmod):
    """more flagged tiles per warp than the epilogue remembers individually -> every tile of that warp is redone"""
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(512 * 296 * 17 + 512 * 40, 1024, 512), S=1, bias=True)
    t_key = [k for k in sc.inputs if k[1] == 1 and k[2] == "AMOI"][0]
    sc.inputs[t_key][::512] = 1e-310                 # one denormal operand in every tile
    fc, o_out, g_out, _, _ = run_both(fcmod, sc, "device", diagnostics=1, staged=2)
    compare(sc, o_out, g_out)
    _diag_check(fc, sc, g_out, 1)


@pytest.mark.parametrize("n", [(512, 300000, 1024), (150000, 512, 0), (1024, 1024, 400000), (152064, 152064, 152064)])
@pytest.mark.parametrize("fset", ["MOM5", "RCO"])
def test_spec_kernel_schedules(fcmod, n, fset):
    """persistent schedule corner cases: CTAs without t tiles, empty grids, t->u/v ring hand-over with few tiles,
    exactly one tile per CTA"""
    from synthetic import Scenario
    sc = Scenario(fset, n=n, S=1, bias=True)
    _, o_out, d_out, _, _ = run_both(fcmod, sc, "device", staged=0)
    fc, _, s_out, _, _ = run_both(fcmod, sc, "device", staged=2, diagnostics=2)
    compare(sc, o_out, s_out)
    _diag_check(fc, sc, s_out, 2)
    for k in d_out:
        assert np.array_equal(d_out[k], s_out[k], equal_nan=True), k


def test_repeated_steps_reuse_diagnostics_buffers(fcmod):
    """the in-kernel last-CTA reduction resets its counter: many steps in a row give the same diagnostics"""
    from components.flux_calculator_b200 import DeviceArray
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(200000, 200000, 200000 + 3), S=1, bias=True)
    g_in, g_out = sc.clone()
    fc = fcmod.FluxCalculator(sc.n, sc.S)
    fc.set_option("staged", 2)
    sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a))
    for g in (1, 2, 3):
        fc.set_area(g, sc.area[g])
    fc.set_option("diagnostics", 2)
    fc.prepare()
    first = None
    for k in range(7):
        fc.step_all(0)
        d = fc.diagnostics(1, 3, "VMOM")
        if first is None:
            first = d
        assert d == first


@pytest.mark.parametrize("staged", [0, 2])
@pytest.mark.parametrize("S", [1, 2])
def test_chunked_host_pipeline_with_diagnostics(fcmod, S, staged):
    """host-pointer pipeline in several chunks: every chunk reduces its own diagnostics vector (concurrently, on
    three streams), a combine kernel folds them in chunk order"""
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(300001, 299999, 300003), S=S, bias=True, averaging=True)
    fc1, o_out, g1, _, _ = run_both(fcmod, sc, "host", chunks=1, diagnostics=2, staged=staged)
    fc7, _, g7, _, _ = run_both(fcmod, sc, "host", chunks=7, diagnostics=2, staged=staged)
    compare(sc, o_out, g7)
    _diag_check(fc7, sc, g7, 2)
    for k in g1:
        assert np.array_equal(g1[k], g7[k], equal_nan=True), k
        if g1[k].size:
            d1, d7 = fc1.diagnostics(*k), fc7.diagnostics(*k)
            assert d1[1:] == d7[1:] and abs(d1[0] - d7[0]) <= 1e-12 * abs(d1[0]) + 1e-300, k


@pytest.mark.parametrize("fset", ["CCLM", "MOM5", "RCO"])
@pytest.mark.parametrize("level", [0, 1, 2])
def test_spec_kernel_two_surface_types_long_schedule(fcmod, fset, level):
    """two surface types: one CTA per SM, two consumer teams sharing the ring (one barrier per (team, stage) pair);
    several tiles per team and per stage so that the barrier phases wrap, ragged remainders, averaging of the sent
    fluxes; bitwise equal to the direct-load kernel, within tolerance of the oracle"""
    from synthetic import Scenario
    n = (512 * 148 * 9 + 300, 512 * 148 * 5 + 1, 512 * 148 * 6 + 511)
    sc = Scenario(fset, n=n, S=2, bias=True, averaging=True)
    _, o_out, d_out, _, _ = run_both(fcmod, sc, "device", staged=0, diagnostics=level)
    fc, _, s_out, _, _ = run_both(fcmod, sc, "device", staged=2, diagnostics=level)
    assert fc.info("spec_kernel") == 1
    compare(sc, o_out, s_out)
    if level:
        _diag_check(fc, sc, s_out, level)
    for k in d_out:
        assert np.array_equal(d_out[k], s_out[k], equal_nan=True), k


def test_spec_kernel_two_surface_types_without_averaging(fcmod):
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(200000, 100001, 99999), S=2, bias=True, averaging=False)
    _, o_out, d_out, _, _ = run_both(fcmod, sc, "device", staged=0)
    fc, _, s_out, _, _ = run_both(fcmod, sc, "device", staged=2)
    assert fc.info("spec_kernel") == 1
    compare(sc, o_out, s_out)
    for k in d_out:
        assert np.array_equal(d_out[k], s_out[k], equal_nan=True), k


@pytest.mark.parametrize("mode", ["device", "host"])
@pytest.mark.parametrize("fset,S", [("CCLM", 1), ("RCO", 1), ("MOM5", 2), ("RCO", 2)])
def test_dynamic_tile_schedule(fcmod, fset, S, mode):
    """without diagnostics the specialised kernel claims its tiles from a global counter on large grids; forced here on a
    small one (option dyn_min_tiles = 1): partial tiles on every grid, more flagged tiles than a warp's list holds, several
    consecutive steps (the counter is never reset).  In host mode the step runs as three chunks, each with its own counter.
    The steps before the last compute from other inputs, so a tile that the last step fails to claim because the host's
    idea of a counter's base drifted keeps a wrong result.  Bit-identical to the static schedule, and within tolerance of
    the oracle"""
    from components.flux_calculator_b200 import DeviceArray
    from synthetic import Scenario
    sc = Scenario(fset, n=(512 * 700 + 37, 512 * 650 + 1, 512 * 600 + 511), S=S, bias=True, averaging=True)
    a_t = {"CCLM": "AMOI", "MOM5": "CMOI", "RCO": "QATM"}[fset]
    t_key = [k for k in sc.inputs if k[1] == 1 and k[2] == a_t][0]
    sc.inputs[t_key][::1024] = 1e-310                # a denormal operand in every second t tile: the cold path, list overflow included
    sc.inputs[(0, 3, "UATM")][77777] = 1e-160
    sc.inputs[(0, 3, "VATM")][77777] = -1e-160
    o_in, o_out = sc.clone()
    orc = Oracle(sc.n, sc.S)
    sc.apply(orc, o_in, o_out)
    orc.step_all(86400 * 40)
    res = {}
    for dyn in (1, 1 << 30):
        g_in, g_out = sc.clone()
        fc = fcmod.FluxCalculator(sc.n, sc.S)
        if mode == "host":
            fc.set_option("h2d_chunks", 3)
            sc.apply(fc, g_in, g_out)
            wrapped = {}
        else:
            wrapped = sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a))
        fc.set_option("dyn_min_tiles", dyn)
        fc.prepare()
        assert fc.info("spec_kernel") == 1
        ins = list({id(a): a for a in g_in.values()}.values())
        exact = [a.copy() for a in ins]
        for k in range(5):
            fc.synchronize()
            for a, e in zip(ins, exact):
                np.multiply(e, 1.0 + 2.0 ** -12 if k < 4 else 1.0, out=a)
                if wrapped:
                    wrapped[id(a)].upload(a)
            fc.step_all(86400 * 10 * k)
        fc.synchronize()
        for k, a in g_out.items():
            if wrapped:
                wrapped[id(a)].download(a)
        res[dyn] = g_out
        fc.close()
        for w in wrapped.values():
            w.free()
    compare(sc, o_out, res[1])
    for k in res[1]:
        assert np.array_equal(res[1][k], res[1 << 30][k], equal_nan=True), k


@pytest.mark.parametrize("S,diag", [(1, 0), (1, 2), (2, 0), (2, 1)])
def test_run_steps_equals_single_steps(fcmod, S, diag):
    """fc_run_steps (CUDA graphs of 32 step launches per calendar month, the rest issued directly) == the same steps
    issued one by one, bit for bit, with the bias month rolling over twice (flux_calculator.F90:859-1028)"""
    from components.flux_calculator_b200 import DeviceArray
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(60000 + 5, 50000, 70000 + 300), S=S, bias=True, averaging=True, init_date=19610101)
    nsteps, dt = 300, 21600      # 75 days in steps of 6 hours: January -> February -> March
    res, dg = {}, {}
    for mode in ("graph", "single"):
        g_in, g_out = sc.clone()
        fc = fcmod.FluxCalculator(sc.n, sc.S)
        wrapped = sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a))
        if diag:
            for g in (1, 2, 3):
                fc.set_area(g, sc.area[g])
            fc.set_option("diagnostics", diag)
        fc.prepare()
        l0 = fc.info("launches")
        if mode == "graph":
            fc.run_steps(0, dt, nsteps)
            assert fc.info("graph_launches") == (124 // 32) + (112 // 32) + (64 // 32)      # 124 + 112 + 64 steps per month
        else:
            for k in range(nsteps):
                fc.step_all(k * dt)
        fc.synchronize()
        assert fc.info("launches") - l0 >= nsteps
        for k, a in g_out.items():
            wrapped[id(a)].download(a)
        res[mode] = g_out
        if diag:
            dg[mode] = {k: fc.diagnostics(*k) for k in g_out}
        fc.close()
        for w in wrapped.values():
            w.free()
    o_in, o_out = sc.clone()
    orc = Oracle(sc.n, sc.S)
    sc.apply(orc, o_in, o_out)
    orc.step_all((nsteps - 1) * dt)
    compare(sc, o_out, res["graph"])
    for k in res["graph"]:
        assert np.array_equal(res["graph"][k], res["single"][k], equal_nan=True), k
    if diag:
        for k in dg["graph"]:
            a, b = dg["graph"][k], dg["single"][k]
            assert a[0] == b[0] and (diag < 2 or (a[1] == b[1] and a[2] == b[2])), k


def test_static_inputs_and_sent_only_download(fcmod):
    """host-pointer mode: arrays marked static travel once (the reference's namelist constants, val_*), with option
    download = 1 only registered output fields come back; the sent fields are bit-identical to the everything-travels mode"""
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(300000, 300000, 300000), S=1, bias=True)
    sent = [(1, 1, "MEVA"), (1, 1, "HLAT"), (1, 1, "HSEN"), (1, 1, "RBBR"), (1, 1, "RSDR"), (1, 2, "UMOM"), (1, 3, "VMOM")]
    a_in, a_out = sc.clone()
    fa = fcmod.FluxCalculator(sc.n, sc.S)
    sc.apply(fa, a_in, a_out)
    fa.step_all(0)
    full_h2d, full_d2h = fa.info("h2d_bytes_per_step"), fa.info("d2h_bytes_per_step")
    b_in, b_out = sc.clone()
    fb = fcmod.FluxCalculator(sc.n, sc.S)
    sc.apply(fb, b_in, b_out)
    for key in sent:
        fb.add_output_field(*key)
    for g in (1, 2, 3):
        fb.mark_static(1, g, "FICE")
    fb.set_option("download", 1)
    fb.step_all(0)
    first_h2d = fb.info("h2d_bytes_per_step")
    fb.step_all(0)
    n8 = 8 * 300000
    assert first_h2d == full_h2d and fb.info("h2d_bytes_per_step") == full_h2d - 3 * n8      # FICE x 3 grids stays on the device
    assert fb.info("d2h_bytes_per_step") == len(sent) * n8 and full_d2h == len(a_out) * n8
    for key in a_out:
        if key in sent:
            assert np.array_equal(a_out[key], b_out[key]), key
        else:
            assert np.isnan(b_out[key]).all(), key      # QSUR never left the device
    # a static array rewritten by the host is picked up only after fc_mark_dirty
    b_in[(1, 1, "FICE")][:] = 1.0
    fb.step_all(0)
    assert np.array_equal(a_out[(1, 1, "MEVA")], b_out[(1, 1, "MEVA")])
    fb.mark_dirty(1, 1, "FICE")
    fb.step_all(0)
    assert not np.array_equal(a_out[(1, 1, "MEVA")], b_out[(1, 1, "MEVA")])
    a_in[(1, 1, "FICE")][:] = 1.0
    fa.step_all(0)
    assert np.array_equal(a_out[(1, 1, "MEVA")], b_out[(1, 1, "MEVA")])
    fa.close()
    fb.close()


@pytest.mark.parametrize("S,diag", [(1, 0), (1, 1), (2, 1)])
def test_chained_steps_keep_the_stream_order(fcmod, S, diag):
    """consecutive device-resident steps of one plan hand over per CTA instead of waiting for the whole previous grid:
    the results of the LAST step must win in every cell (the bias month alternates from step to step, so a stale store
    of the step before would show), with and without the option, and the diagnostics are those of the last step"""
    from components.flux_calculator_b200 import DeviceArray
    from synthetic import Scenario
    sc = Scenario("CCLM", n=(512 * 900 + 3, 512 * 900, 512 * 901), S=S, bias=True, averaging=True, init_date=19610101)
    times = [0 if k % 2 == 0 else 86400 * 45 for k in range(101)]      # January / February alternating; the last one is January
    res = {}
    for chain in (1, 0):
        g_in, g_out = sc.clone()
        fc = fcmod.FluxCalculator(sc.n, sc.S)
        wrapped = sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a))
        if diag:
            for g in (1, 2, 3):
                fc.set_area(g, sc.area[g])
            fc.set_option("diagnostics", diag)
        fc.set_option("chain", chain)
        fc.set_option("dyn_min_tiles", 1 << 30)      # static schedule (the dynamic one never chains)
        fc.prepare()
        for t in times:
            fc.step_all(t)
        fc.synchronize()
        for k, a in g_out.items():
            wrapped[id(a)].download(a)
        res[chain] = (g_out, {k: fc.diagnostics(*k)[0] for k in g_out} if diag else None)
        fc.close()
        for w in wrapped.values():
            w.free()
    o_in, o_out = sc.clone()
    orc = Oracle(sc.n, sc.S)
    sc.apply(orc, o_in, o_out)
    orc.step_all(times[-1])
    compare(sc, o_out, res[1][0])
    for k in res[1][0]:
        assert np.array_equal(res[1][0][k], res[0][0][k], equal_nan=True), k
    if diag:
        assert res[1][1] == res[0][1]
