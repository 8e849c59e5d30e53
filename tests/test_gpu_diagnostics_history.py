"""Per-step diagnostics history (option "diagnostics_history", fc_get_diagnostics_history): the vector of every step,
bit-identical to fc_get_diagnostics read right after that step, on every step path -- graph replays of fc_run_steps,
directly issued steps, the generic kernel, the host-pointer pipeline and the split phases -- and no change with it off."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FC_ERR_ARG, FC_ERR_STATE = 1, 6
DT = 21600                          # 6 hours: January (124 steps) -> February (112) -> March (64) in 300 steps
CALLS = (45, 64, 33, 158)           # fc_run_steps calls: graph replays mixed with directly issued remainders
GRAPHS = 1 + 2 + 0 + 2 + 2          # replays of 32 steps: 45 | 64 | 15 + 18 | 94 + 64, split at the month boundaries


def same_bits(a, b):
    """equal bit for bit, NaN where the other is NaN"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def scenario(S, averaging):
    from synthetic import Scenario
    return Scenario("CCLM", n=(60000 + 5, 50000, 70000 + 300), S=S, bias=True, averaging=averaging, init_date=19610101)


def context(fcmod, sc, level, history=0, device=True, options=()):
    from components.flux_calculator_b200 import DeviceArray
    g_in, g_out = sc.clone()
    fc = fcmod.FluxCalculator(sc.n, sc.S)
    wrapped = sc.apply(fc, g_in, g_out, wrap=(lambda a: DeviceArray.from_numpy(a)) if device else (lambda a: a))
    for g in (1, 2, 3):
        fc.set_area(g, sc.area[g])
    fc.set_option("diagnostics", level)
    for name, value in options:
        fc.set_option(name, value)
    if history:
        fc.set_option("diagnostics_history", history)
    fc.prepare()
    return fc, wrapped, g_in, g_out


def close(fc, wrapped):
    fc.close()
    for w in wrapped.values():
        if hasattr(w, "free"):
            w.free()


def run_calls(fc, wrapped, g_in, one_by_one, per_step=None):
    """the steps of CALLS, either through fc_run_steps or as fc_step_all one at a time (then per_step(k) after step k);
    before every call TSUR of surface type 1 is rewritten with a call-specific factor, so that no two calls agree"""
    tsur = g_in[(1, 1, "TSUR")]
    base = tsur.copy()
    k = 0
    for j, n in enumerate(CALLS):
        fc.synchronize()
        wrapped[id(tsur)].upload(base * (1.0 + 1e-3 * j))
        if one_by_one:
            for _ in range(n):
                fc.step_all(k * DT)
                per_step(k)
                k += 1
        else:
            fc.run_steps(k * DT, DT, n)
            k += n
    fc.synchronize()
    return k


def read_or_nan(fcmod, fc, k):
    """fc_get_diagnostics, or NaN for a field the last step did not compute"""
    try:
        return fc.diagnostics(*k)
    except fcmod.FluxCalcError as e:
        assert e.code == FC_ERR_STATE
        return (np.nan,) * 3


def reference_series(fcmod, sc, level, options=()):
    """fc_get_diagnostics after each of the steps of CALLS issued one by one, without the history: key -> (steps, 3)"""
    fc, wrapped, g_in, g_out = context(fcmod, sc, level, options=options)
    series = {k: [] for k in g_out}
    run_calls(fc, wrapped, g_in, True, lambda _: [series[k].append(fc.diagnostics(*k)) for k in g_out])
    close(fc, wrapped)
    return {k: np.array(v) for k, v in series.items()}


@pytest.mark.parametrize("S,averaging,level,options", [
    (1, False, 1, ()),
    (1, False, 2, ()),
    (2, True, 1, ()),                 # the specialised kernel: captured steps fold their predecessors' rows
    (2, True, 2, ()),
    (3, True, 2, ()),                 # the generic kernel: captured finalize launches
    (1, False, 2, (("staged", 0),)),  # the generic kernel at one surface type
])
def test_run_steps_history_equals_per_step_reads(fcmod, S, averaging, level, options):
    """the history of 300 steps of fc_run_steps (graph replays and direct steps, two month changes, inputs rewritten
    between the calls) == fc_get_diagnostics after each of the same steps issued one by one, bit for bit"""
    sc = scenario(S, averaging)
    ref = reference_series(fcmod, sc, level, options)
    nsteps = sum(CALLS)
    fc, wrapped, g_in, g_out = context(fcmod, sc, level, history=nsteps, options=options)
    run_calls(fc, wrapped, g_in, False)
    assert fc.info("graph_launches") == GRAPHS      # as without the history
    assert fc.info("diagnostics_history_steps") == nsteps
    for k in g_out:
        h = fc.diagnostics_history(*k)
        assert h.shape == (nsteps, 3)
        assert same_bits(h, ref[k]), k
        if level < 2:
            assert np.isnan(h[:, 1:]).all()
    # the months differ in their corrections, the calls in TSUR: no two consecutive calls give the same MEVA sum
    meva = fc.diagnostics_history(1, 1, "MEVA")[:, 0]
    ends = np.cumsum(CALLS) - 1
    assert len(set(meva[ends].tolist())) == len(CALLS)
    close(fc, wrapped)


def test_history_ring_keeps_the_last_h_steps(fcmod):
    """H = 50 over 300 steps: steps [250, 300) are retained and equal the per-step reads; any window reaching outside
    them is refused with FC_ERR_ARG, naming the retained range"""
    sc = scenario(1, False)
    ref = reference_series(fcmod, sc, 2)
    fc, wrapped, g_in, g_out = context(fcmod, sc, 2, history=50)
    run_calls(fc, wrapped, g_in, False)
    assert fc.info("diagnostics_history_steps") == 300
    for k in g_out:
        h = fc.diagnostics_history(*k)
        assert h.shape == (50, 3) and same_bits(h, ref[k][250:]), k
        assert same_bits(fc.diagnostics_history(*k, first=262, count=7), ref[k][262:269]), k
    for first, count in ((249, 1), (249, 51), (260, 41), (300, 1), (0, 300)):
        with pytest.raises(fcmod.FluxCalcError) as e:
            fc.diagnostics_history(1, 1, "MEVA", first=first, count=count)
        assert e.value.code == FC_ERR_ARG and "[250, 300)" in e.value.message
    close(fc, wrapped)


def test_history_of_host_pointer_steps_and_split_phases(fcmod):
    """host arrays through the four-chunk pipeline, fc_step_early and fc_step_normal alternating: the RBBR entries of the
    early steps and the flux entries of the normal steps are what fc_get_diagnostics returned after them, the entries a
    phase did not compute are NaN"""
    sc = scenario(2, True)
    fc, wrapped, g_in, g_out = context(fcmod, sc, 2, history=16, device=False, options=(("h2d_chunks", 4),))
    phases = ["early", "normal"] * 4
    expect = {k: [] for k in g_out}
    for j, ph in enumerate(phases):
        t = j * 86400 * 20      # the month changes along the way
        l0 = fc.info("launches")
        (fc.step_early if ph == "early" else fc.step_normal)(t)
        # four chunks, each a step launch and a fold or finalize, then the combine that also writes the history row
        # (one chunk would be at most three launches)
        assert fc.info("launches") - l0 >= 4 * 2 + 1, ph
        for k in g_out:
            expect[k].append(read_or_nan(fcmod, fc, k))
    assert fc.info("diagnostics_history_steps") == len(phases)
    for k in g_out:
        h = fc.diagnostics_history(*k)
        assert same_bits(h, np.array(expect[k])), k
        early = k[2] == "RBBR"
        for j, ph in enumerate(phases):
            assert np.isnan(h[j]).all() == ((ph == "early") != early), (k, j)
    close(fc, wrapped)


def test_run_steps_around_a_step_of_another_phase(fcmod):
    """fc_run_steps (the graph is captured), an fc_step_early step (the early bundle's diagnostics rows have a layout of
    their own), then fc_run_steps again in the same month, starting with a replay of that graph: the history of all 81
    steps, the graph's last steps included, == fc_get_diagnostics after each of the same steps issued one by one"""
    sc = scenario(2, True)
    plan = [("run", 40), ("early", 1), ("run", 40)]      # January: one replay + 8 direct steps on either side
    fc, wrapped, g_in, g_out = context(fcmod, sc, 2)
    ref = {k: [] for k in g_out}
    k = 0
    for what, n in plan:
        for _ in range(n):
            (fc.step_all if what == "run" else fc.step_early)(k * DT)
            for key in g_out:
                ref[key].append(read_or_nan(fcmod, fc, key))
            k += 1
    close(fc, wrapped)
    fc, wrapped, g_in, g_out = context(fcmod, sc, 2, history=128)
    k = 0
    for what, n in plan:
        if what == "run":
            fc.run_steps(k * DT, DT, n)
        else:
            fc.step_early(k * DT)
        k += n
    fc.synchronize()
    assert fc.info("graph_launches") == 2 and fc.info("diagnostics_history_steps") == k
    for key in g_out:
        assert same_bits(fc.diagnostics_history(*key), np.array(ref[key])), key
    close(fc, wrapped)


def test_history_off_changes_nothing(fcmod):
    """by default there is no history; with it on, every output array, the final fc_get_diagnostics, the graph replays
    and the launches are those of the run without it -- plus exactly one launch per graph replay (the replay's first
    step number)"""
    sc = scenario(2, True)
    res = {}
    for H in (0, 400):
        fc, wrapped, g_in, g_out = context(fcmod, sc, 2, history=H)
        if not H:
            assert fc.info("diagnostics_history_steps") == 0
            with pytest.raises(fcmod.FluxCalcError) as e:
                fc.diagnostics_history(1, 1, "MEVA", first=0, count=0)
            assert e.value.code == FC_ERR_STATE
        l0 = fc.info("launches")
        run_calls(fc, wrapped, g_in, False)
        for k, a in g_out.items():
            wrapped[id(a)].download(a)
        res[H] = (g_out, {k: fc.diagnostics(*k) for k in g_out}, fc.info("launches") - l0, fc.info("graph_launches"))
        close(fc, wrapped)
    (out0, d0, l0, g0), (out1, d1, l1, g1) = res[0], res[400]
    for k in out0:
        assert same_bits(out0[k], out1[k]), k
        assert same_bits(d0[k], d1[k]), k
    assert g0 == g1 == GRAPHS
    assert l1 == l0 + GRAPHS


def test_history_restarts_at_a_reset(fcmod):
    """a new plan (set_method + prepare) and setting the option again both restart the numbering at 0 and drop the
    older steps"""
    sc = scenario(1, False)
    fc, wrapped, g_in, g_out = context(fcmod, sc, 2, history=64)
    fc.run_steps(0, DT, 40)
    assert fc.info("diagnostics_history_steps") == 40
    fc.set_method("which_flux_radiation_blackbody", 1, "StBo")
    fc.prepare()
    assert fc.info("diagnostics_history_steps") == 0
    with pytest.raises(fcmod.FluxCalcError) as e:
        fc.diagnostics_history(1, 1, "MEVA", first=0, count=1)
    assert e.value.code == FC_ERR_ARG
    for reset in ("plan", "option"):
        fc.run_steps(86400 * 40, DT, 37)      # February: one graph replay and five direct steps
        assert fc.info("diagnostics_history_steps") == 37
        for k in g_out:
            h = fc.diagnostics_history(*k)
            assert h.shape == (37, 3) and same_bits(h[-1], fc.diagnostics(*k)), k
        if reset == "plan":
            fc.set_option("diagnostics_history", 64)
            assert fc.info("diagnostics_history_steps") == 0
            assert fc.diagnostics_history(1, 1, "MEVA").shape == (0, 3)
    close(fc, wrapped)
