"""bench.py on a box without a GPU: the reference arm (the CPU oracle, rank 0 only) prints the contract's JSON line, the
product arm refuses to run -- there is no CPU fallback to time."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True, timeout=300, env=e)


def tree_files():
    return sorted(os.path.join(dp, fn) for dp, dns, fns in os.walk(ROOT) for fn in fns
                  if "__pycache__" not in dp and ".pytest_cache" not in dp)


def test_reference_arm_line():
    before = tree_files()
    r = run_bench("--impl", "reference", "--workload", "C1", "--steps", "3", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    assert tree_files() == before      # the host-specific oracle builds go to a temporary directory
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1      # ONE JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "cell-updates/s" and d["higher_is_better"] is True
    assert d["steps"] == 3 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and abs(d["value"] - 20000 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "20000 cells" in cb["sample"]
    assert set(cb["variants"]) == {"fast_build_1_rank", "parity_build_all_ranks", "parity_build_1_rank"}
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        assert d["metric"] == json.load(f)["metric"]


def test_reference_arm_other_ranks_do_nothing():
    r = run_bench("--impl", "reference", "--workload", "C1", "--steps", "1", "--gpus", "2", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_refuses_without_a_gpu(fcmod):
    if fcmod.lib.fc_device_count() >= 1:
        import pytest
        pytest.skip("a GPU is visible")
    r = run_bench("--workload", "C2", "--steps", "1", "--no-e2e", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not any(l.startswith("{") for l in r.stdout.splitlines())      # and no number is printed


def test_steps_below_one_are_refused():
    r = run_bench("--impl", "reference", "--workload", "C1", "--steps", "0")
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


class _Shard:
    """stands in for a DeviceArray: what one rank's output field holds"""
    def __init__(self, a):
        self.a, self.n = a, a.size

    def download(self):
        return self.a.copy()


class _Gather:
    """stands in for torch.distributed.gather_object: keeps what this rank sends; on rank 0, the other ranks' parts follow"""
    def __init__(self, others=()):
        self.others, self.sent = list(others), None

    def gather_object(self, obj, out, dst=0):
        self.sent = obj
        if out is not None:
            out[:] = [obj] + self.others


def test_dump_outputs_sample_and_shards(tmp_path, monkeypatch):
    import numpy as np
    import bench
    keys = [(1, 1, "HSEN"), (1, 2, "UMOM"), (0, 1, "MEVA")]
    full = {k: np.arange(3000, dtype=np.float64) + 10000 * j for j, k in enumerate(keys)}     # field j holds 10000 j + cell
    name = lambda d, k: tmp_path / d / ("type%d_grid%d_%s.npy" % k)      # noqa: E731
    # grids within the budget are written whole, with the diagnostics sums in sorted field order
    bench.dump_outputs(str(tmp_path / "whole"), {k: _Shard(a) for k, a in full.items()}, 3000, 0, [3.0, 1.0, 2.0], None, 0, 1)
    for k, a in full.items():
        got = np.load(name("whole", k))
        assert got.dtype == np.float64 and np.array_equal(got, a)
    assert np.array_equal(np.load(tmp_path / "whole" / "diagnostics_sum.npy"), [3.0, 1.0, 2.0])
    # larger grids: the same seeded sample of cells in every field, within the budget, and the same from two ranks as from one
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 8 * 500)
    bench.dump_outputs(str(tmp_path / "one"), {k: _Shard(a) for k, a in full.items()}, 3000, 0, None, None, 0, 1)
    g1 = _Gather()
    bench.dump_outputs(str(tmp_path / "rank1"), {k: _Shard(a[1536:]) for k, a in full.items()}, 3000, 1536, None, g1, 1, 2)
    assert not (tmp_path / "rank1").exists()
    bench.dump_outputs(str(tmp_path / "two"), {k: _Shard(a[:1536]) for k, a in full.items()}, 3000, 0, None, _Gather([g1.sent]), 0, 2)
    assert not (tmp_path / "one" / "diagnostics_sum.npy").exists()
    cells = np.load(name("one", keys[0]))
    assert cells.size == 500 and np.all(np.diff(cells) > 0)
    total = 0
    for j, k in enumerate(keys):
        one = np.load(name("one", k))
        assert np.array_equal(one, cells + 10000 * j) and np.array_equal(np.load(name("two", k)), one)
        total += one.nbytes
    assert total <= 3 * 8 * 500


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(fcmod, tmp_path):
    """--dump-outputs: two runs with the same arguments write the same fields, and they are the oracle's outputs of the
    last timed step (the profiling loop that follows the timed region must not have overwritten them)"""
    import numpy as np
    from bench import build_scenario
    from oracle_py import Oracle
    from tolerances import check_scenario
    if fcmod.lib.fc_device_count() < 1:
        pytest.skip("no GPU")
    args = ("--cells", "20000", "--steps", "5", "--warmup", "3", "--no-e2e", "--no-cpu-baseline", "--no-parity")
    for run in ("a", "b"):
        r = run_bench(*args, "--dump-outputs", str(tmp_path / run))
        assert r.returncode == 0, r.stderr[-2000:]
    sc = build_scenario("C4", cells=20000)
    o_in, o_out = sc.clone()
    orc = Oracle(sc.n, sc.S)
    sc.apply(orc, o_in, o_out)
    orc.step_all(600 * (3 + 5 - 1))
    sc.inputs = o_in
    got = {}
    for k in o_out:
        a = np.load(tmp_path / "a" / ("type%d_grid%d_%s.npy" % k))
        assert a.dtype == np.float64 and np.array_equal(a, np.load(tmp_path / "b" / ("type%d_grid%d_%s.npy" % k)))
        got[k] = a
    check_scenario(sc, got, o_out)
    sums = np.load(tmp_path / "a" / "diagnostics_sum.npy")
    assert sums.dtype == np.float64 and sums.size == len(o_out)
    for s, k in zip(sums, sorted(o_out)):
        ax = sc.area[k[1]] * got[k]
        assert abs(s - np.sum(ax)) <= 1e-11 * np.sum(np.abs(ax)), k     # the bound bench.py checks its diagnostics against
