#!/usr/bin/env python3
"""bench.py -- flux cell-updates/s of the fused per-cell flux chain (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C2|C3|C5] [--impl reference] [--dump-outputs DIR]

A "step" is one coupling step (early + normal phase fused: fc_step_all) over the synthetic exchange grid.
Default workload C4 = BASELINE.json configs[3], the configuration the metric's roofline target is quoted on:
10^7 cells per grid (t,u,v), CCLM formula set, all fluxes fused, monthly evaporation bias, area-weighted
diagnostics; for N>1 the grid is sharded into contiguous ranges (strong scaling: the 10^7 cells are fixed) and
the diagnostics are reduced with NCCL.  One JSON line on stdout (rank 0).

`value`  : device-resident throughput, CUDA events on the launching stream, max over ranks.
`e2e`    : same metric through the C ABI with HOST (pinned) arrays: H2D + kernel + D2H inside the timed region.
`roofline`: fused kernel only (event pairs around launches of the same loop continued after the timed region, and the
timed region's own time per step = per launch) vs measured HBM peak.
`cpu_baseline` / --impl reference: the CPU oracle arranged like the reference (one pass per quantity, one
scalar call per cell), P independent ranks = all host threads, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (formula_set, cells per grid, S, bias, averaging, diagnostics, description)
    "C1": ("CCLM", 20_000, 1, False, False, False, "Baltic stand-in 20k cells/grid, CCLM set, single instance (BASELINE configs[0]: the reference's own CPU-runnable case; use --impl reference)"),
    "C2": ("MOM5", 20_000, 1, True, False, False, "Baltic stand-in 20k cells/grid, MOM5 coefficients + monthly evaporation bias"),
    "C3": ("RCO", 1_000_000, 1, False, False, False, "RCO (Meier 1999) formula set, 1e6 cells/grid"),
    "C4": ("CCLM", 10_000_000, 1, True, False, True, "1e7 cells/grid, CCLM set, all fluxes fused + bias + diagnostics (NCCL all-reduce for N>1)"),
    "C5": ("CCLM", 10_000_000, 2, True, True, False, "1e7 cells/grid, CCLM set, open water + ice (S=2) with area-fraction averaging, 1000 consecutive steps device resident (fc_run_steps)"),
    # not a BASELINE.json configuration: the generic fused kernel (more than two surface types)
    "S3": ("CCLM", 10_000_000, 3, True, True, False, "1e7 cells/grid, CCLM set, three surface types with area-fraction averaging: the generic fused kernel"),
}
METRIC = "flux cell-updates/s per coupling step; achieved HBM GB/s vs B200 peak"
UNIT = "cell-updates/s"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every ~10 ms from a
    thread (the timed region of the default run lasts tens of milliseconds, too short for `nvidia-smi -lms`);
    falls back to one `nvidia-smi` query per poll when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.thr, self.stop_flag, self.h, self.nv = index, [], None, False, None, None
        self.period = 0.01      # NVML queries disturb the GPU slightly: keep them sparse
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _poll_nvml(self):
        nv = self.nv
        sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
            pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        except Exception:
            pw = float("nan")
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = []
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                names.append(name)
        return sm, self.max_sm, pw, names

    def _poll_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip().split(",")
        r = [x.strip() for x in out]
        names = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7])
                 if v.lower().startswith("active")]
        return float(r[0]), float(r[1]), float(r[2]), names

    def start(self):
        def pump():
            while not self.stop_flag:
                try:
                    self.rows.append(self._poll_nvml() if self.nv else self._poll_smi())
                except Exception:
                    pass
                time.sleep(self.period)
        self.thr = threading.Thread(target=pump, daemon=True)
        self.thr.start()

    def stop(self):
        self.stop_flag = True
        if self.thr:
            self.thr.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples (NVML and nvidia-smi unavailable)"]}
        sm = [r[0] for r in self.rows]
        reasons = sorted({n for r in self.rows for n in r[3]})
        pw = [r[2] for r in self.rows if r[2] == r[2]]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(r[1] for r in self.rows),
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons,
                "how": "NVML polled every ~10 ms during the timed region" if self.nv else "nvidia-smi polled during the timed region"}


SENT = [(1, "MEVA"), (1, "HLAT"), (1, "HSEN"), (1, "RBBR"), (1, "RSDR"), (2, "UMOM"), (3, "VMOM")]      # (grid, flux): what goes to oasis_put


def build_scenario(workload, offset_size=None, cells=None):
    """the workload's fields + the send list of the reference's configuration: the seven fluxes, per surface type (and their
    area-fraction averages on surface type 0 when there are two types); QSUR is an intermediate, never sent"""
    from synthetic import Scenario
    fset, n, S, bias, avg, diag, _ = WORKLOADS[workload]
    if cells is not None:
        n = cells
    off, size = offset_size if offset_size else (0, n)
    sc = Scenario(fset, n=(size, size, size), S=S, bias=bias, averaging=avg, offset=(off, off, off))
    for i in range(1, S + 1):
        for g, name in SENT:
            if (i, g, name) in sc.outputs and (i, g, name) not in sc.send:
                sc.send.append((i, g, name))
    return sc


DUMP_BYTES = 48 << 20      # --dump-outputs: all files together stay below 64 MB
DUMP_SEED = 20240601


def dump_outputs(out_dir, fields, n_total, off, diag_sums, dist, rank, world):
    """what the timed path computed in its last step, written by rank 0: every output field as type<i>_grid<g>_<name>.npy
    (float64, in global cell order) and, with diagnostics, their area-weighted sums in the same (sorted) field order as
    diagnostics_sum.npy.  When the whole grids would exceed DUMP_BYTES, every field holds the same fixed, seeded sample of
    global cells, so two builds run with the same arguments can be compared value for value."""
    keys = sorted(fields)
    m = min(n_total, DUMP_BYTES // (8 * len(keys)))
    cells = np.arange(n_total) if m == n_total else np.sort(np.random.default_rng(DUMP_SEED).choice(n_total, m, replace=False))
    mine = cells[(cells >= off) & (cells < off + fields[keys[0]].n)] - off
    local = {k: fields[k].download()[mine] for k in keys}
    parts = [local]
    if dist:
        parts = [None] * world if rank == 0 else None
        dist.gather_object(local, parts, dst=0)      # the shards are contiguous ranges in rank order
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k in keys:
            np.save(os.path.join(out_dir, "type%d_grid%d_%s.npy" % k), np.concatenate([p[k] for p in parts]))
        if diag_sums is not None:
            np.save(os.path.join(out_dir, "diagnostics_sum.npy"), np.asarray(diag_sums, dtype=np.float64))


_native_dir = None      # the host-specific oracle builds: a temporary directory, the tree may be read-only


def native_oracle(build="fast"):
    """the oracle built for THIS host: 'fast' = -O3 -march=native -ffast-math (the reference's release flags, -O3 -fp-model fast=2
    -xHost, build_hlrng.sh:26), 'parity' = -O2 -ffp-contract=off (its debug / -fp-model precise build, :23); falls back to
    the shipped builds"""
    global _native_dir
    import ctypes as C
    from oracle_py import ORACLE_DIR
    flags = {"fast": ["-O3", "-march=native", "-ffast-math"], "parity": ["-O2", "-march=native", "-ffp-contract=off"]}[build]
    try:
        if _native_dir is None:
            _native_dir = tempfile.TemporaryDirectory(prefix="fluxcalc_oracle_")
        so = os.path.join(_native_dir.name, "liboracle_%s.so" % build)
        subprocess.check_call(["gcc", "-std=c11"] + flags + ["-fPIC", "-shared", "-o", so,
                               os.path.join(ORACLE_DIR, "flux_oracle.c"), os.path.join(ORACLE_DIR, "cpu_baseline.c"),
                               "-lm", "-lpthread"], stderr=subprocess.DEVNULL)
        C.CDLL(so)
        return so, " ".join(flags)
    except Exception:
        return (os.path.join(ORACLE_DIR, "liboracle_fast.so" if build == "fast" else "liboracle.so"),
                "-O3 -march=x86-64-v3 -ffast-math" if build == "fast" else "-O2 -ffp-contract=off")


def cpu_arm(workload, steps, warmup, sample_cells=None, variants=True):
    """the reference's CPU path: the oracle port in the reference's loop structure (one pass per quantity and surface
    type, one scalar call per cell, corrections at stride 12), P ranks each owning a contiguous range (threads standing in
    for the MPI-parallel flux_calculator instances), on the workload's FULL grid.  Headline: release-like build on all
    host threads; beside it the parity build (what the golden files pin) and one rank."""
    import oracle_py
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    fset, n, S, bias, avg, diag, _ = WORKLOADS[workload]
    cells = min(n, sample_cells) if sample_cells else n
    sc = build_scenario(workload, cells=cells)

    def timed(build, P, nsteps, nwarm):
        so, flags = native_oracle(build)
        ins, outs = sc.clone()
        orc = oracle_py.Oracle(sc.n, sc.S, fast=(build == "fast"), lib_path=so)
        sc.apply(orc, ins, outs)
        for _ in range(nwarm):
            orc.run_ranks(P, 1, 600, 0)
        times = []
        for k in range(nsteps):
            t0 = time.perf_counter()
            orc.run_ranks(P, 1, 600, 600 * k)
            times.append(time.perf_counter() - t0)
        t = float(np.mean(times))
        return {"value": cells / t, "ms_per_step": t * 1e3, "ranks": P, "steps": nsteps, "build": "gcc " + flags}

    head = timed("fast", ncores, max(steps, 1), max(1, min(warmup, 3)))
    res = {"value": head["value"], "unit": UNIT, "cores": ncores, "kind": "port",
           "sample": "%d cells/grid (%s) x %d steps of workload %s, %d ranks (threads) each owning a contiguous range, %s"
                     % (cells, "the full grid" if cells == n else "a sample", head["steps"], workload, ncores, head["build"]),
           "ms_per_step": head["ms_per_step"]}
    if variants:
        one = max(1, min(3, steps))
        res["variants"] = {"fast_build_1_rank": timed("fast", 1, one, 1), "parity_build_all_ranks": timed("parity", ncores, max(3, min(steps, 10)), 1),
                           "parity_build_1_rank": timed("parity", 1, one, 1)}
    return res


def run_reference(args, rank):
    if rank != 0:
        return 0
    wl = args.workload
    res = cpu_arm(wl, args.steps, args.warmup, args.cpu_sample_cells)
    fset, n, S, bias, avg, diag, desc = WORKLOADS[wl]
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: %s" % (wl, desc), "cells_per_grid": n, "formula_set": fset, "surface_types": S,
                   "note": "reference cannot be compiled here (Fortran+MPI+netCDF+OASIS, no Fortran compiler): CPU arm is the oracle port in the reference's loop structure"},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "variants") if k in res},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 1000 for C5, BASELINE.json configs[4])")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--cells", type=int, default=None, help="override cells per grid (debug)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample-cells", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--diag", type=int, default=None, help="override the workload's diagnostics switch (0/1)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--prefetch", type=int, default=None, help="L2 prefetch distance in blocks (tuning)")
    ap.add_argument("--staged", type=int, default=None, help="0/1: forbid/allow the staged kernel (tuning)")
    ap.add_argument("--opt", action="append", default=[], help="name=value passed to fc_set_option (tuning)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE.json configs[3]: the 10^7-cell grid is fixed and sharded over the GPUs) or weak "
                         "(every GPU gets the workload's full cell count)")
    ap.add_argument("--profile-stride", type=int, default=4,
                    help="bracket every n-th fused launch of the profiling loop with an event pair for the roofline's kernel time (an "
                         "event between two launches switches their programmatic overlap off, so not every launch is bracketed)")
    ap.add_argument("--profile-steps", type=int, default=64, help="steps of the profiling loop that follows the timed region")
    ap.add_argument("--preheat-ms", type=float, default=0.0,
                    help="run untimed steps for this long BEFORE the W warm-up steps (tuning aid: separates clock / TLB ramp-up from the "
                         "step time when W and K are small; reported in config.preheat_ms)")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="N>1 diagnostics exchange: peer mailboxes written by the step's kernel over NVLink (default; falls back "
                         "to NCCL when CUDA IPC is unavailable) or ncclAllReduce on a side stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64; a fixed, seeded sample of the cells "
                         "when the whole grids would exceed 48 MiB) to compare two builds")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 1000 if (args.workload == "C5" and args.impl == "b200") else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    dist = None
    if world > 1:
        import torch.distributed as dist   # control plane only (barrier, max over ranks, unique-id broadcast)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="gloo", rank=rank, world_size=world)

    import components.flux_calculator_b200 as m
    from components.flux_calculator_b200 import DeviceArray, pinned_empty

    if m.lib.fc_device_count() < 1:
        raise SystemExit("bench.py: no sm_100 device visible; the flux calculator has no CPU fallback")
    device = local_rank
    # host buffers of this rank next to its GPU (pinned allocations below are first touched by this thread)
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_bound = m.lib.fc_bind_thread_to_device_numa(device) == 0
    fset, n_total, S, bias, avg, diag, desc = WORKLOADS[args.workload]
    if args.cells:
        n_total = args.cells
    if args.scaling == "weak":
        n_total *= world
    if args.diag is not None:
        diag = bool(args.diag)
    off, size = m.shard_range(n_total, rank, world, 512)
    sc = build_scenario(args.workload, (off, size), cells=n_total)

    # ---------------- device-resident context (value, roofline) ----------------
    g_in, g_out = sc.clone()
    fc = m.FluxCalculator(sc.n, sc.S, device=device)
    wrapped = sc.apply(fc, g_in, g_out, wrap=lambda a: DeviceArray.from_numpy(a, device))
    if diag:
        for g in (1, 2, 3):
            fc.set_area(g, sc.area[g])
        fc.set_option("diagnostics", 1)
    if args.prefetch is not None:
        fc.set_option("prefetch_distance", args.prefetch)
    if args.staged is not None:
        fc.set_option("staged", args.staged)
    for kv in args.opt:
        fc.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    fc.prepare()
    assert fc.info("fused") == 1, "bench workload must run on the fused kernel"
    comm_used = None
    if world > 1 and diag:
        import torch
        comm_used = args.comm
        if comm_used == "p2p":
            hs = [None] * world
            dist.all_gather_object(hs, fc.comm_p2p_handle())
            try:
                fc.comm_p2p_connect(hs, rank, world)
                ok = 1
            except Exception as e:      # no IPC / no peer access in this container
                sys.stderr.write("rank %d: peer mailboxes unavailable (%s), falling back to NCCL\n" % (rank, e))
                ok = 0
            t = torch.tensor([ok], dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t[0]) == 0:
                if ok:
                    raise SystemExit("bench.py: peer mailboxes connected on some ranks only")
                comm_used = "nccl"
        if comm_used == "nccl":
            os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout (one JSON line only)
            uid = [m.comm_get_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            fc.comm_init(uid[0], rank, world)

    # C5 (BASELINE.json configs[4]): "batched consecutive coupling steps, device resident" = ONE fc_run_steps call for the
    # whole timed region (CUDA graphs of 32 step launches per calendar month; the bias month advances with timestep = 600 s)
    batched = args.workload == "C5"

    def one_step(k):
        fc.step_all(600 * k)
        if diag and world > 1:
            fc.allreduce_diagnostics()

    def barrier():
        fc.synchronize()
        if dist:
            dist.barrier()

    if args.preheat_ms > 0:
        t_end = time.perf_counter() + args.preheat_ms * 1e-3
        while time.perf_counter() < t_end:
            for k in range(16):
                one_step(0)
            fc.synchronize()
    for k in range(args.warmup):
        one_step(k)
    barrier()
    launches0 = fc.info("launches")
    fc.set_option("profile_kernel", 0)      # nothing but the K steps between the two events of the timed region (see below)
    sampler = ClockSampler(device)
    if os.environ.get("FC_BENCH_NO_SAMPLER") != "1":      # tuning aid: rule out the NVML polling as a perturbation
        sampler.start()
    barrier()
    if batched:
        fc.run_steps(600 * args.warmup, 600, 64)      # graphs captured and instantiated before the clock starts
        barrier()
        launches0 = fc.info("launches")
    fc.event_record(0)
    if batched:
        fc.run_steps(600 * (args.warmup + 64), 600, args.steps)
        if diag and world > 1:
            fc.allreduce_diagnostics()
    else:
        for k in range(args.steps):
            one_step(args.warmup + k)
    fc.event_record(1)
    ms_total = fc.event_elapsed_ms()
    barrier()
    clocks = sampler.stop()
    graph_launches = fc.info("graph_launches")
    launches = fc.info("launches") - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: wrapped[id(a)] for k, a in g_out.items()}, n_total, off,
                     [fc.diagnostics(*k)[0] for k in sorted(g_out)] if diag else None, dist, rank, world)
    # kernel time for the roofline: the SAME step loop continued right after the timed region, every n-th launch between an
    # event pair.  Not inside the timed region: an event between two launches switches their programmatic overlap, the early
    # ring fill and the per-CTA hand-over off, which costs 7-18 us per bracketed launch on an 8-GPU shard (call 14: three
    # bracketed launches in a 20-step run made ms_per_step 2-3 % worse) -- `value` must not carry the profiler's footprint.
    k0 = args.warmup + args.steps + (64 if batched else 0)
    last_t = 600 * (k0 - 1)
    fc.set_option("profile_kernel", args.profile_stride)
    for k in range(args.profile_steps):
        last_t = 600 * (k0 + k)
        fc.step_all(last_t)
        if diag and world > 1:
            fc.allreduce_diagnostics()
    fc.synchronize()
    kern_ms, kern_cnt = fc.kernel_time_ms()
    fc.set_option("profile_kernel", 0)
    exact_calls = fc.info("exact_path_calls")
    if os.environ.get("FC_BENCH_PER_RANK") == "1":
        sys.stderr.write("rank %d: %.4f ms/step, bracketed kernel %.4f ms, cells %d\n" % (rank, ms_total / args.steps, kern_ms / max(kern_cnt, 1), size))
    if dist:
        import torch
        t = torch.tensor([ms_total, kern_ms / max(kern_cnt, 1)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, kern_avg_ms = float(t[0]), float(t[1])
        lt = torch.tensor([launches], dtype=torch.int64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])
    else:
        kern_avg_ms = kern_ms / max(kern_cnt, 1)
    ms_per_step = ms_total / args.steps
    value = n_total / (ms_per_step * 1e-3)
    if kern_avg_ms <= 0.0:      # --profile-steps 0
        kern_avg_ms = ms_per_step

    bytes_per_cell = fc.info("bytes_per_cell")
    peak, peak_src = measured_peaks()
    # the slowest rank's kernel processes `size` cells of each grid per launch
    max_size = max(m.shard_range(n_total, r, world, 512)[1] for r in range(world))
    achieved = bytes_per_cell * max_size / (kern_avg_ms * 1e-3) / 1e9
    achieved_step = bytes_per_cell * max_size / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "achieved_from_ms_per_step": achieved_step, "frac_from_ms_per_step": achieved_step / peak,
                "note": "frac: launches bracketed by event pairs in the same step loop continued right after the timed region (an event "
                        "between two launches switches their programmatic overlap off, so the timed region itself carries none); "
                        "frac_from_ms_per_step: the same bytes over the timed region's time per step (one launch per step)",
                "kernel_launches_timed": int(kern_cnt),
                "traffic": None, "kernel": "flux_spec_kernel" if fc.info("spec_kernel") == 1 else "fused_step_kernel",
                "kernel_ms": kern_avg_ms,
                "algorithmic_bytes_per_cell": bytes_per_cell, "cells_per_launch": max_size, "peak_source": peak_src}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tr = json.load(f)
        if tr.get("workload") == args.workload and tr.get("cells_per_launch") == max_size:
            roofline["traffic"] = tr["dram_bytes_per_launch"]
            roofline["traffic_source"] = tr.get("source")
    except Exception:
        pass

    # parity spot check of what was just timed (first 4096 cells of every output vs the oracle)
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle_py import Oracle
        from tolerances import check_scenario, K_ULP
        ns = min(4096, size)
        small = build_scenario(args.workload, (off, ns), cells=n_total)
        o_in, o_out = small.clone()
        orc = Oracle(small.n, small.S)
        small.apply(orc, o_in, o_out)
        orc.step_all(last_t)
        small.inputs = o_in
        got = {k: wrapped[id(g_out[k])].download()[:ns] for k in o_out}
        worst = max(check_scenario(small, got, o_out).values())
        parity = {"checked_fields": len(o_out), "cells": ns, "worst_error_over_tolerance": worst,
                  "tolerance": "bit-exact without a transcendental upstream, else %g ulp of (|ref| + cancelling terms) per cell (tests/tolerances.py)" % K_ULP}

    diag_sample = None
    diag_check = None
    if diag:
        s_, mn_, mx_ = fc.diagnostics(1, 1, "HSEN")
        nn = lambda v: None if v != v else v      # NaN (min/max are only computed at diagnostics level 2) -> null
        diag_sample = {"HSEN_type1": {"sum_area_x": s_, "min": nn(mn_), "max": nn(mx_)}}
        # the (global) diagnostics of the last step against numpy over the outputs of ALL ranks
        local = {}
        for k in sorted(g_out):
            x = wrapped[id(g_out[k])].download()
            a = sc.area[k[1]]
            local[k] = (float(np.sum(a * x)), float(np.sum(np.abs(a * x))))
        parts = [local]
        if dist:
            parts = [None] * world
            dist.all_gather_object(parts, local)
        worst = 0.0
        for k in sorted(local):
            ref = sum(p_[k][0] for p_ in parts)
            mag = sum(p_[k][1] for p_ in parts)
            got = fc.diagnostics(*k)[0]
            dev = abs(got - ref) / mag if mag > 0 else abs(got - ref)
            worst = max(worst, dev)
            if dev > 1e-11:
                raise SystemExit("bench.py: rank %d: global diagnostics of %s differ from numpy over all ranks: %r vs %r" % (rank, k, got, ref))
        diag_check = {"fields": len(local), "ranks": world, "worst_deviation_over_sum_abs": worst, "bound": 1e-11,
                      "what": "sum_j area_j * x_j of every output of the last step: the library's (all-reduced) value against numpy over the outputs gathered from all ranks"}

    # ---------------- end-to-end through the C ABI with host arrays ----------------
    e2e = None
    if not args.no_e2e:
        for w in wrapped.values():
            w.free()
        fc.close()
        h_in, h_out = {}, {}
        memo = {}
        def pin(a):
            if id(a) not in memo:
                p = pinned_empty(a.size)
                p[:] = a
                memo[id(a)] = p
            return memo[id(a)]
        for k, a in g_in.items():
            h_in[k] = pin(a)
        for k, a in g_out.items():
            h_out[k] = pin(a)
        fh = m.FluxCalculator(sc.n, sc.S, device=device)
        sc.apply(fh, h_in, h_out)
        if diag:
            for g in (1, 2, 3):
                fh.set_area(g, sc.area[g])
            fh.set_option("diagnostics", 1)
        # what the reference's own configuration would move: the ice fraction of a surface type is a namelist constant
        # (val_bottom_var_*, flux_calculator.F90:444-449: written once, never received), and only the send list goes back
        # to the coupler (oasis_put) -- QSUR is an intermediate
        for (i, g, name) in h_in:
            if name == "FICE" and i >= 1:
                fh.mark_static(i, g, "FICE")
        fh.set_option("download", 1)
        fh.prepare()
        fh.step_all(0)
        fh.synchronize()
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        for k in range(args.e2e_steps):
            fh.step_all(600 * (k + 1))
            chk = float(h_out[(1, 1, "HSEN")][0])     # the host reads a result of every step
        fh.synchronize()
        dt = time.perf_counter() - t0
        h2d, d2h = fh.info("h2d_bytes_per_step"), fh.info("d2h_bytes_per_step")
        if dist:
            import torch
            t = torch.tensor([dt], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t[0])
            b = torch.tensor([h2d, d2h], dtype=torch.int64)
            dist.all_reduce(b, op=dist.ReduceOp.SUM)
            h2d, d2h = int(b[0]), int(b[1])
        e2e = {"value": n_total * args.e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": dt / args.e2e_steps * 1e3, "steps": args.e2e_steps,
               "how": "fc_step_all on pinned host arrays: chunked H2D -> fused kernel -> D2H over 3 streams, wall clock with sync on both sides, max over ranks; "
                      "every received field travels every step (FICE is a namelist constant: once), the send list comes back",
               "check": chk}
        fh.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if all_cpus:
            os.sched_setaffinity(0, all_cpus)      # the CPU arm gets every core the job has, not just the GPU's socket
        cpu = cpu_arm(args.workload, 10, 2, args.cpu_sample_cells, variants=False)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, desc), "cells_per_grid": n_total, "formula_set": fset,
                       "surface_types": S, "bias": bias, "averaging": avg, "diagnostics": diag,
                       "parallelism": "contiguous range per GPU (fc_shard_range), %d rank(s)" % world,
                       "diagnostics_exchange": {None: "none (1 rank)", "p2p": "peer mailboxes over NVLink, written by the fold of the step's diagnostics rows inside the next step's kernel",
                                                "nccl": "ncclAllReduce on a side stream"}[comm_used],
                       "preheat_ms": args.preheat_ms,
                       "l2": "inputs exceed L2 (%.0f MB per step per GPU vs 126 MB), no flush" % (bytes_per_cell * max_size / 1e6)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "parity": parity, "diagnostics_sample": diag_sample, "diagnostics_check": diag_check, "exact_path_calls": exact_calls,
            "graph_launches": graph_launches, "host_numa_bound": numa_bound,
        }
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
