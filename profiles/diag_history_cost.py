#!/usr/bin/env python3
"""Cost of the per-step diagnostics history (option "diagnostics_history") in device-resident runs.

  python profiles/diag_history_cost.py [--steps 1000] [--reps 5] [--out FILE]

Two shapes through fc_run_steps, diagnostics level 1, 10^7 cells per grid:
  C5: CCLM, open water + ice (S = 2) with area-fraction averaging (the specialised kernel; with the history on, every
      captured step folds its predecessor's diagnostics rows in its producer warps)
  C4: CCLM, one surface type, bias corrections
each with the history off and on (H = steps).  Both arms are contexts over the same device arrays; their timed runs
alternate within one process, every arm is repeated --reps times, and each run is one fc_run_steps call of --steps steps
(600 s apart: one calendar month, graph replays of 32 steps) between CUDA events on the context's stream.  Prints ms per
step (median, min, max over the repetitions) and the card's name, power limit and maximum SM clock read in the same run.
Writes nothing into the tree unless --out names a file.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = "unavailable (%s)" % e
    return "%s: %s" % (q, out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cells", type=int, default=10_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import components.flux_calculator_b200 as m
    from components.flux_calculator_b200 import DeviceArray
    from synthetic import Scenario
    if m.lib.fc_device_count() < 1:
        raise SystemExit("diag_history_cost.py: no sm_100 device visible; the flux calculator has no CPU fallback")

    lines = ["# diagnostics history cost: fc_run_steps of %d steps, diagnostics level 1, %d cells per grid" % (args.steps, args.cells),
             "# " + card()]
    shapes = {"C5": dict(S=2, bias=True, averaging=True), "C4": dict(S=1, bias=True, averaging=False)}
    for name, kw in shapes.items():
        sc = Scenario("CCLM", n=(args.cells,) * 3, **kw)
        g_in, g_out = sc.clone()
        dev, arms = {}, {}

        def wrap(a):      # both arms bind the same device arrays
            if id(a) not in dev:
                dev[id(a)] = DeviceArray.from_numpy(a)
            return dev[id(a)]
        for H in (0, args.steps):
            fc = m.FluxCalculator(sc.n, sc.S)
            sc.apply(fc, g_in, g_out, wrap=wrap)
            for g in (1, 2, 3):
                fc.set_area(g, sc.area[g])
            fc.set_option("diagnostics", 1)
            fc.set_option("diagnostics_history", H)
            fc.prepare()
            assert fc.info("spec_kernel") == 1
            fc.run_steps(0, 600, 64)      # graphs captured, first launches done
            fc.synchronize()
            arms[H] = fc
        ms = {H: [] for H in arms}
        for _ in range(args.reps):
            for H, fc in arms.items():
                fc.synchronize()
                fc.event_record(0)
                fc.run_steps(64 * 600, 600, args.steps)
                fc.event_record(1)
                ms[H].append(fc.event_elapsed_ms() / args.steps)
        # the history of the last run is what fc_get_diagnostics returned after its last step
        on = arms[args.steps]
        assert on.diagnostics_history(1, 1, "MEVA")[-1, 0] == on.diagnostics(1, 1, "MEVA")[0]
        med = {H: float(np.median(v)) for H, v in ms.items()}
        for H, v in ms.items():
            lines.append("%s history %-4s  ms/step median %.4f  min %.4f  max %.4f  (%s)" % (
                name, "off" if H == 0 else "on", med[H], min(v), max(v), " ".join("%.4f" % x for x in v)))
        lines.append("%s on/off (medians): %+.2f %%" % (name, 100.0 * (med[args.steps] / med[0] - 1.0)))
        for fc in arms.values():
            fc.close()
        for d in dev.values():
            d.free()
    lines.append("# " + card())
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
