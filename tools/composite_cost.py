#!/usr/bin/env python
"""What the composite over a moving background costs next to the flatten (DESIGN.md 4.5): flatten_ex with a background,
composite with both motions the identity, and composite with a random affine, alternating in one process so that the
three arms see the same card, clocks and neighbours.  Layers: C1 (1 layer) and C2 (4 layers), solved once by the batch
with extras on a reduced schedule (the composite's cost does not depend on how converged its inputs are).

  python tools/composite_cost.py [--reps 7] [--calls 20]

Every call is host buffers in, host buffers out and ends in a device-to-host copy, so a host clock around it is the
call's wall time.  Prints one JSON line: the card's name and power limit (read in the same run) and, per config and arm,
the median, min and max over the reps of the mean wall time per call.
"""
import argparse
import json
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arap_flow_b200 import lib, synth  # noqa: E402
from tools.extras_cost import card  # noqa: E402


def layers(name):
    sp = synth.config(name)
    n = len(sp.masks)
    b = lib.Batch(sp.W, sp.H, n, nCont=2, nGN=2, nPCG=30)
    outs = [b.submit(s, sp.rgb, sp.masks[s], sp.matches, extras=True) for s in range(n)]
    b.run()
    b.close()
    return sp, ([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs], list(sp.masks),
                [o["bflow"] for o in outs])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    a = ap.parse_args()
    res = dict(card=card(), reps=a.reps, calls_per_rep=a.calls, unit="ms per call")
    for name in ("C1", "C2"):
        sp, args = layers(name)
        A, m = synth.background_motion(sp.W, sp.H, 0)
        bg_big = synth.background(sp.W + 2 * m, sp.H + 2 * m, 0)
        bg = bg_big[m:m + sp.H, m:m + sp.W].copy()
        I2 = [[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]
        arms = {
            "flatten_ex": lambda: lib.flatten_ex(*args, background=bg),
            "composite_identity": lambda: lib.composite(*args, bg, I2),
            "composite_affine": lambda: lib.composite(*args, bg_big, A, origin=(m, m)),
        }
        for f in arms.values():   # warm-up: module load, the workspace at its largest size
            f()
        rec = {k: [] for k in arms}
        for _ in range(a.reps):
            for k, f in arms.items():
                t0 = time.perf_counter()
                for _ in range(a.calls):
                    f()
                rec[k].append((time.perf_counter() - t0) * 1e3 / a.calls)
        res[name] = {k: dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3))
                     for k, v in rec.items()}
        res[name]["layers"] = len(args[0])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
