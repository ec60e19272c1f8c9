#!/usr/bin/env python
"""What the opt-in backward flow and occlusion outputs cost (DESIGN.md 4.3): C1 (854x480), batch 8 = two cooperative
launches of four, the full 19 x 8 x 400 schedule, with and without extras, alternating in one process so that both arms
see the same card, clocks and neighbours.

  python tools/extras_cost.py [--reps 5]

Prints one JSON line: the card's name and power limit (read in the same run), and per arm the median of the reps of
Batch.timing_ms() (device ms: total, solve, warp -- the warp span includes the extra kernels) and pairs/s from a host
clock around submit + run (the run ends in a device synchronise).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arap_flow_b200 import lib, synth  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, limit = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return dict(name=name, power_limit=limit)
    except Exception as e:  # the numbers are still reported, flagged as unattributed
        return dict(name="unknown", power_limit="unknown", error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    a = ap.parse_args()
    sps = [synth.config("C1", i) for i in range(a.batch)]
    b = lib.Batch(854, 480, a.batch)
    outs = {False: [None] * a.batch, True: [None] * a.batch}

    def step(extras):
        t0 = time.perf_counter()
        for i, s in enumerate(sps):
            outs[extras][i] = b.submit(i, s.rgb, s.masks[0], s.matches, out=outs[extras][i], extras=extras)
        b.run()
        dt = time.perf_counter() - t0
        return dict(b.timing_ms(), pairs_per_s=a.batch / dt, launches=b.launches())

    step(False), step(True)                      # warm-up: module load, buffers, the extras' lazy allocation
    rec = {False: [], True: []}
    for _ in range(a.reps):
        for extras in (False, True):
            rec[extras].append(step(extras))
    res = dict(card=card(), workload="C1", batch=a.batch, schedule="19x8x400", reps=a.reps)
    for extras, name in ((False, "plain"), (True, "extras")):
        res[name] = {k: round(statistics.median(r[k] for r in rec[extras]), 4) for k in rec[extras][0]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
