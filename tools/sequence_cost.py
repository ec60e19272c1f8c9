#!/usr/bin/env python
"""What frame sequences cost (DESIGN.md 4.4): C1 (854x480), batch 8 = two cooperative launches of four, the full
19 x 8 x 400 schedule, in three arms that alternate in one process so that they see the same card, clocks and
neighbours: no frames, 4 evenly spaced frames, all 19.

  python tools/sequence_cost.py [--reps 5]

Prints one JSON line: the card's name and power limit (read in the same run), and per arm the median of the reps of
Batch.timing_ms() (device ms: total, solve, warp -- the solve span holds the per-step launches, the warp span the
frames' kernels), pairs/s from a host clock around submit + run (the run ends in a device synchronise and includes the
frames' copies to host memory), and the launch count.
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

ARMS = {"none": None, "four": [4, 9, 13, 18], "all": list(range(19))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    a = ap.parse_args()
    sps = [synth.config("C1", i) for i in range(a.batch)]
    b = lib.Batch(854, 480, a.batch)
    outs = {arm: [None] * a.batch for arm in ARMS}

    def step(arm):
        t0 = time.perf_counter()
        for i, s in enumerate(sps):
            outs[arm][i] = b.submit(i, s.rgb, s.masks[0], s.matches, out=outs[arm][i], frames=ARMS[arm])
        b.run()
        dt = time.perf_counter() - t0
        return dict(b.timing_ms(), pairs_per_s=a.batch / dt, launches=b.launches())

    for arm in ARMS:                             # warm-up: module load, buffers, the frames' lazy allocation
        step(arm)
    rec = {arm: [] for arm in ARMS}
    for _ in range(a.reps):
        for arm in ARMS:
            rec[arm].append(step(arm))
    res = dict(card=card(), workload="C1", batch=a.batch, schedule="19x8x400", reps=a.reps,
               frames={arm: ARMS[arm] for arm in ARMS})
    for arm in ARMS:
        res[arm] = {k: round(statistics.median(r[k] for r in rec[arm]), 4) for k in rec[arm][0]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
