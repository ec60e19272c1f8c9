#!/usr/bin/env python
"""What tracks from frame 0 add to a scene (DESIGN.md 4.9): C2 (854x480, four segments), three pairs per run as bench.py
runs C2, the full 19 x 8 x 400 schedule with all 19 frames, each pair over its own synth.background_motion.  Three arms
alternate in one process so that all see the same card, clocks and neighbours:
  frames:   Batch.submit_scene(..., frames=all 19) per pair, run();
  dense:    the same with tracks=True: flow0, bflow0 and occ0 of every frame copied out;
  queries:  the same with 2048 queries and no dense tracks: only the gathered positions and occlusion copied out.

  python tools/track_cost.py [--reps 5] [--out profiles/track_cost.json]

Every arm ends in host memory after a device synchronise, so a host clock around it is its wall time.  Prints one JSON
line (and writes it to --out): the card's name and power limit (read in the same run) and, per arm, the median, min and
max over the reps of the wall time per pair, and the last run's Batch.timing_ms() and launch count.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arap_flow_b200 import lib, synth  # noqa: E402
from tools.extras_cost import card  # noqa: E402

PAIRS = 3
NCONT, NGN, NPCG = 19, 8, 400
ALL = list(range(NCONT))
N_QUERIES = 2048
ARMS = {"frames": dict(), "dense": dict(tracks=True), "queries": dict(queries=True)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sps = [synth.config("C2", i) for i in range(PAIRS)]
    n = len(sps[0].masks)
    W, H = sps[0].W, sps[0].H
    rng = np.random.default_rng(0)
    queries = np.stack([rng.integers(0, W, N_QUERIES), rng.integers(0, H, N_QUERIES)], -1).astype(np.int32)
    moves = []
    for i, sp in enumerate(sps):
        A, m = synth.background_motion(sp.W, sp.H, 100 + i)
        moves.append((A, synth.background(sp.W + 2 * m, sp.H + 2 * m, 100 + i), m))
    b = lib.Batch(W, H, PAIRS * n, NCONT, NGN, NPCG)
    outs = {k: [None] * PAIRS for k in ARMS}

    def run(arm):
        kw = ARMS[arm]
        for i, (sp, (A, bg, m)) in enumerate(zip(sps, moves)):
            outs[arm][i] = b.submit_scene(i * n, sp.rgb, sp.masks, [sp.matches] * n, bg, A, origin=(m, m), frames=ALL,
                                          frame_motions=synth.motion_path(A, ALL, NCONT), out=outs[arm][i],
                                          tracks=kw.get("tracks", False),
                                          queries=queries if kw.get("queries") else None)
        b.run()

    res = dict(card=card(), workload=f"C2 x{PAIRS} pairs per run, {NCONT}x{NGN}x{NPCG}, all {NCONT} frames",
               reps=a.reps, unit="ms per pair (host wall clock)",
               arms=dict(frames="no tracks", dense="tracks=True (flow0, bflow0, occ0 copied out)",
                         queries=f"{N_QUERIES} queries, no dense tracks copied out"))
    for arm in ARMS:   # warm-up: module load, every buffer of every arm
        run(arm)
    rec = {k: [] for k in ARMS}
    dev = {}
    for _ in range(a.reps):
        for arm in ARMS:
            t0 = time.perf_counter()
            run(arm)
            rec[arm].append((time.perf_counter() - t0) * 1e3 / PAIRS)
            dev[arm] = dict(timing_ms={t: round(v, 3) for t, v in b.timing_ms().items()}, launches=b.launches())
    for arm, v in rec.items():
        res[arm] = dict(median=round(statistics.median(v), 2), min=round(min(v), 2), max=round(max(v), 2), **dev[arm])
    b.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
