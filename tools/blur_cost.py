#!/usr/bin/env python
"""What motion blur adds to a scene (DESIGN.md 4.8): C2 (854x480, four segments), three pairs per run as bench.py runs
C2, the full 19 x 8 x 400 schedule, each pair over its own synth.background_motion.  Three arms alternate in one process
so that all see the same card, clocks and neighbours:
  sharp:      Batch.submit_scene(...) per pair, run();
  blur:       the same with blur=(8, 0.5): the blurred pair;
  blur_all:   blur=(8, 0.5) with all 19 frames and input_frame=True: the blurred pair, frame 0 and 19 frames.

  python tools/blur_cost.py [--reps 5]

Every arm ends in host memory after a device synchronise, so a host clock around it is its wall time.  Prints one JSON
line: the card's name and power limit (read in the same run) and, per arm, the median, min and max over the reps of the
wall time per pair, and the last run's Batch.timing_ms() and launch count.
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

PAIRS = 3
NCONT, NGN, NPCG = 19, 8, 400
ALL = list(range(NCONT))
ARMS = {"sharp": dict(), "blur": dict(blur=(8, 0.5)),
        "blur_all": dict(blur=(8, 0.5), frames=ALL, input_frame=True)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    sps = [synth.config("C2", i) for i in range(PAIRS)]
    n = len(sps[0].masks)
    moves = []
    for i, sp in enumerate(sps):
        A, m = synth.background_motion(sp.W, sp.H, 100 + i)
        moves.append((A, synth.background(sp.W + 2 * m, sp.H + 2 * m, 100 + i), m))
    b = lib.Batch(sps[0].W, sps[0].H, PAIRS * n, NCONT, NGN, NPCG)
    outs = {k: [None] * PAIRS for k in ARMS}

    def run(arm):
        kw = ARMS[arm]
        frames = kw.get("frames")
        for i, (sp, (A, bg, m)) in enumerate(zip(sps, moves)):
            outs[arm][i] = b.submit_scene(i * n, sp.rgb, sp.masks, [sp.matches] * n, bg, A, origin=(m, m),
                                          frames=frames,
                                          frame_motions=synth.motion_path(A, frames, NCONT) if frames else None,
                                          input_frame=kw.get("input_frame", False), blur=kw.get("blur"),
                                          out=outs[arm][i])
        b.run()

    res = dict(card=card(), workload=f"C2 x{PAIRS} pairs per run, {NCONT}x{NGN}x{NPCG}", reps=a.reps,
               unit="ms per pair (host wall clock)", arms={k: str(v.get("blur")) + (" all frames + frame 0" if
                                                                                  "frames" in v else "")
                                                           for k, v in ARMS.items()})
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
    print(json.dumps(res))


if __name__ == "__main__":
    main()
