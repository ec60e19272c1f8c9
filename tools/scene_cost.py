#!/usr/bin/env python
"""What a scene saves over the host path it replaces (DESIGN.md 4.6): C2 (854x480, four segments), three pairs per run as
bench.py runs C2, the full 19 x 8 x 400 schedule, each pair over its own synth.background_motion, with no frames, 4
frames (steps 4, 9, 13, 18) and all 19.  Two arms alternate in one process so that both see the same card, clocks and
neighbours:
  host:  Batch.submit(..., extras=True, frames=...) per segment, run(), then per pair lib.composite, lib.composite_seq
         with frames, and frame 0 in numpy;
  scene: Batch.submit_scene(..., input_frame=True) per pair, run().
Both produce the same composited pair, frames and frame 0 (tests/test_gpu_scene.py).

  python tools/scene_cost.py [--reps 5]

Every arm ends in host memory after a device synchronise, so a host clock around it is its wall time.  Prints one JSON
line: the card's name and power limit (read in the same run) and, per frame count and arm, the median, min and max over
the reps of the wall time per pair, and the last run's Batch.timing_ms() and launch count.
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
FRAMES = {"none": None, "4": [4, 9, 13, 18], "19": list(range(NCONT))}


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
    host_out = [None] * (PAIRS * n)
    scene_out = [None] * PAIRS

    def host(steps):
        for i, sp in enumerate(sps):
            for s in range(n):
                host_out[i * n + s] = b.submit(i * n + s, sp.rgb, sp.masks[s], sp.matches, extras=True, frames=steps,
                                               out=host_out[i * n + s])
        b.run()
        for i, (sp, (A, bg, m)) in enumerate(zip(sps, moves)):
            outs = host_out[i * n:(i + 1) * n]
            lib.composite([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs], sp.masks,
                          [o["bflow"] for o in outs], bg, A, origin=(m, m))
            if steps:
                lib.composite_seq([o["seq"] for o in outs], sp.masks, bg, synth.motion_path(A, steps, NCONT),
                                  origin=(m, m))
            obj = np.any([k == 0 for k in sp.masks], axis=0)
            np.where(obj[..., None], sp.rgb, bg[m:m + sp.H, m:m + sp.W])

    def scene(steps):
        for i, (sp, (A, bg, m)) in enumerate(zip(sps, moves)):
            scene_out[i] = b.submit_scene(i * n, sp.rgb, sp.masks, [sp.matches] * n, bg, A, origin=(m, m), frames=steps,
                                          frame_motions=synth.motion_path(A, steps, NCONT) if steps else None,
                                          input_frame=True, out=scene_out[i])
        b.run()

    res = dict(card=card(), workload=f"C2 x{PAIRS} pairs per run, {NCONT}x{NGN}x{NPCG}", reps=a.reps,
               unit="ms per pair (host wall clock)")
    arms = {"host": host, "scene": scene}
    for name, steps in FRAMES.items():
        for f in arms.values():   # warm-up: module load, every buffer at this frame count
            f(steps)
        rec = {k: [] for k in arms}
        dev = {}
        for _ in range(a.reps):
            for k, f in arms.items():
                t0 = time.perf_counter()
                f(steps)
                rec[k].append((time.perf_counter() - t0) * 1e3 / PAIRS)
                dev[k] = dict(timing_ms={t: round(v, 3) for t, v in b.timing_ms().items()}, launches=b.launches())
        res[f"frames_{name}"] = {k: dict(median=round(statistics.median(v), 2), min=round(min(v), 2),
                                         max=round(max(v), 2), **dev[k]) for k, v in rec.items()}
    b.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
