#!/usr/bin/env python
"""bench.py -- flow pairs/sec @854x480 (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path (19 continuation x 8 Gauss-Newton x 400 PCG iterations + forward
warp) over one batch of synthetic 854x480 pairs (config C1: single segment, fd=1, DeepMatching-like
matches) per GPU.  Pairs are independent: ranks shard them with no collective (para_gen.py --gpu style),
so scaling is weak (per-GPU work fixed).

  python bench.py [--gpus N --steps K --warmup W]            # our arm (libarapb200.so), batched API
  python bench.py --path opt_h [...]                          # our arm through the reference's own Opt.h call sequence
  python bench.py --impl reference [...]                      # the reference arm: CPU oracle port
  python bench.py --dump-outputs DIR [...]                    # also write the last timed step's outputs (rank 0)
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_ITER = 156.0            # algorithmic bytes / active pixel / PCG iteration (SURVEY.md 8d, DESIGN.md 5)
B_GN_EXTRA = 132.0        # init + update + cost per GN step
NCONT, NGN, NPCG = 19, 8, 400
WORKLOADS = {"C1": (854, 480, 1, 1, 1000), "C3": (1024, 436, 1, 5, 3000), "C0": (64, 64, 1, 1, 0),
             "C4": (1920, 1080, 1, 1, 4000), "C2": (854, 480, 4, 3, 2000),
             "C1s": (854, 480, 1, 1, 1000)}   # C1 geometry with a DAVIS-typical small object (8 % of the frame)
AXES = {"C4": (0.46, 0.46),   # SURVEY.md 8d: C4 enlarges the ellipse to 66 % coverage
        "C1s": (0.15, 0.17)}


def make_pairs(workload: str, count: int, first: int):
    from arap_flow_b200 import synth
    W, H, nseg, fd, seed0 = WORKLOADS[workload]
    return [synth.synth(W, H, nseg, fd, seed0 + first + i, axes=AXES.get(workload)) for i in range(count)]


def workload_config(workload: str, pairs):
    """The `config` object: identical for our arm and the reference arm (what is solved, not how)."""
    W, H, nseg, fd, seed0 = WORKLOADS[workload]
    act = [int(sum((m == 0).sum() for m in p.masks)) for p in pairs]
    return {"workload": f"{workload} {W}x{H}, {nseg} segment(s) per pair, fd={fd}, synth seeds {seed0}+",
            "schedule": f"{NCONT}x{NGN}x{NPCG}", "active_px_per_pair": float(np.mean(act)),
            "matches_per_pair": float(np.mean([len(p.matches) for p in pairs])), "warp": "forward warp of RGB + mask per segment"}


DUMP_BYTES = 64_000_000     # --dump-outputs budget: all files together
DUMP_SEED = 0               # seeds the pixel sample taken when the full outputs exceed the budget


def dump_outputs(out_dir: str, outs, flats):
    """Write what the timed path returned in its last step as float32 .npy files, one array per output field with the
    problems stacked on axis 0: flow, rgb, mask (and costs) per problem, plus flat_flow, flat_rgb, flat_mask per pair
    when a pair has several segments.  If the per-pixel arrays exceed DUMP_BYTES, every one of them keeps the same fixed,
    seeded sample of pixels (row-major indices in pixel_index.npy) instead of the full image: the two pixel axes
    [H, W] become one axis [n], e.g. flow.npy [problems, n, 2] and mask.npy [problems, n]."""
    fields = {k: [o[k] for o in outs] for k in ("flow", "rgb", "mask")}
    if flats:
        fields.update({"flat_" + k: [f[i] for f in flats] for i, k in enumerate(("flow", "rgb", "mask"))})
    H, W = outs[0]["mask"].shape
    # float32 bytes of one pixel in every array; 1 MB is left for costs.npy and the .npy headers
    px_bytes = sum(4 * len(v) * v[0][0, 0].size for v in fields.values())
    budget = DUMP_BYTES - 1_000_000
    n = H * W if px_bytes * H * W <= budget else budget // (px_bytes + 8)   # + 8: the float64 pixel_index entry
    idx = None if n == H * W else np.sort(np.random.default_rng(DUMP_SEED).choice(H * W, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in fields.items():
        a = np.stack([np.asarray(x).reshape(H * W, -1) for x in v]).astype(np.float32)
        pixels = (H, W) if idx is None else (n,)
        a = (a if idx is None else a[:, idx]).reshape((len(v),) + pixels + np.shape(v[0])[2:])
        np.save(os.path.join(out_dir, k + ".npy"), a)
    if idx is not None:
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    if all("costs" in o for o in outs):
        np.save(os.path.join(out_dir, "costs.npy"), np.stack([o["costs"] for o in outs]).astype(np.float32))


def measured_traffic(problems_per_launch: int):
    """DRAM bytes of one k_resident launch of that many co-resident problems, from the committed ncu captures
    (profiles/r1_traffic.json), or None."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return int(json.load(f)["launches"][str(problems_per_launch)]["dram_bytes_per_launch"])
        except Exception:
            continue
    return None


def committed_profile_numbers():
    """Numbers that only a profiler or a separate probe can give, read from committed files under profiles/ (never
    measured under ncu in this run): issue-slot utilisation of k_resident and the L2-resident copy peak."""
    out = {}
    for name in ("r2_ncu_resident.json", "r1_ncu_resident.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                out["issue_active_pct"] = float(json.load(f)["smsp__issue_active.avg.pct_of_peak_sustained_active"])
            out["issue_active_source"] = "profiles/" + name
            break
        except Exception:
            continue
    for name in ("r2_copy_peaks.json", "r1_copy_peaks.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                out["l2_copy_gbs"] = float(json.load(f)["l2_copy_gbs_32MiB"])
            out["l2_peak_source"] = "profiles/" + name + " (32 MiB L2-resident copy, same method as MEASURED_PEAKS.json)"
            break
        except Exception:
            continue
    return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class CpuArm:
    """The CPU arm: oracle/arap_oracle.c (port of the reference algorithm, OpenMP over all host threads) advancing the
    solve of ONE pair one continuation step per call, state carried from step to step exactly as
    CombinedSolverBase::singleSolve does (ARAP/shared/CombinedSolverBase.h:108-117).  19 consecutive calls are one full
    solve; fewer are a sample of it (continuation steps cost the same: every one runs 8 x 400 PCG iterations)."""

    def __init__(self, workload: str):
        # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm runs on rank 0 alone)
        # (ARAP_CPU_THREADS caps it, for trying the arm out on a machine that is busy with something else)
        os.environ["OMP_NUM_THREADS"] = os.environ.get("ARAP_CPU_THREADS", str(len(os.sched_getaffinity(0))))
        from oracle import pyoracle as O
        O.build()
        self.O = O
        self.workload = workload
        self.sp = make_pairs(workload, 1, 0)[0]
        sp = self.sp
        self.m = O.with_border_pins(sp.matches, sp.W, sp.H)
        self.U = O.grid(sp.W, sp.H)
        self.t = 0
        self.reset()

    def reset(self):
        sp = self.sp
        self.state = [(self.U.copy(), np.zeros((sp.H, sp.W), np.float32)) for _ in sp.masks]

    def step(self) -> float:
        """one continuation step of every segment of the pair; returns the seconds it took"""
        O, sp = self.O, self.sp
        if self.t == 0:
            self.reset()
        alpha = np.float32(self.t + 1) / np.float32(NCONT)
        dt = 0.0
        for k, mask in enumerate(sp.masks):
            Cn = O.constraint_image(mask, self.m, alpha)
            X, A = self.state[k]
            t0 = time.perf_counter()
            X, A, costs, _ = O.gn_solve(X, A, self.U, Cn, mask.astype(np.float32), NGN, NPCG)
            dt += time.perf_counter() - t0
            self.state[k] = (X, A)
        self.t = (self.t + 1) % NCONT
        return dt

    def warp_seconds(self) -> float:
        t0 = time.perf_counter()
        for k, mask in enumerate(self.sp.masks):
            self.O.warp(self.state[k][0], self.sp.rgb, mask)
        return time.perf_counter() - t0

    def info(self, step_seconds, warp_s):
        n = len(step_seconds)
        per_pair = NCONT * float(np.mean(step_seconds)) + warp_s
        return {"value": 1.0 / per_pair, "unit": "pairs/s", "cores": self.O.num_threads(), "kind": "port",
                "extrapolated": n < NCONT, "sampled_seconds": float(np.sum(step_seconds)),
                "sample": f"{self.workload}: {n} consecutive continuation step(s) of one pair's solve ({NGN}x{NPCG} PCG iterations "
                          f"each, {len(self.sp.masks)} segment(s)), mean {np.mean(step_seconds):.2f} s per step; a pair = {NCONT} such steps "
                          f"+ forward warp ({warp_s:.3f} s)" + ("" if n < NCONT else "; the timed steps contain a complete 19-step solve") +
                          "; oracle/arap_oracle.c, OpenMP"}


def cpu_leg(workload: str, n_steps: int = 3):
    """cpu_baseline of our arm: a bounded sample (n_steps continuation steps, about 10 s) of one pair on the host cores."""
    arm = CpuArm(workload)
    secs = [arm.step() for _ in range(n_steps)]
    return arm.info(secs, arm.warp_seconds())


def run_reference_arm(args, rank, world):
    """--impl reference.  A "step" here is ONE continuation step of one pair's solve (1/19 of a pair: the bounded sample
    the contract asks for); `ms_per_step` is the time of that step as executed, `value` = 1 / (19 x mean step + warp).
    With --steps >= 19 the timed region holds a complete solve and nothing is extrapolated."""
    if rank != 0:
        return
    W, H = WORKLOADS[args.workload][:2]
    arm = CpuArm(args.workload)
    for _ in range(args.warmup):
        arm.step()
    arm.t = 0                   # the timed steps start a fresh solve
    secs = [arm.step() for _ in range(args.steps)]
    info = arm.info(secs, arm.warp_seconds())
    v = info["value"]
    line = {"impl": "reference", "metric": f"flow pairs/sec @{W}x{H}", "value": v, "unit": "pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * float(np.mean(secs)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, [arm.sp]),
            "step_definition": f"one of the {NCONT} continuation steps of one pair (bounded sample of the workload); "
                               "pairs per step = 1/19",
            "extrapolated": info["extrapolated"],
            "note": "the reference has no CPU path (ARAP/API/src/o.t:121-124 accepts GPU solver kinds only; SURVEY.md 8c): "
                    "this is the oracle port on the host cores; rank 0 alone runs it at any N",
            "cpu_baseline": info,
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def opt_h_image(cs, p, mask):
    """one (image, segment) through the reference's own API sequence (CombinedSolver -> OptSolver -> Opt.h)"""
    from arap_flow_b200.combined_solver import with_border_pins
    cs.add_image(p.rgb, mask, with_border_pins(p.matches, p.W, p.H))
    cs.solve_all()


def single_problem_gn_step_ms(pair, mask):
    """SURVEY.md 8d (ii): device time of ONE Opt_ProblemStep (PCGInit + 400 PCG iterations + update + cost) of ONE problem,
    median over the steps of a few continuation steps -- through Opt_ProblemInit / Opt_ProblemStep, outside the timed region."""
    import ctypes as C
    import torch
    from arap_flow_b200.combined_solver import CombinedSolver, with_border_pins
    cs = CombinedSolver(pair.W, pair.H)
    cs.add_image(pair.rgb, mask, with_border_pins(pair.matches, pair.W, pair.H))
    cs._reset_gpu()
    pp = (C.c_void_p * 7)(cs.d_offset.data_ptr(), cs.d_angle.data_ptr(), cs.d_urshape.data_ptr(),
                          cs.d_constraints.data_ptr(), cs.d_mask.data_ptr(),
                          C.cast(C.byref(cs.w_fit), C.c_void_p), C.cast(C.byref(cs.w_reg), C.c_void_p))
    L, sv = cs.solver.L, cs.solver
    L.Opt_SetSolverParameter(sv.state, sv.plan, b"nIterations", C.byref(cs.nIterations))
    L.Opt_SetSolverParameter(sv.state, sv.plan, b"lIterations", C.byref(cs.lIterations))
    ms = []
    for t in range(3):
        cs._set_constraint_image(np.float32(t + 1) / np.float32(NCONT))
        torch.cuda.synchronize()
        L.Opt_ProblemInit(sv.state, sv.plan, pp)
        while True:
            t0 = time.perf_counter()
            more = L.Opt_ProblemStep(sv.state, sv.plan, pp)     # synchronous: returns after the step's cost read-back
            if not more:
                break
            ms.append((time.perf_counter() - t0) * 1e3)
    cs.close()
    return float(np.median(ms)) if ms else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C1", choices=sorted(WORKLOADS))
    ap.add_argument("--path", default="batch", choices=["batch", "opt_h"],
                    help="batch: arapb200_batch_* (several problems per cooperative launch).  opt_h: the reference's own "
                         "call sequence, one image at a time: 19 x Opt_ProblemSolve with the host-side constraint lerp and "
                         "full-image upload per continuation step (CombinedSolver.h / OptSolver.h)")
    ap.add_argument("--batch", type=int, default=0, help="pairs per GPU per step (0 = backend default)")
    ap.add_argument("--backend", default="auto", choices=["auto", "stream", "resident"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one to DIR/<name>.npy (float32, at most "
                         "64 MB; rank 0's pairs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug output (NCCL_DEBUG=VERSION|INFO) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":   # that banner is printf'ed to stdout regardless
            os.environ["NCCL_DEBUG"] = "WARN"
            if rank == 0:
                print("NCCL version %s" % ".".join(str(v) for v in torch.cuda.nccl.version()), file=sys.stderr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from arap_flow_b200 import lib
    lib.load()
    backend = {"auto": lib.BACKEND_AUTO, "stream": lib.BACKEND_STREAM, "resident": lib.BACKEND_RESIDENT}[args.backend]
    W, H = WORKLOADS[args.workload][:2]
    opt_h = args.path == "opt_h"
    # resident back-end: 3 (168 registers) or 4 (128 registers) C1-sized problems share one cooperative launch; 9 = three
    # launches of three, measured 2 % faster than two launches of four (profiles/r1_batch_choice.txt).  Smaller problems: as
    # many as fill the CTA slots of ONE launch (profiles/r2_batch_sweep.txt): 3 multi-segment pairs = 12 problems, 14 C1s pairs
    # C1: two launches of FOUR co-resident problems (128-register variant; 3 x 3 at 168 registers was the default until the
    # lean variants got their own load hoisting and deferred delta update: profiles/r2_batch_sweep.txt)
    DEFAULT_B = {"C1": 8, "C2": 3, "C1s": 14}
    B = args.batch if args.batch > 0 else (1 if (args.backend == "stream" or args.workload == "C4" or opt_h) else
                                           DEFAULT_B.get(args.workload, 9))
    pairs = make_pairs(args.workload, B, first=rank * B)
    nseg = WORKLOADS[args.workload][2]
    # --multseg (C2): one independent problem per segment, all of them sharing the pair's constraint list
    problems = [(p, m) for p in pairs for m in p.masks]
    active_px = [int(sum((m == 0).sum() for m in p.masks)) for p in pairs]   # per pair
    batch = None if opt_h else lib.Batch(W, H, len(problems), NCONT, NGN, NPCG, backend)
    cs = None
    if opt_h:
        from arap_flow_b200.combined_solver import CombinedSolver
        cs = CombinedSolver(W, H)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    out_bufs = [None] * len(problems)   # output arrays are allocated once and reused, as a caller looping over pairs would
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    io_bytes = [0, 0]
    opt_h_stage_log = []     # wall seconds per stage of every image, warm-up included

    def one_step():
        if opt_h:
            # the library's kernels run on its own stream, but every Opt_ProblemSolve is synchronous and the uploads /
            # download run on the current (default) stream, so events on the default stream bracket the device work
            outs = []
            for (p, m) in problems:
                opt_h_image(cs, p, m)
                opt_h_stage_log.append({k: round(v, 4) for k, v in cs.seconds.items()})
                io_bytes[0] += cs.h2d_bytes
                io_bytes[1] += cs.d2h_bytes
                outs.append({"flow": cs.warp_field(), "rgb": cs.warped_rgb, "mask": cs.warped_mask, "costs": cs.costs})
        else:
            outs = [batch.submit(i, p.rgb, m, p.matches, out=out_bufs[i]) for i, (p, m) in enumerate(problems)]
            out_bufs[:] = outs
            batch.run()
        flats = []
        if nseg > 1:  # layer flatten of every pair (para_gen.py:136-175) belongs to the pair's end-to-end time
            for k in range(len(pairs)):
                o = outs[k * nseg:(k + 1) * nseg]
                flats.append(lib.flatten([x["flow"] for x in o], [x["rgb"] for x in o], [x["mask"] for x in o]))
        return outs, flats

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > the 126 MiB L2

    def flush_l2():
        flush.zero_()

    for _ in range(args.warmup):
        one_step()
        flush_l2()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    dev_ms, solve_ms, launches = 0.0, 0.0, 0
    io_bytes[:] = [0, 0]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush_l2()
        if opt_h:
            ev[0].record()
            last = one_step()
            ev[1].record()
            ev[1].synchronize()
            ms = ev[0].elapsed_time(ev[1])
            dev_ms += ms
            solve_ms += ms
        else:
            last = one_step()
            tm = batch.timing_ms()
            dev_ms += tm["solve"] + tm["warp"]
            solve_ms += tm["solve"]
            launches += batch.launches()
    streamed = (batch.resident_count() == 0) if batch else (args.workload == "C4")
    linfo = batch.launch_info() if batch else None
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    # max over ranks (device-timed region and end-to-end wall)
    t = torch.tensor([dev_ms, wall * 1000.0, solve_ms], dtype=torch.float64, device="cuda")
    lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_ms_max, solve_ms_max = (float(x) for x in t.cpu())
    total_pairs = B * world * args.steps
    if rank == 0:
        value = total_pairs / (dev_ms_max / 1000.0)
        e2e = total_pairs / (wall_ms_max / 1000.0)
        peak, peak_src = measured_peak()
        n_iter = NCONT * NGN * NPCG
        alg_bytes = float(np.mean(active_px)) * (B_ITER * n_iter + B_GN_EXTRA * NCONT * NGN)   # per pair
        achieved = alg_bytes * B * args.steps / (solve_ms_max / 1000.0) / 1e9                  # this rank's GPU
        N = W * H
        prof = committed_profile_numbers()
        if opt_h:
            # per image: 1 check + (first call: 2 strip kernels) + 1 cooperative launch per Opt_ProblemSolve, + 3 warp kernels
            n_launch = len(problems) * args.steps * world * (NCONT * 2 + 2 + 3)
            h2d, d2h = io_bytes[0] // args.steps, io_bytes[1] // args.steps
        else:
            n_launch = int(lt.cpu()[0])
            h2d = int(len(problems) * (4 * N) + nseg * sum(16 * (len(p.matches) + 2 * (W + H)) for p in pairs))
            d2h = int(len(problems) * (12 * N + 4 * NCONT * (NGN + 1)))
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (measured_traffic(4 if B % 4 == 0 else 3) if not streamed and not opt_h and (B % 3 == 0 or B % 4 == 0) and args.workload == "C1" else None),
                "peak_source": peak_src}
        if streamed:
            roof["kernel"] = "k_step_a + k_step_b (streaming PCG iteration; 156 B/active px/iteration algorithmic)"
            roof["model"] = "streaming-HBM: state in HBM/L2, this is the bound that applies"
        else:
            roof["kernel"] = "k_resident (persistent fused GN/PCG solve; 156 B/active px/PCG iteration algorithmic)"
            roof["model"] = ("streaming-HBM figure for comparison only: NOT a bound for the resident kernel, whose PCG state never "
                             "leaves registers/shared memory (traffic << algorithmic bytes, so frac may exceed 1); the bound that "
                             "applies is issue-slot throughput: see issue_active_pct")
            if "l2_copy_gbs" in prof:
                roof["l2_frac"] = achieved / prof["l2_copy_gbs"]
                roof["l2_peak"] = prof["l2_copy_gbs"]
                roof["l2_peak_source"] = prof["l2_peak_source"]
            if "issue_active_pct" in prof:
                roof["issue_active_pct"] = prof["issue_active_pct"]
                roof["issue_active_source"] = prof["issue_active_source"]
        line = {
            "metric": f"flow pairs/sec @{W}x{H}", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, pairs),
            "run": {"path": ("opt_h: CombinedSolver/OptSolver sequence, 19 synchronous Opt_ProblemSolve calls per image, host-side "
                             "constraint lerp + full-image upload per continuation step, one problem per launch" if opt_h else
                             "batch: arapb200_batch_* (whole 19x8x400 schedules, several problems per cooperative launch)"),
                    "pairs_per_gpu_per_step": B, "backend": args.backend + (" (streaming)" if streamed else " (resident)"),
                    "launch": linfo, "opt_h_seconds_last_image": (cs.seconds if cs else None), "opt_h_seconds_every_image": (opt_h_stage_log if cs else None), "parallelism": f"independent pairs x{world}, no collective",
                    "l2_policy": "L2 flushed between steps by writing a 256 MiB buffer; every step also re-uploads its inputs "
                                 "(host->device) and restarts from the reset grid, nothing is reused across steps; within a "
                                 "solve the PCG state lives " + ("in HBM/L2 (tile-interleaved planes)" if streamed else
                                                                 "in registers/shared memory")},
            "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": n_launch,
            # amortised: solve time of the whole step / (problems x GN steps) -- co-resident problems overlap, so this is
            # NOT the latency of one Gauss-Newton step; that is ms_per_gn_step_single_problem below
            "ms_per_gn_step_amortised": solve_ms_max / (B * args.steps * NCONT * NGN),
            "roofline": roof,
            "clocks": clocks,
        }
        if world == 1 and not streamed:
            try:   # SURVEY.md 8d (ii), measured after the timed region
                line["ms_per_gn_step_single_problem"] = single_problem_gn_step_ms(pairs[0], pairs[0].masks[0])
            except Exception as e:
                line["ms_per_gn_step_single_problem"] = None
                print("single-problem GN step timing failed:", e, file=sys.stderr)
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_leg(args.workload)
            except Exception as e:  # the oracle is a checker; never let it sink the GPU number
                line["cpu_baseline"] = {"error": str(e)}
        print(json.dumps(line), flush=True)
    if batch:
        batch.close()
    if cs:
        cs.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
