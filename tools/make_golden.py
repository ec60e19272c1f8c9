#!/usr/bin/env python
"""Generate the committed fixtures under tests/golden/ (run in the build container only).

Needs /root/reference (read-only) and oracle/_ref/warp_image_ref (built by oracle/Makefile from the
reference's own warp sources).  Nothing here is needed at test time: the tests read tests/golden/ only.

  python tools/make_golden.py            # fixtures: cat512 copies + reference-tool warp outputs
  python tools/make_golden.py --solve    # additionally pin the oracle solve on cat512 (minutes of CPU)
  python tools/make_golden.py --para-gen # only: para_gen.py's own valid_cnstr / add_bg / flatten run on seeded inputs
"""
from __future__ import annotations

import argparse
import json
import lzma
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from arap_flow_b200 import flowio, synth  # noqa: E402
from oracle import pyoracle as O  # noqa: E402

REF = "/root/reference/ARAP"
GOLD = os.path.join(ROOT, "tests", "golden")


def ref_warp(rgb, mask, flow, tmp):
    """Run the reference's warp_image on in-memory inputs; returns (rgb, mask_rgb)."""
    pr, pm, pf = (os.path.join(tmp, n) for n in ("i.png", "m.png", "f.flo"))
    orr, om = os.path.join(tmp, "or.png"), os.path.join(tmp, "om.png")
    flowio.write_png(pr, rgb)
    flowio.write_png(pm, np.repeat(mask[..., None], 3, axis=2))
    flowio.write_flo(pf, flow)
    subprocess.check_call([O.REF_WARP_BIN, pr, pm, pf, orr, om], stdout=subprocess.DEVNULL)
    return flowio.read_png_rgb(orr), flowio.read_png_rgb(om)


def ref_function(name):
    """The reference's own top-level function `name` of para_gen.py, compiled from its source text where it lies.
    (para_gen.py is Python 2 -- print statements -- and cannot be imported; the three functions used here are valid
    Python 3 as they stand.)"""
    lines = open("/root/reference/para_gen.py").read().splitlines()
    start = next(i for i, l in enumerate(lines) if l.startswith("def %s(" % name))
    end = next((i for i in range(start + 1, len(lines)) if lines[i] and not lines[i][0].isspace() and not lines[i].startswith("#")), len(lines))
    return "\n".join(lines[start:end])


def para_gen_cases():
    """Run para_gen.valid_cnstr / add_bg / flatten themselves on seeded inputs -> tests/golden/para_gen_cases.npz."""
    from math import sqrt
    rng = np.random.default_rng(7)
    out = {}
    # --- valid_cnstr over raw matches, two label images of different sizes, points in and out of range
    H1, W1, H2, W2 = 60, 90, 64, 88
    yy, xx = np.mgrid[0:H1, 0:W1]
    mk1 = ((xx // 30) + 1).astype(np.uint8) * (yy > 8)          # labels 1..3, background band on top
    mk2 = np.zeros((H2, W2), np.uint8)
    mk2[:H1, :W2] = np.roll(mk1, 3, axis=1)[:, :W2]
    n = 400
    m = np.stack([rng.integers(0, W1 + 6, n), rng.integers(0, H1 + 6, n), np.zeros(n, np.int64), np.zeros(n, np.int64)], 1)
    m[:, 2] = m[:, 0] + rng.integers(-70, 71, n)
    m[:, 3] = m[:, 1] + rng.integers(-70, 71, n)
    m[::7, 2:] = m[::7, :2]                                      # zero-length matches are dropped
    m[:, 2:] = np.abs(m[:, 2:])                                  # the matcher never emits negative coordinates
    ns = {"sqrt": sqrt}
    exec(ref_function("valid_cnstr"), ns)
    keep = np.array([bool(ns["valid_cnstr"](int(a), int(b), int(c), int(d), mk1, mk2)) for a, b, c, d in m])
    out.update(vc_mk1=mk1, vc_mk2=mk2, vc_matches=m.astype(np.int32), vc_keep=keep)
    # --- add_bg
    ns = {"np": np}
    exec(ref_function("add_bg"), ns)
    im = rng.integers(0, 256, (40, 56, 3)).astype(np.uint8)
    mk = (rng.random((40, 56)) < 0.6).astype(np.uint8) * 255
    bg = rng.integers(0, 256, (40, 56, 3)).astype(np.uint8)
    out.update(bg_im=im, bg_mk=mk, bg_bg=bg, bg_out=ns["add_bg"](im, mk, bg))
    # --- flatten: file-based in the reference; run it on an in-memory "file system"
    fs = {}

    class _Img:
        def __init__(self, a): self.a = a
        def save(self, path): fs[path] = np.array(self.a)

    class _Image:
        @staticmethod
        def open(path): return fs[path]
        @staticmethod
        def fromarray(a): return _Img(a)

    class _Sintel:
        @staticmethod
        def flow_read(path): return fs[path][..., 0], fs[path][..., 1]
        @staticmethod
        def flow_write(path, a): fs[path] = np.array(a)

    class _Os:
        @staticmethod
        def remove(path): fs.pop(path)

    ns = {"np": np, "Image": _Image, "sintel_io": _Sintel, "os": _Os}
    exec(ref_function("flatten"), ns)
    L, H, W = 3, 36, 48
    flows = rng.normal(0, 5, (L, H, W, 2)).astype(np.float32)
    rgbs = rng.integers(0, 256, (L, H, W, 3)).astype(np.uint8)
    masks = ((rng.random((L, H, W)) < 0.4) * 255).astype(np.uint8)
    seg = []
    for s_ in range(L):
        fs["f%d" % s_], fs["r%d" % s_], fs["m%d" % s_] = flows[s_], rgbs[s_], masks[s_]
        seg.append("a b c f%d r%d m%d" % (s_, s_, s_))
    ns["flatten"]([("a b c F R M", seg)])
    out.update(fl_flows=flows, fl_rgbs=rgbs, fl_masks=masks, fl_out_flow=fs["F"], fl_out_rgb=fs["R"], fl_out_mask=fs["M"])
    np.savez_compressed(os.path.join(GOLD, "para_gen_cases.npz"), **out)
    print("para_gen_cases.npz:", {k: (v.shape, str(v.dtype)) for k, v in out.items()}, "kept", int(keep.sum()), "of", n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--solve", action="store_true")
    ap.add_argument("--para-gen", action="store_true")
    args = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    if args.para_gen:
        para_gen_cases()
        return
    # 1. the reference's own worked-example fixtures (data, not source)
    for src, dst in (
        ("deformation/cat512_iRGB.png", "cat512_iRGB.png"),
        ("deformation/cat512_iMsk.png", "cat512_iMsk.png"),
        ("deformation/cat512_iCstr.txt", "cat512_iCstr.txt"),
        ("warping/cat512_wRGB.png", "cat512_wRGB.png"),
        ("warping/cat512_wMsk.png", "cat512_wMsk.png"),
    ):
        shutil.copyfile(os.path.join(REF, src), os.path.join(GOLD, dst))
        os.chmod(os.path.join(GOLD, dst), 0o644)
    # the shipped flow is 2 MB raw: stored xz-compressed, byte for byte (tests/helpers.py cat512_flo restores it)
    with open(os.path.join(REF, "warping/cat512_iFlo.flo"), "rb") as f:
        flo_bytes = f.read()
    with open(os.path.join(GOLD, "cat512_iFlo.flo.xz"), "wb") as f:
        f.write(lzma.compress(flo_bytes, preset=9 | lzma.PRESET_EXTREME))
    # 2. reference warp tool outputs: cat512 (its RGB differs from the shipped golden by +-1 on 978 px,
    #    SURVEY.md 4) and synthetic cases with folds / out-of-frame motion / ragged masks.
    with tempfile.TemporaryDirectory() as tmp:
        rgb = flowio.read_png_rgb(os.path.join(GOLD, "cat512_iRGB.png"))
        msk = flowio.read_png_mask_red(os.path.join(GOLD, "cat512_iMsk.png"))
        flo = flowio.read_flo(os.path.join(REF, "warping/cat512_iFlo.flo"))
        wr, wm = ref_warp(rgb, msk, flo, tmp)
        flowio.write_png(os.path.join(GOLD, "cat512_reftool_wRGB.png"), wr)
        cases = {}
        for name, (W, H, seed, amp) in {
            "warp_a": (96, 64, 11, 3.0),     # gentle
            "warp_b": (131, 77, 12, 25.0),   # folds, overlaps, leaves the frame
            "warp_c": (64, 64, 13, 0.0),     # identity flow
        }.items():
            rng = np.random.default_rng(seed)
            p = synth.synth(W, H, 1, 1, seed)
            mask = p.masks[0].copy()
            # ragged mask: punch random holes and let the object touch the border on one side
            holes = rng.random((H, W)) < 0.03
            mask[holes] = 255
            mask[H // 3: H // 2, : W // 4] = 0
            yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
            fl = np.stack([amp * np.sin(yy / 7.0) + amp * 0.5 * np.cos(xx / 5.0),
                           amp * np.cos(xx / 9.0) - amp * 0.25], axis=-1).astype(np.float32)
            fl += (rng.standard_normal((H, W, 2)) * (amp * 0.1)).astype(np.float32)
            r, m = ref_warp(p.rgb, mask, fl, tmp)
            cases[name] = dict(rgb=p.rgb, mask=mask, flow=fl, ref_rgb=r, ref_mask=m[..., 0])
        np.savez_compressed(os.path.join(GOLD, "warp_reftool_cases.npz"),
                            **{f"{k}__{f}": v for k, c in cases.items() for f, v in c.items()})
    print("fixtures written to", GOLD)
    # 3. pin the oracle solve on the only end-to-end golden the tree ships
    if args.solve:
        cstr = flowio.read_constraints(os.path.join(GOLD, "cat512_iCstr.txt"))
        t0 = time.time()
        X, A, costs = O.solve(msk, cstr)
        dt = time.time() - t0
        fl = O.flow(X)
        act = msk == 0
        epe = np.hypot(*(np.moveaxis(fl - flo, -1, 0)))
        cerr = [float(np.hypot(*(fl[y1, x1] - (x2 - x1, y2 - y1)))) for x1, y1, x2, y2 in cstr]
        gcerr = [float(np.hypot(*(flo[y1, x1] - (x2 - x1, y2 - y1)))) for x1, y1, x2, y2 in cstr]
        np.savez_compressed(os.path.join(GOLD, "cat512_oracle_flow.npz"), flow=fl, costs=costs)
        # the rasteriser on the solved positions themselves (positions rebuilt from the float32 flow can differ)
        wr, wm, _ = O.warp(X, rgb, msk)
        flowio.write_png(os.path.join(GOLD, "cat512_oracle_wRGB.png"), wr)
        flowio.write_png(os.path.join(GOLD, "cat512_oracle_wMsk.png"), wm)
        out = dict(
            what="oracle full solve (19x8x400) on cat512 vs the shipped golden cat512_iFlo.flo",
            threads=O.num_threads(), seconds=dt,
            active_px=int(act.sum()),
            mean_epe_px=float(epe[act].mean()), median_epe_px=float(np.median(epe[act])),
            max_epe_px=float(epe.max()),
            mean_flow_px=float(np.hypot(flo[..., 0], flo[..., 1])[act].mean()),
            off_object_max_abs_flow=float(np.abs(fl[~act]).max()),
            constraint_err_px_max=max(cerr), golden_constraint_err_px_max=max(gcerr),
            final_cost=float(costs[-1, -1]), first_cost=float(costs[0, 0]),
        )
        with open(os.path.join(GOLD, "cat512_oracle_pin.json"), "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
