"""Process-level contracts on the GPU box: our arap_deform / warp_image binaries, the reference's OWN host
program linked against libarapb200 (oracle/_ref/arap_deform_refhost), and para_gen-style sharding."""
import os
import subprocess

import numpy as np
import pytest

from arap_flow_b200 import driver, flowio, lib, synth
from tests.helpers import cat512_flo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFHOST = os.path.join(ROOT, "oracle", "_ref", "arap_deform_refhost")


def _write_case(d, name, sp, mask):
    p = {k: str(d / f"{name}_{k}") for k in ("rgb.png", "msk.png", "cstr.txt", "out.flo", "wrgb.png", "wmsk.png")}
    flowio.write_png(p["rgb.png"], sp.rgb)
    flowio.write_png(p["msk.png"], np.repeat(mask[..., None], 3, axis=2))
    flowio.write_constraints(p["cstr.txt"], sp.matches)
    return (p["rgb.png"], p["msk.png"], p["cstr.txt"], p["out.flo"], p["wrgb.png"], p["wmsk.png"])


def test_warp_image_cli_on_cat512(gold, tmp_path):
    out_rgb, out_m = str(tmp_path / "w.png"), str(tmp_path / "m.png")
    r = subprocess.run([driver.WARP_BIN, os.path.join(gold, "cat512_iRGB.png"), os.path.join(gold, "cat512_iMsk.png"),
                        cat512_flo(tmp_path), out_rgb, out_m], capture_output=True, text=True)
    assert r.returncode == 0 and "Saved" in r.stdout
    assert np.array_equal(flowio.read_png_rgb(out_m), flowio.read_png_rgb(os.path.join(gold, "cat512_wMsk.png")))
    assert np.array_equal(flowio.read_png_rgb(out_rgb), flowio.read_png_rgb(os.path.join(gold, "cat512_reftool_wRGB.png")))


def test_arap_deform_cli_list_file_matches_library(tmp_path):
    """list file with two image sizes (re-plan path) and a multi-segment pair sharing one constraint file"""
    a = synth.synth(96, 80, 1, 2, 7)
    b = synth.synth(128, 96, 2, 3, 8)
    items = [_write_case(tmp_path, "a", a, a.masks[0]), _write_case(tmp_path, "b0", b, b.masks[0]),
             _write_case(tmp_path, "b1", b, b.masks[1])]
    lst = str(tmp_path / "list.txt")
    driver.write_list_file(lst, items)
    env = dict(os.environ, ARAP_PLAN=driver.PLAN)
    r = subprocess.run([driver.ARAP_BIN, lst], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count("Saved") == 3 and "re-build plan" in r.stdout
    for it, (sp, mask) in zip(items, [(a, a.masks[0]), (b, b.masks[0]), (b, b.masks[1])]):
        flow, rgb, m, _ = lib.deform(sp.rgb, mask, sp.matches)
        assert np.array_equal(flowio.read_flo(it[3]), flow)
        assert np.array_equal(flowio.read_png_rgb(it[4]), rgb)
        assert np.array_equal(flowio.read_png_rgb(it[5])[..., 0], m)


def _cat512(gold):
    return (flowio.read_png_rgb(os.path.join(gold, "cat512_iRGB.png")),
            flowio.read_png_mask_red(os.path.join(gold, "cat512_iMsk.png")),
            flowio.read_constraints(os.path.join(gold, "cat512_iCstr.txt")))


def _check_cat512_solve(gold, tmp_path, msk, cstr, flo, costs):
    """(2) identical to the recorded oracle solve of the README example (tools/make_golden.py --solve); (3) against the
    shipped golden flow: the weak end-to-end pin (chaotic fixed-budget trajectory, SURVEY.md 8c)"""
    z = np.load(os.path.join(gold, "cat512_oracle_flow.npz"))
    assert np.array_equal(flo, z["flow"]) and np.array_equal(costs, z["costs"])
    gflo = flowio.read_flo(cat512_flo(tmp_path))
    act = msk == 0
    epe = np.hypot(flo[..., 0] - gflo[..., 0], flo[..., 1] - gflo[..., 1])
    assert epe[act].mean() < 0.35 and np.median(epe[act]) < 0.12 and (flo[~act] == 0).all()
    err = [np.hypot(*(flo[y1, x1] - (x2 - x1, y2 - y1))) for x1, y1, x2, y2 in cstr]
    assert max(err) < 5e-3


@pytest.mark.skipif(not os.path.exists(REFHOST), reason="reference host binary not built (needs the reference's sources)")
def test_reference_host_program_runs_on_our_library(oracle, gold, tmp_path):
    """The reference's unmodified main.cpp / CombinedSolver.h / OptSolver.h, compiled against include/Opt.h and
    linked with libarapb200.so, solves the README example (ARAP/deformation/README.md:34-38) end to end:
    19 x Opt_ProblemSolve through the real Opt.h call sequence, then the reference's own CPU rasteriser."""
    out = {k: str(tmp_path / k) for k in ("o.flo", "wrgb.png", "wmsk.png")}
    env = dict(os.environ, ARAP_PLAN=driver.PLAN)
    r = subprocess.run([REFHOST, os.path.join(gold, "cat512_iRGB.png"), os.path.join(gold, "cat512_iMsk.png"),
                        os.path.join(gold, "cat512_iCstr.txt"), out["o.flo"], out["wrgb.png"], out["wmsk.png"]],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Saved" in r.stdout
    flo = flowio.read_flo(out["o.flo"])
    # (1) identical to our own end-to-end path on the same inputs, bit for bit
    rgb, msk, cstr = _cat512(gold)
    flow, wrgb, wm, costs = lib.deform(rgb, msk, cstr)
    assert np.array_equal(flo, flow)
    # ... including the reference's CPU rasteriser vs our z-buffer kernels
    assert np.array_equal(flowio.read_png_rgb(out["wrgb.png"]), wrgb)
    assert np.array_equal(flowio.read_png_rgb(out["wmsk.png"])[..., 0], wm)
    _check_cat512_solve(gold, tmp_path, msk, cstr, flo, costs)


def test_readme_example_matches_recorded_oracle_solve(gold, tmp_path):
    """The README example end to end through the library at the full 19 x 8 x 400 schedule, against stored fixtures
    only: the solve as in test_reference_host_program_runs_on_our_library (2) and (3), and the warped RGB and mask
    against the oracle's rasteriser (bit-exact with the reference's warp tool, tests/test_oracle_golden.py) applied to
    the recorded solve's positions (tools/make_golden.py --solve).  Those positions are not stored: rebuilt from the
    float32 flow they differ in the last bit on some pixels, enough to move warped RGB values."""
    rgb, msk, cstr = _cat512(gold)
    flo, wrgb, wm, costs = lib.deform(rgb, msk, cstr)
    _check_cat512_solve(gold, tmp_path, msk, cstr, flo, costs)
    assert np.array_equal(wrgb, flowio.read_png_rgb(os.path.join(gold, "cat512_oracle_wRGB.png")))
    assert np.array_equal(wm, flowio.read_png_mask_red(os.path.join(gold, "cat512_oracle_wMsk.png")))


def test_sharded_run_is_byte_identical_to_single_gpu(tmp_path):
    """para_gen.py --gpu: N solver processes x CUDA_VISIBLE_DEVICES produce the same files as one process."""
    import torch
    ngpu = torch.cuda.device_count()
    sp = [synth.synth(80, 64, 1, 2, 100 + i) for i in range(5)]
    d1, d2 = tmp_path / "one", tmp_path / "many"
    d1.mkdir(); d2.mkdir()
    it1 = [_write_case(d1, f"p{i}", s, s.masks[0]) for i, s in enumerate(sp)]
    it2 = [_write_case(d2, f"p{i}", s, s.masks[0]) for i, s in enumerate(sp)]
    driver.run_sharded(it1, [0], str(tmp_path / "tmp"))
    gpus = list(range(min(ngpu, 2))) if ngpu > 1 else [0, 0]   # two worker processes even on a 1-GPU box
    driver.run_sharded(it2, gpus, str(tmp_path / "tmp"), batch=2)
    for a, b in zip(it1, it2):
        for k in (3, 4, 5):
            assert open(a[k], "rb").read() == open(b[k], "rb").read()
    assert not os.listdir(tmp_path / "tmp")  # temporary list files are always removed (para_gen.py:197-200)


def test_resident_worker_serves_clients_byte_identically(tmp_path):
    """N2: `arap_deform --serve` keeps context + plan + buffers; clients (the same binary, same argv contract, with
    ARAP_SERVER set) hand their list files over.  Several dispatches, two image sizes, a single-item argv call: every
    output file equals the one a stand-alone process writes, the "Saved" lines and exit codes are the same."""
    sps = [synth.synth(96, 80, 1, 2, 30 + i) for i in range(5)] + [synth.synth(128, 96, 2, 3, 40)]
    jobs = [(s, s.masks[0]) for s in sps] + [(sps[-1], sps[-1].masks[1])]
    d1, d2 = tmp_path / "direct", tmp_path / "served"
    d1.mkdir(); d2.mkdir()
    it1 = [_write_case(d1, f"p{i}", s, m) for i, (s, m) in enumerate(jobs)]
    it2 = [_write_case(d2, f"p{i}", s, m) for i, (s, m) in enumerate(jobs)]
    driver.do_arap(it1, 0, str(tmp_path / "tmp"))
    spool = str(tmp_path / "spool")
    env = dict(os.environ, ARAP_PLAN=driver.PLAN, ARAP_SERVER=spool)
    # no server yet: the client fails loudly instead of solving on its own
    r = subprocess.run([driver.ARAP_BIN] + list(it2[0]), capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "no server" in r.stderr
    with driver.Server(0, spool, warm=(96, 80)) as srv:                        # plan + buffers pre-built for the first size
        driver.do_arap(it2[:3], 0, str(tmp_path / "tmp"), server=spool)        # dispatch 1
        driver.do_arap(it2[3:6], 0, str(tmp_path / "tmp"), server=spool)       # dispatch 2: ends with a size change
        r = subprocess.run([driver.ARAP_BIN] + list(it2[6]), capture_output=True, text=True, env=env)   # argv form
        assert r.returncode == 0 and r.stdout.count("Saved") == 1, r.stdout + r.stderr
        # a bad request is answered with a non-zero code and does not take the worker down
        bad = list(it2[0]); bad[0] = str(tmp_path / "missing.png")
        r = subprocess.run([driver.ARAP_BIN] + bad, capture_output=True, text=True, env=env)
        assert r.returncode != 0
        driver.do_arap(it2[:1], 0, str(tmp_path / "tmp"), server=spool)
        assert srv.proc.poll() is None
    for a, b in zip(it1, it2):
        for k in (3, 4, 5):
            assert open(a[k], "rb").read() == open(b[k], "rb").read()
    assert not [f for f in os.listdir(spool) if f.endswith((".job", ".run", ".done"))]
