"""Motion blur of scenes in the batch (DESIGN.md 4.8): Batch.submit_scene(..., blur=...) against the CPU restatement
(tests/blur_oracle.py) on the oracle's continuation states, against the scene's own sharp outputs where the definition
makes them equal, across the solver paths, in mixed runs, with buffer reuse and after rejections.  Every comparison is
bit for bit."""
import ctypes as C
import functools

import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from tests import blur_oracle as BL
from tests import sequence_oracle as SO

pytestmark = pytest.mark.gpu

KW = dict(nCont=6, nGN=2, nPCG=30)
STEPS = [0, 2, 5]
SCENE_KEYS = ("flow", "rgb", "mask", "bflow", "occ", "costs")


def _moving(sp, seed):
    A, m = synth.background_motion(sp.W, sp.H, seed)
    return A, synth.background(sp.W + 2 * m, sp.H + 2 * m, seed), (m, m)


@functools.lru_cache(maxsize=None)
def _case(name):
    """A config scene over a moving background, with the oracle's state after every continuation step of every layer."""
    sp = synth.config(name)
    A, bg, origin = _moving(sp, 70 + int(name[1]))
    states = []
    for m in sp.masks:
        snaps = SO.solve_states(m, sp.matches, range(KW["nCont"]), **KW)[3]
        states.append({t: snaps[t] for t in range(KW["nCont"])})
    return sp, A, bg, origin, states


def _submit(b, sp, A, bg, origin, frames, blur, input_frame=True, slot=0, out=None):
    path = synth.motion_path(A, frames, KW["nCont"]) if frames else None
    return b.submit_scene(slot, sp.rgb, sp.masks, [sp.matches] * len(sp.masks), bg, A, origin=origin, frames=frames,
                          frame_motions=path, input_frame=input_frame, out=out, blur=blur)


def _same(a, b, keys):
    for k in keys:
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------- against the restatement
@pytest.mark.parametrize("frames", [STEPS, None], ids=["frames", "pair"])
@pytest.mark.parametrize("shutter", [0.3, 1.0])
@pytest.mark.parametrize("S", [2, 5, 8])
@pytest.mark.parametrize("name", ["C1", "C2"])
def test_against_the_restatement(oracle, name, S, shutter, frames):
    sp, A, bg, origin, states = _case(name)
    b = lib.Batch(sp.W, sp.H, len(sp.masks), **KW)
    out = _submit(b, sp, A, bg, origin, frames, (S, shutter))
    b.run()
    b.close()
    path = synth.motion_path(A, frames, KW["nCont"]) if frames else None
    args = (states, sp.rgb, sp.masks, bg, origin, KW["nCont"], frames, A, path, S, shutter)
    assert np.array_equal(out["blur_rgb"], BL.blur_image(*args, 0))
    assert np.array_equal(out["blur_rgb0"], BL.blur_image(*args, -1))
    if frames:
        for k in range(1, len(frames) + 1):
            assert np.array_equal(out["seq"]["blur_rgb"][k - 1], BL.blur_image(*args, k)), k
    assert not np.array_equal(out["blur_rgb"], out["rgb"])


# ------------------------------------------------------------------------------------- clean equality
@pytest.mark.parametrize("S,shutter", [(1, 1.0), (6, 0.0)])
def test_one_sample_or_closed_shutter_gives_the_sharp_images(oracle, S, shutter):
    sp = synth.config("C2")
    A, bg, origin = _moving(sp, 81)
    b = lib.Batch(sp.W, sp.H, 4, **KW)
    out = _submit(b, sp, A, bg, origin, STEPS, (S, shutter))
    b.run()
    b.close()
    assert np.array_equal(out["blur_rgb"], out["rgb"])
    assert np.array_equal(out["seq"]["blur_rgb"], out["seq"]["rgb"])
    grid = oracle.grid(sp.W, sp.H)
    covered = np.any([oracle.warp(grid, sp.rgb, m)[1] != 0 for m in sp.masks], axis=0)
    obj = np.any([m == 0 for m in sp.masks], axis=0)
    keep = covered | ~obj
    assert np.array_equal(out["blur_rgb0"][keep], out["rgb0"][keep])


def test_full_schedule_two_samples_average_consecutive_frames():
    sp = synth.config("C2")
    A, bg, origin = _moving(sp, 82)
    nCont = 19
    steps = list(range(nCont))
    b = lib.Batch(sp.W, sp.H, 4, nCont, 8, 400)
    out = b.submit_scene(0, sp.rgb, sp.masks, [sp.matches] * 4, bg, A, origin=origin, frames=steps,
                         frame_motions=synth.motion_path(A, steps, nCont), blur=(2, 1.0))
    b.run()
    assert b.launch_info()["grid"][1] == 1 and b.resident_count() == 4
    b.close()
    clean, blur = out["seq"]["rgb"].astype(np.int32), out["seq"]["blur_rgb"].astype(np.int32)
    assert np.array_equal(blur[1:], (clean[1:] + clean[:-1] + 1) >> 1)
    assert not np.array_equal(blur[1:], clean[1:])


# ------------------------------------------------------------------------------------- solver paths
def _paths_scene():
    sp = synth.synth(96, 80, 2, 2, 91)
    A, bg, origin = _moving(sp, 83)
    return sp, A, bg, origin


@pytest.mark.parametrize("kind", ["resident", "stream", "lm"])
def test_solver_paths_against_the_restatement(oracle, kind):
    sp, A, bg, origin = _paths_scene()
    b = lib.Batch(sp.W, sp.H, 2, backend=lib.BACKEND_STREAM if kind == "stream" else lib.BACKEND_AUTO, **KW)
    if kind == "lm":
        b.set_option("lm", 1)
    _submit(b, sp, A, bg, origin, None, None)
    b.run()
    sharp = b.launches()
    got = []
    for frames in (None, [1, 4]):   # without frames only the blur asks the resident path for per-step launches
        got.append(_submit(b, sp, A, bg, origin, frames, (5, 0.8)))
        b.run()
        if kind == "resident":
            assert b.resident_count() == 2 and b.launch_info()["problems_per_launch"] == 2
            if frames is None:   # one launch per step: nCont - 1 more group launches and constraint images (2 each)
                assert b.launches() == sharp + 2 * 5 * 2 + (KW["nCont"] - 1) * (1 + 2 * 2)
        else:
            assert b.resident_count() == 0
    b.close()
    states = []
    for m in sp.masks:
        snaps = SO.solve_states(m, sp.matches, range(KW["nCont"]), lm=kind == "lm", **KW)[3]
        states.append(dict(enumerate(snaps)))
    for out, frames in zip(got, (None, [1, 4])):
        path = synth.motion_path(A, frames, KW["nCont"]) if frames else None
        args = (states, sp.rgb, sp.masks, bg, origin, KW["nCont"], frames, A, path, 5, 0.8)
        assert np.array_equal(out["blur_rgb"], BL.blur_image(*args, 0))
        assert np.array_equal(out["blur_rgb0"], BL.blur_image(*args, -1))
        if frames:
            for k in (1, 2):
                assert np.array_equal(out["seq"]["blur_rgb"][k - 1], BL.blur_image(*args, k))


def test_streaming_and_resident_blur_alike():
    sp, A, bg, origin = _paths_scene()
    outs = []
    for backend in (lib.BACKEND_STREAM, lib.BACKEND_AUTO):
        b = lib.Batch(sp.W, sp.H, 2, backend=backend, **KW)
        outs.append(_submit(b, sp, A, bg, origin, [0, 3, 5], (7, 1.0)))
        b.run()
        b.close()
    _same(outs[0], outs[1], SCENE_KEYS + ("rgb0", "blur_rgb", "blur_rgb0"))
    _same(outs[0]["seq"], outs[1]["seq"], ("rgb", "blur_rgb"))


# ------------------------------------------------------------------------------------- a mixed run
def test_mixed_run_changes_nothing_else():
    sp1, sp2 = synth.synth(160, 120, 3, 2, 92), synth.synth(160, 120, 2, 2, 93)
    plain = synth.synth(160, 120, 1, 2, 94)
    m1, m2 = _moving(sp1, 84), _moving(sp2, 85)
    S, frames = 4, [1, 3, 5]
    runs = []
    for blur in (None, (S, 0.6)):
        b = lib.Batch(160, 120, 7, **KW)
        o1 = _submit(b, sp1, *m1, frames, blur)
        o2 = _submit(b, sp2, *m2, [2, 5], None, input_frame=False, slot=3)
        op = [b.submit(5 + j, plain.rgb, plain.masks[0], plain.matches, extras=j == 1) for j in range(2)]
        b.run()
        runs.append((o1, o2, op, b.launches(), b.resident_count()))
        b.close()
    (a1, a2, ap, la, ra), (g1, g2, gp, lg, rg) = runs
    assert lg == la + 2 * S * (1 + len(frames) + 1) and rg == ra == 7
    _same(g1, a1, SCENE_KEYS + ("rgb0",))
    _same(g1["seq"], a1["seq"], ("flow", "rgb", "mask", "bflow", "occ"))
    _same(g2, a2, SCENE_KEYS)
    _same(g2["seq"], a2["seq"], ("flow", "rgb", "mask", "bflow", "occ"))
    for j, (g, a) in enumerate(zip(gp, ap)):
        _same(g, a, ("flow", "rgb", "mask", "costs") + (("bflow", "occ") if j == 1 else ()))
    assert "blur_rgb" not in a1 and "blur_rgb" not in g2


# ------------------------------------------------------------------------------------- buffer reuse
def test_one_batch_reuses_its_buffers():
    small, big = synth.synth(160, 120, 2, 2, 95), synth.synth(200, 150, 3, 2, 96)
    b = lib.Batch(200, 150, 3, **KW)
    out = None
    for sp, blur, frames, seed in ((small, (8, 1.0), STEPS, 86), (small, (2, 0.5), STEPS, 87), (small, None, STEPS, 88),
                                   (big, (3, 0.9), [0, 4], 89)):
        A, bg, origin = _moving(sp, seed)
        fresh = lib.Batch(200, 150, 3, **KW)
        want = _submit(fresh, sp, A, bg, origin, frames, blur)
        fresh.run()
        fresh.close()
        out = _submit(b, sp, A, bg, origin, frames, blur, out=out)
        b.run()
        assert set(out) == set(want) and set(out["seq"]) == set(want["seq"])
        _same(out, want, [k for k in want if k != "seq"])
        _same(out["seq"], want["seq"], list(want["seq"]))
        assert ("blur_rgb" in out) == (blur is not None) and ("blur_rgb" in out["seq"]) == (blur is not None)
    b.close()


# ------------------------------------------------------------------------------------- rejections
def test_rejections_change_nothing():
    sp = synth.synth(96, 80, 2, 2, 97)
    A, bg, origin = _moving(sp, 90)
    W, H = sp.W, sp.H
    L = lib.load()
    L.arapb200_batch_scene_blur.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 3
    b = lib.Batch(W, H, 5, **KW)
    out = _submit(b, sp, A, bg, origin, [1, 3], (3, 0.5))             # a valid request that the rejections must keep
    two = 2 * np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])              # frame 0 at u = 1 extrapolates to 0: singular
    still = b.submit_scene(2, sp.rgb, sp.masks, [sp.matches] * 2, bg, two, origin=origin, input_frame=True)
    no_rgb0 = b.submit_scene(4, sp.rgb, sp.masks[:1], [sp.matches], bg, A, origin=origin)
    buf = np.zeros((3, H, W, 3), np.uint8)
    p = buf.ctypes.data
    cases = {
        "null batch": (None, 0, 3, 0.5, p, None, None), "second slot of a scene": (b.h, 1, 3, 0.5, p, None, None),
        "slot -1": (b.h, -1, 3, 0.5, p, None, None), "slot past the batch": (b.h, 5, 3, 0.5, p, None, None),
        "S 0": (b.h, 0, 0, 0.5, p, None, None), "S 65": (b.h, 0, 65, 0.5, p, None, None),
        "shutter nan": (b.h, 0, 3, float("nan"), p, None, None), "shutter -0.1": (b.h, 0, 3, -0.1, p, None, None),
        "shutter 1.1": (b.h, 0, 3, 1.1, p, None, None), "null blur_rgb": (b.h, 0, 3, 0.5, None, None, None),
        "blur_rgb0 without rgb0": (b.h, 4, 3, 0.5, p, p, None), "frames of a scene without": (b.h, 2, 3, 0.5, p, None, p),
        "singular frame-0 sub-frame": (b.h, 2, 2, 1.0, p, p, None),
    }
    for what, args in cases.items():
        assert L.arapb200_batch_scene_blur(*args) != 0, what
    assert L.arapb200_batch_scene_blur(b.h, 2, 2, 0.5, p, p, None) == 0   # the same scene at a shorter shutter is fine
    assert L.arapb200_batch_scene_blur(b.h, 2, 2, 0.5, None, None, None) != 0
    L.arapb200_batch_scene_blur(b.h, 2, 1, 0.0, p, None, None)               # replaces the request above
    b.run()
    b.close()
    fresh = lib.Batch(W, H, 5, **KW)
    want = _submit(fresh, sp, A, bg, origin, [1, 3], (3, 0.5))
    fresh.run()
    fresh.close()
    _same(out, want, SCENE_KEYS + ("rgb0", "blur_rgb", "blur_rgb0"))
    _same(out["seq"], want["seq"], ("rgb", "blur_rgb"))
    assert np.array_equal(buf[0], still["rgb"]) and not buf[1:].any()
    assert "blur_rgb" not in no_rgb0
    # the run dropped every request: the next run of the same scenes blurs nothing
    b2 = lib.Batch(W, H, 5, **KW)
    o = _submit(b2, sp, A, bg, origin, [1, 3], None)
    b2.run()
    l0 = b2.launches()
    _submit(b2, sp, A, bg, origin, [1, 3], (3, 0.5))
    b2.run()
    _submit(b2, sp, A, bg, origin, [1, 3], None, out=o)
    b2.run()
    assert b2.launches() == l0
    b2.close()


def test_python_blur_rejection_queues_nothing_and_reuse_drops_stale_keys():
    sp = synth.synth(96, 80, 2, 2, 98)
    A, bg, origin = _moving(sp, 91)
    two = 2 * np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])   # frame 0 at u = 1 extrapolates to 0: singular
    b = lib.Batch(sp.W, sp.H, 2, **KW)
    with pytest.raises(RuntimeError):
        _submit(b, sp, two, bg, origin, None, (2, 1.0))
    b.submit(0, sp.rgb, sp.masks[0], sp.matches)              # the slots are free: the scene was not queued
    b.submit(1, sp.rgb, sp.masks[1], sp.matches)
    b.run()
    out = _submit(b, sp, A, bg, origin, [1, 4], (3, 0.5))
    b.run()
    assert {"rgb0", "blur_rgb0"} <= set(out)
    out = _submit(b, sp, A, bg, origin, [1, 4], (3, 0.5), input_frame=False, out=out)
    b.run()
    b.close()
    assert "rgb0" not in out and "blur_rgb0" not in out and "blur_rgb" in out and "blur_rgb" in out["seq"]
    fresh = lib.Batch(sp.W, sp.H, 2, **KW)
    want = _submit(fresh, sp, A, bg, origin, [1, 4], (3, 0.5), input_frame=False)
    fresh.run()
    fresh.close()
    assert set(out) == set(want)
    _same(out, want, SCENE_KEYS + ("blur_rgb",))
    _same(out["seq"], want["seq"], ("rgb", "blur_rgb"))
