"""Scenes in the batch (DESIGN.md 4.6): Batch.submit_scene against the host path it replaces -- Batch.submit(...,
extras=True, frames=...) per segment, then lib.flatten_ex / lib.composite / lib.composite_seq, which are pinned against
their numpy restatements elsewhere.  Every comparison is bit for bit."""
import ctypes as C

import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from oracle import pycomposite as PC

pytestmark = pytest.mark.gpu

KEYS = ("flow", "rgb", "mask", "bflow", "occ")
KW = dict(nCont=6, nGN=2, nPCG=30)
I2 = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def _same(a, b, keys=KEYS):
    for k in keys:
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k], b[k]), k


def _scene(name, index=0):
    sp = synth.config(name, index)
    return sp, [sp.matches] * len(sp.masks)


def _host(b, rgb, masks, matches, bg, motion, origin=(0, 0), frames=None, path=None, slot=0):
    """The host path: one submit per segment, run, then the library composite."""
    outs = [b.submit(slot + s, rgb, m, mt, extras=True, frames=frames) for s, (m, mt) in enumerate(zip(masks, matches))]
    b.run()
    return _compose(outs, masks, bg, motion, origin, path)


def _compose(outs, masks, bg, motion, origin=(0, 0), path=None):
    args = ([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs], list(masks),
            [o["bflow"] for o in outs])
    res = lib.composite(*args, bg, motion, origin=origin)
    res["costs"] = np.stack([o["costs"] for o in outs])
    if path is not None:
        res["seq"] = lib.composite_seq([o["seq"] for o in outs], masks, bg, path, origin=origin)
    return res


def _check(got, want, frames=False):
    _same(got, want)
    assert np.array_equal(got["costs"], want["costs"])
    if frames:
        _same(got["seq"], want["seq"])
    else:
        assert "seq" not in got


def _moving(sp, seed):
    A, m = synth.background_motion(sp.W, sp.H, seed)
    return A, synth.background(sp.W + 2 * m, sp.H + 2 * m, seed), (m, m)


# ------------------------------------------------------------------------------------- 1, 2, 4: the pair and frame 0
@pytest.mark.parametrize("name", ["C1", "C2"])
def test_still_background_is_flatten_and_composite(name):
    sp, matches = _scene(name)
    n = len(sp.masks)
    bg = synth.background(sp.W, sp.H, 11)
    b = lib.Batch(sp.W, sp.H, n, **KW)
    outs = [b.submit(s, sp.rgb, sp.masks[s], matches[s], extras=True) for s in range(n)]
    b.run()
    want = _compose(outs, sp.masks, bg, I2)
    flat = lib.flatten_ex([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs],
                          list(sp.masks), [o["bflow"] for o in outs])
    flat["rgb"] = PC.add_bg(flat["rgb"], flat["mask"], bg)
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, I2)
    b.run()
    b.close()
    _check(got, want)
    _same(got, flat)


@pytest.mark.parametrize("name,seed", [("C1", 21), ("C2", 22)])
def test_moving_background_and_input_frame(name, seed):
    sp, matches = _scene(name)
    A, bg, origin = _moving(sp, seed)
    b = lib.Batch(sp.W, sp.H, len(sp.masks), **KW)
    want = _host(b, sp.rgb, sp.masks, matches, bg, A, origin)
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, input_frame=True)
    b.run()
    b.close()
    _check(got, want)
    obj = np.any([m == 0 for m in sp.masks], axis=0)
    ox, oy = origin
    assert np.array_equal(got["rgb0"], np.where(obj[..., None], sp.rgb, bg[oy:oy + sp.H, ox:ox + sp.W]))
    assert (got["flow"][~obj] != 0).any() and (got["occ"] == 255).any() and (got["occ"] == 0).any()


# ------------------------------------------------------------------------------------- 3: frames
def test_frames_c2_against_composite_seq():
    sp, matches = _scene("C2")
    A, bg, origin = _moving(sp, 23)
    steps = [0, 2, 5]
    path = synth.motion_path(A, steps, KW["nCont"])
    b = lib.Batch(sp.W, sp.H, 4, **KW)
    want = _host(b, sp.rgb, sp.masks, matches, bg, A, origin, steps, path)
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path)
    b.run()
    b.close()
    _check(got, want, frames=True)
    for k in ("rgb", "mask"):   # t_K = nCont - 1 and A_K = A: the last frame is the pair
        assert np.array_equal(got["seq"][k][-1], got[k]), k


def test_frames_c2_full_schedule_all_frames():
    sp, matches = _scene("C2")
    A, bg, origin = _moving(sp, 24)
    nCont, nGN, nPCG = 19, 8, 400
    steps = list(range(nCont))
    path = synth.motion_path(A, steps, nCont)
    b = lib.Batch(sp.W, sp.H, 4, nCont, nGN, nPCG)
    want = _host(b, sp.rgb, sp.masks, matches, bg, A, origin, steps, path)
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path)
    b.run()
    assert b.launch_info()["grid"][1] == 1 and b.resident_count() == 4
    b.close()
    _check(got, want, frames=True)
    for k in ("rgb", "mask"):
        assert np.array_equal(got["seq"][k][-1], got[k]), k


# ------------------------------------------------------------------------------------- 5: a mixed run
def test_three_c2_scenes_and_plain_problems_in_one_run():
    scenes = [_scene("C2", i) for i in range(3)]
    moves = [_moving(sp, 30 + i) for i, (sp, _) in enumerate(scenes)]
    plain = [synth.config("C2", 3 + i) for i in range(2)]
    steps = [1, 4]
    paths = [synth.motion_path(A, steps, KW["nCont"]) for A, _, _ in moves]
    # alone: each scene in its own batch; the plain problems in a run without scenes
    alone = []
    for i, ((sp, mt), (A, bg, org)) in enumerate(zip(scenes, moves)):
        b1 = lib.Batch(854, 480, 4, **KW)
        fr = dict(frames=steps, frame_motions=paths[i]) if i == 1 else {}
        alone.append(b1.submit_scene(0, sp.rgb, sp.masks, mt, bg, A, origin=org, input_frame=i == 2, **fr))
        b1.run()
        b1.close()
    b0 = lib.Batch(854, 480, 2, **KW)
    ref = [b0.submit(j, p.rgb, p.masks[j], p.matches, extras=j == 1) for j, p in enumerate(plain)]
    b0.run()
    b0.close()
    # together: 12 scene problems, then two plain ones
    b = lib.Batch(854, 480, 14, **KW)
    got = []
    for i, ((sp, mt), (A, bg, org)) in enumerate(zip(scenes, moves)):
        fr = dict(frames=steps, frame_motions=paths[i]) if i == 1 else {}
        got.append(b.submit_scene(4 * i, sp.rgb, sp.masks, mt, bg, A, origin=org, input_frame=i == 2, **fr))
    outs = [b.submit(12 + j, p.rgb, p.masks[j], p.matches, extras=j == 1) for j, p in enumerate(plain)]
    b.run()
    info = b.launch_info()
    assert info["grid"][1] == 1 and b.resident_count() == 14, info
    b.close()
    for i, (g, a) in enumerate(zip(got, alone)):
        _check(g, a, frames=i == 1)
        if i == 2:
            assert np.array_equal(g["rgb0"], a["rgb0"])
    for j, (o, r) in enumerate(zip(outs, ref)):
        _same(o, r, ("flow", "rgb", "mask", "costs") + (("bflow", "occ") if j == 1 else ()))


# ------------------------------------------------------------------------------------- 6: solver paths
@pytest.mark.parametrize("kind", ["stream", "lm", "resident_small"])
def test_solver_paths(kind):
    sp = synth.synth(160, 120, 2, 2, 90) if kind != "resident_small" else synth.synth(96, 80, 2, 2, 91)
    matches = [sp.matches] * 2
    A, bg, origin = _moving(sp, 40)
    steps = [0, 3, 5]
    path = synth.motion_path(A, steps, KW["nCont"])
    b = lib.Batch(sp.W, sp.H, 2, backend=lib.BACKEND_STREAM if kind == "stream" else lib.BACKEND_AUTO, **KW)
    if kind == "lm":
        b.set_option("lm", 1)
    want = _host(b, sp.rgb, sp.masks, matches, bg, A, origin, steps, path)
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path)
    b.run()
    if kind == "resident_small":
        assert b.resident_count() == 2
    else:
        assert b.resident_count() == 0
    b.close()
    _check(got, want, frames=True)


# ------------------------------------------------------------------------------------- 7: buffer reuse
def test_one_batch_reuses_its_buffers():
    kw = dict(nCont=19, nGN=1, nPCG=10)
    small = synth.synth(160, 120, 2, 2, 95)
    big = synth.synth(200, 150, 3, 2, 96)
    b = lib.Batch(200, 150, 3, **kw)
    out = None
    for sp, K, seed in ((small, 19, 50), (small, 4, 51), (small, 0, 52), (big, 19, 53)):
        n = len(sp.masks)
        matches = [sp.matches] * n
        A, bg, origin = _moving(sp, seed)
        steps = list(range(19))[-K:] if K else None
        path = synth.motion_path(A, steps, kw["nCont"]) if K else None
        fresh = lib.Batch(200, 150, 3, **kw)
        want = _host(fresh, sp.rgb, sp.masks, matches, bg, A, origin, steps, path)
        fresh.close()
        out = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path,
                             input_frame=K == 4, out=out)
        b.run()
        _check(out, want, frames=bool(K))
        assert ("rgb0" in out) == (K == 4)
    b.close()


def test_ordinary_submits_after_a_scene_are_ordinary():
    """A slot that was a scene layer in one run is an ordinary problem in the next: same outputs, copies and launches
    as in a batch that never ran a scene."""
    sp = synth.synth(160, 120, 3, 2, 98)
    A, bg, origin = _moving(sp, 61)
    b = lib.Batch(sp.W, sp.H, 3, **KW)
    b.submit_scene(0, sp.rgb, sp.masks, [sp.matches] * 3, bg, A, origin=origin, frames=[1, 5],
                   frame_motions=synth.motion_path(A, [1, 5], KW["nCont"]))
    b.run()
    kinds = [dict(), dict(extras=True), dict(frames=[2, 5])]
    got = [b.submit(s, sp.rgb, sp.masks[s], sp.matches, **k) for s, k in enumerate(kinds)]
    b.run()
    fresh = lib.Batch(sp.W, sp.H, 3, **KW)
    want = [fresh.submit(s, sp.rgb, sp.masks[s], sp.matches, **k) for s, k in enumerate(kinds)]
    fresh.run()
    assert b.launches() == fresh.launches()
    b.close()
    fresh.close()
    for g, w, k in zip(got, want, kinds):
        assert set(g) == set(w)
        _same(g, w, ("flow", "rgb", "mask", "costs") + (("bflow", "occ") if "extras" in k else ()))
        if "frames" in k:
            _same(g["seq"], w["seq"], lib.SEQ_KEYS)


# ------------------------------------------------------------------------------------- 8: rejections
def _call(b, slot, n, W, H, rgb, masks, matches, counts, bg, origin, motion, K, steps, fm, outs):
    L = b.L
    L.arapb200_batch_submit_scene.argtypes = ([C.c_void_p] + [C.c_int] * 4 + [C.c_void_p] * 4 + [C.c_int] * 2 +
                                              [C.c_void_p] + [C.c_int] * 2 + [C.c_void_p, C.c_int] + [C.c_void_p] * 14)
    return L.arapb200_batch_submit_scene(b.h, slot, n, W, H, rgb, masks, matches, counts, bg.shape[1], bg.shape[0],
                                         bg.ctypes.data, origin[0], origin[1], motion, K, steps, fm, *outs)


def test_rejections_queue_nothing_and_leave_the_batch_usable():
    sp = synth.synth(96, 80, 2, 2, 97)
    W, H, n = sp.W, sp.H, 2
    A, bg, origin = _moving(sp, 60)
    matches = [sp.matches] * n
    steps = [1, 3]
    path = np.ascontiguousarray(synth.motion_path(A, steps, KW["nCont"]), np.float64)
    b = lib.Batch(W, H, 3, **KW)
    rgb = np.ascontiguousarray(sp.rgb)
    mk = [np.ascontiguousarray(m) for m in sp.masks]
    mt = [np.ascontiguousarray(m, np.int32) for m in matches]
    P = C.c_void_p * n
    masks_p, matches_p = P(*[m.ctypes.data for m in mk]), P(*[m.ctypes.data for m in mt])
    counts = (C.c_int * n)(*[len(m) for m in mt])
    A64 = np.ascontiguousarray(A, np.float64)
    st = np.array(steps, np.int32)
    bufs = dict(flow=np.zeros((H, W, 2), np.float32), rgb=np.zeros((H, W, 3), np.uint8), mask=np.zeros((H, W), np.uint8),
                srgb=np.zeros((2, H, W, 3), np.uint8), smask=np.zeros((2, H, W), np.uint8),
                sflow=np.zeros((2, H, W, 2), np.float32))
    outs = [bufs["flow"].ctypes.data, bufs["rgb"].ctypes.data, bufs["mask"].ctypes.data, None, None, None, None,
            bufs["srgb"].ctypes.data, bufs["smask"].ctypes.data, None, None, None]
    good = dict(slot=0, n=n, W=W, H=H, rgb=rgb.ctypes.data, masks=masks_p, matches=matches_p, counts=counts, bg=bg,
                origin=origin, motion=A64.ctypes.data, K=2, steps=st.ctypes.data, fm=path.ctypes.data, outs=outs)

    def with_outs(**o):
        names = ("flow", "rgb", "mask", "bflow", "occ", "rgb0", "costs", "srgb", "smask", "sflow", "sbflow", "socc")
        return [o.get(k, v) for k, v in zip(names, outs)]

    nan = A64.copy()
    nan[0, 2] = np.nan
    singular = np.zeros((2, 3))
    bad_path = path.copy()
    bad_path[1, 0, :2] = 0.0
    null_mask = P(mk[0].ctypes.data, None)
    null_matches = P(mt[0].ctypes.data, None)
    neg = (C.c_int * n)(len(mt[0]), -1)
    repeated, past = np.array([3, 3], np.int32), np.array([1, 6], np.int32)
    cases = {
        "n_layers 0": dict(n=0), "n_layers 33": dict(n=33), "slot -1": dict(slot=-1), "slots past the batch": dict(slot=2),
        "W 0": dict(W=0), "too large": dict(W=W + 1), "null rgb": dict(rgb=None), "null masks": dict(masks=None),
        "null mask entry": dict(masks=null_mask), "null matches": dict(matches=None),
        "null match entry": dict(matches=null_matches), "negative match count": dict(counts=neg),
        "null counts": dict(counts=None), "empty background": dict(bg=np.zeros((0, 4, 3), np.uint8)),
        "null motion": dict(motion=None), "nan motion": dict(motion=nan.ctypes.data),
        "singular motion": dict(motion=singular.ctypes.data), "singular frame motion": dict(fm=bad_path.ctypes.data),
        "null out_flow": dict(outs=with_outs(flow=None)), "null out_rgb": dict(outs=with_outs(rgb=None)),
        "null out_mask": dict(outs=with_outs(mask=None)), "negative frames": dict(K=-1),
        "outputs without frames": dict(K=0), "frames without steps": dict(steps=None),
        "frames without motions": dict(fm=None), "frames without seq_rgb": dict(outs=with_outs(srgb=None)),
        "frames without seq_mask": dict(outs=with_outs(smask=None)),
        "steps not increasing": dict(steps=repeated.ctypes.data), "step past nCont": dict(steps=past.ctypes.data),
    }
    for what, change in cases.items():
        assert _call(b, **{**good, **change}) != 0, what
    # a queued scene owns its slots until the next run: another scene over them, or an ordinary submit, is refused
    assert _call(b, **good) == 0
    assert _call(b, **{**good, "slot": 1}) != 0
    with pytest.raises(RuntimeError):
        b.submit(1, sp.rgb, sp.masks[1], sp.matches)
    b.submit(2, sp.rgb, sp.masks[0], sp.matches)   # a slot outside the scene is free
    b.run()
    # after all that, a valid run equals a fresh batch's
    got = b.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path)
    b.run()
    b.close()
    fresh = lib.Batch(W, H, 3, **KW)
    want = fresh.submit_scene(0, sp.rgb, sp.masks, matches, bg, A, origin=origin, frames=steps, frame_motions=path)
    fresh.run()
    fresh.close()
    _check(got, want, frames=True)
    _same(got, {k: bufs[k] for k in ("flow", "rgb", "mask")}, ("flow", "rgb", "mask"))
