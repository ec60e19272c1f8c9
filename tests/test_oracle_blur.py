"""The CPU restatement of motion blur (tests/blur_oracle.py, DESIGN.md 4.8) against cases that do not use its formulas,
the library's host schedule (lib.blur_schedule) against the restatement's bit for bit, and the rejections of both C
entry points, which happen before any CUDA call.  CPU only."""
import ctypes as C

import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from tests import background_oracle as BO
from tests import blur_oracle as BL

F = np.float32
I2 = BL.I2


def _tr(tx, ty, a=1.0):
    return np.array([[a, 0.0, tx], [0.0, a, ty]])


def _box(images):
    acc = np.sum([im.astype(np.int64) for im in images], axis=0)
    return ((acc + len(images) // 2) // len(images)).astype(np.uint8)


def _shifted(img, fill, dx, dy):
    """img moved by the integer (dx, dy): out[q] = img[q - d] where that is inside, else fill[q]."""
    H, W = img.shape[:2]
    out = fill.copy()
    ys, xs = slice(max(dy, 0), min(H, H + dy)), slice(max(dx, 0), min(W, W + dx))
    out[ys, xs] = img[max(-dy, 0):min(H, H - dy), max(-dx, 0):min(W, W - dx)]
    return out


def _scene(seed, nCont):
    """Two layers of synth's masks with smooth random states X_t = grid + (t + 1) / nCont * field."""
    sp = synth.synth(40, 32, 2, 2, seed)
    rng = np.random.default_rng(seed)
    from oracle import pyoracle as O
    grid = O.grid(sp.W, sp.H)
    states = []
    for _ in sp.masks:
        field = np.repeat(np.repeat(rng.uniform(-3, 3, (5, 6, 2)), 8, 0), 8, 1)[:sp.H, :sp.W].astype(F)
        states.append({t: (grid + F((t + 1) / nCont) * field).astype(F) for t in range(nCont)})
    bg = synth.background(sp.W + 8, sp.H + 8, seed)
    return sp, states, bg


def _clean(sp, states, t, bg, A_hi, origin):
    from oracle import pyoracle as O
    warps = [O.warp(st[t], sp.rgb, m) for st, m in zip(states, sp.masks)]
    cf = BO.coeffs(A_hi)
    return BO.composite([O.flow(st[t]) for st in states], [w[0] for w in warps], [w[1] for w in warps], list(sp.masks),
                        None, bg, cf, origin)["rgb"]


# ------------------------------------------------------------------------------------- the definition's consequences
@pytest.mark.parametrize("S,shutter", [(1, 0.7), (5, 0.0)])
def test_one_sample_or_closed_shutter_is_the_clean_composite(oracle, S, shutter):
    nCont, steps = 5, [1, 4]
    sp, states, bg = _scene(3, nCont)
    A = _tr(1.5, -0.75, 1.02)
    path = synth.motion_path(A, steps, nCont)
    args = (sp.rgb, sp.masks, bg, (4, 4), nCont, steps, A, path, S, shutter)
    assert np.array_equal(BL.blur_image(states, *args, 0), _clean(sp, states, nCont - 1, bg, A, (4, 4)))
    for k, t in enumerate(steps, 1):
        assert np.array_equal(BL.blur_image(states, *args, k), _clean(sp, states, t, bg, path[k - 1], (4, 4)))


def test_still_scene_is_unchanged(oracle):
    from oracle import pyoracle as O
    sp, _, bg = _scene(4, 4)
    still = [{t: O.grid(sp.W, sp.H) for t in range(4)} for _ in sp.masks]
    sharp = BL.render([O.grid(sp.W, sp.H)] * 2, sp.rgb, sp.masks, bg, I2)
    for image in (-1, 0):
        assert np.array_equal(BL.blur_image(still, sp.rgb, sp.masks, bg, (0, 0), 4, None, I2, None, 7, 1.0, image),
                              sharp)


def _translating_layer(W, H, d, nCont):
    from oracle import pyoracle as O
    g = O.grid(W, H)
    return [{t: (g + F(t + 1) * np.array(d, F)).astype(F) for t in range(nCont)}]


@pytest.mark.parametrize("d", [(1, 0), (0, -2), (2, 1)])
def test_rigid_integer_translation_is_the_box_average_of_shifted_copies(oracle, d):
    """One all-object layer moving by d per continuation step; nCont = 4, S = 5, shutter 1: the pair's sub-frames sit on
    states 3, 2, 1, 0 and the grid."""
    W, H, nCont = 36, 28, 4
    rgb = synth.background(W, H, 7)
    bg = synth.background(W, H, 8)
    mask = np.zeros((H, W), np.uint8)
    states = _translating_layer(W, H, d, nCont)
    got = BL.blur_image(states, rgb, [mask], bg, (0, 0), nCont, None, I2, None, 5, 1.0, 0)
    want = _box([_shifted(rgb, bg, s * d[0], s * d[1]) for s in (4, 3, 2, 1, 0)])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("t", [(4, 0), (-8, 4)])
def test_empty_layer_over_a_translating_background_is_the_box_average_of_the_background(oracle, t):
    """The pair motion translates by t; with S = 5 and shutter 1 the sub-frames translate by t, 3t/4, t/2, t/4, 0."""
    W, H, m = 30, 20, 10
    bg = synth.background(W + 2 * m, H + 2 * m, 9)
    mask = np.full((H, W), 255, np.uint8)
    states = _translating_layer(W, H, (1, 1), 4)
    got = BL.blur_image(states, bg[:H, :W], [mask], bg, (m, m), 4, None, _tr(*t), None, 5, 1.0, 0)
    crops = [bg[m - k * t[1] // 4:m - k * t[1] // 4 + H, m - k * t[0] // 4:m - k * t[0] // 4 + W] for k in (4, 3, 2, 1, 0)]
    assert np.array_equal(got, _box(crops))


def test_mean_rounds_half_up(oracle):
    """Columns alternate 0 / 1 and the background moves by one column: every pixel averages a 0 and a 1 and gets 1."""
    W, H = 16, 6
    bg = np.zeros((H, W + 2, 3), np.uint8)
    bg[:, 1::2] = 1
    mask = np.full((H, W), 255, np.uint8)
    states = _translating_layer(W, H, (0, 0), 3)
    got = BL.blur_image(states, bg[:, :W], [mask], bg, (1, 0), 3, None, _tr(1, 0), None, 2, 1.0, 0)
    assert (got == 1).all()


def test_lerp_selects_a_state_exactly_even_next_to_nan_and_inf():
    a = np.array([[[1.25, -3.5]]], F)
    bad = np.array([[[np.nan, np.inf]]], F)
    assert np.array_equal(BL.lerp(a, bad, F(0)), a) and np.array_equal(BL.lerp(bad, a, F(1)), a)
    assert np.isnan(BL.lerp(a, bad, F(0.5))[..., 0]).all()


def test_frame_zero_extrapolates_below_the_grid(oracle):
    nCont, S = 4, 5
    j0, w, _ = BL.schedule(nCont, None, I2, None, S, 1.0, -1)
    assert (j0 == -1).all() and np.array_equal(w, np.array([0, -1, -2, -3, -4], F))
    W, H, d = 36, 28, (1, 1)
    rgb, bg = synth.background(W, H, 10), synth.background(W, H, 11)
    mask = np.zeros((H, W), np.uint8)
    got = BL.blur_image(_translating_layer(W, H, d, nCont), rgb, [mask], bg, (0, 0), nCont, None, I2, None, S, 1.0, -1)
    assert np.array_equal(got, _box([_shifted(rgb, bg, -s, -s) for s in range(S)]))


def _inexact_end():
    """a with a + (1 - a) != 1 and (p, q) with q + (p - q) != p in binary64"""
    rng = np.random.default_rng(0)
    a = next(v for v in rng.uniform(-3, 3, 10000) if v + (1.0 - v) != 1.0)
    p, q = next((p, q) for p, q in rng.uniform(-3, 3, (10000, 2)) if q + (p - q) != p)
    return a, p, q


def test_closed_interval_end_uses_the_previous_motion_exactly():
    a, p, q = _inexact_end()
    A = np.array([[a, 0.0, 3.0], [0.0, 1.0, -2.0]])
    fm = [_tr(p, 0.0), _tr(q, 0.0)]
    for image, steps, prev in ((0, None, I2), (2, [1, 3], fm[0])):
        for smap in (BL.schedule(4, steps, A, fm if steps else None, 3, 1.0, image)[2],
                     lib.blur_schedule(4, steps, A, fm if steps else None, 3, 1.0, image)[2]):
            assert np.array_equal(smap[-1], BO.inverse(prev).astype(F))
    # the sum would not have given them
    assert A[0, 0] + 1.0 * (I2 - A)[0, 0] != 1.0 and q + 1.0 * (p - q) != p


# ------------------------------------------------------------------------------------- the library's host schedule
CASES = [
    (6, None, 0, 2, 1.0), (6, None, 0, 5, 0.3), (6, None, -1, 8, 1.0), (6, [0, 2, 5], 1, 8, 0.3),
    (6, [0, 2, 5], 2, 5, 1.0), (6, [0, 2, 5], 3, 2, 1.0), (6, [0, 2, 5], -1, 5, 0.3), (19, list(range(19)), 7, 2, 1.0),
    (19, list(range(19)), 19, 64, 0.77), (1, None, 0, 3, 1.0), (3, [2], -1, 1, 0.5), (5, [1, 4], 0, 3, 0.0),
]


@pytest.mark.parametrize("nCont,steps,image,S,shutter", CASES)
def test_library_schedule_equals_the_restatement(nCont, steps, image, S, shutter):
    A, _ = synth.background_motion(854, 480, nCont + S)
    fm = synth.motion_path(A, steps, nCont) if steps else None
    got = lib.blur_schedule(nCont, steps, A, fm, S, shutter, image)
    want = BL.schedule(nCont, steps, A, fm, S, shutter, image)
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w)
    assert got[0].min() >= -1 and got[0].max() <= max(nCont - 2, -1)


def test_schedule_rejections_need_no_gpu():
    L = lib.load()
    L.arapb200_blur_schedule.argtypes = lib.BLUR_SCHEDULE_ARGTYPES
    A = np.ascontiguousarray(_tr(1.0, 2.0, 1.01))
    steps = np.array([1, 3], np.int32)
    fm = np.ascontiguousarray(np.stack(synth.motion_path(A, [1, 3], 5)))
    o_s, o_w, o_m = np.zeros(64, np.int32), np.zeros(64, np.float32), np.zeros(64 * 6, np.float32)
    good = dict(nCont=5, K=2, steps=steps.ctypes.data, motion=A.ctypes.data, fm=fm.ctypes.data, S=4, shutter=0.5,
                image=1, o_s=o_s.ctypes.data, o_w=o_w.ctypes.data, o_m=o_m.ctypes.data)

    def call(**kw):
        a = {**good, **kw}
        return L.arapb200_blur_schedule(a["nCont"], a["K"], a["steps"], a["motion"], a["fm"], a["S"], a["shutter"],
                                        a["image"], a["o_s"], a["o_w"], a["o_m"])

    assert call() == 0
    singular, nan = np.zeros((2, 3)), A.copy()
    nan[1, 1] = np.nan
    flip = np.ascontiguousarray(2 * I2)   # frame 0 at u = 1 extrapolates to 2I - A_1 = 0: singular
    bad_steps, past = np.array([3, 1], np.int32), np.array([1, 5], np.int32)
    cases = {
        "nCont 0": dict(nCont=0), "negative frames": dict(K=-1), "null motion": dict(motion=None),
        "frames without steps": dict(steps=None), "frames without motions": dict(fm=None),
        "steps decreasing": dict(steps=bad_steps.ctypes.data), "step past nCont": dict(steps=past.ctypes.data),
        "S 0": dict(S=0), "S 65": dict(S=65), "shutter nan": dict(shutter=float("nan")), "shutter -0.1": dict(shutter=-0.1),
        "shutter 1.5": dict(shutter=1.5), "image -2": dict(image=-2), "image 3": dict(image=3),
        "null out_state": dict(o_s=None), "null out_w": dict(o_w=None), "null out_smap": dict(o_m=None),
        "singular motion": dict(K=0, motion=singular.ctypes.data, image=0),
        "nan motion": dict(K=0, motion=nan.ctypes.data, image=0),
        "frame 0 extrapolates to a singular motion": dict(K=0, motion=flip.ctypes.data, image=-1, S=2, shutter=1.0),
    }
    o_s[:], o_w[:], o_m[:] = -7, -7, -7
    before = (o_s.copy(), o_w.copy(), o_m.copy())
    for what, change in cases.items():
        assert call(**change) != 0, what
        assert all(np.array_equal(x, y) for x, y in zip((o_s, o_w, o_m), before)), what
    # the same flip without extrapolation is fine: the pair interpolates between 2I and I
    assert call(K=0, motion=flip.ctypes.data, image=0, S=2, shutter=1.0) == 0
    with pytest.raises(RuntimeError):
        lib.blur_schedule(5, None, flip, None, 2, 1.0, -1)


def test_scene_blur_rejects_a_null_batch_without_a_gpu():
    L = lib.load()
    L.arapb200_batch_scene_blur.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 3
    buf = np.zeros(12, np.uint8)
    assert L.arapb200_batch_scene_blur(None, 0, 4, 0.5, buf.ctypes.data, None, None) != 0
