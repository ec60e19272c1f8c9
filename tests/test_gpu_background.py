"""The composite over a moving background on the GPU (DESIGN.md 4.5): the analytic cases of test_oracle_background.py
through the library, the binary32 maps against their binary64 derivation, then the library against the restatement
(tests/background_oracle.py, fed the library's own maps) bit for bit -- random affines and layers, Batch outputs of C1 and
C2, and composite_seq on a C2 frame sequence."""
import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from oracle import pycomposite as PC
from tests import background_cases as BC
from tests import background_oracle as BO

pytestmark = pytest.mark.gpu

KEYS = ("flow", "rgb", "mask", "bflow", "occ")


def _same(a, b, keys=KEYS):
    for k in keys:   # NaN layer flows pass through to the output
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


def _vs_oracle(out, flows, rgbs, masks, srcs, bflows, bg, origin=(0, 0), shape=None):
    _same(out, BO.composite(flows, rgbs, masks, srcs, bflows, bg, out["coeffs"], origin, shape))


# ------------------------------------------------------------------------------------- analytic cases
@pytest.mark.parametrize("n", [1, 2])
def test_identity_is_flatten_ex_with_add_bg(n):
    BC.check_identity_is_flatten(lib.composite, lib.warp_ex, n)


def test_identity_without_layers_is_the_crop():
    BC.check_identity_no_layers(lib.composite)


@pytest.mark.parametrize("t", BC.BG_SHIFTS)
def test_integer_background_translation(t):
    BC.check_integer_translation(lib.composite, t)


def test_half_pixel_shift_rounds_to_nearest_even():
    BC.check_half_pixel(lib.composite)


def test_half_scale_pins_the_strict_bound():
    BC.check_half_scale(lib.composite)


@pytest.mark.parametrize("deg,scale", BC.ZOOMS)
def test_rotation_and_zoom_in(deg, scale):
    BC.check_rotation_zoom(lib.composite, deg, scale)


def test_moving_object_over_moving_background():
    BC.check_object_over_background(lib.composite, lib.warp_ex)


@pytest.mark.parametrize("t", BC.CLAMP_SHIFTS)
def test_clamping_replicates_the_edge(t):
    BC.check_clamping(lib.composite, t)


def test_same_motion_is_a_still_background():
    BC.check_same_motion_is_still(lib.composite)


def test_chord_path_composes_to_the_pair():
    BC.check_chord_path_composes(lib.composite)


# ------------------------------------------------------------------------------------- bit for bit against the oracle
def _random_affine(rng, kind, W, H):
    """A random linear map of the given kind about the frame centre, plus a shift of up to 30 px."""
    a = rng.uniform(-np.pi, np.pi)
    R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
    if kind == "reflection":
        R = R @ np.diag([-1.0, 1.0]) * rng.uniform(0.7, 1.4)
    elif kind == "near_singular":
        R = R @ np.diag([rng.uniform(1e-4, 1e-3), rng.uniform(0.5, 2.0)])
    elif kind == "shear":
        R = R @ np.array([[1.0, rng.uniform(-0.8, 0.8)], [0.0, rng.uniform(0.6, 1.6)]])
    c = np.array([(W - 1) / 2.0, (H - 1) / 2.0])
    return np.hstack([R, (c - R @ c + rng.uniform(-30, 30, 2))[:, None]])


def _random_layers(rng, W, H, n):
    """n layers of random content: flows and backward flows with NaN and inf, random warped and source masks."""
    flows, rgbs, masks, srcs, bflows = [], [], [], [], []
    for _ in range(n):
        f = (rng.standard_normal((H, W, 2)) * 4).astype(np.float32)
        b = (rng.standard_normal((H, W, 2)) * 1.5).astype(np.float32)
        for a in (f, b):
            a[rng.random((H, W)) < 0.02] = np.nan
            a[rng.random((H, W)) < 0.02] = np.inf
            a[rng.random((H, W)) < 0.02] = -np.inf
        flows.append(f)
        bflows.append(b)
        rgbs.append(rng.integers(0, 256, (H, W, 3), dtype=np.uint8))
        masks.append(np.where(rng.random((H, W)) < 0.3, 255, 0).astype(np.uint8))
        srcs.append(np.where(rng.random((H, W)) < 0.3, 0, 255).astype(np.uint8))
    return flows, rgbs, masks, srcs, bflows


CASES = [(3, 2, 0, "rotation", 0), (3, 2, 2, "reflection", 1), (97, 61, 1, "near_singular", 2),
         (97, 61, 3, "shear", 3), (200, 120, 0, "reflection", 4), (200, 120, 2, "rotation", 5),
         (854, 480, 4, "rotation", 6), (854, 480, 1, "near_singular", 7)]


@pytest.mark.parametrize("W,H,n,kind,seed", CASES)
def test_random_affines_and_layers_vs_oracle(W, H, n, kind, seed):
    rng = np.random.default_rng(seed)
    args = _random_layers(rng, W, H, n)
    A_to, A_from = _random_affine(rng, kind, W, H), _random_affine(rng, "rotation", W, H)
    bg = rng.integers(0, 256, (H + 13, W + 7, 3), dtype=np.uint8)
    origin = (int(rng.integers(-5, 10)), int(rng.integers(-5, 10)))
    for mf in (None, A_from):
        out = lib.composite(*args, bg, A_to, motion_from=mf, origin=origin, shape=(H, W))
        assert np.array_equal(out["coeffs"], BO.coeffs(A_to, mf))    # the binary64 derivation, rounded once
        _vs_oracle(out, *args, bg, origin, (H, W))
        plain = lib.composite(*args, bg, A_to, motion_from=mf, origin=origin, shape=(H, W), extras=False)
        _same(plain, out, ("flow", "rgb", "mask", "coeffs"))
        assert "occ" not in plain
        if W * H > 1000 and kind != "near_singular":   # a near-singular map leaves almost nothing visible
            assert 0 < (out["occ"] == 255).sum() < W * H


# ------------------------------------------------------------------------------------- Batch outputs
KW = dict(nCont=2, nGN=2, nPCG=30)


def test_batch_c1_over_a_synth_background_motion():
    sp = synth.config("C1")
    b = lib.Batch(sp.W, sp.H, 1, **KW)
    o = b.submit(0, sp.rgb, sp.masks[0], sp.matches, extras=True)
    b.run()
    b.close()
    A, m = synth.background_motion(sp.W, sp.H, 1)
    bg = synth.background(sp.W + 2 * m, sp.H + 2 * m, 1)
    args = ([o["flow"]], [o["rgb"]], [o["mask"]], [sp.masks[0]], [o["bflow"]])
    out = lib.composite(*args, bg, A, origin=(m, m))
    _vs_oracle(out, *args, bg, (m, m))
    front = o["mask"] != 0
    obj = sp.masks[0] == 0
    assert np.array_equal(out["rgb"][front], o["rgb"][front]) and (out["mask"][front] == 255).all()
    assert np.array_equal(out["flow"][obj], o["flow"][obj]) and np.array_equal(out["bflow"][front], o["bflow"][front])
    xx, yy = BC.grid64(sp.W, sp.H)
    fx, fy = BC.affine_np(A, xx, yy)
    assert np.abs(out["flow"][~obj][:, 0] - (fx - xx)[~obj]).max() < 1e-3
    assert np.abs(out["flow"][~obj][:, 1] - (fy - yy)[~obj]).max() < 1e-3
    s = BO.apply(out["coeffs"][2], sp.W, sp.H) + np.float32(m)     # the sample points the kernel used
    assert (s >= 0).all() and (s[..., 0] <= bg.shape[1] - 1).all() and (s[..., 1] <= bg.shape[0] - 1).all()
    assert (out["occ"][~obj] == 255).any() and (out["occ"][~obj] == 0).any()


def _c2_batch(frames=None, nCont=2):
    sp = synth.config("C2")
    b = lib.Batch(sp.W, sp.H, 4, nCont=nCont, nGN=2, nPCG=30)
    outs = [b.submit(s, sp.rgb, sp.masks[s], sp.matches, extras=True, frames=frames) for s in range(4)]
    b.run()
    b.close()
    return sp, outs


def test_batch_c2_four_segments():
    sp, outs = _c2_batch()
    A, m = synth.background_motion(sp.W, sp.H, 2)
    bg = synth.background(sp.W + 2 * m, sp.H + 2 * m, 2)
    args = ([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs], list(sp.masks),
            [o["bflow"] for o in outs])
    out = lib.composite(*args, bg, A, origin=(m, m))
    _vs_oracle(out, *args, bg, (m, m))
    obj = np.any([s == 0 for s in sp.masks], axis=0)
    assert (out["occ"][obj] == 255).any() and (out["occ"][~obj] == 255).any() and (out["occ"] == 0).any()


def test_composite_seq_c2_frames():
    steps, nCont = [0, 2, 5], 6
    sp, outs = _c2_batch(frames=steps, nCont=nCont)
    seqs = [o["seq"] for o in outs]
    A, m = synth.background_motion(sp.W, sp.H, 3)
    bg = synth.background(sp.W + 2 * m, sp.H + 2 * m, 3)
    crop = bg[m:m + sp.H, m:m + sp.W]
    # identity path: the layer recipe of DESIGN.md 4.4 per frame, plus the background crop
    still = lib.composite_seq(seqs, sp.masks, bg, [BC.I2] * len(steps), origin=(m, m))
    for k in range(len(steps)):
        src = list(sp.masks) if k == 0 else [255 - q["mask"][k - 1] for q in seqs]
        flat = lib.flatten_ex([q["flow"][k] for q in seqs], [q["rgb"][k] for q in seqs], [q["mask"][k] for q in seqs],
                              src, [q["bflow"][k] for q in seqs])
        flat["rgb"] = PC.add_bg(flat["rgb"], flat["mask"], crop)
        _same({key: still[key][k] for key in KEYS}, flat)
    # the chord path: every frame against the restatement with the maps the library used
    path = synth.motion_path(A, steps, nCont)
    seq = lib.composite_seq(seqs, sp.masks, bg, path, origin=(m, m))
    for k in range(len(steps)):
        src = list(sp.masks) if k == 0 else [255 - q["mask"][k - 1] for q in seqs]
        assert np.array_equal(seq["coeffs"][k], BO.coeffs(path[k], None if k == 0 else path[k - 1]))
        ref = BO.composite([q["flow"][k] for q in seqs], [q["rgb"][k] for q in seqs], [q["mask"][k] for q in seqs],
                           src, [q["bflow"][k] for q in seqs], bg, seq["coeffs"][k], (m, m))
        _same({key: seq[key][k] for key in KEYS}, ref)
