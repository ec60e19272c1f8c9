"""Analytic cases of the backward flow and the occlusion of frame 1 (DESIGN.md 4.3), shared by the oracle tests and the
GPU tests.  Every expectation here comes from the geometry of the case, not from the formulas the oracle or the kernels
evaluate; every comparison is exact except the rotation's, whose bound is derived where it is asserted."""
import numpy as np

from tests import helpers


def grid(W, H):
    yy, xx = np.mgrid[0:H, 0:W]
    return np.stack([xx, yy], -1).astype(np.float32)


def rgb_for(W, H, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def cov(mask):
    """Pixels that are a corner of a quad whose four corners are on the object: what the rasteriser draws at rest."""
    act = mask == 0
    H, W = act.shape
    quad = act[:-1, :-1] & act[1:, :-1] & act[:-1, 1:] & act[1:, 1:]
    c = np.zeros_like(act)
    for dy in (0, 1):
        for dx in (0, 1):
            c[dy:H - 1 + dy, dx:W - 1 + dx] |= quad
    return c


def shift(a, t, fill=False):
    """out[p + t] = a[p] (integer t = (tx, ty)); pixels shifted in from outside the frame get `fill`."""
    tx, ty = t
    H, W = a.shape[:2]
    out = np.full_like(a, fill)
    ys, yd = (slice(0, H - ty), slice(ty, H)) if ty >= 0 else (slice(-ty, H), slice(0, H + ty))
    xs, xd = (slice(0, W - tx), slice(tx, W)) if tx >= 0 else (slice(-tx, W), slice(0, W + tx))
    out[yd, xd] = a[ys, xs]
    return out


def in_frame_after(W, H, t):
    """p + t inside the frame, per frame-1 pixel p."""
    g = grid(W, H).astype(np.int64)
    x, y = g[..., 0] + t[0], g[..., 1] + t[1]
    return (x >= 0) & (x < W) & (y >= 0) & (y < H)


W_T, H_T = 150, 97
TRANSLATION_MASKS = {
    "ellipse": lambda: helpers._as_mask(helpers.ellipse(W_T, H_T, 70, 45, 40, 30)),
    "border": lambda: helpers.mask_border(W_T, H_T, 3, "left"),
    "holes": lambda: helpers.mask_holes(W_T, H_T, 4),
    "lines_pixels": lambda: np.minimum(helpers.mask_lines(W_T, H_T, 5), helpers.mask_pixels(W_T, H_T, 6)),
}
SHIFTS = [(3, -2), (-7, 5), (60, 0)]   # the last one moves a large part of every object out of the frame


def check_translation(out, mask, t):
    """Integer translation by t: out is a warp_ex result dict for flow = t everywhere."""
    H, W = mask.shape
    c = cov(mask)
    landed = shift(c, t)
    assert np.array_equal(out["mask"] == 255, landed)
    exp_b = np.zeros((H, W, 2), np.float32)
    exp_b[landed] = (-t[0], -t[1])
    assert np.array_equal(out["bflow"], exp_b)
    obj = mask == 0
    occluded = out["occ"] == 255
    assert set(np.unique(out["occ"])) <= {0, 255}
    assert np.array_equal(occluded[obj], (~c | ~in_frame_after(W, H, t))[obj])
    assert np.array_equal(occluded[~obj], landed[~obj])   # background: occluded iff cov(p - t)


def check_identity(out, mask):
    c = cov(mask)
    assert (out["occ"][c] == 0).all()
    assert (out["occ"][(mask == 0) & ~c] == 255).all()
    assert not out["bflow"].any()


# ---- small rigid rotation --------------------------------------------------------------------------------------------
W_R = H_R = 128
ROT_DEG = 3.0


def rotation_case():
    """3 degrees about the centre of a 128 x 128 frame; the object (an ellipse) stays well inside the frame."""
    mask = helpers._as_mask(helpers.ellipse(W_R, H_R, 63.5, 63.5, 40, 30))
    a = np.deg2rad(ROT_DEG)
    c = (W_R - 1) / 2.0
    g = grid(W_R, H_R).astype(np.float64) - c
    pos = np.stack([np.cos(a) * g[..., 0] - np.sin(a) * g[..., 1], np.sin(a) * g[..., 0] + np.cos(a) * g[..., 1]], -1) + c
    return mask, pos.astype(np.float32)


def check_rotation(out, mask):
    a = np.deg2rad(ROT_DEG)
    c = (W_R - 1) / 2.0
    # every object pixel at least 2 px (Chebyshev) from the mask edge
    obj = mask == 0
    inner = obj.copy()
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            inner &= shift(obj, (dx, dy), fill=False)
    assert inner.sum() > 2000
    assert (out["occ"][inner] == 0).all()
    # analytic inverse rotation of every covered frame-2 pixel
    covd = out["mask"] == 255
    q = grid(W_R, H_R).astype(np.float64) - c
    src = np.stack([np.cos(a) * q[..., 0] + np.sin(a) * q[..., 1], -np.sin(a) * q[..., 0] + np.cos(a) * q[..., 1]], -1)
    err = np.abs(out["bflow"].astype(np.float64) - (src - q))[covd]
    # The mesh map is affine on every triangle, so barycentric interpolation of the undeformed vertices inverts it exactly
    # up to rounding: the positions are float32 below 128, off by at most half an ulp (< 8e-6 px), and the float32
    # barycentric arithmetic adds a few ulps of 128 (~1e-5 px).  1e-3 px leaves two orders of magnitude of margin.
    assert err.max() < 1e-3
    assert not out["bflow"][~covd].any()


# ---- 2:1 horizontal compression --------------------------------------------------------------------------------------
W_C, H_C = 41, 9


def compression_case():
    """X = (px / 2, py) on an all-object frame."""
    pos = grid(W_C, H_C)
    pos[..., 0] *= np.float32(0.5)
    return np.zeros((H_C, W_C), np.uint8), pos


def check_compression(out):
    px = grid(W_C, H_C)[..., 0].astype(np.int64)
    # even px lands on the vertex whose source is p (error 0): visible.  Odd px sits at k + 0.5, rounds to q = (px + 1)/2,
    # whose source is px + 1: error exactly 1, so the strict < 1 makes p occluded.
    assert np.array_equal(out["occ"] == 255, px % 2 == 1)
    covd = px <= (W_C - 1) // 2
    assert np.array_equal(out["mask"] == 255, covd)
    exp = np.zeros((H_C, W_C, 2), np.float32)
    exp[..., 0] = np.where(covd, px, 0)        # source 2 qx, minus qx
    assert np.array_equal(out["bflow"], exp)


# ---- two layers, integer translations --------------------------------------------------------------------------------
W_L, H_L = 120, 80
T_LAYERS = [(6, 2), (-9, 1)]


def layer_masks():
    """Segment 0: a wide ellipse on the left; segment 1: a disc on the right that moves over segment 0's right part."""
    m0 = helpers.ellipse(W_L, H_L, 40, 40, 28, 20)
    m1 = helpers.ellipse(W_L, H_L, 82, 40, 14, 14) & ~m0
    return [helpers._as_mask(m0), helpers._as_mask(m1)]


def layer_inputs(warp_ex):
    """Per-segment inputs of the flatten from a warp_ex implementation: flows, rgbs, warped masks, src masks, bflows."""
    srcs = layer_masks()
    rgb = rgb_for(W_L, H_L, 7)
    flows, outs = [], []
    for m, t in zip(srcs, T_LAYERS):
        fl = np.zeros((H_L, W_L, 2), np.float32) + np.float32(t)
        flows.append(fl)
        outs.append(warp_ex(fl, rgb, m, is_flow=True))
    return flows, [o["rgb"] for o in outs], [o["mask"] for o in outs], srcs, [o["bflow"] for o in outs]


def check_layers(flat, srcs):
    landed = [shift(cov(m), t) for m, t in zip(srcs, T_LAYERS)]
    assert (landed[0] & landed[1]).sum() > 100      # the upper layer really covers part of the lower one
    front = np.where(landed[1], 1, np.where(landed[0], 0, -1))
    exp_b = np.zeros((H_L, W_L, 2), np.float32)
    for s, t in enumerate(T_LAYERS):
        exp_b[front == s] = (-t[0], -t[1])
    assert np.array_equal(flat["bflow"], exp_b)
    occ = flat["occ"] == 255
    for s, (m, t) in enumerate(zip(srcs, T_LAYERS)):
        obj = m == 0
        exp = ~cov(m) | ~in_frame_after(W_L, H_L, t)
        if s == 0:   # under the upper layer's footprint after the move
            exp |= shift(landed[1], (-t[0], -t[1]))
        assert np.array_equal(occ[obj], exp[obj]), s
    bg = (srcs[0] != 0) & (srcs[1] != 0)
    assert np.array_equal(occ[bg], (front >= 0)[bg])
    # the lower layer's pixels that end up under the upper layer are occluded
    under = (srcs[0] == 0) & cov(srcs[0]) & shift(landed[1], (-T_LAYERS[0][0], -T_LAYERS[0][1]))
    assert under.sum() > 100 and occ[under].all()
