"""Analytic cases of the composite over a moving background (DESIGN.md 4.5), shared by the oracle tests and the GPU
tests.  `comp` is lib.composite or tests.background_oracle.composite_api, `warp_ex` lib.warp_ex or
tests.occlusion_oracle.warp_ex.  Every expectation comes from the geometry of the case or from the existing flatten, not
from the formulas the oracle or the kernels evaluate; the comparisons are exact except where a bound is derived."""
import numpy as np

from arap_flow_b200 import synth
from oracle import pycomposite as PC
from tests import occlusion_cases as OC
from tests import occlusion_oracle as OO

I2 = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def translation(t):
    return np.array([[1.0, 0.0, t[0]], [0.0, 1.0, t[1]]])


def about_centre(W, H, deg, scale):
    """A(u) = c + scale R(deg) (u - c), c the frame centre."""
    a = np.deg2rad(deg)
    R = scale * np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
    c = np.array([(W - 1) / 2.0, (H - 1) / 2.0])
    return np.hstack([R, (c - R @ c)[:, None]])


def affine_np(A, x, y):
    """A at points (x, y) in binary64."""
    A = np.asarray(A, np.float64)
    return A[0, 0] * x + A[0, 1] * y + A[0, 2], A[1, 0] * x + A[1, 1] * y + A[1, 2]


def grid64(W, H):
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    return xx, yy


def layer_inputs(warp_ex, n):
    """The first n layers of OC.layer_masks() moved by OC.T_LAYERS through warp_ex, with every layer's flow zero off its
    own object (as every solver or warp output is): flows, rgbs, warped masks, src masks, bflows."""
    srcs = OC.layer_masks()[:n]
    rgb = OC.rgb_for(OC.W_L, OC.H_L, 7)
    flows, outs = [], []
    for m, t in zip(srcs, OC.T_LAYERS):
        fl = np.zeros((OC.H_L, OC.W_L, 2), np.float32) + np.float32(t)
        fl[m != 0] = 0
        flows.append(fl)
        outs.append(warp_ex(fl, rgb, m, is_flow=True))
    return flows, [o["rgb"] for o in outs], [o["mask"] for o in outs], srcs, [o["bflow"] for o in outs]


# ---- both motions the identity ---------------------------------------------------------------------------------------
def check_identity_is_flatten(comp, warp_ex, n):
    """n = 1, 2: flatten_ex with add_bg of a same-size background, bit for bit (flow included: the flows vanish off the
    objects)."""
    args = layer_inputs(warp_ex, n)
    bg = synth.background(OC.W_L, OC.H_L, 11)
    ref = OO.flatten_ex(*args)
    ref["rgb"] = PC.add_bg(ref["rgb"], ref["mask"], bg)
    for motion_from in (None, I2):
        out = comp(*args, bg, I2, motion_from=motion_from)
        for k in ("flow", "rgb", "mask", "bflow", "occ"):
            assert np.array_equal(out[k], ref[k]), k
        assert np.array_equal(out["coeffs"], np.stack([I2, I2, I2]).astype(np.float32))
    assert (ref["occ"] == 255).any() and (ref["occ"] == 0).any()


def check_identity_no_layers(comp):
    """No layers: the background crop, zero flow both ways, nothing occluded."""
    W, H, o = 37, 23, (5, 3)
    bg = synth.background(W + 9, H + 7, 12)
    out = comp([], [], [], [], [], bg, I2, origin=o, shape=(H, W))
    assert np.array_equal(out["rgb"], bg[o[1]:o[1] + H, o[0]:o[0] + W])
    assert not out["flow"].any() and not out["bflow"].any() and not out["mask"].any() and not out["occ"].any()


# ---- integer background translation ----------------------------------------------------------------------------------
W_B, H_B, M_B = 37, 23, 8
BG_SHIFTS = [(3, -2), (-7, 5), (0, 0)]


def check_integer_translation(comp, t):
    bg = synth.background(W_B + 2 * M_B, H_B + 2 * M_B, 13)
    out = comp([], [], [], [], [], bg, translation(t), origin=(M_B, M_B), shape=(H_B, W_B))
    xx, yy = np.mgrid[0:H_B, 0:W_B][::-1]
    assert np.array_equal(out["rgb"], bg[yy - t[1] + M_B, xx - t[0] + M_B])          # rgb[q] = bg[q - t + o]
    assert (out["flow"] == np.float32(t)).all() and (out["bflow"] == -np.float32(t)).all()
    assert np.array_equal(out["occ"] == 255, ~OC.in_frame_after(W_B, H_B, t))
    assert set(np.unique(out["occ"])) <= {0, 255}


# ---- half-pixel shift: pins round-to-nearest-even of the colour --------------------------------------------------
def check_half_pixel(comp):
    bg = synth.background(W_B + 2, H_B + 2, 14)
    out = comp([], [], [], [], [], bg, translation((0.5, 0.0)), origin=(1, 1), shape=(H_B, W_B))
    xx, yy = np.mgrid[0:H_B, 0:W_B][::-1]
    c0, c1 = bg[yy + 1, xx].astype(np.int64), bg[yy + 1, xx + 1].astype(np.int64)  # sample at x + 0.5 in the background
    assert ((c0 + c1) % 4 == 3).any() and ((c0 + c1) % 4 == 1).any()              # halves that round up and down
    assert np.array_equal(out["rgb"], np.rint((c0 + c1) / 2).astype(np.uint8))


# ---- scale 0.5 about the origin: pins the strict < 1 for the background -------------------------------------------
def check_half_scale(comp):
    W, H = 40, 30
    A = np.array([[0.5, 0.0, 0.0], [0.0, 0.5, 0.0]])
    out = comp([], [], [], [], [], synth.background(W, H, 15), A, shape=(H, W))
    xx, yy = np.mgrid[0:H, 0:W][::-1]
    # p goes to p/2 and the nearest pixel q = floor(p/2 + 0.5) shows the point 2q: p itself for even coordinates, an
    # error of exactly 1 for odd ones, which the strict bound makes occluded
    assert np.array_equal(out["occ"] == 255, (xx % 2 == 1) | (yy % 2 == 1))
    assert np.array_equal(out["flow"], -np.stack([xx, yy], -1).astype(np.float32) / 2)
    assert np.array_equal(out["bflow"], np.stack([xx, yy], -1).astype(np.float32))


# ---- rotation and zoom-in --------------------------------------------------------------------------------------------
W_Z, H_Z = 96, 64
ZOOMS = [(20.0, 1.0), (-35.0, 1.25), (170.0, 1.5)]


def check_rotation_zoom(comp, deg, scale):
    A = about_centre(W_Z, H_Z, deg, scale)
    m = synth.background_margin(A, W_Z, H_Z)
    bg = synth.background(W_Z + 2 * m, H_Z + 2 * m, 16)
    out = comp([], [], [], [], [], bg, A, origin=(m, m), shape=(H_Z, W_Z))
    xx, yy = grid64(W_Z, H_Z)
    fx, fy = affine_np(A, xx, yy)
    Ai = np.linalg.inv(np.vstack([A, [0, 0, 1]]))[:2]
    bx, by = affine_np(Ai, xx, yy)
    # binary32 maps and coordinates below 200 px: a few ulps of 200 (~1e-5 px); 1e-3 leaves two orders of margin
    assert np.abs(out["flow"][..., 0] - (fx - xx)).max() < 1e-3 and np.abs(out["flow"][..., 1] - (fy - yy)).max() < 1e-3
    assert np.abs(out["bflow"][..., 0] - (bx - xx)).max() < 1e-3 and np.abs(out["bflow"][..., 1] - (by - yy)).max() < 1e-3
    # a p that stays in the frame is visible: the nearest pixel q is within 0.71 px of A(p) and inv(A) shrinks that by
    # the scale (>= 1), so q shows a point within 0.71 px of p.  Pixels within 1e-3 px of the frame's edge are skipped.
    tx, ty = fx + 0.5, fy + 0.5
    inside = (tx >= 1e-3) & (tx < W_Z - 1e-3) & (ty >= 1e-3) & (ty < H_Z - 1e-3)
    outside = (tx < -1e-3) | (tx >= W_Z + 1e-3) | (ty < -1e-3) | (ty >= H_Z + 1e-3)
    assert inside.sum() > W_Z * H_Z // 3 and outside.any()
    assert (out["occ"][inside] == 0).all() and (out["occ"][outside] == 255).all()


# ---- a moving object over a moving background ------------------------------------------------------------------------
T_OBJ, T_BG, M_L = (6, 2), (-3, 4), 8


def check_object_over_background(comp, warp_ex):
    src = OC.layer_masks()[0]
    rgb = OC.rgb_for(OC.W_L, OC.H_L, 7)
    fl = np.zeros((OC.H_L, OC.W_L, 2), np.float32) + np.float32(T_OBJ)
    w = warp_ex(fl, rgb, src, is_flow=True)
    bg = synth.background(OC.W_L + 2 * M_L, OC.H_L + 2 * M_L, 17)
    out = comp([fl], [w["rgb"]], [w["mask"]], [src], [w["bflow"]], bg, translation(T_BG), origin=(M_L, M_L))
    landed = OC.shift(OC.cov(src), T_OBJ)
    assert np.array_equal(out["mask"] == 255, landed)
    xx, yy = np.mgrid[0:OC.H_L, 0:OC.W_L][::-1]
    exp_rgb = bg[yy - T_BG[1] + M_L, xx - T_BG[0] + M_L]
    exp_rgb[landed] = w["rgb"][landed]
    assert np.array_equal(out["rgb"], exp_rgb)
    obj = src == 0
    exp_flow = np.where(obj[..., None], np.float32(T_OBJ), np.float32(T_BG))
    assert np.array_equal(out["flow"], exp_flow)
    assert np.array_equal(out["bflow"], np.where(landed[..., None], -np.float32(T_OBJ), -np.float32(T_BG)))
    occ = out["occ"] == 255
    assert np.array_equal(occ[obj], (~OC.cov(src) | ~OC.in_frame_after(OC.W_L, OC.H_L, T_OBJ))[obj])
    # a background p is occluded iff p + t_b leaves the frame or lands on the object's frame-2 footprint
    exp_bg = ~OC.in_frame_after(OC.W_L, OC.H_L, T_BG) | OC.shift(landed, (-T_BG[0], -T_BG[1]), fill=True)
    assert np.array_equal(occ[~obj], exp_bg[~obj])
    assert (occ[~obj] & OC.in_frame_after(OC.W_L, OC.H_L, T_BG)[~obj]).sum() > 100   # really hidden by the object


# ---- clamping --------------------------------------------------------------------------------------------------------
CLAMP_SHIFTS = [(5, -4), (-6, 3)]   # beyond the 2-px margin on one side in x and one in y


def check_clamping(comp, t):
    m = 2
    bg = synth.background(W_B + 2 * m, H_B + 2 * m, 18)
    out = comp([], [], [], [], [], bg, translation(t), origin=(m, m), shape=(H_B, W_B))
    xx, yy = np.mgrid[0:H_B, 0:W_B][::-1]
    sx, sy = xx - t[0] + m, yy - t[1] + m
    assert ((sx < 0) | (sx >= W_B + 2 * m)).any() and ((sy < 0) | (sy >= H_B + 2 * m)).any()
    assert np.array_equal(out["rgb"], bg[np.clip(sy, 0, H_B + 2 * m - 1), np.clip(sx, 0, W_B + 2 * m - 1)])


# ---- sequences -------------------------------------------------------------------------------------------------------
def check_same_motion_is_still(comp):
    """A_from = A_to: a background that does not move between the two frames.  A dyadic map composes with its inverse
    to the identity exactly; a rotation to within the rounding of binary64 (~1e-13 px here)."""
    W, H = 64, 48
    bg = synth.background(W, H, 19)
    dyadic = np.array([[2.0, 0.0, 3.0], [0.0, 0.5, -1.0]])
    out = comp([], [], [], [], [], bg, dyadic, motion_from=dyadic, shape=(H, W))
    assert not out["flow"].any() and not out["bflow"].any() and not out["occ"].any()
    A = synth.background_motion(W, H, 3)[0]
    out = comp([], [], [], [], [], bg, A, motion_from=A, shape=(H, W))
    assert np.abs(out["flow"]).max() < 1e-6 and np.abs(out["bflow"]).max() < 1e-6 and not out["occ"].any()


def _bilinear(f, x, y):
    x0, y0 = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    x1, y1 = np.minimum(x0 + 1, f.shape[1] - 1), np.minimum(y0 + 1, f.shape[0] - 1)
    ax, ay = (x - x0)[..., None], (y - y0)[..., None]
    f = f.astype(np.float64)
    return (f[y0, x0] * (1 - ax) + f[y0, x1] * ax) * (1 - ay) + (f[y1, x0] * (1 - ax) + f[y1, x1] * ax) * ay


def check_chord_path_composes(comp, seed=4):
    """The frame-to-frame flows of the chord path, chained (bilinearly: each is affine), give the pair's flow."""
    W, H, nCont, steps = 96, 64, 6, [1, 3, 5]
    A, m = synth.background_motion(W, H, seed)
    path = synth.motion_path(A, steps, nCont)
    assert np.array_equal(path[-1], A)
    bg = synth.background(W + 2 * m, H + 2 * m, 20)
    kw = dict(origin=(m, m), shape=(H, W))
    pair = comp([], [], [], [], [], bg, A, **kw)["flow"].astype(np.float64)
    xx, yy = grid64(W, H)
    x, y = xx.copy(), yy.copy()
    ok = np.ones((H, W), bool)
    prev = None
    for Ak in path:
        f = comp([], [], [], [], [], bg, Ak, motion_from=prev, **kw)["flow"]
        ok &= (x >= 0) & (x <= W - 1) & (y >= 0) & (y <= H - 1)
        d = _bilinear(f, np.clip(x, 0, W - 1), np.clip(y, 0, H - 1))
        x, y = x + d[..., 0], y + d[..., 1]
        prev = Ak
    assert ok.sum() > W * H // 2
    assert np.abs((x - xx) - pair[..., 0])[ok].max() < 1e-3 and np.abs((y - yy) - pair[..., 1])[ok].max() < 1e-3
