"""Analytic cases of tracks from frame 0 (DESIGN.md 4.9), shared by the oracle tests and the GPU tests.  Each case is a
list of position fields with no solve; every expectation comes from the motion, not from the formulas the restatement or
the kernels evaluate.  `warp_tracks(positions, mask) -> dict` is an implementation: the restatement or lib.warp_tracks."""
import numpy as np

from tests import occlusion_cases as OC
from tests import sequence_cases as SC

F = np.float32


def offsets_positions(offsets, W=OC.W_T, H=OC.H_T):
    """P_k = grid + offsets[k - 1] (integer offsets from frame 0)."""
    g = OC.grid(W, H)
    return np.stack([g + np.asarray(t, F) for t in offsets])


def _landed(mask, t):
    H, W = mask.shape
    return OC.shift(OC.cov(mask), t) if abs(t[0]) < W and abs(t[1]) < H else np.zeros((H, W), bool)


def check_offsets(tr, mask, offsets):
    """A rigid integer translation by offsets[k - 1] from frame 0 to frame k: flow0 is the offset everywhere, bflow0 its
    negative where the object landed and (0, 0) elsewhere; an object pixel is visible iff the rasteriser draws it and its
    target is in the frame, a background pixel iff nothing landed on it."""
    H, W = mask.shape
    for k, t in enumerate(offsets, 1):
        landed = _landed(mask, t)
        assert np.array_equal(tr["flow0"][k - 1], np.zeros((H, W, 2), F) + np.asarray(t, F)), k
        exp_b = np.zeros((H, W, 2), F)
        exp_b[landed] = (-t[0], -t[1])
        assert np.array_equal(tr["bflow0"][k - 1], exp_b), k
        obj = mask == 0
        exp_occ = np.where(obj, ~OC.cov(mask) | ~OC.in_frame_after(W, H, t), landed)
        assert np.array_equal(tr["occ0"][k - 1] == 255, exp_occ), k
        assert set(np.unique(tr["occ0"][k - 1])) <= {0, 255}


# a translation by t per frame, and an object that leaves the frame at frame 2 and comes back at frame 3
CONSTANT = [(3, -2), (6, -4), (9, -6)]
LEAVE_RETURN = [(4, 1), (OC.W_T, 0), (8, 2)]


def check_leave_return(tr, mask):
    """Visible, occluded, visible: the part of the object that is drawn and stays in the frame at frames 1 and 3."""
    H, W = mask.shape
    keep = (mask == 0) & OC.cov(mask) & OC.in_frame_after(W, H, LEAVE_RETURN[0]) & OC.in_frame_after(W, H, LEAVE_RETURN[2])
    assert keep.sum() > 500
    assert (tr["occ0"][0][keep] == 0).all() and (tr["occ0"][1][keep] == 255).all() and (tr["occ0"][2][keep] == 0).all()


def rotation_positions():
    """3 degrees per frame about the centre (sequence_cases.rotation_positions), with its mask."""
    return OC.rotation_case()[0], SC.rotation_positions()


def check_rotation(tr, seq_mask):
    """Within 1e-3 px of binary64: flow0[k] = R(3k)(p - c) + c - p, bflow0[k] = R(-3k)(q - c) + c - q where something
    landed (both frames are affine images of the same undeformed triangle; the bound is sequence_cases.check_rotation's)."""
    for k in range(1, SC.K + 1):
        dst = seq_mask[k - 1] == 255
        assert dst.sum() > 3000
        eb = np.abs(tr["bflow0"][k - 1].astype(np.float64) - SC._rot_flow(-OC.ROT_DEG * k))[dst]
        ef = np.abs(tr["flow0"][k - 1].astype(np.float64) - SC._rot_flow(OC.ROT_DEG * k))
        assert eb.max() < 1e-3 and ef.max() < 1e-3, (k, eb.max(), ef.max())
        assert not tr["bflow0"][k - 1][~dst].any()


def check_repeated(tr):
    """P_2 = P_1 (sequence_cases.repeated_positions): frame 2's tracks are frame 1's."""
    for key in ("flow0", "bflow0", "occ0"):
        assert np.array_equal(tr[key][1], tr[key][0]), key
    assert not np.array_equal(tr["bflow0"][2], tr["bflow0"][1])


# two layers on a 120 x 80 frame: A, a static block; B, a smaller block in front of it (a later layer) that starts to its
# left, lies on A at frame 2 and has passed it at frame 3
W_X, H_X = 120, 80
B_OFFSETS = [(0, 0), (40, 0), (80, 0)]


def crossing_layers():
    """(masks, positions per layer [K, H, W, 2]): A = x 40..79, y 20..59; B = x 2..21, y 30..49."""
    a = np.full((H_X, W_X), 255, np.uint8)
    a[20:60, 40:80] = 0
    b = np.full((H_X, W_X), 255, np.uint8)
    b[30:50, 2:22] = 0
    g = OC.grid(W_X, H_X)
    return [a, b], [np.stack([g] * 3), offsets_positions(B_OFFSETS, W_X, H_X)]


def crossed_pixels():
    """A's pixels that B lies on at frame 2 (B's drawn block x 2..21, y 30..49 shifted by 40)."""
    m = np.zeros((H_X, W_X), bool)
    m[30:50, 42:62] = True
    return m


def check_crossing(tr, masks):
    """A's pixels under B at frame 2 are occluded there and visible at frames 1 and 3; their flow0 is A's (zero), not
    B's, at every frame."""
    hit = crossed_pixels()
    assert (tr["occ0"][1][hit] == 255).all()
    assert (tr["occ0"][0][hit] == 0).all() and (tr["occ0"][2][hit] == 0).all()
    assert not tr["flow0"][:, hit].any()
    on_a = (masks[0] == 0) & (masks[1] != 0)
    assert (tr["occ0"][0][on_a & OC.cov(masks[0])] == 0).all()
