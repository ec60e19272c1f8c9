"""Analytic frame sequences (DESIGN.md 4.4), shared by the oracle tests and the GPU tests.  Each case is a list of
position fields with no solve; every expectation comes from the motion, not from the formulas the oracle or the kernels
evaluate.  `warp_seq` is an implementation: tests.sequence_oracle.warp_seq or arap_flow_b200.lib.warp_seq."""
import numpy as np

from tests import occlusion_cases as OC

K = 3


def translation_positions(t):
    """Constant velocity: P_k = grid + k t."""
    g = OC.grid(OC.W_T, OC.H_T)
    return np.stack([g + np.float32(k) * np.float32(t) for k in range(1, K + 1)])


def _shift(a, t):
    """OC.shift, also for motions that leave the frame entirely."""
    H, W = a.shape[:2]
    return OC.shift(a, t) if abs(t[0]) < W and abs(t[1]) < H else np.zeros_like(a)


def check_translation(out, mask, t):
    H, W = mask.shape
    landed = [_shift(OC.cov(mask), (k * t[0], k * t[1])) for k in range(K + 1)]   # landed[0]: the object at rest
    leaves = ~OC.in_frame_after(W, H, t)
    for k in range(1, K + 1):
        assert np.array_equal(out["mask"][k - 1] == 255, landed[k]), k
        exp_f = np.zeros((H, W, 2), np.float32)
        exp_b = np.zeros((H, W, 2), np.float32)
        exp_b[landed[k]] = (-t[0], -t[1])
        if k == 1:
            exp_f[...] = t                    # the forward flow of the input grid, object or not
        else:
            exp_f[landed[k - 1]] = t
        assert np.array_equal(out["flow"][k - 1], exp_f), k
        assert np.array_equal(out["bflow"][k - 1], exp_b), k
        assert np.array_equal(out["flow0"][k - 1], np.zeros((H, W, 2), np.float32) + np.float32(k) * np.float32(t)), k
        # frame k - 1's object: occluded iff it was never rasterised (k = 1) or it leaves the frame;
        # its background: occluded iff something lands on it
        obj = (mask == 0) if k == 1 else landed[k - 1]
        exp_occ = np.where(obj, leaves | ((~OC.cov(mask)) if k == 1 else False), landed[k])
        assert np.array_equal(out["occ"][k - 1] == 255, exp_occ), k
        assert set(np.unique(out["occ"][k - 1])) <= {0, 255}


def rotation_positions(deg=OC.ROT_DEG):
    """A rotation by `deg` per frame about the centre of the rotation case's frame."""
    c = (OC.W_R - 1) / 2.0
    g = OC.grid(OC.W_R, OC.H_R).astype(np.float64) - c
    out = []
    for k in range(1, K + 1):
        a = np.deg2rad(deg * k)
        out.append(np.stack([np.cos(a) * g[..., 0] - np.sin(a) * g[..., 1],
                             np.sin(a) * g[..., 0] + np.cos(a) * g[..., 1]], -1) + c)
    return np.stack(out).astype(np.float32)


def _rot_flow(deg):
    """The analytic flow of a rotation by deg about the centre, at every pixel: R(q - c) + c - q."""
    c = (OC.W_R - 1) / 2.0
    q = OC.grid(OC.W_R, OC.H_R).astype(np.float64) - c
    a = np.deg2rad(deg)
    return np.stack([np.cos(a) * q[..., 0] - np.sin(a) * q[..., 1], np.sin(a) * q[..., 0] + np.cos(a) * q[..., 1]], -1) - q


def check_rotation(out):
    # Both frames are affine images of the same undeformed triangle, so the frame-(k-1) weights carry a frame-(k-1)
    # pixel to its frame-k position exactly up to rounding: positions below 128 px are off by half an ulp (< 8e-6 px)
    # and the float32 weights add a few ulps of 128 (~1e-5 px).  1e-3 px leaves two orders of magnitude of margin.
    for k in range(2, K + 1):
        src = out["mask"][k - 2] == 255
        dst = out["mask"][k - 1] == 255
        assert src.sum() > 3000 and dst.sum() > 3000
        ef = np.abs(out["flow"][k - 1].astype(np.float64) - _rot_flow(OC.ROT_DEG))[src]
        eb = np.abs(out["bflow"][k - 1].astype(np.float64) - _rot_flow(-OC.ROT_DEG))[dst]
        assert ef.max() < 1e-3 and eb.max() < 1e-3, (k, ef.max(), eb.max())
        assert not out["flow"][k - 1][~src].any() and not out["bflow"][k - 1][~dst].any()


def repeated_positions():
    """P_1 = a 3 degree rotation, P_2 = P_1 (a frame that does not move), P_3 = a 6 degree rotation."""
    r = rotation_positions()
    return np.stack([r[0], r[0], r[1]])


def check_repeated(out):
    landed = out["mask"][0] == 255
    assert np.array_equal(out["mask"][1], out["mask"][0]) and np.array_equal(out["rgb"][1], out["rgb"][0])
    assert np.abs(out["flow"][1]).max() <= 1e-4 and np.abs(out["bflow"][1]).max() <= 1e-4
    assert landed.sum() > 3000
    assert (out["occ"][1] == 0).all()          # every rasterised pixel stays put; nothing lands on the background


def compression_positions():
    """P_1 = the grid (identity), P_2 = (px / 2, py): frame 1 -> 2 is the 2:1 compression of DESIGN.md 4.3."""
    mask, pos = OC.compression_case()
    return mask, np.stack([OC.grid(OC.W_C, OC.H_C), pos])


def check_compression(out):
    OC.check_identity({k: out[k][0] for k in ("occ", "bflow")}, np.zeros((OC.H_C, OC.W_C), np.uint8))
    OC.check_compression({k: out[k][1] for k in ("occ", "mask", "bflow")})
    px = OC.grid(OC.W_C, OC.H_C)[..., 0]
    assert np.array_equal(out["flow"][1][..., 0], px * np.float32(0.5) - px) and not out["flow"][1][..., 1].any()
