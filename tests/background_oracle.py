"""CPU restatement of the composite over a moving background (DESIGN.md 4.5), for the tests.

Built on tests/occlusion_oracle.py (its occlusion rule and the layer flatten of oracle.pycomposite).  The maps are
derived in binary64 in the documented order and rounded once to binary32; everything per pixel is numpy float32, one
rounding per operation in the documented order (numpy never contracts a * b + c into an FMA), so it can be compared with
the CUDA kernels bit for bit.  Held to analytic cases by tests/test_oracle_background.py.
"""
import numpy as np

from oracle import pycomposite as PC
from tests import occlusion_oracle as OO

F = np.float32
IDENTITY = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def inverse(A):
    a00, a01, a02, a10, a11, a12 = np.asarray(A, np.float64).ravel()
    det = a00 * a11 - a01 * a10
    i00, i01, i10, i11 = a11 / det, -a01 / det, -a10 / det, a00 / det
    return np.array([[i00, i01, -(i00 * a02 + i01 * a12)], [i10, i11, -(i10 * a02 + i11 * a12)]])


def compose(P, Q):
    """P o Q"""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    return np.array([[P[r, 0] * Q[0, 0] + P[r, 1] * Q[1, 0], P[r, 0] * Q[0, 1] + P[r, 1] * Q[1, 1],
                      (P[r, 0] * Q[0, 2] + P[r, 1] * Q[1, 2]) + P[r, 2]] for r in range(2)])


def coeffs(motion, motion_from=None):
    """float32 [3, 2, 3]: F = A_to o inv(A_from), B = A_from o inv(A_to), S = inv(A_to)."""
    Af = IDENTITY if motion_from is None else np.asarray(motion_from, np.float64)
    It = inverse(motion)
    return np.stack([compose(motion, inverse(Af)), compose(Af, It), It]).astype(F)


def apply(M, W, H):
    """M(x, y) on the W x H pixel grid: ((m00 x + m01 y) + m02, (m10 x + m11 y) + m12), float32 [H, W, 2]."""
    yy, xx = np.mgrid[0:H, 0:W].astype(F)
    with np.errstate(all="ignore"):
        return np.stack([(M[0, 0] * xx + M[0, 1] * yy) + M[0, 2], (M[1, 0] * xx + M[1, 1] * yy) + M[1, 2]], -1)


def sample(bg, s):
    """Bilinear sample of uint8 bg[bgH, bgW, 3] at float32 points s[..., 2], clamped (NaN -> 0), rounded to nearest even."""
    bgH, bgW = bg.shape[:2]
    sx = np.fmin(np.fmax(s[..., 0], F(0)), F(bgW - 1))     # fmax / fmin drop a NaN, as fmaxf / fminf do
    sy = np.fmin(np.fmax(s[..., 1], F(0)), F(bgH - 1))
    x0, y0 = np.floor(sx).astype(np.int64), np.floor(sy).astype(np.int64)
    x1, y1 = np.minimum(x0 + 1, bgW - 1), np.minimum(y0 + 1, bgH - 1)
    fx, fy = (sx - x0.astype(F))[..., None], (sy - y0.astype(F))[..., None]
    gx, gy = F(1) - fx, F(1) - fy
    c = [bg[y, x].astype(F) for y, x in ((y0, x0), (y0, x1), (y1, x0), (y1, x1))]
    v = ((c[0] * gx + c[1] * fx) * gy) + ((c[2] * gx + c[3] * fx) * fy)
    return np.minimum(255, np.rint(v)).astype(np.uint8)


def composite(flows, rgbs, masks, src_masks, bflows, background, cf, origin=(0, 0), shape=None):
    """What arapb200_composite computes with the float32 maps cf = (F, B, S).  Returns a dict flow, rgb, mask, bflow, occ."""
    n = len(masks)
    H, W = masks[0].shape if n else shape
    F_, B_, S_ = (np.asarray(m, F) for m in cf)
    front = np.full((H, W), -1)                # last layer whose warped mask is non-zero
    for s, m in enumerate(masks):
        front[m != 0] = s
    owner = np.full((H, W), -1)                # the (last) layer whose frame-a input mask has p on the object
    for s, m in enumerate(src_masks):
        owner[m == 0] = s
    if n:
        _, rgb, mask = PC.flatten(flows, rgbs, masks)
        # the flatten's flow as the kernel selects it (PC.flatten's x * 0 would carry a covered layer's NaN through)
        flow = np.stack([np.asarray(f, F) for f in flows])[np.maximum(front, 0), np.arange(H)[:, None], np.arange(W)]
    else:
        flow, rgb, mask = np.zeros((H, W, 2), F), np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.uint8)
    grid = apply(np.array([[1, 0, 0], [0, 1, 0]], F), W, H)
    s = apply(S_, W, H)
    with np.errstate(all="ignore"):
        s = np.stack([s[..., 0] + F(origin[0]), s[..., 1] + F(origin[1])], -1)
        rgb = np.where((front >= 0)[..., None], rgb, sample(background, s))
        bflow = apply(B_, W, H) - grid
        fbg = apply(F_, W, H) - grid
    for k, b in enumerate(bflows or []):
        bflow[front == k] = b[front == k]
    flow = np.where((owner >= 0)[..., None], flow, fbg)
    # the background is surface n: every p has a surface, so the static-background branch of the rule never applies
    seg = np.where(owner >= 0, owner, n)
    occ = OO.occlusion(seg, list(flows) + [fbg], [bflow] * (n + 1), np.where(front >= 0, front, n))
    return dict(flow=flow.astype(F), rgb=rgb, mask=mask, bflow=bflow.astype(F), occ=occ)


def composite_api(flows, rgbs, masks, src_masks, bflows, background, motion, motion_from=None, origin=(0, 0),
                  extras=True, shape=None):
    """composite() behind lib.composite's signature, with the maps derived here."""
    cf = coeffs(motion, motion_from)
    out = composite(flows, rgbs, masks, src_masks, bflows if extras else None, background, cf, origin, shape)
    if not extras:
        del out["bflow"], out["occ"]
    return dict(out, coeffs=cf)
