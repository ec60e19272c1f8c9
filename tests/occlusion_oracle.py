"""CPU restatement of the backward flow, the occlusion of frame 1 and their layer flatten (DESIGN.md 4.3), for the tests.

Built on the oracle's sequential last-writer rasteriser (oracle.pyoracle.warp: splat indices bit-exact with the
reference's warp tool) and its flow extraction; the new quantities are computed here in numpy float32, one rounding per
operation in the order DESIGN.md 4.3 gives (numpy never contracts a * b + c into an FMA), so they can be compared with the
CUDA kernels bit for bit.  Held to analytic cases by tests/test_oracle_occlusion.py.
"""
import numpy as np

from oracle import pycomposite as PC
from oracle import pyoracle as O

F = np.float32


def _lk(pa, pb, pc, sx, sy):
    """PointInTriangleLK with w = 1 (warp.cu lk / arap_oracle.c point_in_triangle_lk): the weights (b0, b1, b2)."""
    X0, X1, X2 = pa[:, 0] - sx, pb[:, 0] - sx, pc[:, 0] - sx
    Y0, Y1, Y2 = pa[:, 1] - sy, pb[:, 1] - sy, pc[:, 1] - sy
    d01 = X0 * Y1 - Y0 * X1
    d12 = X1 * Y2 - Y1 * X2
    d20 = X2 * Y0 - Y2 * X0
    inv = F(1) / ((d01 + d12) + d20)
    return d12 * inv, d20 * inv, d01 * inv


def backward_flow(pos, splat):
    """bflow[q] = (the winning triangle's weights applied to its undeformed vertices) - q; (0, 0) where nothing landed."""
    H, W = splat.shape
    out = np.zeros((H, W, 2), F)
    qy, qx = np.nonzero(splat)
    sid = splat[qy, qx].astype(np.int64) - 1
    t, i00 = sid & 1, sid >> 1
    x0, y0 = i00 % W, i00 // W
    # triangle t = 0: (x0, y0), (x0+1, y0), (x0, y0+1); t = 1: (x0, y0+1), (x0+1, y0), (x0+1, y0+1)
    ax, ay, bx, by, cx, cy = x0, y0 + t, x0 + 1, y0, x0 + t, y0 + 1
    with np.errstate(all="ignore"):
        b0, b1, b2 = _lk(pos[ay, ax], pos[by, bx], pos[cy, cx], qx.astype(F), qy.astype(F))
        sx = (ax.astype(F) * b0 + bx.astype(F) * b1) + cx.astype(F) * b2
        sy = (ay.astype(F) * b0 + by.astype(F) * b1) + cy.astype(F) * b2
        out[qy, qx, 0] = sx - qx.astype(F)
        out[qy, qx, 1] = sy - qy.astype(F)
    return out


def occlusion(seg, flows, bflows, front):
    """Occlusion of frame 1 (0 visible, 255 not).  seg[p]: p's surface (-1 background); flows[s] / bflows[s]: forward /
    backward flow of surface s; front[q]: the surface in front at frame-2 pixel q (-1 = nothing landed)."""
    H, W = seg.shape
    occ = np.full((H, W), 255, np.uint8)
    occ[(seg < 0) & (front < 0)] = 0           # static background, nothing landed on it
    for s in range(len(flows)):
        py, px = np.nonzero(seg == s)
        f = flows[s][py, px].astype(F)
        with np.errstate(invalid="ignore"):
            tx = (px.astype(F) + f[:, 0]) + F(0.5)
            ty = (py.astype(F) + f[:, 1]) + F(0.5)
            inside = (tx >= 0) & (tx < F(W)) & (ty >= 0) & (ty < F(H))   # NaN compares false: left the frame
        px, py, tx, ty = px[inside], py[inside], tx[inside], ty[inside]
        qx, qy = np.floor(tx).astype(np.int64), np.floor(ty).astype(np.int64)
        b = bflows[s][qy, qx].astype(F)
        ex = b[:, 0] + (qx - px).astype(F)
        ey = b[:, 1] + (qy - py).astype(F)
        vis = (front[qy, qx] == s) & (np.abs(ex) < 1) & (np.abs(ey) < 1)
        occ[py[vis], px[vis]] = 0
    return occ


def warp_ex(pos_or_flow, rgb, mask_red, is_flow=False):
    """What arapb200_warp_ex computes.  Returns a dict rgb, mask, splat (oracle.pyoracle.warp), bflow, occ."""
    pf = np.ascontiguousarray(pos_or_flow, F)
    pos, flow = (O.flow_to_pos(pf), pf) if is_flow else (pf, O.flow(pf))
    rgb_w, mask_w, splat = O.warp(pos, rgb, mask_red)
    bflow = backward_flow(pos, splat)
    seg = np.where(np.asarray(mask_red) == 0, 0, -1)
    occ = occlusion(seg, [flow], [bflow], np.where(splat != 0, 0, -1))
    return dict(rgb=rgb_w, mask=mask_w, splat=splat, bflow=bflow, occ=occ)


def flatten_ex(flows, rgbs, masks, src_masks, bflows):
    """What arapb200_flatten_ex computes: pycomposite.flatten plus the flattened backward flow and the occlusion of
    frame 1 across the layers.  Returns a dict flow, rgb, mask, bflow, occ."""
    flow, rgb, mask = PC.flatten(flows, rgbs, masks)
    H, W = masks[0].shape
    front = np.full((H, W), -1)                # last layer whose warped mask is non-zero
    for s, m in enumerate(masks):
        front[m != 0] = s
    bflow = np.zeros((H, W, 2), F)
    for s, b in enumerate(bflows):
        bflow[front == s] = b[front == s]
    seg = np.full((H, W), -1)                  # p's surface: the (last) layer whose input mask has p on the object
    for s, m in enumerate(src_masks):
        seg[m == 0] = s
    occ = occlusion(seg, flows, bflows, front)
    return dict(flow=flow, rgb=rgb, mask=mask, bflow=bflow, occ=occ)
