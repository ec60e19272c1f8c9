"""CPU restatement of frame sequences (DESIGN.md 4.4), for the tests.

Built on tests/occlusion_oracle.py (_lk, occlusion) and the oracle's rasteriser and flow extraction (oracle.pyoracle.warp,
.flow); the new quantities are computed in numpy float32 with one rounding per operation in the order DESIGN.md 4.4
gives, so they can be compared with the CUDA kernels bit for bit.  The solver states come from a Python loop over the
continuation schedule that makes the same oracle calls arap_oracle_solve makes.  Held to analytic cases by
tests/test_oracle_sequence.py.
"""
import numpy as np

from oracle import pyoracle as O
from tests import occlusion_oracle as OO

F = np.float32
KEYS = ("rgb", "mask", "flow", "bflow", "occ", "flow0")


def interp(splat_a, P_a, V):
    """interp(z_a, P_a, V)[q]: the weights of q's winning triangle in frame a (against P_a) applied to that triangle's
    vertices in V, (Va*b0 + Vb*b1) + Vc*b2, minus q; (0, 0) where nothing landed."""
    H, W = splat_a.shape
    out = np.zeros((H, W, 2), F)
    qy, qx = np.nonzero(splat_a)
    sid = splat_a[qy, qx].astype(np.int64) - 1
    t, i00 = sid & 1, sid >> 1
    x0, y0 = i00 % W, i00 // W
    ax, ay, bx, by, cx, cy = x0, y0 + t, x0 + 1, y0, x0 + t, y0 + 1
    V = np.asarray(V, F)
    with np.errstate(all="ignore"):
        b0, b1, b2 = OO._lk(P_a[ay, ax], P_a[by, bx], P_a[cy, cx], qx.astype(F), qy.astype(F))
        for c in (0, 1):
            s = (V[ay, ax, c] * b0 + V[by, bx, c] * b1) + V[cy, cx, c] * b2
            out[qy, qx, c] = s - (qx if c == 0 else qy).astype(F)
    return out


def warp_seq(positions, rgb, mask_red):
    """What arapb200_warp_seq computes for P_1 .. P_K = positions[0 .. K-1].  Returns a dict of [K, ...] arrays
    (KEYS) plus splat[K, H, W], the winning triangle of every frame."""
    H, W = mask_red.shape
    out = {k: [] for k in KEYS + ("splat",)}
    prev_P = prev_z = None
    for P in np.asarray(positions, F):
        rgb_w, mask_w, z = O.warp(P, rgb, mask_red)
        if prev_z is None:            # frame 0 is the pixel grid and its object is the input mask
            flow = O.flow(P)
            bflow = interp(z, P, O.grid(W, H))
            seg = np.where(np.asarray(mask_red) == 0, 0, -1)
        else:
            flow = interp(prev_z, prev_P, P)
            bflow = interp(z, P, prev_P)
            seg = np.where(prev_z != 0, 0, -1)
        occ = OO.occlusion(seg, [flow], [bflow], np.where(z != 0, 0, -1))
        for k, v in zip(KEYS + ("splat",), (rgb_w, mask_w, flow, bflow, occ, O.flow(P), z)):
            out[k].append(v)
        prev_P, prev_z = P, z
    return {k: np.stack(v) for k, v in out.items()}


def solve_states(mask_red, matches, steps, nCont, nGN, nPCG, lm=False):
    """The continuation schedule as arap_oracle_solve runs it (resetGPU, then per step t the constraint image for
    alpha = (t+1)/nCont and one Opt_ProblemSolve), keeping X after every step in `steps`.  Returns (X, A, costs[nCont,
    nGN+1], snapshots[len(steps), H, W, 2])."""
    H, W = mask_red.shape
    m = O.with_border_pins(matches, W, H)
    U = O.grid(W, H)
    M = np.asarray(mask_red, np.uint8).astype(F)
    X, A = U.copy(), np.zeros((H, W), F)
    costs = np.zeros((nCont, nGN + 1), F)
    snaps = []
    solve = O.lm_solve if lm else O.gn_solve
    for t in range(nCont):
        alpha = F(t + 1) / F(nCont)
        X, A, costs[t] = solve(X, A, U, O.constraint_image(mask_red, m, alpha), M, nGN, nPCG)[:3]
        if t in steps:
            snaps.append(X.copy())
    return X, A, costs, np.stack(snaps) if snaps else np.zeros((0, H, W, 2), F)
