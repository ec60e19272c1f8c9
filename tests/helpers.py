"""Shared problem builders for the parity tests (seeded, small enough for the oracle to finish in seconds)."""
import lzma
import os
import shutil

import numpy as np

from arap_flow_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def cat512_flo(tmp_dir):
    """Path of the reference's shipped cat512_iFlo.flo, restored byte for byte into tmp_dir from the xz-compressed copy
    under tests/golden (the raw file is 2 MB)."""
    path = os.path.join(str(tmp_dir), "cat512_iFlo.flo")
    with lzma.open(os.path.join(GOLD, "cat512_iFlo.flo.xz")) as src, open(path, "wb") as dst:
        shutil.copyfileobj(src, dst)
    return path


def random_problem(W, H, seed, p_inactive=0.25, n_cstr=10, angle_amp=0.3, x_amp=0.5):
    """A ragged random mask with random state, for unit-level (single kernel) parity."""
    rng = np.random.default_rng(seed)
    M = ((rng.random((H, W)) < p_inactive).astype(np.float32)) * 255.0
    yy, xx = np.mgrid[0:H, 0:W]
    U = np.ascontiguousarray(np.stack([xx, yy], -1).astype(np.float32))
    X = (U + rng.standard_normal((H, W, 2)) * x_amp).astype(np.float32)
    A = (rng.standard_normal((H, W)) * angle_amp).astype(np.float32)
    Cn = np.full((H, W, 2), -1.0, np.float32)
    for _ in range(n_cstr):
        x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
        Cn[y, x] = (abs(x + rng.uniform(-2, 2)), abs(y + rng.uniform(-2, 2)))
    p = rng.standard_normal((H, W, 3)).astype(np.float32)
    p[M != 0] = 0
    return dict(W=W, H=H, M=M, U=U, X=X, A=A, C=Cn, p=p)


def synth_gn_problem(oracle, W, H, seed, fd=2, alpha=1.0, nseg=1):
    """Opt_ProblemSolve-level inputs from the synthetic generator at continuation weight alpha."""
    sp = synth.synth(W, H, nseg, fd, seed)
    mask = sp.masks[0]
    m = oracle.with_border_pins(sp.matches, W, H)
    Cn = oracle.constraint_image(mask, m, alpha)
    U = oracle.grid(W, H)
    return dict(W=W, H=H, M=mask.astype(np.float32), U=U, X=U.copy(), A=np.zeros((H, W), np.float32), C=Cn,
                sp=sp, mask=mask)


def epe(a, b, sel=None):
    d = np.hypot(a[..., 0] - b[..., 0], a[..., 1] - b[..., 1])
    return d[sel] if sel is not None else d


def optimal_angles(X, U, active):
    """argmin over a_i of sum_j |(X_i - X_j) - R(a_i)(u_i - u_j)|^2 over valid 4-neighbours (arap_plan.t:16-20): the
    energy is separable in the angles for fixed positions, a_i = atan2(sum d x e, sum d . e).  float64 numpy."""
    H, W = active.shape
    X = X.astype(np.float64)
    Ud = U.astype(np.float64)
    num = np.zeros((H, W))
    den = np.zeros((H, W))
    for dy, dx in ((0, 1), (0, -1), (1, 0), (-1, 0)):
        ys = slice(max(0, -dy), H - max(0, dy)); xs = slice(max(0, -dx), W - max(0, dx))
        yn = slice(max(0, dy), H - max(0, -dy)); xn = slice(max(0, dx), W - max(0, -dx))
        v = np.zeros((H, W), bool)
        v[ys, xs] = active[ys, xs] & active[yn, xn]
        e = np.zeros((H, W, 2)); d = np.zeros((H, W, 2))
        e[ys, xs] = X[ys, xs] - X[yn, xn]
        d[ys, xs] = Ud[ys, xs] - Ud[yn, xn]
        num += np.where(v, d[..., 0] * e[..., 1] - d[..., 1] * e[..., 0], 0.0)
        den += np.where(v, d[..., 0] * e[..., 0] + d[..., 1] * e[..., 1], 0.0)
    return np.arctan2(num, den)
