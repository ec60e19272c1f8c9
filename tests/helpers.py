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


# ---- mask geometries (uint8 HxW, 0 = object): what real segments look like, unlike synth's inset convex ellipses ----
def ellipse(W, H, cx, cy, ax, ay):
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    return ((xx - cx) / max(ax, 0.5)) ** 2 + ((yy - cy) / max(ay, 0.5)) ** 2 <= 1.0


def _as_mask(obj):
    return np.where(obj, 0, 255).astype(np.uint8)


def mask_border(W, H, seed, side):
    """An ellipse centred just outside one edge (side = left/right/top/bottom) plus a band two pixels inside the opposite
    edge, so that exactly that border is touched; side = all: a cross of full-width and full-height bands plus a corner
    ellipse, touching all four borders."""
    rng = np.random.default_rng(seed)
    obj = np.zeros((H, W), bool)
    if side == "all":
        y0, x0 = int(rng.integers(0, H - 3)), int(rng.integers(0, W - 4))
        obj[y0:y0 + max(2, H // 8)] = True
        obj[:, x0:x0 + max(2, W // 10)] = True
        return _as_mask(obj | ellipse(W, H, W - 1, H - 1, 0.3 * W, 0.35 * H))
    cx = {"left": -0.05 * W, "right": 1.05 * W - 1}.get(side, rng.uniform(0.35, 0.65) * W)
    cy = {"top": -0.05 * H, "bottom": 1.05 * H - 1}.get(side, rng.uniform(0.35, 0.65) * H)
    horiz = side in ("left", "right")
    obj |= ellipse(W, H, cx, cy, (0.35 if horiz else 0.3) * W, (0.3 if horiz else 0.35) * H)
    bw, bh = max(1, W // 12), max(1, H // 12)
    if side == "left":
        obj[2:H - 2, W - 2 - bw:W - 2] = True
    elif side == "right":
        obj[2:H - 2, 2:2 + bw] = True
    elif side == "top":
        obj[H - 2 - bh:H - 2, 2:W - 2] = True
    else:
        obj[2:2 + bh, 2:W - 2] = True
    return _as_mask(obj)


def mask_full(W, H, seed=0):
    return np.zeros((H, W), np.uint8)


def mask_empty(W, H, seed=0):
    return np.full((H, W), 255, np.uint8)


def mask_holes(W, H, seed):
    """A large ellipse with three rectangular holes of at least 33x9 pixels (one strip is 32x8): strips inside the object
    whose neighbour strip is absent."""
    rng = np.random.default_rng(seed)
    obj = ellipse(W, H, W / 2, H / 2, 0.48 * W, 0.48 * H)
    for _ in range(3):
        hw, hh = int(rng.integers(33, 48)), int(rng.integers(9, 16))
        x0 = int(rng.integers(W // 6, max(W // 6 + 1, W - W // 6 - hw)))
        y0 = int(rng.integers(H // 6, max(H // 6 + 1, H - H // 6 - hh)))
        obj[y0:y0 + hh, x0:x0 + hw] = False
    return _as_mask(obj)


def mask_components(W, H, seed):
    """Many small disconnected blobs (radius 0..4) on a jittered 16x12 lattice."""
    rng = np.random.default_rng(seed)
    obj = np.zeros((H, W), bool)
    for y in range(6, H - 5, 12):
        for x in range(8, W - 7, 16):
            if rng.random() < 0.7:
                obj |= ellipse(W, H, x + rng.integers(-2, 3), y + rng.integers(-1, 2), rng.uniform(0, 5), rng.uniform(0, 4))
    return _as_mask(obj)


def mask_lines(W, H, seed):
    """One-pixel-wide lines: a random row and column, the last row of a strip row (y % 8 == 7) and the last lane of a strip
    column (x % 32 == 31)."""
    rng = np.random.default_rng(seed)
    obj = np.zeros((H, W), bool)
    obj[int(rng.integers(1, H - 1)), 3:W - 3] = True
    obj[2:H - 2, int(rng.integers(1, W - 1))] = True
    obj[8 * int(rng.integers(0, max(1, (H - 7) // 8))) + 7, :] = True
    obj[:, 32 * int(rng.integers(0, max(1, (W - 31) // 32))) + 31] = True
    return _as_mask(obj)


def mask_pixels(W, H, seed):
    """Isolated single pixels: one in each corner of several strips (lane 0 / 31, row 0 / 7), the image corners, and random
    ones on even coordinates (no two 4-adjacent)."""
    rng = np.random.default_rng(seed)
    obj = np.zeros((H, W), bool)
    for sx in range(0, W // 32, 2):
        for sy in range(0, H // 8, 2):
            k = (sx + sy) // 2 % 4
            obj[8 * sy + 7 * (k & 1), 32 * sx + 31 * (k >> 1)] = True
    obj[0, 0] = obj[H - 1, W - 1] = obj[0, W - 1] = obj[H - 1, 0] = True
    ys, xs = 2 * rng.integers(0, H // 2, 40), 2 * rng.integers(0, W // 2, 40)
    obj[ys, xs] = True
    act = obj.copy()          # keep isolation: drop any pixel that got a 4-neighbour
    nb = np.zeros_like(act)
    nb[1:] |= act[:-1]; nb[:-1] |= act[1:]; nb[:, 1:] |= act[:, :-1]; nb[:, :-1] |= act[:, 1:]
    return _as_mask(act & ~nb)


def mask_ragged(W, H, seed):
    rng = np.random.default_rng(seed)
    return ((rng.random((H, W)) < 0.25) * 255).astype(np.uint8)


def mask_single(W, H, seed):
    rng = np.random.default_rng(seed)
    m = mask_empty(W, H)
    m[int(rng.integers(0, H)), int(rng.integers(0, W))] = 0
    return m


MASKS = {
    **{f"border_{s}": (lambda s: lambda W, H, seed: mask_border(W, H, seed, s))(s)
       for s in ("left", "right", "top", "bottom", "all")},
    "full": mask_full, "holes": mask_holes, "components": mask_components, "lines": mask_lines, "pixels": mask_pixels,
    "ragged": mask_ragged, "single": mask_single, "empty": mask_empty,
}

# (mask, W, H): every builder at two sizes with W % 32 != 0 and H % 8 != 0, plus images smaller than one strip
GEOMETRY_CASES = [(name, W, H) for name in MASKS for (W, H) in ((203, 77), (150, 97))] + \
                 [("full", 5, 3), ("ragged", 5, 3), ("full", 31, 7), ("ragged", 31, 7), ("single", 31, 7)]



def geometry_matches(mask, seed, fd=2.0):
    """DeepMatching-like matches on the 8-px lattice of the object: a smooth displacement of about fd pixels."""
    rng = np.random.default_rng(seed)
    H, W = mask.shape
    ph = rng.uniform(0, 2 * np.pi, 2)
    rows = []
    for y in range(3, H, 8):
        for x in range(3, W, 8):
            if mask[y, x] == 0:
                tx = int(round(x + fd * (1.0 + np.sin(2 * np.pi * y / 97.0 + ph[0]))))
                ty = int(round(y + fd * np.cos(2 * np.pi * x / 131.0 + ph[1])))
                rows.append((x, y, min(max(tx, 0), W - 1), min(max(ty, 0), H - 1)))
    return np.asarray(rows, np.int32).reshape(-1, 4)


def geometry_gn_problem(oracle, mask, seed, perturbed, alpha=0.5):
    """Opt_ProblemSolve-level inputs on `mask`: lattice matches + border pins at continuation weight alpha; the rest state
    (X = U, A = 0) or a perturbed one (X = U + N(0, 0.5), A ~ N(0, 0.3))."""
    H, W = mask.shape
    rng = np.random.default_rng(seed + 7919)
    U = oracle.grid(W, H)
    Cn = oracle.constraint_image(mask, oracle.with_border_pins(geometry_matches(mask, seed), W, H), alpha)
    X, A = U.copy(), np.zeros((H, W), np.float32)
    if perturbed:
        X = (U + rng.standard_normal((H, W, 2)) * 0.5).astype(np.float32)
        A = (rng.standard_normal((H, W)) * 0.3).astype(np.float32)
    return dict(W=W, H=H, M=mask.astype(np.float32), U=U, X=X, A=A, C=Cn)


def energy_f64(oracle, X, A, pr):
    """0.5 * sum of the squared residuals, evaluated in float64 at (X, A): the energy the solvers' cost reports."""
    r = oracle.residuals_f64(X, A, pr["U"], pr["C"], pr["M"])
    return 0.5 * float((r * r).sum())


def energy_bound(E, E_start):
    """How far a float32 cost may be from the float64 energy E of the same state: 1e-6 relative, plus 1e-12 of the energy
    the solve started from.  The floor matters only near convergence: a residual is still the float32 difference of
    positions as large as at the start, so its rounding error does not shrink with it.  Measured on the oracle over the
    geometry cases of test_oracle_geometry.py: 1e-6 relative alone fails (3.8e-4 relative at E = 1.5e-11, a fully
    converged 5x3 image); the largest error is 11 % of this bound."""
    return 1e-6 * E + 1e-12 * E_start


# ---- the resident back-end's launch arithmetic, mirrored (solver_resident.cu: k_strip_active, prepare_finish) ----
STRIP_W, STRIP_H, MAX_WARPS, MAX_CTAS = 32, 8, 12, 160


def strip_count(mask, sms):
    """Strips (32x8 tiles with at least one object pixel), warps per CTA (NW), CTAs (G) and whether the problem fits on
    chip on a device with `sms` SMs.  Occupancy (pick_variant) is not mirrored: a problem that passes these checks can
    still be refused by it."""
    H, W = mask.shape
    SX, SY = -(-W // STRIP_W), -(-H // STRIP_H)
    act = np.zeros((SY * STRIP_H, SX * STRIP_W), bool)
    act[:H, :W] = mask == 0
    n = int(act.reshape(SY, STRIP_H, SX, STRIP_W).any(axis=(1, 3)).sum())
    if n == 0:
        return dict(strips=0, NW=1, G=1, fits=True)
    NW = max(4, -(-n // sms))
    if NW > MAX_WARPS:
        return dict(strips=n, NW=NW, G=0, fits=False)
    G = min(-(-n // NW), sms)
    fits = G <= MAX_CTAS and -(-n // G) <= NW
    return dict(strips=n, NW=NW, G=G, fits=fits)


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
