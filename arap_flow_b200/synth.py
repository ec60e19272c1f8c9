"""Synthetic inputs of the shapes BASELINE.json names (SURVEY.md 8d).

Everything is produced in the reference's own formats: an RGB image (uint8 HxWx3), an ARAP mask per
segment (uint8 HxW, 0 = deform this pixel, 255 = static background; para_gen.py:515-517, 526-527) and
a DeepMatching-like match list (int32 n x 4: x1 y1 x2 y2; para_gen.py:476-479).  The app itself adds
the image-border pins (ARAP/deformation/src/main.cpp:130-136), so they are NOT part of the list.
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np


@dataclasses.dataclass
class SynthPair:
    W: int
    H: int
    rgb: np.ndarray          # uint8 [H, W, 3]
    labels: np.ndarray       # int32 [H, W], 0 = background, s = segment id
    masks: list              # list of uint8 [H, W] ARAP masks (0 on the segment, 255 elsewhere)
    matches: np.ndarray      # int32 [n, 4]
    seed: int
    fd: int


def _value_noise(rng: np.random.Generator, W: int, H: int) -> np.ndarray:
    out = np.zeros((H, W), dtype=np.float64)
    ys = np.arange(H, dtype=np.float64)
    xs = np.arange(W, dtype=np.float64)
    for cell, amp in ((64, 1.0), (32, 0.5), (16, 0.25), (8, 0.125)):
        gh, gw = H // cell + 2, W // cell + 2
        g = rng.random((gh, gw))
        fy, fx = ys / cell, xs / cell
        iy, ix = fy.astype(np.int64), fx.astype(np.int64)
        ty, tx = (fy - iy)[:, None], (fx - ix)[None, :]
        a = g[iy[:, None], ix[None, :]]
        b = g[iy[:, None], ix[None, :] + 1]
        c = g[iy[:, None] + 1, ix[None, :]]
        d = g[iy[:, None] + 1, ix[None, :] + 1]
        out += amp * ((a * (1 - tx) + b * tx) * (1 - ty) + (c * (1 - tx) + d * tx) * ty)
    return out


def _texture(rng: np.random.Generator, W: int, H: int) -> np.ndarray:
    chans = []
    for _ in range(3):
        v = _value_noise(rng, W, H)
        v = (v - v.min()) / max(v.max() - v.min(), 1e-12)
        chans.append(16.0 + v * (240.0 - 16.0))
    return np.clip(np.rint(np.stack(chans, axis=-1)), 0, 255).astype(np.uint8)


def synth(W: int, H: int, nseg: int = 1, fd: int = 1, seed: int = 0, axes=None) -> SynthPair:
    """`axes` = (ax, ay) as fractions of (W, H) overrides the single-segment ellipse (C4 uses 0.46, 0.46)."""
    rng = np.random.default_rng(seed)
    rgb = _texture(rng, W, H)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    labels = np.zeros((H, W), dtype=np.int32)
    g = int(math.ceil(math.sqrt(nseg)))
    inside = (xx >= 2) & (xx < W - 2) & (yy >= 2) & (yy < H - 2)
    for s in range(1, nseg + 1):
        if nseg == 1:
            cx, cy = W / 2.0, H / 2.0
            fa = axes if axes is not None else (0.30, 0.35)
            ax, ay, th = fa[0] * W, fa[1] * H, 0.0
        else:
            gi, gj = (s - 1) % g, (s - 1) // g
            cx = (gi + 0.5 + rng.uniform(-0.15, 0.15)) * W / g
            cy = (gj + 0.5 + rng.uniform(-0.15, 0.15)) * H / g
            ax = rng.uniform(0.18, 0.28) * min(W, H)
            ay = rng.uniform(0.18, 0.28) * min(W, H)
            th = rng.uniform(0.0, math.pi)
        c, sn = math.cos(th), math.sin(th)
        u = (xx - cx) * c + (yy - cy) * sn
        v = -(xx - cx) * sn + (yy - cy) * c
        sel = ((u / ax) ** 2 + (v / ay) ** 2 <= 1.0) & inside
        labels[sel] = s
    masks = []
    if nseg == 1:
        masks.append(np.where(labels > 0, 0, 255).astype(np.uint8))
    else:
        for s in range(1, nseg + 1):
            masks.append(np.where(labels == s, 0, 255).astype(np.uint8))
    # DeepMatching-like matches on the 8-px lattice
    rows = []
    rot = math.radians(1.5)
    rc, rs = math.cos(rot) - 1.0, math.sin(rot)
    for s in range(1, nseg + 1):
        seg = labels == s
        if not seg.any():
            continue
        cyx = np.argwhere(seg).mean(axis=0)
        ccy, ccx = cyx[0], cyx[1]
        for y in range(4, H, 8):
            for x in range(4, W, 8):
                if not seg[y, x]:
                    continue
                rx, ry = x - ccx, y - ccy
                dx = fd * ((rc * rx - rs * ry) + 2.0) + 1.5 * fd * math.sin(2 * math.pi * y / (W / 2.0))
                dy = fd * ((rs * rx + rc * ry) - 1.0) + 1.5 * fd * math.cos(2 * math.pi * x / (W / 2.0))
                nrm = math.hypot(dx, dy)
                tx, ty = x + int(round(dx)), y + int(round(dy))
                if 0.0 < nrm < 60.0 and 0 <= tx < W and 0 <= ty < H:
                    rows.append((x, y, tx, ty))
    matches = np.asarray(rows, dtype=np.int32).reshape(-1, 4)
    return SynthPair(W, H, rgb, labels, masks, matches, seed, fd)


# The five BASELINE.json configurations (SURVEY.md 8d table)
def config(name: str, index: int = 0) -> SynthPair:
    if name == "C0":
        return synth(64, 64, 1, 1, 0 + index)
    if name == "C1":
        return synth(854, 480, 1, 1, 1000 + index)
    if name == "C2":
        return synth(854, 480, 4, 3, 2000 + index)
    if name == "C3":
        return synth(1024, 436, 1, 5, 3000 + index)
    if name == "C4":
        return synth(1920, 1080, 1, 1, 4000 + index, axes=(0.46, 0.46))
    raise ValueError(name)


# ---- background motion (DESIGN.md 4.5): own generators, so that synth()'s draws stay as they are -------------------
def background(W: int, H: int, seed: int = 0) -> np.ndarray:
    """A background image (uint8 [H, W, 3]) textured as synth()'s images are."""
    return _texture(np.random.default_rng(seed), W, H)


SHIFT_FRAC = 0.05   # translation: uniform in +-5 % of W (x) and of H (y)
ROT_DEG = 5.0       # rotation: uniform in +-5 degrees
SCALE = 0.05        # scale: uniform in [0.95, 1.05]


def background_margin(A, W: int, H: int) -> int:
    """The smallest integer m such that a (W+2m) x (H+2m) background at origin (m, m) covers inv(A) of the whole frame
    with 0.01 px to spare for binary32 evaluation, i.e. such that the composite never clamps a sample."""
    A = np.asarray(A, np.float64)
    Ai = np.linalg.inv(np.vstack([A, [0.0, 0.0, 1.0]]))[:2]
    corners = np.array([[0, 0, 1], [W - 1, 0, 1], [0, H - 1, 1], [W - 1, H - 1, 1]], np.float64)
    u = corners @ Ai.T          # the preimage of the frame is the parallelogram of its corners' preimages
    over = max(0.0, -u[:, 0].min(), -u[:, 1].min(), u[:, 0].max() - (W - 1), u[:, 1].max() - (H - 1))
    return int(math.ceil(over + 0.01)) if over > 0 else 0


def background_motion(W: int, H: int, seed: int = 0):
    """A random affine background motion about the frame centre, FlyingChairs-style: A(u) = c + s R(th) (u - c) + t with
    t uniform in +-SHIFT_FRAC (W, H), th in +-ROT_DEG degrees, s in [1 - SCALE, 1 + SCALE].  Returns (A float64 [2, 3],
    m = background_margin(A, W, H))."""
    rng = np.random.default_rng(seed)
    t = rng.uniform(-SHIFT_FRAC, SHIFT_FRAC, 2) * (W, H)
    th = math.radians(rng.uniform(-ROT_DEG, ROT_DEG))
    s = rng.uniform(1.0 - SCALE, 1.0 + SCALE)
    c = np.array([(W - 1) / 2.0, (H - 1) / 2.0])
    R = s * np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])
    A = np.hstack([R, (c - R @ c + t)[:, None]])
    return A, background_margin(A, W, H)


def motion_path(A, steps, nCont: int) -> list:
    """The chord path of a pair motion A for the frames of a sequence (DESIGN.md 4.4): A_k = (1 - a_k) I + a_k A with
    a_k = (t_k + 1) / nCont for the continuation steps t_k, as the match constraints move.  Returns [A_1 .. A_K]."""
    A = np.asarray(A, np.float64)
    I = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])
    return [(1.0 - (t + 1) / nCont) * I + ((t + 1) / nCont) * A for t in steps]
