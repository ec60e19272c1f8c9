"""CPU restatement of a scene's motion blur (DESIGN.md 4.8), for the tests.

The schedule is binary64 in the documented order (numpy never contracts a * b + c into an FMA) with S_map derived by
tests/background_oracle.py's inverse and rounded once to binary32; the lerp is numpy float32, one rounding per
operation; each sub-frame warps every layer with the oracle's rasteriser (oracle.pyoracle.warp), takes the front layer
from the warped masks and samples the background with background_oracle.sample; the mean is integer arithmetic.  Held to
cases that do not use these formulas by tests/test_oracle_blur.py.
"""
import math

import numpy as np

from oracle import pyoracle as O
from tests import background_oracle as BO

F = np.float32
I2 = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def schedule(nCont, steps, motion, frame_motions, n_samples, shutter, image):
    """(j0 int32[S], w float32[S], smap float32[S,2,3]) of image -1 (frame 0), 0 (the pair) or k (frame k)."""
    steps = [] if steps is None else [int(t) for t in steps]
    K = len(steps)
    fm = [np.asarray(m, np.float64) for m in (frame_motions if K else [])]
    A = np.asarray(motion, np.float64)
    if image == 0:
        i_hi, delta, A_hi, A_prev = nCont - 1, nCont, A, I2
    elif image > 0:
        i_hi = steps[image - 1]
        delta = i_hi - (steps[image - 2] if image > 1 else -1)
        A_hi, A_prev = fm[image - 1], (fm[image - 2] if image > 1 else I2)
    else:
        i_hi, delta, A_hi, A_prev = -1, (steps[0] + 1 if K else nCont), I2, None
    D = A_prev - A_hi if A_prev is not None else I2 - (fm[0] if K else A)
    S = n_samples
    j0, w, smap = np.zeros(S, np.int32), np.zeros(S, F), np.zeros((S, 2, 3), F)
    for j in range(S):
        u = 0.0 if S == 1 else (shutter * j) / (S - 1)
        i = i_hi - u * delta
        Ai = A_prev if (A_prev is not None and u == 1.0) else A_hi + u * D
        j0[j] = min(max(math.floor(i), -1), nCont - 2)
        w[j] = F(i - int(j0[j]))
        smap[j] = BO.inverse(Ai).astype(F)
    return j0, w, smap


def lerp(Qa, Qb, w):
    """State positions at weight w: Qa at w == 0, Qb at w == 1, else Qa + w (Qb - Qa) in float32."""
    if w == 0:
        return np.asarray(Qa, F)
    if w == 1:
        return np.asarray(Qb, F)
    Qa, Qb = np.asarray(Qa, F), np.asarray(Qb, F)
    with np.errstate(all="ignore"):
        return Qa + F(w) * (Qb - Qa)


def render(positions, rgb, masks, background, smap, origin=(0, 0)):
    """One sub-frame: every layer warped at its positions, the last layer with a non-zero warped mask in front, the
    background sampled through smap elsewhere."""
    H, W = masks[0].shape
    with np.errstate(all="ignore"):
        out = BO.sample(background, BO.apply(np.asarray(smap, F), W, H) + np.array(origin, F))
    for P, m in zip(positions, masks):
        r, wm, _ = O.warp(P, rgb, m)
        out = np.where((wm != 0)[..., None], r, out)
    return out


def blur_image(states, rgb, masks, background, origin, nCont, steps, motion, frame_motions, n_samples, shutter, image):
    """The blurred image: states[s] maps a continuation step t to layer s's X after it (the grid is state -1)."""
    H, W = masks[0].shape
    j0, w, smap = schedule(nCont, steps, motion, frame_motions, n_samples, shutter, image)
    grid = O.grid(W, H)
    acc = np.zeros((H, W, 3), np.int64)
    for j in range(n_samples):
        def at(s, t):
            return grid if t < 0 else states[s][t]
        pos = [lerp(at(s, j0[j]) if w[j] != 1 else None, at(s, j0[j] + 1) if w[j] != 0 else None, w[j])
               for s in range(len(masks))]
        acc += render(pos, rgb, masks, background, smap[j], origin)
    return ((acc + n_samples // 2) // n_samples).astype(np.uint8)
