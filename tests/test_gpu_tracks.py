"""Tracks from frame 0 on the GPU (DESIGN.md 4.9): the analytic cases of test_oracle_tracks.py through lib.warp_tracks,
then the library against the CPU restatement (tests/track_oracle.py) bit for bit -- warp_tracks on random, degenerate and
non-finite positions, Batch.submit with tracks on every solver path, scenes with and without queries, the frame-1 and
last-frame identities, a mixed run, buffer reuse and every rejection of arapb200_batch_tracks."""
import ctypes as C
import functools

import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from tests import occlusion_cases as OC
from tests import sequence_cases as SC
from tests import sequence_oracle as SO
from tests import track_cases as TC
from tests import track_oracle as TO

pytestmark = pytest.mark.gpu

KW = dict(nCont=6, nGN=2, nPCG=30)
STEPS = [0, 2, 5]
DENSE = ("flow0", "bflow0", "occ0")
QUERY = ("query_pos", "query_occ")


def _same(a, b, keys):
    for k in keys:
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


def _queries(W, H, n, seed):
    rng = np.random.default_rng(seed)
    q = np.stack([rng.integers(0, W, n), rng.integers(0, H, n)], -1).astype(np.int32)
    return np.concatenate([q, [[0, 0], [W - 1, H - 1]]]).astype(np.int32)


# ------------------------------------------------------------------------------------- analytic cases
@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
def test_integer_translation(name):
    mask = OC.TRANSLATION_MASKS[name]()
    pos = TC.offsets_positions(TC.CONSTANT)
    tr = lib.warp_tracks(pos, mask)
    tr["flow0"] = lib.warp_seq(pos, OC.rgb_for(OC.W_T, OC.H_T), mask)["flow0"]
    TC.check_offsets(tr, mask, TC.CONSTANT)


def test_leaving_the_frame_and_coming_back():
    mask = OC.TRANSLATION_MASKS["ellipse"]()
    pos = TC.offsets_positions(TC.LEAVE_RETURN)
    tr = dict(lib.warp_tracks(pos, mask), flow0=lib.warp_seq(pos, OC.rgb_for(OC.W_T, OC.H_T), mask)["flow0"])
    TC.check_offsets(tr, mask, TC.LEAVE_RETURN)
    TC.check_leave_return(tr, mask)


def test_rotation_and_repeated_frame():
    mask, pos = TC.rotation_positions()
    seq = lib.warp_seq(pos, OC.rgb_for(OC.W_R, OC.H_R), mask)
    TC.check_rotation(dict(lib.warp_tracks(pos, mask), flow0=seq["flow0"]), seq["mask"])
    rep = SC.repeated_positions()
    TC.check_repeated(dict(lib.warp_tracks(rep, mask), flow0=lib.warp_seq(rep, OC.rgb_for(OC.W_R, OC.H_R), mask)["flow0"]))


# ------------------------------------------------------------------------------------- warp_tracks bit for bit
@pytest.mark.parametrize("W,H,amp,seed", [(97, 61, 4.0, 0), (200, 120, 40.0, 1), (64, 64, 0.0, 2), (3, 2, 1.0, 3)])
def test_warp_tracks_random_vs_restatement(oracle, W, H, amp, seed):
    """Random walks of the positions, with NaN, inf and degenerate corners in the large-amplitude case."""
    rng = np.random.default_rng(seed)
    mask = np.where(rng.random((H, W)) < 0.2, 255, 0).astype(np.uint8)
    pos = (oracle.grid(W, H) + np.cumsum(rng.standard_normal((4, H, W, 2)) * amp / 2, axis=0)).astype(np.float32)
    if amp > 10:
        pos[1, 5, 5] = pos[1, 5, 6]
        pos[2, 10, 10] = np.nan
        pos[3, 12, 12] = np.inf
        pos[2, 30:33, 40:43] = pos[1, 30:33, 40:43]
    got = lib.warp_tracks(pos, mask)
    want, seq = TO.warp_tracks(pos, mask)
    _same(got, want, ("bflow0", "occ0"))
    lseq = lib.warp_seq(pos, np.zeros((H, W, 3), np.uint8), mask)
    assert np.array_equal(got["bflow0"][0], lseq["bflow"][0]) and np.array_equal(got["occ0"][0], lseq["occ"][0])
    if amp > 0 and W * H > 1000:
        assert (got["occ0"][1:] == 255).any() and (got["occ0"][1:] == 0).any() and got["bflow0"][1:].any()


# ------------------------------------------------------------------------------------- the batch, one problem
@functools.lru_cache(maxsize=None)
def _plain_want(W, H, nseg, fd, seed, steps, lm=False):
    sp = synth.synth(W, H, nseg, fd, seed) if W else synth.config("C1")
    snaps = SO.solve_states(sp.masks[0], sp.matches, list(steps), lm=lm, **KW)[3]
    seq = SO.warp_seq(snaps, sp.rgb, sp.masks[0])
    return sp, TO.tracks(snaps, seq, sp.masks[0])


def _check_plain(out, want, q=None):
    t = out["tracks"]
    _same(t, want, DENSE)
    assert np.array_equal(t["flow0"], out["seq"]["flow0"])
    if q is not None:
        _same(t, TO.gather(want, q), QUERY)


def test_submit_c1_two_launches_of_four(oracle):
    sp, want = _plain_want(0, 0, 0, 0, 0, tuple(STEPS))
    q = _queries(sp.W, sp.H, 300, 1)
    b = lib.Batch(sp.W, sp.H, 8, **KW)
    outs = [b.submit(j, sp.rgb, sp.masks[0], sp.matches, frames=STEPS, tracks=j % 2 == 0,
                     queries=q if j % 3 == 0 else None) for j in range(8)]
    b.run()
    assert b.resident_count() == 8 and b.launch_info()["problems_per_launch"] == 4
    b.close()
    for j, out in enumerate(outs):
        if j % 2 == 0:
            _same(out["tracks"], want, DENSE)
        elif j % 3 == 0:
            assert set(out["tracks"]) == set(QUERY)
        else:
            assert "tracks" not in out
        if j % 3 == 0:
            _same(out["tracks"], TO.gather(want, q), QUERY)


@pytest.mark.parametrize("kind", ["resident", "stream", "lm"])
def test_submit_three_small_problems(oracle, kind):
    b = lib.Batch(96, 80, 3, backend=lib.BACKEND_STREAM if kind == "stream" else lib.BACKEND_AUTO, **KW)
    if kind == "lm":
        b.set_option("lm", 1)
    cases = [(96, 80, 1, 2, 40 + j, (1, 3, 5) if j else (0, 4)) for j in range(3)]
    outs = []
    for j, c in enumerate(cases):
        sp = _plain_want(*c, lm=kind == "lm")[0]
        outs.append(b.submit(j, sp.rgb, sp.masks[0], sp.matches, frames=list(c[5]), tracks=True,
                             queries=_queries(96, 80, 50, j)))
    b.run()
    if kind == "resident":
        assert b.resident_count() == 3 and b.launch_info()["problems_per_launch"] == 3
    b.close()
    for j, (c, out) in enumerate(zip(cases, outs)):
        _check_plain(out, _plain_want(*c, lm=kind == "lm")[1], _queries(96, 80, 50, j))


# ------------------------------------------------------------------------------------- scenes
def _moving(sp, seed):
    A, m = synth.background_motion(sp.W, sp.H, seed)
    return A, synth.background(sp.W + 2 * m, sp.H + 2 * m, seed), (m, m)


@functools.lru_cache(maxsize=None)
def _scene_case(name, steps):
    sp = synth.config(name) if isinstance(name, str) else synth.synth(*name)
    A, bg, origin = _moving(sp, 60 + (int(name[1]) if isinstance(name, str) else name[-1]))
    path = synth.motion_path(A, steps, KW["nCont"])
    seqs, trs = [], []
    for m in sp.masks:
        snaps = SO.solve_states(m, sp.matches, list(steps), **KW)[3]
        seqs.append(SO.warp_seq(snaps, sp.rgb, m))
        trs.append(TO.tracks(snaps, seqs[-1], m))
    return sp, A, bg, origin, path, TO.scene_tracks(seqs, trs, sp.masks, path)


def _submit_scene(b, sp, A, bg, origin, frames, slot=0, out=None, nCont=KW["nCont"], **kw):
    path = synth.motion_path(A, frames, nCont) if frames else None
    return b.submit_scene(slot, sp.rgb, sp.masks, [sp.matches] * len(sp.masks), bg, A, origin=origin, frames=frames,
                          frame_motions=path, out=out, **kw)


@pytest.mark.parametrize("queries", [False, True], ids=["dense", "queries"])
@pytest.mark.parametrize("name", ["C1", "C2"])
def test_scene_against_the_restatement(oracle, name, queries):
    sp, A, bg, origin, path, want = _scene_case(name, tuple(STEPS))
    q = _queries(sp.W, sp.H, 500, 2) if queries else None
    b = lib.Batch(sp.W, sp.H, len(sp.masks), **KW)
    out = _submit_scene(b, sp, A, bg, origin, STEPS, tracks=True, queries=q)
    b.run()
    b.close()
    _same(out["tracks"], want, DENSE)
    if queries:
        _same(out["tracks"], TO.gather(want, q), QUERY)
    # frame 1 is the scene's first frame
    assert np.array_equal(out["tracks"]["bflow0"][0], out["seq"]["bflow"][0])
    assert np.array_equal(out["tracks"]["occ0"][0], out["seq"]["occ"][0])
    assert (out["tracks"]["occ0"] == 0).any() and (out["tracks"]["occ0"] == 255).any()


def test_scene_queries_only(oracle):
    sp, A, bg, origin, path, want = _scene_case("C1", tuple(STEPS))
    q = _queries(sp.W, sp.H, 2048, 3)
    b = lib.Batch(sp.W, sp.H, 1, **KW)
    out = _submit_scene(b, sp, A, bg, origin, STEPS, queries=q)
    b.run()
    b.close()
    assert set(out["tracks"]) == set(QUERY)
    _same(out["tracks"], TO.gather(want, q), QUERY)


# ------------------------------------------------------------------------------------- identities
def test_plain_frame_one_and_last_frame():
    sp = synth.synth(160, 120, 1, 2, 50)
    steps = [1, 3, KW["nCont"] - 1]
    b = lib.Batch(sp.W, sp.H, 1, **KW)
    out = b.submit(0, sp.rgb, sp.masks[0], sp.matches, extras=True, frames=steps, tracks=True)
    b.run()
    b.close()
    t, s = out["tracks"], out["seq"]
    assert np.array_equal(t["bflow0"][0], s["bflow"][0]) and np.array_equal(t["occ0"][0], s["occ"][0])
    assert np.array_equal(t["bflow0"][-1], out["bflow"]) and np.array_equal(t["occ0"][-1], out["occ"])
    assert np.array_equal(t["flow0"][-1], out["flow"])


def test_scene_last_frame_at_the_full_schedule():
    """C2 at 19 x 8 x 400 with all 19 frames: A_19 = A, so frame 19's tracks are the pair's bflow and occ."""
    sp = synth.config("C2")
    A, bg, origin = _moving(sp, 71)
    steps = list(range(19))
    b = lib.Batch(sp.W, sp.H, 4, 19, 8, 400)
    out = _submit_scene(b, sp, A, bg, origin, steps, nCont=19, tracks=True)
    b.run()
    assert b.resident_count() == 4
    b.close()
    t = out["tracks"]
    assert np.array_equal(t["bflow0"][-1], out["bflow"]) and np.array_equal(t["occ0"][-1], out["occ"])
    assert np.array_equal(t["bflow0"][0], out["seq"]["bflow"][0]) and np.array_equal(t["occ0"][0], out["seq"]["occ"][0])


# ------------------------------------------------------------------------------------- a mixed run
def test_mixed_run_changes_nothing_else():
    sp1, sp2 = synth.synth(160, 120, 3, 2, 52), synth.synth(160, 120, 2, 2, 53)
    plain = synth.synth(160, 120, 1, 2, 54)
    m1, m2 = _moving(sp1, 72), _moving(sp2, 73)
    f1, fp = [1, 3, 5], [0, 2, 4, 5]
    q = _queries(160, 120, 40, 4)
    runs = []
    for tracks in (False, True):
        b = lib.Batch(160, 120, 7, **KW)
        o1 = _submit_scene(b, sp1, *m1, f1, input_frame=True, tracks=tracks, queries=q if tracks else None)
        o2 = _submit_scene(b, sp2, *m2, [2, 5], slot=3)
        op = [b.submit(5, plain.rgb, plain.masks[0], plain.matches, extras=True, frames=fp, tracks=tracks,
                       queries=q if tracks else None),
              b.submit(6, plain.rgb, plain.masks[0], plain.matches, frames=[1, 5])]
        b.run()
        runs.append((o1, o2, op, b.launches(), b.resident_count()))
        b.close()
    (a1, a2, ap, la, ra), (g1, g2, gp, lg, rg) = runs
    K1, Kp, n1 = len(f1), len(fp), len(sp1.masks)
    assert lg == la + (n1 * (K1 - 1) + 2 * K1 + 1) + (2 * (Kp - 1) + 1) and rg == ra == 7
    keys = ("flow", "rgb", "mask", "bflow", "occ", "costs")
    _same(g1, a1, keys + ("rgb0",))
    _same(g1["seq"], a1["seq"], ("flow", "rgb", "mask", "bflow", "occ"))
    _same(g2, a2, keys)
    _same(g2["seq"], a2["seq"], ("flow", "rgb", "mask", "bflow", "occ"))
    _same(gp[0], ap[0], ("flow", "rgb", "mask", "costs", "bflow", "occ"))
    _same(gp[0]["seq"], ap[0]["seq"], SO.KEYS)
    _same(gp[1], ap[1], ("flow", "rgb", "mask", "costs"))
    _same(gp[1]["seq"], ap[1]["seq"], SO.KEYS)
    assert "tracks" in g1 and "tracks" not in g2 and "tracks" in gp[0] and "tracks" not in gp[1]
    assert np.array_equal(gp[0]["tracks"]["flow0"], gp[0]["seq"]["flow0"])
    _same(gp[0]["tracks"], TO.gather(gp[0]["tracks"], q), QUERY)
    _same(g1["tracks"], TO.gather(g1["tracks"], q), QUERY)


# ------------------------------------------------------------------------------------- buffer reuse
def test_one_batch_reuses_its_buffers():
    small, big = synth.synth(160, 120, 2, 2, 55), synth.synth(200, 150, 3, 2, 56)
    nCont = 19
    b = lib.Batch(200, 150, 3, nCont, 2, 20)
    out = None
    for sp, frames, tracks, seed in ((small, list(range(19)), True, 74), (small, [2, 9, 18], True, 75),
                                     (small, [2, 9, 18], False, 76), (big, [0, 4, 18], True, 77)):
        A, bg, origin = _moving(sp, seed)
        q = _queries(sp.W, sp.H, 30, seed) if tracks else None
        fresh = lib.Batch(200, 150, 3, nCont, 2, 20)
        want = _submit_scene(fresh, sp, A, bg, origin, frames, nCont=nCont, tracks=tracks, queries=q)
        fresh.run()
        fresh.close()
        out = _submit_scene(b, sp, A, bg, origin, frames, nCont=nCont, out=out, tracks=tracks, queries=q)
        b.run()
        assert set(out) == set(want) and ("tracks" in out) == tracks
        _same(out, want, [k for k in want if k not in ("seq", "tracks")])
        _same(out["seq"], want["seq"], list(want["seq"]))
        if tracks:
            assert set(out["tracks"]) == set(DENSE + QUERY)
            _same(out["tracks"], want["tracks"], DENSE + QUERY)
    b.close()


# ------------------------------------------------------------------------------------- rejections
def test_rejections_change_nothing():
    sp = synth.synth(96, 80, 2, 2, 57)
    A, bg, origin = _moving(sp, 78)
    W, H = sp.W, sp.H
    L = lib.load()
    L.arapb200_batch_tracks.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3
    b = lib.Batch(W, H, 7, **KW)
    q = _queries(W, H, 20, 5)
    out = _submit_scene(b, sp, A, bg, origin, [1, 3], tracks=True, queries=q)   # valid requests the rejections keep
    po = b.submit(2, sp.rgb, sp.masks[0], sp.matches, frames=[0, 4], tracks=True)
    b.submit(3, sp.rgb, sp.masks[1], sp.matches)                                   # no frames
    b.submit_scene(4, sp.rgb, sp.masks, [sp.matches] * 2, bg, A, origin=origin)    # a scene without frames
    buf = np.zeros((2, 3, H, W, 2), np.float32)
    p = buf.ctypes.data
    qq = np.ascontiguousarray(q)
    one = lambda x, y: np.array([[x, y]], np.int32)  # noqa: E731
    cases = {
        "null batch": (None, 0, p, None, None, 0, None, None, None),
        "slot -1": (b.h, -1, p, None, None, 0, None, None, None),
        "slot past the batch": (b.h, 7, p, None, None, 0, None, None, None),
        "second slot of a scene": (b.h, 1, p, None, None, 0, None, None, None),
        "problem without frames": (b.h, 3, p, None, None, 0, None, None, None),
        "scene without frames": (b.h, 4, p, None, None, 0, None, None, None),
        "empty slot": (b.h, 6, p, None, None, 0, None, None, None),
        "nothing asked for": (b.h, 0, None, None, None, 0, None, None, None),
        "negative n_queries": (b.h, 0, p, None, None, -1, qq.ctypes.data, p, None),
        "queries without query_pos": (b.h, 0, None, None, None, 2, qq.ctypes.data, None, p),
        "queries array missing": (b.h, 0, None, None, None, 2, None, p, None),
        "query_pos without queries": (b.h, 0, p, None, None, 0, None, p, None),
        "query_occ without queries": (b.h, 2, p, None, None, 0, None, None, p),
    }
    outside = [one(W, 0), one(-1, 0), one(0, H), one(0, -1)]
    for i, o in enumerate(outside):
        cases[f"query outside {i}"] = (b.h, 0, None, None, None, 1, o.ctypes.data, p, None)
    for what, args in cases.items():
        assert L.arapb200_batch_tracks(*args) != 0, what
    b.run()
    b.close()
    assert not buf.any()
    fresh = lib.Batch(W, H, 7, **KW)
    want = _submit_scene(fresh, sp, A, bg, origin, [1, 3], tracks=True, queries=q)
    pw = fresh.submit(2, sp.rgb, sp.masks[0], sp.matches, frames=[0, 4], tracks=True)
    fresh.run()
    fresh.close()
    _same(out["tracks"], want["tracks"], DENSE + QUERY)
    _same(po["tracks"], pw["tracks"], DENSE)
    # a second call replaces the first: queries only, so the dense arrays of the first stay untouched; the run drops it
    b2 = lib.Batch(W, H, 2, **KW)
    o = _submit_scene(b2, sp, A, bg, origin, [1, 3])
    b2.run()
    l0 = b2.launches()
    first = _submit_scene(b2, sp, A, bg, origin, [1, 3], tracks=True)["tracks"]
    pos = np.zeros((2, 1, 2), np.float32)
    assert L.arapb200_batch_tracks(b2.h, 0, None, None, None, 1, one(5, 7).ctypes.data, pos.ctypes.data, None) == 0
    b2.run()
    assert b2.launches() == l0 + 2 * (2 - 1) + 2 * 2 + 1          # two layers, two frames, one gather
    assert not any(v.any() for v in first.values())
    assert np.array_equal(pos, TO.gather(want["tracks"], one(5, 7))["query_pos"])
    _submit_scene(b2, sp, A, bg, origin, [1, 3], out=o)
    b2.run()
    assert b2.launches() == l0
    b2.close()
