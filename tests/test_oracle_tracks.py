"""The CPU restatement of tracks from frame 0 (tests/track_oracle.py, DESIGN.md 4.9) against analytic cases that do not
use its formulas (tests/track_cases.py), the consecutive outputs it must reproduce at frame 1, and the rejections of the
Python binding that come before any library call.  CPU only."""
import numpy as np
import pytest

from arap_flow_b200 import lib
from tests import background_oracle as BO
from tests import occlusion_cases as OC
from tests import sequence_cases as SC
from tests import sequence_oracle as SO
from tests import track_cases as TC
from tests import track_oracle as TO

IDENTITY = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
def test_integer_translation(oracle, name):
    mask = OC.TRANSLATION_MASKS[name]()
    TC.check_offsets(TO.warp_tracks(TC.offsets_positions(TC.CONSTANT), mask)[0], mask, TC.CONSTANT)


def test_leaving_the_frame_and_coming_back(oracle):
    mask = OC.TRANSLATION_MASKS["ellipse"]()
    tr, seq = TO.warp_tracks(TC.offsets_positions(TC.LEAVE_RETURN), mask)
    TC.check_offsets(tr, mask, TC.LEAVE_RETURN)
    TC.check_leave_return(tr, mask)
    # the chain of consecutive occlusions has lost the object by frame 3: nothing of frame 2 was drawn to follow
    assert not (seq["mask"][1] == 255).any()


def test_rotation_per_frame(oracle):
    mask, pos = TC.rotation_positions()
    tr, seq = TO.warp_tracks(pos, mask)
    TC.check_rotation(tr, seq["mask"])


def test_repeated_frame(oracle):
    mask = OC.rotation_case()[0]
    TC.check_repeated(TO.warp_tracks(SC.repeated_positions(), mask)[0])


def test_frame_one_is_the_consecutive_pair(oracle):
    mask, pos = TC.rotation_positions()
    tr, seq = TO.warp_tracks(pos, mask)
    assert np.array_equal(tr["bflow0"][0], seq["bflow"][0]) and np.array_equal(tr["occ0"][0], seq["occ"][0])
    assert np.array_equal(tr["flow0"], seq["flow0"])
    assert not np.array_equal(tr["bflow0"][2], seq["bflow"][2])


def _crossing_scene():
    masks, positions = TC.crossing_layers()
    rgb = OC.rgb_for(TC.W_X, TC.H_X)
    seqs = [SO.warp_seq(p, rgb, m) for p, m in zip(positions, masks)]
    trs = [TO.tracks(p, q, m) for p, q, m in zip(positions, seqs, masks)]
    return masks, seqs, trs, TO.scene_tracks(seqs, trs, masks, [IDENTITY] * 3)


def test_crossing_layers(oracle):
    masks, seqs, trs, tr = _crossing_scene()
    TC.check_crossing(tr, masks)


def test_owner_selection_is_not_the_flatten(oracle):
    """Where B lies on A at frame 2, the flatten's rule gives A's pixel B's flow; a track keeps A's."""
    masks, seqs, trs, tr = _crossing_scene()
    hit = TC.crossed_pixels()
    flat = BO.composite([t["flow0"][1] for t in trs], [q["rgb"][1] for q in seqs], [q["mask"][1] for q in seqs], masks,
                        [t["bflow0"][1] for t in trs], np.zeros((1, 1, 3), np.uint8), BO.coeffs(IDENTITY))
    assert (flat["flow"][hit] == (40, 0)).all()
    assert not tr["flow0"][1][hit].any()
    assert np.array_equal(flat["bflow"], tr["bflow0"][1]) and np.array_equal(flat["occ"], tr["occ0"][1])


def test_scene_frame_one_is_the_consecutive_composite(oracle):
    """Frame 1 of a scene over a moving background: the scene's frame-1 composite (lib.composite_seq's rule)."""
    masks, positions = TC.crossing_layers()
    rgb = OC.rgb_for(TC.W_X, TC.H_X)
    seqs = [SO.warp_seq(p, rgb, m) for p, m in zip(positions, masks)]
    trs = [TO.tracks(p, q, m) for p, q, m in zip(positions, seqs, masks)]
    th = np.deg2rad(2.0)
    motions = [np.array([[np.cos(k * th), -np.sin(k * th), 1.5 * k], [np.sin(k * th), np.cos(k * th), -0.5 * k]])
               for k in (1, 2, 3)]
    tr = TO.scene_tracks(seqs, trs, masks, motions)
    c1 = BO.composite([q["flow"][0] for q in seqs], [q["rgb"][0] for q in seqs], [q["mask"][0] for q in seqs], masks,
                      [q["bflow"][0] for q in seqs], np.zeros((1, 1, 3), np.uint8), BO.coeffs(motions[0]))
    assert np.array_equal(tr["bflow0"][0], c1["bflow"]) and np.array_equal(tr["occ0"][0], c1["occ"])
    own = TO.owner(masks, masks[0].shape)
    assert np.array_equal(tr["flow0"][0][own < 0], c1["flow"][own < 0])
    # the background's flow from frame 0 is A_k(p) - p, to within binary32 rounding of the analytic map
    g = OC.grid(TC.W_X, TC.H_X).astype(np.float64)
    for k, A in enumerate(motions):
        exact = g @ A[:, :2].T + A[:, 2] - g
        assert np.abs(tr["flow0"][k][own < 0] - exact[own < 0]).max() < 1e-3


def test_gather():
    rng = np.random.default_rng(3)
    K, H, W = 4, 7, 9
    tr = dict(flow0=rng.standard_normal((K, H, W, 2)).astype(np.float32) * 5,
              occ0=rng.integers(0, 2, (K, H, W)).astype(np.uint8) * 255)
    q = np.array([[0, 0], [W - 1, H - 1], [3, 5], [3, 5], [8, 0]], np.int32)
    g = TO.gather(tr, q)
    for k in range(K):
        for i, (x, y) in enumerate(q):
            assert g["query_pos"][k, i, 0] == np.float32(x) + tr["flow0"][k, y, x, 0]
            assert g["query_pos"][k, i, 1] == np.float32(y) + tr["flow0"][k, y, x, 1]
            assert g["query_occ"][k, i] == tr["occ0"][k, y, x]
    assert g["query_pos"].shape == (K, len(q), 2) and g["query_occ"].shape == (K, len(q))


def _unbound_batch():
    """A Batch whose handle is NULL: any call that reaches the library fails with RuntimeError, so a ValueError proves the
    binding refused the request before calling it."""
    b = lib.Batch.__new__(lib.Batch)
    b.L, b.h, b.nCont, b.nGN, b._keep = lib.load(), None, 6, 2, {}
    return b


@pytest.mark.parametrize("kw", [dict(tracks=True), dict(queries=[[1, 1]]), dict(tracks=True, frames=[]),
                                dict(tracks=True, frames=[0, 2], queries=[[9, 0]]),
                                dict(frames=[0, 2], queries=[[0, -1]]), dict(frames=[1], queries=[[0.5, 1]])],
                         ids=["tracks", "queries", "empty frames", "x past the frame", "negative y", "sub-pixel"])
def test_python_rejections_before_the_library(kw):
    b = _unbound_batch()
    rgb, mask = np.zeros((6, 9, 3), np.uint8), np.zeros((6, 9), np.uint8)
    with pytest.raises(ValueError):
        b.submit(0, rgb, mask, np.zeros((0, 4), np.int32), **kw)
    with pytest.raises(ValueError):
        b.submit_scene(0, rgb, [mask], [np.zeros((0, 4), np.int32)], np.zeros((6, 9, 3), np.uint8), IDENTITY,
                       frame_motions=[IDENTITY] * len(kw.get("frames") or []), **kw)
    assert not b._keep
