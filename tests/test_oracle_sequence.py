"""The CPU restatement of frame sequences (tests/sequence_oracle.py, DESIGN.md 4.4) against the oracle's own solve, the
single-warp restatement of DESIGN.md 4.3 and analytic sequences that do not use its formulas (tests/sequence_cases.py).
CPU only."""
import numpy as np
import pytest

from arap_flow_b200 import synth
from tests import occlusion_cases as OC
from tests import occlusion_oracle as OO
from tests import sequence_cases as SC
from tests import sequence_oracle as SO

KW = dict(nCont=4, nGN=2, nPCG=20)


@pytest.mark.parametrize("lm", [False, True])
def test_schedule_loop_is_the_oracle_solve(oracle, lm):
    s = synth.synth(96, 80, 1, 2, 11)
    X, A, costs, snaps = SO.solve_states(s.masks[0], s.matches, range(KW["nCont"]), lm=lm, **KW)
    if lm:
        Xo, Ao, co = oracle.solve_lm(s.masks[0], s.matches, **KW)[:3]
    else:
        Xo, Ao, co = oracle.solve(s.masks[0], s.matches, **KW)
    assert np.array_equal(X, Xo) and np.array_equal(A, Ao) and np.array_equal(costs, co)
    assert np.array_equal(snaps[-1], Xo) and len(snaps) == KW["nCont"]
    assert not np.array_equal(snaps[0], snaps[-1])
    part = SO.solve_states(s.masks[0], s.matches, [1, 3], lm=lm, **KW)[3]
    assert np.array_equal(part, snaps[[1, 3]])


def test_interp_against_the_grid_is_the_backward_flow(oracle):
    rng = np.random.default_rng(5)
    W, H = 97, 61
    mask = np.where(rng.random((H, W)) < 0.2, 255, 0).astype(np.uint8)
    pos = (oracle.grid(W, H) + rng.standard_normal((H, W, 2)) * 3).astype(np.float32)
    z = oracle.warp(pos, OC.rgb_for(W, H), mask)[2]
    assert np.array_equal(SO.interp(z, pos, oracle.grid(W, H)), OO.backward_flow(pos, z))


def test_frame_one_is_the_single_warp(oracle):
    mask, pos = OC.rotation_case()
    rgb = OC.rgb_for(OC.W_R, OC.H_R)
    seq = SO.warp_seq(SC.rotation_positions(), rgb, mask)
    ex = OO.warp_ex(pos, rgb, mask)
    for k in ("rgb", "mask", "splat", "bflow", "occ"):
        assert np.array_equal(seq[k][0], ex[k]), k
    assert np.array_equal(seq["flow"][0], oracle.flow(pos)) and np.array_equal(seq["flow0"][0], oracle.flow(pos))


@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
@pytest.mark.parametrize("t", OC.SHIFTS)
def test_constant_velocity_translation(oracle, name, t):
    mask = OC.TRANSLATION_MASKS[name]()
    SC.check_translation(SO.warp_seq(SC.translation_positions(t), OC.rgb_for(OC.W_T, OC.H_T), mask), mask, t)


def test_rotation_per_frame(oracle):
    mask = OC.rotation_case()[0]
    SC.check_rotation(SO.warp_seq(SC.rotation_positions(), OC.rgb_for(OC.W_R, OC.H_R), mask))


def test_repeated_frame(oracle):
    mask = OC.rotation_case()[0]
    SC.check_repeated(SO.warp_seq(SC.repeated_positions(), OC.rgb_for(OC.W_R, OC.H_R), mask))


def test_compression_pins_the_strict_bound(oracle):
    mask, pos = SC.compression_positions()
    SC.check_compression(SO.warp_seq(pos, OC.rgb_for(OC.W_C, OC.H_C), mask))


def test_frames_are_sampled_from_frame_zero(oracle):
    """Frame k is the warp of P_k from the input image, whatever the frames before it were."""
    mask = OC.rotation_case()[0]
    rgb = OC.rgb_for(OC.W_R, OC.H_R)
    P = SC.rotation_positions()
    seq = SO.warp_seq(P, rgb, mask)
    r, m, z = oracle.warp(P[2], rgb, mask)
    assert np.array_equal(seq["rgb"][2], r) and np.array_equal(seq["mask"][2], m) and np.array_equal(seq["splat"][2], z)
