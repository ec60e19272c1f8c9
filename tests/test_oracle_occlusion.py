"""The CPU restatement of the backward flow and occlusion (tests/occlusion_oracle.py: warp_ex on the oracle's rasteriser,
flatten_ex on pycomposite.flatten) against analytic cases that do not use its formulas (tests/occlusion_cases.py,
DESIGN.md 4.3).  CPU only."""
import numpy as np
import pytest

from oracle import pycomposite as PC
from tests import occlusion_cases as OC
from tests import occlusion_oracle as OO


@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
@pytest.mark.parametrize("t", OC.SHIFTS)
def test_integer_translation(oracle, name, t):
    mask = OC.TRANSLATION_MASKS[name]()
    flow = np.zeros((OC.H_T, OC.W_T, 2), np.float32) + np.float32(t)
    out = OO.warp_ex(flow, OC.rgb_for(OC.W_T, OC.H_T), mask, is_flow=True)
    OC.check_translation(out, mask, t)
    # the same motion given as positions
    pos = OO.warp_ex(OC.grid(OC.W_T, OC.H_T) + np.float32(t), OC.rgb_for(OC.W_T, OC.H_T), mask)
    assert all(np.array_equal(pos[k], out[k]) for k in out)


@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
def test_identity(oracle, name):
    mask = OC.TRANSLATION_MASKS[name]()
    OC.check_identity(OO.warp_ex(OC.grid(OC.W_T, OC.H_T), OC.rgb_for(OC.W_T, OC.H_T), mask), mask)


def test_small_rigid_rotation(oracle):
    mask, pos = OC.rotation_case()
    OC.check_rotation(OO.warp_ex(pos, OC.rgb_for(OC.W_R, OC.H_R), mask), mask)


def test_compression_pins_the_strict_bound(oracle):
    mask, pos = OC.compression_case()
    OC.check_compression(OO.warp_ex(pos, OC.rgb_for(OC.W_C, OC.H_C), mask))


def test_warp_ex_keeps_the_warp(oracle):
    mask, pos = OC.rotation_case()
    rgb = OC.rgb_for(OC.W_R, OC.H_R)
    out = OO.warp_ex(pos, rgb, mask)
    r, m, sp = oracle.warp(pos, rgb, mask)
    assert np.array_equal(out["rgb"], r) and np.array_equal(out["mask"], m) and np.array_equal(out["splat"], sp)


def test_two_layers_numpy_rules(oracle):
    flows, rgbs, masks, srcs, bflows = OC.layer_inputs(OO.warp_ex)
    flat = OO.flatten_ex(flows, rgbs, masks, srcs, bflows)
    OC.check_layers(flat, srcs)
    f, r, m = PC.flatten(flows, rgbs, masks)
    assert np.array_equal(flat["flow"], f) and np.array_equal(flat["rgb"], r) and np.array_equal(flat["mask"], m)


@pytest.mark.parametrize("case", ["rotation", "translation"])
def test_one_layer_flatten_is_the_warp(oracle, case):
    if case == "rotation":
        mask, pos = OC.rotation_case()
        out = OO.warp_ex(pos, OC.rgb_for(OC.W_R, OC.H_R), mask)
        flow = oracle.flow(pos)                  # the forward flow warp_ex used: pos - grid
    else:
        mask = OC.TRANSLATION_MASKS["holes"]()
        flow = np.zeros((OC.H_T, OC.W_T, 2), np.float32) + np.float32((4, -3))
        out = OO.warp_ex(flow, OC.rgb_for(OC.W_T, OC.H_T), mask, is_flow=True)
    flat = OO.flatten_ex([flow], [out["rgb"]], [out["mask"]], [mask], [out["bflow"]])
    assert np.array_equal(flat["bflow"], out["bflow"]) and np.array_equal(flat["occ"], out["occ"])
