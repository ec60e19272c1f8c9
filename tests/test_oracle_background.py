"""The CPU restatement of the composite over a moving background (tests/background_oracle.py) against analytic cases
that do not use its formulas (tests/background_cases.py, DESIGN.md 4.5), and the argument checks of arapb200_composite,
which reject before any CUDA call.  CPU only."""
import ctypes as C

import numpy as np
import pytest

from arap_flow_b200 import lib, synth
from tests import background_cases as BC
from tests import background_oracle as BO
from tests import occlusion_oracle as OO

comp = BO.composite_api


@pytest.mark.parametrize("n", [1, 2])
def test_identity_is_flatten_ex_with_add_bg(oracle, n):
    BC.check_identity_is_flatten(comp, OO.warp_ex, n)


def test_identity_without_layers_is_the_crop():
    BC.check_identity_no_layers(comp)


@pytest.mark.parametrize("t", BC.BG_SHIFTS)
def test_integer_background_translation(t):
    BC.check_integer_translation(comp, t)


def test_half_pixel_shift_rounds_to_nearest_even():
    BC.check_half_pixel(comp)


def test_half_scale_pins_the_strict_bound():
    BC.check_half_scale(comp)


@pytest.mark.parametrize("deg,scale", BC.ZOOMS)
def test_rotation_and_zoom_in(deg, scale):
    BC.check_rotation_zoom(comp, deg, scale)


def test_moving_object_over_moving_background(oracle):
    BC.check_object_over_background(comp, OO.warp_ex)


@pytest.mark.parametrize("t", BC.CLAMP_SHIFTS)
def test_clamping_replicates_the_edge(t):
    BC.check_clamping(comp, t)


def test_same_motion_is_a_still_background():
    BC.check_same_motion_is_still(comp)


def test_chord_path_composes_to_the_pair():
    BC.check_chord_path_composes(comp)


def test_identity_maps_are_exact():
    for A in (BC.I2, np.eye(2, 3) * 1.0):
        assert np.array_equal(BO.coeffs(A), np.stack([BC.I2] * 3).astype(np.float32))
        assert np.array_equal(BO.coeffs(A, A), np.stack([BC.I2] * 3).astype(np.float32))


def test_synth_background_keeps_synth_draws():
    """The background helpers draw from their own generators: synth()'s outputs stay as they were."""
    a = synth.synth(64, 48, 2, 2, 5)
    synth.background(64, 48, 5), synth.background_motion(64, 48, 5)
    b = synth.synth(64, 48, 2, 2, 5)
    assert np.array_equal(a.rgb, b.rgb) and np.array_equal(a.matches, b.matches)
    assert np.array_equal(synth.background(64, 48, 5), synth._texture(np.random.default_rng(5), 64, 48))


@pytest.mark.parametrize("seed", range(8))
def test_background_motion_margin_needs_no_clamping(seed):
    """At the margin m every binary32 sample point is inside the background; at m - 1 some point is outside or within
    the 0.01 px kept spare."""
    W, H = 854, 480
    A, m = synth.background_motion(W, H, seed)
    assert m > 0
    s = BO.apply(BO.coeffs(A)[2], W, H)

    def fits(m, spare):
        return ((s + np.float32(m) >= spare).all() and (s[..., 0] + m <= W + 2 * m - 1 - spare).all()
                and (s[..., 1] + m <= H + 2 * m - 1 - spare).all())

    assert fits(m, 0) and not fits(m - 1, 0.01)


# ------------------------------------------------------------------------------------- argument rejection
def _call(**over):
    """arapb200_composite on a valid 8 x 6 two-layer case with `over` replacing arguments; returns (rc, outputs), the
    outputs pre-filled with a sentinel."""
    W, H, n = 8, 6, 2
    keep = []

    def arr(shape, dt):
        a = np.zeros(shape, dt)
        keep.append(a)
        return a.ctypes.data

    P = C.c_void_p * n
    layers = {k: P(*[arr(s, dt) for _ in range(n)]) for k, s, dt in
              (("flows", (H, W, 2), np.float32), ("rgbs", (H, W, 3), np.uint8), ("masks", (H, W), np.uint8),
               ("src_masks", (H, W), np.uint8), ("bflows", (H, W, 2), np.float32))}
    outs = dict(out_flow=np.full((H, W, 2), 7, np.float32), out_rgb=np.full((H, W, 3), 7, np.uint8),
                out_mask=np.full((H, W), 7, np.uint8), out_bflow=np.full((H, W, 2), 7, np.float32),
                out_occ=np.full((H, W), 7, np.uint8), out_coeffs=np.full((3, 2, 3), 7, np.float32))
    motion_to = np.array([[1.0, 0.1, 2.0], [0.0, 0.9, -1.0]])
    a = dict(W=W, H=H, n_layers=n, **layers, bgW=W, bgH=H, background=arr((H, W, 3), np.uint8), bg_x=0, bg_y=0,
             motion_from=None, motion_to=motion_to.ctypes.data, **{k: v.ctypes.data for k, v in outs.items()})
    a.update(over)
    L = lib.load()
    L.arapb200_composite.argtypes = lib.COMPOSITE_ARGTYPES
    order = ("W H n_layers flows rgbs masks src_masks bflows bgW bgH background bg_x bg_y motion_from motion_to "
             "out_flow out_rgb out_mask out_bflow out_occ out_coeffs").split()
    rc = L.arapb200_composite(*[a[k] for k in order])
    return rc, outs


def _m(a):
    a = np.asarray(a, np.float64)
    _m.keep.append(a)
    return a.ctypes.data


_m.keep = []
NULL2 = (C.c_void_p * 2)(None, None)
REJECTED = {
    "W": dict(W=0), "H": dict(H=-3), "n_negative": dict(n_layers=-1), "n_too_many": dict(n_layers=33),
    "no_flows": dict(flows=None), "no_rgbs": dict(rgbs=None), "no_masks": dict(masks=None),
    "no_src_masks": dict(src_masks=None), "null_layer_entry": dict(src_masks=NULL2),
    "bflow_without_bflows": dict(bflows=None, out_occ=None), "occ_without_bflows": dict(bflows=None, out_bflow=None),
    "no_background": dict(background=None), "bgW": dict(bgW=0), "bgH": dict(bgH=-1), "no_motion_to": dict(motion_to=None),
    "nan_motion": dict(motion_to=_m([[1, 0, np.nan], [0, 1, 0]])),
    "inf_motion_from": dict(motion_from=_m([[1, 0, 0], [0, np.inf, 0]])),
    "singular_to": dict(motion_to=_m([[1, 2, 0], [2, 4, 0]])), "singular_from": dict(motion_from=_m([[0, 0, 0], [0, 0, 0]])),
    "overflowing_maps": dict(motion_to=_m([[1e-300, 0, 0], [0, 1e-300, 0]])),
    "no_out_flow": dict(out_flow=None), "no_out_rgb": dict(out_rgb=None), "no_out_mask": dict(out_mask=None),
}


@pytest.mark.parametrize("case", sorted(REJECTED))
def test_bad_arguments_are_rejected_before_any_cuda_call(case):
    """Return code 1 (a CUDA call on a machine without a GPU would give 2), and nothing written."""
    rc, outs = _call(**REJECTED[case])
    assert rc == 1, rc
    for k, v in outs.items():
        assert (v == 7).all(), k


def test_lib_composite_raises_on_rejection():
    bg = np.zeros((6, 8, 3), np.uint8)
    with pytest.raises(RuntimeError, match="code 1"):
        lib.composite([], [], [], [], [], bg, [[1, 0, 0], [0, 0, 0]], shape=(6, 8))
    with pytest.raises(ValueError):
        lib.composite([], [], [], [], [], bg, np.eye(3), shape=(6, 8))
