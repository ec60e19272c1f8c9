"""The oracle against the reference's own golden vectors (SURVEY.md 8c) -- CPU only."""
import json
import os

import numpy as np
import pytest

from arap_flow_b200 import flowio

from .helpers import cat512_flo


def _cat(gold, tmp_path):
    rgb = flowio.read_png_rgb(os.path.join(gold, "cat512_iRGB.png"))
    msk = flowio.read_png_mask_red(os.path.join(gold, "cat512_iMsk.png"))
    flo = flowio.read_flo(cat512_flo(tmp_path))
    return rgb, msk, flo


def test_warp_oracle_matches_shipped_golden_mask(oracle, gold, tmp_path):
    rgb, msk, flo = _cat(gold, tmp_path)
    o_rgb, o_m, sp = oracle.warp(oracle.flow_to_pos(flo), rgb, msk)
    g_m = flowio.read_png_rgb(os.path.join(gold, "cat512_wMsk.png"))
    assert np.array_equal(o_m, g_m[..., 0]) and np.array_equal(g_m[..., 0], g_m[..., 2])
    assert int((sp != 0).sum()) == int((o_m == 255).sum()) == 105530
    # shipped RGB golden was rasterised from un-rounded positions: +-1 level on < 0.5 % of pixels (SURVEY.md 4)
    g_rgb = flowio.read_png_rgb(os.path.join(gold, "cat512_wRGB.png")).astype(int)
    d = np.abs(o_rgb.astype(int) - g_rgb)
    assert d.max() <= 1 and (d.max(-1) > 0).mean() < 0.005


def test_warp_oracle_bit_exact_vs_reference_tool(oracle, gold, tmp_path):
    """cat512 RGB and three synthetic cases (folds, out-of-frame motion, ragged masks, identity) produced by the
    reference's own warp_image binary (tools/make_golden.py)."""
    rgb, msk, flo = _cat(gold, tmp_path)
    o_rgb, _, _ = oracle.warp(oracle.flow_to_pos(flo), rgb, msk)
    assert np.array_equal(o_rgb, flowio.read_png_rgb(os.path.join(gold, "cat512_reftool_wRGB.png")))
    z = np.load(os.path.join(gold, "warp_reftool_cases.npz"))
    for name in ("warp_a", "warp_b", "warp_c"):
        r, m, sp = oracle.warp(oracle.flow_to_pos(z[f"{name}__flow"]), z[f"{name}__rgb"], z[f"{name}__mask"])
        assert np.array_equal(r, z[f"{name}__ref_rgb"]), name
        assert np.array_equal(m, z[f"{name}__ref_mask"]), name


def test_warp_oracle_live_reference_binary(oracle, gold, tmp_path):
    """When oracle/_ref/warp_image_ref is present (build container, or shipped prebuilt), run it live."""
    if not os.path.exists(oracle.REF_WARP_BIN):
        pytest.skip("reference warp binary not built")
    import subprocess
    from arap_flow_b200 import synth
    sp = synth.synth(80, 60, 1, 3, 77)
    rng = np.random.default_rng(5)
    fl = (rng.standard_normal((60, 80, 2)) * 2.0).astype(np.float32)
    p = {k: str(tmp_path / k) for k in ("i.png", "m.png", "f.flo", "o.png", "om.png")}
    flowio.write_png(p["i.png"], sp.rgb)
    flowio.write_png(p["m.png"], np.repeat(sp.masks[0][..., None], 3, 2))
    flowio.write_flo(p["f.flo"], fl)
    subprocess.check_call([oracle.REF_WARP_BIN, p["i.png"], p["m.png"], p["f.flo"], p["o.png"], p["om.png"]],
                          stdout=subprocess.DEVNULL)
    r, m, _ = oracle.warp(oracle.flow_to_pos(fl), sp.rgb, sp.masks[0])
    assert np.array_equal(r, flowio.read_png_rgb(p["o.png"]))
    assert np.array_equal(m, flowio.read_png_rgb(p["om.png"])[..., 0])


def test_solve_pin_record(gold):
    """The recorded full-schedule oracle solve on cat512 (tools/make_golden.py --solve): weak end-to-end pin."""
    with open(os.path.join(gold, "cat512_oracle_pin.json")) as f:
        pin = json.load(f)
    assert pin["active_px"] == 101406
    assert pin["off_object_max_abs_flow"] == 0.0
    assert pin["constraint_err_px_max"] < 5e-3          # golden itself: 3.9e-3
    assert pin["mean_epe_px"] < 0.35                      # chaotic regime, SURVEY.md 8c expects 0.2-0.3
    assert pin["median_epe_px"] < 0.12


def test_solve_energy_pin_vs_shipped_golden(oracle, gold, tmp_path):
    """Energy-level anchor for the solve (the trajectory-level one is chaotic, see test_solve_pin_record): evaluate the
    ARAP energy AS DEFINED (arap_plan.t:13-23; float64 residuals, angles at their closed-form optimum for the given
    positions) at the reference's shipped result cat512_iFlo.flo and at the oracle's recorded full-schedule result.  Both
    must have minimised the same energy to the same level."""
    from .helpers import optimal_angles
    rgb, msk, flo_gold = _cat(gold, tmp_path)
    flo_ours = np.load(os.path.join(gold, "cat512_oracle_flow.npz"))["flow"]
    cstr = flowio.read_constraints(os.path.join(gold, "cat512_iCstr.txt"))
    H, W = msk.shape
    U = oracle.grid(W, H)
    Cn = oracle.constraint_image(msk, oracle.with_border_pins(cstr, W, H), 1.0)
    act = msk == 0
    E = {}
    for name, fl in (("golden", flo_gold), ("oracle", flo_ours)):
        X = (U + np.where(act[..., None], fl, 0)).astype(np.float32)
        A = optimal_angles(X, U, act)
        r = oracle.residuals_f64(X, A, U, Cn, msk.astype(np.float32))
        E[name] = (0.5 * float((r[..., :8] ** 2).sum()), 0.5 * float((r[..., 8:] ** 2).sum()))
    (rg, fg), (ro, fo) = E["golden"], E["oracle"]
    # recorded when the fixture was made: rigidity 44.762 vs 45.413, fit 2.78e-3 vs 2.73e-3
    assert abs(ro - rg) / rg < 0.02, E
    assert abs(fo - fg) / fg < 0.05, E
    assert 40.0 < rg < 50.0 and fg < 5e-3, E


@pytest.mark.slow
def test_solve_cat512_full(oracle, gold, tmp_path):
    rgb, msk, flo = _cat(gold, tmp_path)
    cstr = flowio.read_constraints(os.path.join(gold, "cat512_iCstr.txt"))
    X, A, costs = oracle.solve(msk, cstr)
    fl = oracle.flow(X)
    z = np.load(os.path.join(gold, "cat512_oracle_flow.npz"))
    assert np.array_equal(fl, z["flow"])  # the oracle is deterministic


def test_composite_restatement_vs_para_gen_itself(gold):
    """oracle/pycomposite.py against para_gen.py's OWN valid_cnstr / add_bg / flatten, executed on seeded inputs by
    tools/make_golden.py --para-gen (fixture para_gen_cases.npz)."""
    from oracle import pycomposite as PC
    z = np.load(os.path.join(gold, "para_gen_cases.npz"))
    mk1, mk2, m = z["vc_mk1"], z["vc_mk2"], z["vc_matches"]
    keep = np.array([PC.valid_cnstr(int(a), int(b), int(c), int(d), mk1, mk2) for a, b, c, d in m])
    assert np.array_equal(keep, z["vc_keep"]) and 0 < keep.sum() < len(keep)
    km, kl = PC.filter_matches(m, mk1, mk2)
    assert np.array_equal(km, m[z["vc_keep"]]) and np.array_equal(kl, mk1[km[:, 1], km[:, 0]])
    assert np.array_equal(PC.add_bg(z["bg_im"], z["bg_mk"], z["bg_bg"]), z["bg_out"])
    f, r, k = PC.flatten(list(z["fl_flows"]), list(z["fl_rgbs"]), list(z["fl_masks"]))
    assert np.array_equal(f, z["fl_out_flow"]) and np.array_equal(r, z["fl_out_rgb"]) and np.array_equal(k, z["fl_out_mask"])
