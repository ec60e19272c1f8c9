"""Backward flow and occlusion of frame 1 on the GPU (DESIGN.md 4.3): the analytic cases of test_oracle_occlusion.py
through the library's entry points, then the library against the oracle bit for bit -- warp_ex, the Batch path with
extras on every solver kind, flatten_ex, and arap_deform with 8-token list lines (directly and through --serve)."""
import os
import subprocess

import numpy as np
import pytest

from arap_flow_b200 import driver, flowio, lib, synth
from tests import occlusion_cases as OC
from tests import occlusion_oracle as OO
from tests.helpers import cat512_flo

pytestmark = pytest.mark.gpu

KEYS = ("rgb", "mask", "splat", "bflow", "occ")


def _same(a, b, keys=KEYS):
    for k in keys:
        assert np.array_equal(a[k], b[k]), k


@pytest.fixture(params=["oracle", "lib"])
def impl(request, oracle):
    """(warp_ex, flatten_ex) of the oracle / of the library: the analytic cases must hold for both."""
    if request.param == "oracle":
        return OO.warp_ex, OO.flatten_ex
    return lib.warp_ex, lib.flatten_ex


# ------------------------------------------------------------------------------------- analytic cases
@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
@pytest.mark.parametrize("t", OC.SHIFTS)
def test_integer_translation(impl, name, t):
    mask = OC.TRANSLATION_MASKS[name]()
    flow = np.zeros((OC.H_T, OC.W_T, 2), np.float32) + np.float32(t)
    OC.check_translation(impl[0](flow, OC.rgb_for(OC.W_T, OC.H_T), mask, is_flow=True), mask, t)


@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
def test_identity(impl, name):
    mask = OC.TRANSLATION_MASKS[name]()
    OC.check_identity(impl[0](OC.grid(OC.W_T, OC.H_T), OC.rgb_for(OC.W_T, OC.H_T), mask), mask)


def test_small_rigid_rotation(impl):
    mask, pos = OC.rotation_case()
    OC.check_rotation(impl[0](pos, OC.rgb_for(OC.W_R, OC.H_R), mask), mask)


def test_compression_pins_the_strict_bound(impl):
    mask, pos = OC.compression_case()
    OC.check_compression(impl[0](pos, OC.rgb_for(OC.W_C, OC.H_C), mask))


def test_two_layers(impl):
    flows, rgbs, masks, srcs, bflows = OC.layer_inputs(impl[0])
    OC.check_layers(impl[1](flows, rgbs, masks, srcs, bflows), srcs)


def test_one_layer_flatten_is_the_warp(impl, oracle):
    mask, pos = OC.rotation_case()
    out = impl[0](pos, OC.rgb_for(OC.W_R, OC.H_R), mask)
    flat = impl[1]([oracle.flow(pos)], [out["rgb"]], [out["mask"]], [mask], [out["bflow"]])
    _same(flat, out, ("bflow", "occ"))


# ------------------------------------------------------------------------------------- bit for bit against the oracle
@pytest.mark.parametrize("W,H,amp,seed", [(97, 61, 4.0, 0), (200, 120, 40.0, 1), (64, 64, 0.0, 2), (3, 2, 1.0, 3)])
def test_warp_ex_random_vs_oracle(oracle, W, H, amp, seed):
    """The cases of test_warp_random_vs_oracle, including NaN, inf and degenerate corners."""
    rng = np.random.default_rng(seed)
    rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mask = np.where(rng.random((H, W)) < 0.2, 255, 0).astype(np.uint8)
    pos = (oracle.grid(W, H) + rng.standard_normal((H, W, 2)) * amp).astype(np.float32)
    if amp > 10:
        pos[5, 5] = pos[5, 6]
        pos[10, 10] = np.nan
        pos[12, 12] = np.inf
    out = lib.warp_ex(pos, rgb, mask)
    _same(out, OO.warp_ex(pos, rgb, mask))
    r, m, sp = lib.warp(pos, rgb, mask)
    _same(out, dict(rgb=r, mask=m, splat=sp), ("rgb", "mask", "splat"))
    if amp > 0 and W * H > 1000:   # a non-trivial mix (3x2 has no all-object quad: everything is occluded)
        assert 0 < (out["occ"][mask == 0] == 255).sum() < (mask == 0).sum()


def test_warp_ex_reference_tool_cases_and_cat512(oracle, gold, tmp_path):
    z = np.load(os.path.join(gold, "warp_reftool_cases.npz"))
    cases = [(z[f"{n}__flow"], z[f"{n}__rgb"], z[f"{n}__mask"]) for n in ("warp_a", "warp_b", "warp_c")]
    cases.append((flowio.read_flo(cat512_flo(tmp_path)), flowio.read_png_rgb(os.path.join(gold, "cat512_iRGB.png")),
                  flowio.read_png_mask_red(os.path.join(gold, "cat512_iMsk.png"))))
    for flo, rgb, msk in cases:
        out = lib.warp_ex(flo, rgb, msk, is_flow=True)
        _same(out, OO.warp_ex(flo, rgb, msk, is_flow=True))
        r, m, sp = lib.warp_flow(flo, rgb, msk)
        _same(out, dict(rgb=r, mask=m, splat=sp), ("rgb", "mask", "splat"))


KW = dict(nCont=2, nGN=2, nPCG=30)


def _check_problem(oracle, o, rgb, mask, matches, solve=None):
    X, _, co = (solve or oracle.solve)(mask, matches, **KW)[:3]
    assert np.array_equal(o["flow"], oracle.flow(X)) and np.array_equal(o["costs"], co)
    _same(o, OO.warp_ex(X, rgb, mask), ("rgb", "mask", "bflow", "occ"))


def test_batch_extras_c1_two_launches_of_four(oracle):
    sps = [synth.config("C1", i) for i in range(8)]
    b = lib.Batch(854, 480, 8, **KW)
    outs = [b.submit(i, s.rgb, s.masks[0], s.matches, extras=True) for i, s in enumerate(sps)]
    b.run()
    assert b.launch_info()["problems_per_launch"] == 4 and b.resident_count() == 8
    n_extras = b.launches()
    for o, s in zip(outs, sps):
        _check_problem(oracle, o, s.rgb, s.masks[0], s.matches)
    # the same batch object without extras: same results; as many launches as a batch that never used extras
    plain = [b.submit(i, s.rgb, s.masks[0], s.matches) for i, s in enumerate(sps)]
    b.run()
    assert "bflow" not in plain[0]
    for p, o in zip(plain, outs):
        _same(p, o, ("flow", "rgb", "mask", "costs"))
    fresh = lib.Batch(854, 480, 8, **KW)
    for i, s in enumerate(sps):
        fresh.submit(i, s.rgb, s.masks[0], s.matches)
    fresh.run()
    assert b.launches() == fresh.launches() == n_extras - 8
    b.close()
    fresh.close()


def test_batch_extras_c2_segments_and_flatten(oracle):
    """C2 (854x480, four segments) on the compact grid, then the layers flattened with their extras."""
    sp = synth.config("C2")
    b = lib.Batch(sp.W, sp.H, 4, **KW)
    outs = [b.submit(s, sp.rgb, sp.masks[s], sp.matches, extras=True) for s in range(4)]
    b.run()
    for s, o in enumerate(outs):
        _check_problem(oracle, o, sp.rgb, sp.masks[s], sp.matches)
    args = ([o["flow"] for o in outs], [o["rgb"] for o in outs], [o["mask"] for o in outs], list(sp.masks),
            [o["bflow"] for o in outs])
    flat = lib.flatten_ex(*args)
    ref = OO.flatten_ex(*args)
    _same(flat, ref, ("flow", "rgb", "mask", "bflow", "occ"))
    assert (flat["occ"] == 0).any() and (flat["occ"] == 255).any()
    off = lib.flatten_ex(*args, extras=False)
    f, r, m = lib.flatten(*args[:3])
    assert np.array_equal(off["flow"], f) and np.array_equal(off["rgb"], r) and np.array_equal(off["mask"], m)
    assert "bflow" not in off
    b.close()


@pytest.mark.parametrize("kind", ["stream", "lm"])
def test_batch_extras_streaming_and_lm(oracle, kind):
    s = synth.synth(160, 120, 1, 2, 77)
    backend = lib.BACKEND_STREAM if kind == "stream" else lib.BACKEND_AUTO
    b = lib.Batch(160, 120, 1, backend=backend, **KW)
    if kind == "lm":
        b.set_option("lm", 1)
    o = b.submit(0, s.rgb, s.masks[0], s.matches, extras=True)
    b.run()
    assert b.resident_count() == 0
    _check_problem(oracle, o, s.rgb, s.masks[0], s.matches, solve=oracle.solve_lm if kind == "lm" else None)
    b.close()


# ------------------------------------------------------------------------------------- arap_deform with 8-token lines
def _case(d, name, sp, mask, extras):
    p = {k: str(d / f"{name}_{k}") for k in ("rgb.png", "msk.png", "cstr.txt", "out.flo", "wrgb.png", "wmsk.png",
                                             "bflo.flo", "occ.png")}
    flowio.write_png(p["rgb.png"], sp.rgb)
    flowio.write_png(p["msk.png"], np.repeat(mask[..., None], 3, axis=2))
    flowio.write_constraints(p["cstr.txt"], sp.matches)
    keys = ("rgb.png", "msk.png", "cstr.txt", "out.flo", "wrgb.png", "wmsk.png") + (("bflo.flo", "occ.png") if extras else ())
    return tuple(p[k] for k in keys)


def test_arap_deform_mixed_list(tmp_path):
    sps = [synth.synth(96, 80, 1, 2, 50 + i) for i in range(4)]
    extras = [True, False, True, False]
    dirs = {k: tmp_path / k for k in ("mixed", "six", "served")}
    for d in dirs.values():
        d.mkdir()
    mixed = [_case(dirs["mixed"], f"p{i}", s, s.masks[0], e) for i, (s, e) in enumerate(zip(sps, extras))]
    six = [_case(dirs["six"], f"p{i}", s, s.masks[0], False) for i, s in enumerate(sps)]
    served = [_case(dirs["served"], f"p{i}", s, s.masks[0], e) for i, (s, e) in enumerate(zip(sps, extras))]
    driver.do_arap(mixed, 0, str(tmp_path / "tmp"))
    driver.do_arap(six, 0, str(tmp_path / "tmp"))
    for it, s, e in zip(mixed, sps, extras):
        flow, rgb, m, _ = lib.deform(s.rgb, s.masks[0], s.matches)
        assert np.array_equal(flowio.read_flo(it[3]), flow)
        assert np.array_equal(flowio.read_png_rgb(it[4]), rgb) and np.array_equal(flowio.read_png_rgb(it[5])[..., 0], m)
        if e:
            ref = lib.warp_ex(flow, s.rgb, s.masks[0], is_flow=True)
            b = lib.Batch(96, 80, 1)
            o = b.submit(0, s.rgb, s.masks[0], s.matches, extras=True)
            b.run()
            b.close()
            assert np.array_equal(flowio.read_flo(it[6]), o["bflow"])
            occ = flowio.read_png_rgb(it[7])
            assert all(np.array_equal(occ[..., c], o["occ"]) for c in range(3))
            assert np.array_equal(o["rgb"], ref["rgb"]) and np.array_equal(o["mask"], ref["mask"])
    for a, b6 in zip(mixed, six):   # the 6-token outputs do not depend on what else the list asks for
        for k in (3, 4, 5):
            assert open(a[k], "rb").read() == open(b6[k], "rb").read()
    spool = str(tmp_path / "spool")
    with driver.Server(0, spool):
        driver.do_arap(served, 0, str(tmp_path / "tmp"), server=spool)
        r = subprocess.run([driver.ARAP_BIN] + list(served[0]), capture_output=True, text=True,
                           env=dict(os.environ, ARAP_PLAN=driver.PLAN, ARAP_SERVER=spool))
        assert r.returncode == 0 and r.stdout.count("Saved") == 1, r.stdout + r.stderr
    for a, b in zip(mixed, served):
        assert len(a) == len(b)
        for k in range(3, len(a)):
            assert open(a[k], "rb").read() == open(b[k], "rb").read()
