"""Frame sequences on the GPU (DESIGN.md 4.4): the analytic cases of test_oracle_sequence.py through lib.warp_seq, then
the library against the CPU restatement (tests/sequence_oracle.py) bit for bit -- warp_seq on random, degenerate and
non-finite positions and on scaled reference flows, the Batch path with frames on every solver path, the full schedule
against its committed fixtures, mixed batches, the layer recipe and the rejection of bad step lists."""
import ctypes as C
import os

import numpy as np
import pytest

from arap_flow_b200 import flowio, lib, synth
from tests import occlusion_cases as OC
from tests import occlusion_oracle as OO
from tests import sequence_cases as SC
from tests import sequence_oracle as SO
from tests import test_gpu_full_schedule as FS
from tests.helpers import cat512_flo

pytestmark = pytest.mark.gpu


def _same(a, b, keys=SO.KEYS):
    """Equal outputs; a NaN position gives a NaN flow0 in both, and NaN never compares equal to itself."""
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


@pytest.fixture(params=["oracle", "lib"])
def warp_seq(request, oracle):
    return SO.warp_seq if request.param == "oracle" else lib.warp_seq


# ------------------------------------------------------------------------------------- analytic cases
@pytest.mark.parametrize("name", sorted(OC.TRANSLATION_MASKS))
@pytest.mark.parametrize("t", OC.SHIFTS)
def test_constant_velocity_translation(warp_seq, name, t):
    mask = OC.TRANSLATION_MASKS[name]()
    SC.check_translation(warp_seq(SC.translation_positions(t), OC.rgb_for(OC.W_T, OC.H_T), mask), mask, t)


def test_rotation_per_frame(warp_seq):
    SC.check_rotation(warp_seq(SC.rotation_positions(), OC.rgb_for(OC.W_R, OC.H_R), OC.rotation_case()[0]))


def test_repeated_frame(warp_seq):
    SC.check_repeated(warp_seq(SC.repeated_positions(), OC.rgb_for(OC.W_R, OC.H_R), OC.rotation_case()[0]))


def test_compression_pins_the_strict_bound(warp_seq):
    mask, pos = SC.compression_positions()
    SC.check_compression(warp_seq(pos, OC.rgb_for(OC.W_C, OC.H_C), mask))


# ------------------------------------------------------------------------------------- warp_seq bit for bit
@pytest.mark.parametrize("W,H,amp,seed", [(97, 61, 4.0, 0), (200, 120, 40.0, 1), (64, 64, 0.0, 2), (3, 2, 1.0, 3)])
def test_warp_seq_random_vs_oracle(oracle, W, H, amp, seed):
    """Random walks of the positions, with NaN, inf and degenerate corners in the large-amplitude case."""
    rng = np.random.default_rng(seed)
    rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mask = np.where(rng.random((H, W)) < 0.2, 255, 0).astype(np.uint8)
    pos = oracle.grid(W, H) + np.cumsum(rng.standard_normal((4, H, W, 2)) * amp / 2, axis=0)
    pos = pos.astype(np.float32)
    if amp > 10:
        pos[1, 5, 5] = pos[1, 5, 6]
        pos[2, 10, 10] = np.nan
        pos[3, 12, 12] = np.inf
        pos[2, 30:33, 40:43] = pos[1, 30:33, 40:43]
    out = lib.warp_seq(pos, rgb, mask)
    _same(out, SO.warp_seq(pos, rgb, mask))
    if amp > 0 and W * H > 1000:
        assert (out["occ"][1:] == 255).any() and (out["occ"][1:] == 0).any() and out["flow"][1:].any()


def test_warp_seq_reference_tool_flows_and_cat512(oracle, gold, tmp_path):
    z = np.load(os.path.join(gold, "warp_reftool_cases.npz"))
    cases = [(z[f"{n}__flow"], z[f"{n}__rgb"], z[f"{n}__mask"]) for n in ("warp_a", "warp_b", "warp_c")]
    cases.append((flowio.read_flo(cat512_flo(tmp_path)), flowio.read_png_rgb(os.path.join(gold, "cat512_iRGB.png")),
                  flowio.read_png_mask_red(os.path.join(gold, "cat512_iMsk.png"))))
    for flo, rgb, msk in cases:
        H, W = msk.shape
        pos = np.stack([oracle.flow_to_pos((np.float32(s) * flo).astype(np.float32)) for s in (0.25, 0.5, 1.0)])
        out = lib.warp_seq(pos, rgb, msk)
        _same(out, SO.warp_seq(pos, rgb, msk))


def test_one_frame_is_warp_ex(oracle):
    mask, pos = OC.rotation_case()
    rgb = OC.rgb_for(OC.W_R, OC.H_R)
    seq = lib.warp_seq(pos[None], rgb, mask)
    ex = lib.warp_ex(pos, rgb, mask)
    for k in ("rgb", "mask", "bflow", "occ"):
        assert np.array_equal(seq[k][0], ex[k]), k
    assert np.array_equal(seq["flow"][0], oracle.flow(pos)) and np.array_equal(seq["flow0"][0], oracle.flow(pos))


# ------------------------------------------------------------------------------------- the Batch path
KW = dict(nCont=6, nGN=2, nPCG=30)
STEPS = ([0, 2, 5], list(range(6)))


def _check_problem(o, rgb, mask, matches, steps, lm=False):
    """Costs and ordinary outputs against the oracle's solve; flow0 against the oracle's snapshots; every sequence
    output against the restatement run on those snapshots."""
    X, _, co, snaps = SO.solve_states(mask, matches, steps, lm=lm, **KW)
    assert np.array_equal(o["costs"], co)
    from oracle import pyoracle as O
    assert np.array_equal(o["flow"], O.flow(X))
    r, m, _ = O.warp(X, rgb, mask)
    assert np.array_equal(o["rgb"], r) and np.array_equal(o["mask"], m)
    assert np.array_equal(o["seq"]["flow0"], np.stack([O.flow(s) for s in snaps]))
    _same(o["seq"], SO.warp_seq(snaps, rgb, mask))
    if steps[-1] == KW["nCont"] - 1:
        for k in ("rgb", "mask", "flow"):
            assert np.array_equal(o["seq"][k if k != "flow" else "flow0"][-1], o[k]), k


def test_batch_frames_c1_two_launches_of_four(oracle):
    sps = [synth.config("C1", i) for i in range(8)]
    b = lib.Batch(854, 480, 8, **KW)
    outs = [b.submit(i, s.rgb, s.masks[0], s.matches, frames=STEPS[i % 2]) for i, s in enumerate(sps)]
    b.run()
    info = b.launch_info()
    assert info["problems_per_launch"] == 4 and info["grid"][1] == 4 and b.resident_count() == 8, info
    for i, (o, s) in enumerate(zip(outs, sps)):
        _check_problem(o, s.rgb, s.masks[0], s.matches, STEPS[i % 2])


def test_batch_frames_c2_segments_compact_grid_and_flatten(oracle):
    """C2 (854x480, four segments) on the compact 1-D grid; then the layer recipe of DESIGN.md 4.4 per frame."""
    sp = synth.config("C2")
    b = lib.Batch(sp.W, sp.H, 4, **KW)
    steps = STEPS[1]
    outs = [b.submit(s, sp.rgb, sp.masks[s], sp.matches, frames=steps) for s in range(4)]
    b.run()
    info = b.launch_info()
    assert info["grid"][1] == 1 and info["problems_per_launch"] == 4 and b.resident_count() == 4, info
    for s, o in enumerate(outs):
        _check_problem(o, sp.rgb, sp.masks[s], sp.matches, steps)
    seqs = [o["seq"] for o in outs]
    for k in range(len(steps)):
        src = list(sp.masks) if k == 0 else [255 - q["mask"][k - 1] for q in seqs]
        args = ([q["flow"][k] for q in seqs], [q["rgb"][k] for q in seqs], [q["mask"][k] for q in seqs], src,
                [q["bflow"][k] for q in seqs])
        flat = lib.flatten_ex(*args)
        _same(flat, OO.flatten_ex(*args), ("flow", "rgb", "mask", "bflow", "occ"))
        assert (flat["occ"] == 0).any() and (flat["occ"] == 255).any()
    b.close()


def test_batch_frames_small_problems_one_launch(oracle):
    sps = [synth.synth(96, 80, 1, 2, 60 + i) for i in range(3)]
    b = lib.Batch(96, 80, 3, **KW)
    outs = [b.submit(i, s.rgb, s.masks[0], s.matches, frames=STEPS[i % 2]) for i, s in enumerate(sps)]
    b.run()
    info = b.launch_info()
    assert info["problems_per_launch"] == 3 and b.resident_count() == 3, info
    for i, (o, s) in enumerate(zip(outs, sps)):
        _check_problem(o, s.rgb, s.masks[0], s.matches, STEPS[i % 2])
    b.close()


@pytest.mark.parametrize("kind", ["stream", "lm"])
def test_batch_frames_streaming_and_lm(oracle, kind):
    s = synth.synth(160, 120, 1, 2, 77)
    b = lib.Batch(160, 120, 1, backend=lib.BACKEND_STREAM if kind == "stream" else lib.BACKEND_AUTO, **KW)
    if kind == "lm":
        b.set_option("lm", 1)
    for steps in STEPS:
        o = b.submit(0, s.rgb, s.masks[0], s.matches, frames=steps, extras=True)
        b.run()
        assert b.resident_count() == 0
        _check_problem(o, s.rgb, s.masks[0], s.matches, steps, lm=kind == "lm")
        ex = lib.warp_ex(o["seq"]["flow0"][-1], s.rgb, s.masks[0], is_flow=True)
        assert np.array_equal(o["bflow"], ex["bflow"]) and np.array_equal(o["occ"], ex["occ"])
    b.close()


# ------------------------------------------------------------------------------------- nothing else changes
def test_full_schedule_all_frames_keeps_the_fixtures():
    """bench.py's C1 batch of eight at 19 x 8 x 400 with every step as a frame: the committed fixtures, the same launch
    shape, and the last frame equal to the ordinary outputs."""
    db = FS._db()
    pairs = [FS._pair("C1", s) for s in range(1000, 1008)]
    keys = [f"C1:{p.seed}:0" for p in pairs]
    if any(k not in db for k in keys):
        pytest.skip("no full-schedule oracle fixture for C1")
    nCont, nGN, nPCG = db[keys[0]]["schedule"]
    b = lib.Batch(854, 480, 8, nCont, nGN, nPCG)
    outs = [b.submit(i, p.rgb, p.masks[0], p.matches, frames=list(range(nCont))) for i, p in enumerate(pairs)]
    b.run()
    info = b.launch_info()
    assert info["variant"] == (160, 3) and info["grid"][1] == 4 and info["problems_per_launch"] == 4, info
    for k, o in zip(keys, outs):
        want = db[k]
        assert np.array_equal(np.ascontiguousarray(o["costs"], np.float32).view(np.uint32),
                              np.asarray(want["costs_bits"], np.uint32)), k
        assert FS._digest(o["flow"]) == want["flow_sha256"], k
        assert FS._digest(o["rgb"]) == want["rgb_sha256"] and FS._digest(o["mask"]) == want["mask_sha256"], k
        assert np.array_equal(o["seq"]["flow0"][-1], o["flow"])
        assert np.array_equal(o["seq"]["rgb"][-1], o["rgb"]) and np.array_equal(o["seq"]["mask"][-1], o["mask"])
    b.close()


def test_mixed_batch_plain_slots_unchanged_and_launch_count():
    KW4 = dict(nCont=4, nGN=2, nPCG=30)
    sps = [synth.config("C1", i) for i in range(8)]
    plain = lib.Batch(854, 480, 8, **KW4)
    ref = [plain.submit(i, s.rgb, s.masks[0], s.matches) for i, s in enumerate(sps)]
    plain.run()
    n_plain = plain.launches()
    b = lib.Batch(854, 480, 8, **KW4)
    kinds = ["frames", "extras", "plain", "both", "plain", "frames", "extras", "plain"]
    outs = [b.submit(i, s.rgb, s.masks[0], s.matches, frames=[1, 3] if k in ("frames", "both") else None,
                     extras=k in ("extras", "both")) for i, (s, k) in enumerate(zip(sps, kinds))]
    b.run()
    assert b.launch_info()["problems_per_launch"] == 4
    for o, r, k in zip(outs, ref, kinds):
        _same(o, r, ("flow", "rgb", "mask", "costs"))
        assert ("seq" in o) == (k in ("frames", "both"))
    # the same batch object, asked for nothing: as many launches as a batch that never asked
    for i, s in enumerate(sps):
        b.submit(i, s.rgb, s.masks[0], s.matches)
    b.run()
    assert b.launches() == n_plain
    plain.close()
    b.close()


# ------------------------------------------------------------------------------------- bad step lists
def _submit_seq(b, s, n_frames, steps, seq_rgb=True, seq_mask=True, any_out=True):
    H, W = s.masks[0].shape
    L = b.L
    L.arapb200_batch_submit_seq.argtypes = L.arapb200_batch_submit.argtypes + [C.c_void_p, C.c_void_p, C.c_int] + \
        [C.c_void_p] * 7
    keep = [np.ascontiguousarray(x) for x in (s.rgb, s.masks[0], np.asarray(s.matches, np.int32).reshape(-1, 4))]
    outs = [np.zeros(max(len(steps or []), 1) * H * W * 8, np.uint8) for _ in range(6)]
    ptr = [o.ctypes.data for o in outs]
    if not seq_rgb:
        ptr[0] = None
    if not seq_mask:
        ptr[1] = None
    if not any_out:
        ptr = [None] * 6
    st = np.asarray(steps if steps is not None else [0], np.int32)
    o = [np.zeros((H, W, 2), np.float32), np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.uint8)]
    return L.arapb200_batch_submit_seq(b.h, 0, W, H, keep[0].ctypes.data, keep[1].ctypes.data, keep[2].ctypes.data,
                                       len(keep[2]), o[0].ctypes.data, o[1].ctypes.data, o[2].ctypes.data, None, None,
                                       None, n_frames, st.ctypes.data if steps is not None else None, *ptr)


def test_bad_step_lists_are_rejected_and_the_batch_still_runs(oracle):
    s = synth.synth(96, 80, 1, 2, 42)
    b = lib.Batch(96, 80, 1, nCont=3, nGN=2, nPCG=50)
    bad = [dict(n_frames=-1, steps=[0]), dict(n_frames=0, steps=[]), dict(n_frames=2, steps=[1, 1]),
           dict(n_frames=2, steps=[2, 1]), dict(n_frames=1, steps=[3]), dict(n_frames=1, steps=[-1]),
           dict(n_frames=1, steps=None), dict(n_frames=1, steps=[0], seq_rgb=False),
           dict(n_frames=1, steps=[0], seq_mask=False)]
    for kw in bad:
        assert _submit_seq(b, s, **kw) != 0, kw
    with pytest.raises(RuntimeError):
        b.submit(0, s.rgb, s.masks[0], s.matches, frames=[2, 0])
    assert _submit_seq(b, s, 0, None, any_out=False) == 0   # no frames, no outputs: arapb200_batch_submit_ex
    o = b.submit(0, s.rgb, s.masks[0], s.matches, frames=[0, 2])
    b.run()
    Xo, _, co = oracle.solve(s.masks[0], s.matches, nCont=3, nGN=2, nPCG=50)
    assert np.array_equal(o["costs"], co) and np.array_equal(o["seq"]["flow0"][-1], oracle.flow(Xo))
    b.close()
