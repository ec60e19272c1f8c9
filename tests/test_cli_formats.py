"""File-format codecs of the command-line tools (PNG over zlib, .flo, constraint lists) and the argv contracts
that need no GPU -- CPU only."""
import os
import subprocess

import numpy as np
import pytest

from arap_flow_b200 import flowio
from tests.helpers import cat512_flo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "arap_flow_b200", "bin")
TOOL = os.path.join(BIN, "arap_imgtool")

pytestmark = pytest.mark.skipif(not os.path.exists(TOOL), reason="CLI tools not built (run __graft_entry__.build())")


def _png2raw(path, tmp):
    out = str(tmp / "o.raw")
    subprocess.check_call([TOOL, "png2raw", path, out])
    d = open(out, "rb").read()
    W, H = np.frombuffer(d[:8], "<i4")
    return np.frombuffer(d[8:], np.uint8).reshape(H, W, 3)


@pytest.mark.parametrize("name", ["cat512_iRGB.png", "cat512_iMsk.png", "cat512_wMsk.png", "cat512_wRGB.png"])
def test_png_decoder_matches_pil_on_reference_fixtures(gold, tmp_path, name):
    """iRGB is RGBA, iMsk an 8-bit image, wMsk a 1-bit image written by LodePNG's auto-convert."""
    got = _png2raw(os.path.join(gold, name), tmp_path)
    assert np.array_equal(got, flowio.read_png_rgb(os.path.join(gold, name)))


def test_png_decoder_colour_types_and_depths(tmp_path):
    from PIL import Image
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    cases = {
        "rgb": Image.fromarray(a),
        "rgba": Image.fromarray(np.dstack([a, rng.integers(0, 256, (37, 53, 1), dtype=np.uint8)])),
        "gray": Image.fromarray(a[..., 0]),
        "pal": Image.fromarray(a).quantize(17),
        "bit1": Image.fromarray((a[..., 0] > 127).astype(np.uint8) * 255).convert("1"),
        "i16": Image.fromarray((a[..., 0].astype(np.uint16) << 8) | 7),
    }
    for k, im in cases.items():
        p = str(tmp_path / f"{k}.png")
        im.save(p)
        want = np.asarray(Image.open(p).convert("RGB")) if k != "i16" else np.repeat(a[..., :1], 3, axis=2)
        assert np.array_equal(_png2raw(p, tmp_path), want), k


def test_png_encoder_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (31, 45, 3), dtype=np.uint8)
    raw, png = str(tmp_path / "a.raw"), str(tmp_path / "a.png")
    with open(raw, "wb") as f:
        f.write(np.asarray([45, 31], "<i4").tobytes() + a.tobytes())
    subprocess.check_call([TOOL, "raw2png", raw, png])
    assert np.array_equal(flowio.read_png_rgb(png), a)


def test_flo_and_constraint_readers(gold, tmp_path):
    out = str(tmp_path / "copy.flo")
    flo = cat512_flo(tmp_path)
    subprocess.check_call([TOOL, "flocopy", flo, out])
    assert open(out, "rb").read() == open(flo, "rb").read()
    bad = tmp_path / "bad.flo"
    bad.write_bytes(b"XXXX" + b"\0" * 20)
    assert subprocess.call([TOOL, "flocopy", str(bad), out], stderr=subprocess.DEVNULL) != 0
    got = subprocess.check_output([TOOL, "cstr", os.path.join(gold, "cat512_iCstr.txt")]).split()
    c = flowio.read_constraints(os.path.join(gold, "cat512_iCstr.txt"))
    assert int(got[0]) == len(c) == 9 and int(got[1]) == int(c.sum())
    # python-side .flo round trip
    fl = flowio.read_flo(flo)
    flowio.write_flo(out, fl)
    assert open(out, "rb").read() == open(flo, "rb").read()


def test_argv_contracts_without_gpu(tmp_path):
    """exit code 1 + usage on bad argc (main.cpp:194-198, warping main.cpp:313-317); missing plan -> 1 (main.cpp:206-213)"""
    r = subprocess.run([os.path.join(BIN, "warp_image"), "a"], capture_output=True, text=True)
    assert r.returncode == 1 and "Invalid Input!" in r.stdout
    r = subprocess.run([os.path.join(BIN, "arap_deform"), "a", "b"], capture_output=True, text=True)
    assert r.returncode == 1 and "Invalid Input!" in r.stdout
    empty = tmp_path / "empty.txt"
    empty.write_text("")
    r = subprocess.run([os.path.join(BIN, "arap_deform"), str(empty)], capture_output=True, text=True)
    assert r.returncode == 1 and "No file to be processed" in r.stdout
    env = dict(os.environ, ARAP_PLAN=str(tmp_path / "missing.t"))
    r = subprocess.run([os.path.join(BIN, "arap_deform"), "a", "b", "c", "d", "e", "f"], capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "Optimization plan at" in r.stdout and "Not found!" in r.stdout


def test_resident_worker_contracts_without_gpu(tmp_path):
    """`arap_deform --serve` / ARAP_SERVER (SURVEY.md 8f N2) on a box without a GPU: the client refuses to run when no
    worker watches the spool directory (it never falls back to solving in-process), the worker refuses to start without a
    plan, and without a CUDA device it exits non-zero instead of signalling `ready`."""
    from arap_flow_b200 import driver
    exe = os.path.join(BIN, "arap_deform")
    spool = str(tmp_path / "spool")
    env = dict(os.environ, ARAP_PLAN=driver.PLAN, ARAP_SERVER=spool)
    r = subprocess.run([exe, "a", "b", "c", "d", "e", "f"], capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "no server is watching" in r.stderr
    r = subprocess.run([exe, "--serve", spool], capture_output=True, text=True, env=dict(os.environ, ARAP_PLAN=str(tmp_path / "nope.t")))
    assert r.returncode == 1 and "Not found!" in r.stdout
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            driver.Server(0, spool, timeout=20.0)
        assert not os.path.exists(os.path.join(spool, "ready"))


def test_dispatch_queue_hands_every_dispatch_to_a_free_gpu(tmp_path, monkeypatch):
    """driver.run_dispatches mirrors para_gen's free-GPU queue (para_gen.py:441-445, 560-567): every dispatch runs exactly
    once, never two at a time on one GPU."""
    import threading
    import time
    from arap_flow_b200 import driver
    lock, busy, seen, overlap = threading.Lock(), set(), [], []

    def fake_do_arap(items, gpu, tmp_dir, server=None, **kw):
        with lock:
            if gpu in busy:
                overlap.append(gpu)
            busy.add(gpu)
        time.sleep(0.01)
        with lock:
            busy.discard(gpu)
            seen.append((gpu, tuple(items), server))
        return 0.01

    monkeypatch.setattr(driver, "do_arap", fake_do_arap)
    dispatches = [[("r%d" % k, "m", "c", "f", "wr", "wm")] for k in range(11)]
    driver.run_dispatches(dispatches, [0, 1, 2], str(tmp_path), servers=["s0", "s1", "s2"])
    assert not overlap and sorted(s[1][0][0] for s in seen) == sorted("r%d" % k for k in range(11))
    assert all(s[2] == "s%d" % s[0] for s in seen)
