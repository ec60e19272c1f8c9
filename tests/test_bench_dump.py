"""bench.py --dump-outputs on synthetic outputs of the shapes the benchmark produces -- CPU only."""
import os

import numpy as np
import pytest

import bench


def _outs(P, H, W, seed=0):
    rng = np.random.default_rng(seed)
    return [dict(flow=rng.standard_normal((H, W, 2)).astype(np.float32),
                 rgb=rng.integers(0, 256, (H, W, 3), dtype=np.uint8),
                 mask=(rng.random((H, W)) < 0.5).astype(np.uint8) * 255,
                 costs=rng.random((19, 9)).astype(np.float32)) for _ in range(P)]


def _flats(outs, nseg):
    return [(o["flow"], o["rgb"], o["mask"]) for o in outs[::nseg]]


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _total(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_small_outputs_are_written_whole(tmp_path):
    outs = _outs(3, 24, 40)
    bench.dump_outputs(str(tmp_path), outs, [])
    z = _load(tmp_path)
    assert sorted(z) == ["costs", "flow", "mask", "rgb"]                    # no sample index, no flattened outputs
    assert all(a.dtype == np.float32 for a in z.values())
    for k in ("flow", "rgb", "mask", "costs"):
        assert np.array_equal(z[k], np.stack([o[k] for o in outs])), k


@pytest.mark.parametrize("P,H,W,nseg", [(8, 480, 854, 1),       # bench.py default: C1, batch 8
                                        (12, 480, 854, 4),      # C2: 3 pairs of 4 segments, flattened per pair
                                        (14, 480, 854, 1)])     # C1s, batch 14
def test_large_outputs_share_one_seeded_pixel_sample_within_budget(tmp_path, P, H, W, nseg):
    outs = _outs(P, H, W)
    flats = _flats(outs, nseg) if nseg > 1 else []
    bench.dump_outputs(str(tmp_path / "a"), outs, flats)
    assert _total(tmp_path / "a") <= bench.DUMP_BYTES
    z = _load(tmp_path / "a")
    assert ("flat_flow" in z) == (nseg > 1)
    idx = z["pixel_index"]
    assert idx.dtype == np.float64 and np.array_equal(idx, np.round(idx))
    idx = idx.astype(np.int64)
    n = len(idx)
    assert 0 < n < H * W and np.all(np.diff(idx) > 0) and idx[-1] < H * W
    for k in ("flow", "rgb", "mask"):
        src = [o[k] for o in outs]
        assert z[k].shape == (P, n) + src[0].shape[2:], k
        assert np.array_equal(z[k], np.stack([s.reshape(H * W, -1)[idx].reshape((n,) + s.shape[2:]) for s in src])), k
    for i, k in enumerate(("flow", "rgb", "mask")):
        if nseg > 1:
            want = np.stack([f[i].reshape(H * W, -1)[idx].reshape((n,) + f[i].shape[2:]) for f in flats])
            assert np.array_equal(z["flat_" + k], want), k
    assert np.array_equal(z["costs"], np.stack([o["costs"] for o in outs]))
    # the sample is fixed: a second dump of other values picks the same pixels
    bench.dump_outputs(str(tmp_path / "b"), _outs(P, H, W, seed=1), flats)
    assert np.array_equal(np.load(str(tmp_path / "b" / "pixel_index.npy")).astype(np.int64), idx)
