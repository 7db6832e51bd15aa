"""CPU: the synthetic inputs of bench.py are what SURVEY.md 8(d) / BASELINE.json name. The config-2 clip must be the
reference's own scripts/gradients.py pattern (checked against frames the script drew, tests/golden/bench_gradients.npz,
and against properties of im_function); the config-3 / config-5 block texture must be deterministic."""
import os

import numpy as np

import bench
from helpers import GOLDEN_DIR


def test_gradient_clip_properties():
    fr = bench.gradient_clip(260, 346, 31)
    assert fr.shape == (31, 260, 346) and fr.dtype == np.uint8
    low, high = np.uint8((127 * 2) / 3), np.uint8(2 * (127 * 2) / 3)      # contrast 2 around the background 127
    assert fr.min() == low and fr.max() == high
    assert (fr == fr[:, :1, :]).all()                                  # constant along y
    # the bump's peak moves 300 px/s = 10 px per 30 fps frame
    peaks = [int(np.argmax(f[0, :int(0.5 * 346) + 10 * k + 2])) for k, f in enumerate(fr[:10])]
    assert np.all(np.diff(peaks) == 10), peaks


def test_gradient_clip_equals_reference_script():
    # frames of scripts/gradients.py::im_function at 30 fps, recorded by oracle/make_golden_bench.py
    ref = np.load(os.path.join(GOLDEN_DIR, "bench_gradients.npz"))["frames"]
    assert ref.shape == (8, 260, 346) and ref.dtype == np.uint8
    mine = bench.gradient_clip(260, 346, 8)
    for k in range(8):
        assert np.array_equal(mine[k], ref[k]), k


def test_block_texture_clip_is_deterministic_and_translates():
    a = bench.block_texture_clip(64, 96, 5, seed=0)
    b = bench.block_texture_clip(64, 96, 5, seed=0)
    assert np.array_equal(a, b) and a.dtype == np.uint8
    assert np.array_equal(a[1][:-4, :-8], a[0][4:, 8:])                # (+8, +4) px per source frame
    assert len(np.unique(a[0])) > 50


def test_unet_activation_bytes_matches_a_hand_count():
    # one layer by hand: conv2 of UNet(12, 5) at 1280x704, batch 8: 32 channels in + 32 out, fp16
    tot = bench.unet_activation_bytes(12, 5, 704, 1280, 8)
    conv2 = 8 * 704 * 1280 * (32 + 32) * 2
    assert tot > 5 * conv2 and tot < 12 * conv2


def _dump(d, n, budget, shuffle_seed):
    """Two frames of n // 3 and n - n // 3 event rows (t, x, y, p), each frame's rows in a shuffled order."""
    rng = np.random.default_rng(3)
    offs, t = np.array([0, n // 3, n], np.int64), np.array([1.0, 2.0])
    ev = np.stack([np.repeat(t, np.diff(offs)) - rng.integers(0, 4, n) / 8, rng.integers(0, 64, n),
                   rng.integers(0, 48, n), rng.choice([-1, 1], n)], 1).astype(np.float32)
    want = ev[np.lexsort((ev[:, 3], ev[:, 1], ev[:, 2], ev[:, 0]))]          # sorted by (t, y, x, p)
    shuffle = np.random.default_rng(shuffle_seed)
    rows = np.concatenate([offs[f] + shuffle.permutation(offs[f + 1] - offs[f]) for f in range(2)])
    bench.dump_outputs(str(d), want[rows], offs, t, budget=budget)
    return want, {f[:-4]: np.load(os.path.join(str(d), f)) for f in os.listdir(str(d))}


def test_dump_outputs_writes_small_outputs_whole(tmp_path):
    want, got = _dump(tmp_path, 1000, bench.DUMP_BYTES, 1)
    assert sorted(got) == ["events", "offsets", "times"]
    assert np.array_equal(got["events"], want) and got["events"].dtype == np.float32
    assert got["offsets"].dtype == np.float64 and got["offsets"].tolist() == [0, 333, 1000]
    assert got["times"].tolist() == [1.0, 2.0]


def test_dump_outputs_samples_large_outputs_within_budget(tmp_path):
    budget = 1 << 20
    want, got = _dump(tmp_path / "a", 200000, budget, 1)
    _, again = _dump(tmp_path / "b", 200000, budget, 2)       # same rows, emitted in another order
    assert sum(os.path.getsize(str(p)) for p in (tmp_path / "a").iterdir()) <= budget
    rows = got["events_rows"].astype(np.int64)
    assert len(rows) > 30000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["events"], want[rows])
    assert sorted(again) == sorted(got) and all(np.array_equal(got[k], again[k]) for k in got)
