"""bench.py --dump-outputs on the host: float32 / float64 files within the size bound, a fixed sample of the commits of a
larger probability tensor."""
import os

import numpy as np

import bench


def _arrays(B, Nc):
    P = 3129
    rows = np.arange(B, dtype=np.float32)[:, None, None]
    return {"probs": np.broadcast_to(rows, (B, 2, Nc * (Nc - 1))), "losses": np.ones(3, np.float32),
            "params": np.ones(P, np.float32), "adam_m": np.zeros(P, np.float32), "adam_v": np.zeros(P, np.float32),
            "adam_step": np.array([7], np.int32)}


def test_dump_outputs_small_run_is_written_whole(tmp_path):
    arrays = _arrays(100, 74)
    bench.write_outputs(str(tmp_path), arrays)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in arrays)
    assert np.array_equal(np.load(tmp_path / "probs.npy"), arrays["probs"])
    step = np.load(tmp_path / "adam_step.npy")
    assert step.dtype == np.float64 and step[0] == 7


def test_dump_outputs_large_run_keeps_a_fixed_sample_within_the_bound(tmp_path):
    arrays = _arrays(512, 256)                      # cfg4: 267 MB of probabilities
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(list(k + ".npy" for k in arrays) + ["probs_commits.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= bench.DUMP_BYTES
    for n in names:
        x, y = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y)
    rows = np.load(tmp_path / "a" / "probs_commits.npy").astype(np.int64)
    assert len(rows) > 64 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "probs.npy"), arrays["probs"][rows])
