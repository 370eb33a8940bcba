"""bench.py --dump-outputs: host logic of the writer (no GPU needed)."""
import os

import numpy as np

import bench


def test_dump_outputs_budget_and_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 4096)          # a 4096-byte share per array
    rng = np.random.RandomState(1)
    arrays = {"loss": np.float32(0.5).reshape(()), "x_hat": rng.standard_normal((4, 3, 32, 32)).astype(np.float32),
              "perplexity": np.array(7.0, dtype=np.float32),
              "min_encoding_indices": rng.randint(0, 512, (256, 1)).astype(np.float64)}
    info = bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    total = 0
    for name, a in arrays.items():
        got = np.load(tmp_path / "a" / (name + ".npy"))
        total += os.path.getsize(tmp_path / "a" / (name + ".npy")) - 128     # minus the .npy header
        assert got.dtype == a.dtype and info[name]["shape"] == list(a.shape)
        assert np.array_equal(got, np.load(tmp_path / "b" / (name + ".npy")))   # same positions in every run
        if a.nbytes <= 4096:
            assert np.array_equal(got, a) and "sampled_elements" not in info[name]
        else:
            assert got.size == info[name]["sampled_elements"] == 4096 // a.itemsize
            assert np.isin(got, a.ravel()).all()
    assert total <= bench.DUMP_BYTES
