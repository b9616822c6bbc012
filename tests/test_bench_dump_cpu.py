"""bench.py --dump-outputs, host side: an output under its size cap is written whole, a larger one as the same seeded sample in every
run, both in float32, and the caps keep a dump under 64 MB."""
import numpy as np
import torch

import bench


def test_dump_outputs_whole_and_sampled(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_CAP_BYTES", {"small": 4 * 60, "big": 4 * 50})
    small = torch.arange(60, dtype=torch.bfloat16).view(3, 4, 5)
    big = torch.randn(7, 3, 11, 13, dtype=torch.float64).transpose(0, 1)     # not contiguous, like the feature ring's window
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"small": small, "big": big})
    got = np.load(tmp_path / "a" / "small.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())
    got, again = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert got.dtype == np.float32 and got.shape == (50,) and np.array_equal(got, again)
    flat = big.float().reshape(-1).numpy()
    assert np.array_equal(got, flat[np.sort(np.random.default_rng(0).choice(flat.size, 50, replace=False))])


def test_dump_caps_stay_under_64_mb():
    assert sum(bench.DUMP_CAP_BYTES.values()) + 128 * len(bench.DUMP_CAP_BYTES) <= 64_000_000     # + one .npy header per file
