"""bench.py --dump-outputs: float64 .npy files within the byte budget, arrays over their share written as a seeded sample
of positions (with the positions beside them), and the same outputs giving the same files."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_budget_and_sample(tmp_path):
    rng = np.random.default_rng(1)
    scores = torch.from_numpy(rng.integers(-2**31, 2**31 - 1, 300_000, dtype=np.int32))
    states = torch.from_numpy(rng.integers(0, 2**32, 5000, dtype=np.uint32).view(np.int32))  # u32 held in an i32 tensor
    offs = torch.arange(1001, dtype=torch.int64) * 7
    arrays = {"scores": (scores, np.int32), "states": (states, np.uint32), "offsets": (offs, np.int64)}
    budget = 1_000_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget)
    a, b = tmp_path / "a", tmp_path / "b"
    files = sorted(os.listdir(a))
    assert files == ["offsets.npy", "scores.npy", "scores_index.npy", "states.npy"]
    assert sum(os.path.getsize(a / f) for f in files) <= budget
    for f in files:
        x, y = np.load(a / f), np.load(b / f)
        assert x.dtype == np.float64 and np.array_equal(x, y)
    idx = np.load(a / "scores_index.npy").astype(np.int64)
    assert idx.size > 1000 and np.all(np.diff(idx) > 0) and idx[-1] < scores.numel()
    assert np.array_equal(np.load(a / "scores.npy"), scores.numpy()[idx].astype(np.float64))
    assert np.array_equal(np.load(a / "states.npy"), states.numpy().view(np.uint32).astype(np.float64))
    assert np.array_equal(np.load(a / "offsets.npy"), offs.numpy().astype(np.float64))
