"""CPU: bench.py --dump-outputs writes float32 arrays within its size limit, the whole output when
it fits and otherwise the same seeded sample of pixels on every run."""
import os

import numpy as np
import torch

import bench


def test_small_output_is_written_whole(tmp_path):
    t = torch.arange(2 * 5 * 7 * 3, dtype=torch.int64).reshape(2, 5, 7, 3).to(torch.uint8)
    paths = bench.dump_output(str(tmp_path), "warp_output", t)
    assert paths == [str(tmp_path / "warp_output.npy")]
    a = np.load(paths[0])
    assert a.dtype == np.float32 and np.array_equal(a, t.numpy().astype(np.float32))


def test_large_output_is_a_fixed_sample_within_the_limit(tmp_path):
    g = torch.Generator().manual_seed(1)
    t = torch.randint(0, 256, (4, 64, 96, 3), dtype=torch.uint8, generator=g).to(torch.float16)
    limit = 40_000
    runs = []
    for d in ("a", "b"):
        paths = bench.dump_output(str(tmp_path / d), "warp_output", t, limit=limit)
        assert [os.path.basename(p) for p in paths] == ["warp_output.npy", "warp_output_index.npy"]
        assert sum(os.path.getsize(p) for p in paths) <= limit
        runs.append([np.load(p) for p in paths])
    (vals, idx), (vals2, idx2) = runs
    assert vals.dtype == np.float32 and idx.dtype == np.float64
    assert np.array_equal(vals, vals2) and np.array_equal(idx, idx2)
    assert vals.shape == (len(idx), 3) and len(idx) > 1000
    assert np.all(np.diff(idx) > 0)
    flat = t.reshape(-1, 3).float().numpy()
    assert np.array_equal(vals, flat[idx.astype(np.int64)])
