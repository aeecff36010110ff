"""CPU: bench.py --dump-outputs writes the timed path's outputs as float .npy files, under 64 MB, identical from run to run."""
import os
import types

import numpy as np
import torch

import bench


def _plan(B, K, H, W, heat):
    g = torch.Generator().manual_seed(0)
    return types.SimpleNamespace(heat=heat.reshape(B, K, H, W), yx=torch.randint(0, H, (B, K, 2), generator=g, dtype=torch.int32),
                                 maxval=torch.rand(B, K, generator=g))


def test_dump_small_workload_whole(tmp_path):
    p = _plan(2, 4, 32, 48, torch.rand(2 * 4 * 32 * 48, generator=torch.Generator().manual_seed(1)))
    bench.dump_outputs(str(tmp_path), p)
    assert np.array_equal(np.load(tmp_path / "heatmaps.npy"), p.heat.numpy())
    yx = np.load(tmp_path / "keypoints_yx.npy")
    assert yx.dtype == np.float64 and np.array_equal(yx, p.yx.numpy())
    assert np.array_equal(np.load(tmp_path / "peak_values.npy"), p.maxval.numpy())


def test_dump_default_workload_fixed_sample_under_64mb(tmp_path):
    B, K, H, W = 64, 4, 480, 640
    p = _plan(B, K, H, W, torch.linspace(0.0, 1.0, B * K * H * W))     # increasing in the flat index
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), p)
    bench.dump_outputs(str(b), p)
    assert sorted(os.listdir(a)) == ["heatmaps.npy", "keypoints_yx.npy", "peak_values.npy"]
    assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= 64 << 20
    for f in os.listdir(a):
        x = np.load(a / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(b / f))
    h = np.load(a / "heatmaps.npy")
    assert h.ndim == 1 and h.size > bench.HEAT_DUMP_VALUES // 2
    assert (np.diff(h) >= 0).all() and h[0] < 1e-3 and h[-1] > 1 - 1e-3    # sorted indices spread over the whole tensor
