"""CPU: the numpy references of the peak decode (tests/peaks_ref.py) against each other, numpy's argmax and scipy's maximum filter, and
ops.peak_decode's argument checks (which raise before any kernel or library is touched)."""
import numpy as np
import pytest
import torch
from scipy import ndimage

from hulk_keypoints_b200 import ops
from peaks_ref import peak_decode_ref, peak_mask, peak_mask_brute


def _tie_heavy(rng, H, W, t):
    h = rng.integers(0, 4, (H, W)).astype(np.float32)
    if t % 3 == 0:
        h[rng.random((H, W)) < 0.1] = np.nan
    if t % 4 == 0:
        h[rng.random((H, W)) < 0.1] = np.inf
    if t % 5 == 0:
        h[rng.random((H, W)) < 0.1] = -np.inf
    return h


@pytest.mark.parametrize("r", range(1, 17))
def test_separable_form_equals_definition(r):
    rng = np.random.default_rng(100 + r)
    for t in range(24):
        H, W = (int(v) for v in rng.integers(1, 2 * r + 12, 2))
        h = _tie_heavy(rng, H, W, t)
        thr = float(rng.integers(-1, 3))
        assert np.array_equal(peak_mask(h, r, thr), peak_mask_brute(h, r, thr)), (t, H, W)


def test_constant_map_has_one_peak_at_origin():
    for r in (1, 5, 16):
        m = peak_mask(np.full((20, 30), 0.25, np.float32), r, 0.0)
        assert np.flatnonzero(m).tolist() == [0]


@pytest.mark.parametrize("r", [1, 2, 4, 8, 16])
def test_top1_is_numpy_argmax(r):
    rng = np.random.default_rng(r)
    for t in range(20):
        H, W = (int(v) for v in rng.integers(1, 60, 2))
        h = (rng.integers(0, 5, (H, W)) / 4).astype(np.float32) if t % 2 else rng.random((H, W), dtype=np.float32)
        if t % 5 == 0:
            h[rng.random((H, W)) < 0.05] = np.inf
        yx, score, count = peak_decode_ref(h, 1, float(np.nanmax(h)) if t % 3 == 0 else -1.0, r)
        assert count == 1
        assert tuple(yx[0]) == np.unravel_index(np.argmax(h), h.shape) and score[0] == h.max()


@pytest.mark.parametrize("r", [1, 3, 8, 16])
def test_tie_free_mask_equals_maximum_filter(r):
    rng = np.random.default_rng(7 * r)
    h = rng.permutation(np.arange(150 * 170, dtype=np.float32)).reshape(150, 170) / (150 * 170)   # distinct values
    thr = 0.3
    want = (h == ndimage.maximum_filter(h, size=2 * r + 1, mode="constant", cval=-np.inf)) & (h >= np.float32(thr))
    assert np.array_equal(peak_mask(h, r, thr), want)


def test_reference_order_and_padding():
    h = np.zeros((5, 9), np.float32)
    h[0, 0] = h[4, 8] = 0.7   # tie: lower flat index first
    h[2, 4] = 0.9
    yx, score, count = peak_decode_ref(h[None], 5, 0.5, 1)
    assert count.tolist() == [3]
    assert yx[0].tolist() == [[2, 4], [0, 0], [4, 8], [-1, -1], [-1, -1]]
    assert np.array_equal(score[0], np.array([0.9, 0.7, 0.7, -np.inf, -np.inf], np.float32))


@pytest.mark.parametrize("kw", [dict(max_peaks=0), dict(max_peaks=257), dict(max_peaks=2.5), dict(min_distance=0),
                                dict(min_distance=17), dict(threshold=float("nan")), dict(threshold=float("inf")),
                                dict(threshold=-float("inf")), dict(threshold=1e39)])
def test_peak_decode_rejects_bad_arguments(kw):
    args = {**dict(max_peaks=16, threshold=0.5, min_distance=4), **kw}
    heat = torch.zeros(1, 1, 8, 8)
    with pytest.raises(ValueError):
        ops.peak_decode(heat, **args)


def test_peak_decode_rejects_cpu_tensors():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.peak_decode(torch.zeros(1, 1, 8, 8), 16, 0.5, 4)
