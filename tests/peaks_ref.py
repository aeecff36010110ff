"""numpy restatements of the peak decode (csrc/peaks.cu) that tests/test_peaks_host.py and tests/test_gpu_peaks.py compare against.

Pixel p with value v (NaN read as -inf) is a peak iff v >= threshold, v > q for every neighbour q of its (2r+1)x(2r+1) window (clipped to
the image) that precedes p in row-major order, and v >= q for every neighbour after p.  Per map the peaks are ordered by value descending,
ties by flat index ascending, and the first N are kept.
"""
import numpy as np


def peak_mask_brute(h: np.ndarray, r: int, thr: float) -> np.ndarray:
    """The definition, literally: one (H, W) map -> bool mask.  O(H*W*r^2): small maps only."""
    H, W = h.shape
    v = np.where(np.isnan(h), -np.inf, h)
    out = np.zeros((H, W), bool)
    for y in range(H):
        for x in range(W):
            p = v[y, x]
            if not p >= thr:
                continue
            ok = True
            for yy in range(max(0, y - r), min(H, y + r + 1)):
                for xx in range(max(0, x - r), min(W, x + r + 1)):
                    if (yy, xx) == (y, x):
                        continue
                    q = v[yy, xx]
                    ok &= bool(p > q) if (yy, xx) < (y, x) else bool(p >= q)
            out[y, x] = ok
    return out


def _shift_max(a: np.ndarray, lo: int, hi: int, axis: int) -> np.ndarray:
    """out[..., i, ...] = max of a[..., i+d, ...] over d in [lo, hi] along `axis` (-inf outside)."""
    n = a.shape[axis]
    out = np.full(a.shape, -np.inf, dtype=a.dtype)
    for d in range(max(lo, 1 - n), min(hi, n - 1) + 1):
        src = [slice(None)] * a.ndim
        dst = [slice(None)] * a.ndim
        src[axis] = slice(max(0, d), min(n, n + d))
        dst[axis] = slice(max(0, -d), min(n, n - d))
        np.maximum(out[tuple(dst)], a[tuple(src)], out=out[tuple(dst)])
    return out


def peak_mask(h: np.ndarray, r: int, thr: float) -> np.ndarray:
    """The separable form, vectorised over (..., H, W): Mrow = row max over [x-r, x+r], L = row max over [x-r, x-1], U = max of Mrow over
    rows [y-r, y-1], Dn = max of Mrow over rows [y, y+r]; peak iff v >= thr and v >= max(U, Dn) and v > max(U, L)."""
    v = np.where(np.isnan(h), np.float32(-np.inf), h).astype(np.float32)
    mrow = _shift_max(v, -r, r, -1)
    left = _shift_max(v, -r, -1, -1)
    up = _shift_max(mrow, -r, -1, -2)
    dn = _shift_max(mrow, 0, r, -2)
    return (v >= np.float32(thr)) & (v >= np.maximum(up, dn)) & (v > np.maximum(up, left))


def peak_decode_ref(heat: np.ndarray, max_peaks: int, thr: float, r: int, mask: np.ndarray = None):
    """(..., H, W) fp32 -> (yx int32 (..., N, 2), score fp32 (..., N), count int32 (...)) with the kernel's order and padding.
    `mask` (the peak_mask of heat) may be passed in when several N share one map."""
    heat = np.asarray(heat, dtype=np.float32)
    lead, (H, W) = heat.shape[:-2], heat.shape[-2:]
    if mask is None:
        mask = peak_mask(heat, r, thr)
    flat, fmask = heat.reshape(-1, H * W), mask.reshape(-1, H * W)
    M = flat.shape[0]
    yx = np.full((M, max_peaks, 2), -1, np.int32)
    score = np.full((M, max_peaks), -np.inf, np.float32)
    count = np.zeros(M, np.int32)
    for m in range(M):
        idx = np.flatnonzero(fmask[m])
        vals = flat[m, idx]
        idx = idx[np.lexsort((idx, -vals))][:max_peaks]
        n = idx.size
        yx[m, :n, 0], yx[m, :n, 1] = idx // W, idx % W
        score[m, :n] = flat[m, idx]
        count[m] = n
    return yx.reshape(lead + (max_peaks, 2)), score.reshape(lead + (max_peaks,)), count.reshape(lead)
