"""Host restatements of the augmentation kernels (csrc/augment.cu) that tests/test_augment_host.py and tests/test_gpu_augment.py
compare against: Philox4x32-10 and the Box-Muller normals in numpy, the candidate pick + label map in numpy fp32 with the kernel's
rounding sequence, and the warp and photometric steps in float64."""
import numpy as np
import torch

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key) -> np.ndarray:
    """Random123's Philox4x32-10.  ctr (..., 4) and key (..., 2) of uint32 values (broadcast) -> (..., 4) uint32."""
    ctr, key = np.asarray(ctr, dtype=np.uint64), np.asarray(key, dtype=np.uint64)
    c = [ctr[..., i] for i in range(4)]
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = np.uint64(_M0) * c[0], np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0, k1 = (k0 + np.uint64(_W0)) & _MASK, (k1 + np.uint64(_W1)) & _MASK
    return np.stack(np.broadcast_arrays(*c), -1).astype(np.uint32)


def uniform_open(r: np.ndarray) -> np.ndarray:
    """23 random bits -> (m + 0.5) * 2^-23, strictly inside (0, 1) (exact in fp32 and fp64)."""
    return ((r >> np.uint32(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def noise_normals(key: int, B: int, H: int, W: int) -> np.ndarray:
    """(B, 3, H, W) float64 N(0,1) values of the kernel: counter (x/4, y, channel, b), key (low word, high word), one Philox output
    -> two Box-Muller pairs for pixels x0..x0+3."""
    wq = (W + 3) // 4
    b, ch, y, xq = np.meshgrid(np.arange(B), np.arange(3), np.arange(H), np.arange(wq), indexing="ij")
    r = philox4x32_10(np.stack([xq, y, ch, b], -1), [key & 0xFFFFFFFF, key >> 32])
    u = uniform_open(r)
    rad01, rad23 = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    n = np.stack([rad01 * np.cos(2 * np.pi * u[..., 1]), rad01 * np.sin(2 * np.pi * u[..., 1]),
                  rad23 * np.cos(2 * np.pi * u[..., 3]), rad23 * np.sin(2 * np.pi * u[..., 3])], -1)
    return n.reshape(B, 3, H, 4 * wq)[..., :W]


def _affine_f32(m, x, y):
    """(m0*x + m1*y) + m2 with one fp32 rounding per operation, the kernel's sequence."""
    return (m[..., 0] * x + m[..., 1] * y) + m[..., 2]


def pick_and_move(fwd: np.ndarray, uv: np.ndarray, H: int, W: int):
    """fwd (B,T,2,3) fp32, uv (B,K,2) fp32 -> (pick (B,) int32, first candidate keeping every label in [0,W-1] x [0,H-1] or -1;
    uv' (B,K,2) fp32 under it, uv unchanged for -1)."""
    fwd, uv = np.asarray(fwd, dtype=np.float32), np.asarray(uv, dtype=np.float32)
    B, T = fwd.shape[:2]
    x, y = uv[:, None, :, 0], uv[:, None, :, 1]                                   # (B,1,K)
    xp, yp = _affine_f32(fwd[:, :, None, 0, :], x, y), _affine_f32(fwd[:, :, None, 1, :], x, y)   # (B,T,K)
    ok = ((xp >= 0) & (xp <= np.float32(W - 1)) & (yp >= 0) & (yp <= np.float32(H - 1))).all(-1)
    pick = np.where(ok.any(1), ok.argmax(1), -1).astype(np.int32)
    out = uv.copy()
    for b in range(B):
        if pick[b] >= 0:
            out[b] = np.stack([xp[b, pick[b]], yp[b, pick[b]]], -1)
    return pick, out


def warp_ref(img: torch.Tensor, inv: torch.Tensor, pick) -> torch.Tensor:
    """float64 F.grid_sample(align_corners=True, padding_mode="zeros") at A^-1(p), A^-1 = inv[b, pick[b]] (fp32 values, identity for
    pick -1), p = integer pixel coordinates."""
    img = img.double().cpu()
    B, _, H, W = img.shape
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    out = torch.empty_like(img)
    for b in range(B):
        p = int(pick[b])
        m = inv[b, p].double().cpu() if p >= 0 else torch.tensor([[1., 0., 0.], [0., 1., 0.]], dtype=torch.float64)
        xs = m[0, 0] * xx + m[0, 1] * yy + m[0, 2]
        ys = m[1, 0] * xx + m[1, 1] * yy + m[1, 2]
        grid = torch.stack([xs * 2 / (W - 1) - 1, ys * 2 / (H - 1) - 1], -1)[None]
        out[b] = torch.nn.functional.grid_sample(img[b:b + 1], grid, mode="bilinear", padding_mode="zeros", align_corners=True)[0]
    return out


def photometric_ref(v: torch.Tensor, photo: torch.Tensor, noise_std: float = 0.0, normals=None) -> torch.Tensor:
    """float64 steps after the warp: v = (v - 0.5)*c + 0.5 + beta; v *= g_ch; v += noise_std*n; clamp to [0, 1]."""
    v = v.double().cpu()
    ph = photo.double().cpu()
    c, beta, g = ph[:, 0].view(-1, 1, 1, 1), ph[:, 1].view(-1, 1, 1, 1), ph[:, 2:].view(-1, 3, 1, 1)
    v = ((v - 0.5) * c + 0.5 + beta) * g
    if normals is not None:
        v = v + float(np.float32(noise_std)) * torch.as_tensor(normals, dtype=torch.float64)
    return v.clamp(0.0, 1.0)
