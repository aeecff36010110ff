"""KeypointAugment: random affine warp and photometric jitter of a training batch on the GPU, with the keypoint labels moved along.

The reference carries a domain-randomisation pipeline (src/dataset.py:18-31, imgaug; commented out there) and clips labels into the
image (:63-66).  Here a batch is augmented on the device in two launches (csrc/augment.cu): `hk_augment_pick` moves the (B,K,2) labels
and `hk_augment_images` warps and jitters the (B,3,H,W) fp32 images.  Because the training engine builds its Gaussian targets from the
labels inside the loss kernel, no target tensor is ever warped.

Per image the host draws, from a seeded CPU `torch.Generator` owned by the augmenter:
    rotation theta ~ U[-rotate, rotate] degrees, scale s ~ U[scale], translation tx ~ U[-translate*W, translate*W],
    ty ~ U[-translate*H, translate*H]        (`tries` candidates of these)
    brightness beta ~ U[-brightness, brightness], contrast c ~ U[contrast], gain g_ch ~ U[1 - channel_gain, 1 + channel_gain]
and, once per call, a 64-bit Philox key for the noise.  Geometry, in pixel indices (x in [0, W-1], y in [0, H-1], the dataset's label
convention): A(p) = s*R(theta)*(p - ctr) + ctr + t with ctr = ((W-1)/2, (H-1)/2); labels become A(uv), the image is sampled at
A^-1(p) (bilinear, zero outside).  Positive theta turns x towards y (clockwise on screen).  Each image takes the first candidate that
keeps all its labels inside the frame, or the identity geometry if none does (`last_pick` = -1); the photometric jitter applies either
way.  The forward and inverse matrices are computed in fp64 and rounded once to fp32; the kernels read that table.

Drawing costs no host-device synchronisation: the tables go to the device through a pinned buffer and `copy_(non_blocking=True)`.
A call is a pure function of the generator state and the inputs.  Under `torch.distributed` the rank is folded into the seed at
construction so replicas see different transforms (`rank=` overrides).
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import ops
from ._lib import AUGMENT_MAX_TRIES

_RANK_STRIDE = 0x9E3779B97F4A7C15   # odd 64-bit constant: rank r starts the generator at seed + r * stride (mod 2^64)


class AugmentParams(NamedTuple):
    """The parameter tables of one call (CPU tensors)."""
    fwd: torch.Tensor     # (B, tries, 2, 3) fp32: label maps A
    inv: torch.Tensor     # (B, tries, 2, 3) fp32: image sampling maps A^-1
    photo: torch.Tensor   # (B, 5) fp32: contrast, brightness, gain of channels 0..2
    key: int              # 64-bit Philox key of the noise


def _range(name: str, v) -> Tuple[float, float]:
    lo, hi = (float(x) for x in v)
    if not (math.isfinite(lo) and math.isfinite(hi)):
        raise ValueError(f"KeypointAugment: {name} must be finite")
    if lo > hi:
        raise ValueError(f"KeypointAugment: {name} range has lo {lo} > hi {hi}")
    return lo, hi


def _amount(name: str, v) -> float:
    v = float(v)
    if not math.isfinite(v) or v < 0:
        raise ValueError(f"KeypointAugment: {name} must be a finite value >= 0, got {v}")
    return v


class KeypointAugment:
    """Augmenter of (img (B,3,H,W) fp32 CUDA, uv (B,K,2) labels) batches.  All ranges default to their neutral value, which returns
    the batch unchanged (bit for bit for images in [0, 1]).

    rotate        max |theta| in degrees                      scale       (lo, hi) of the isotropic scale, lo > 0
    translate     max shift as a fraction of W (x) / H (y)   brightness  max |beta| added after the contrast
    contrast      (lo, hi) of c in (v - 0.5)*c + 0.5          channel_gain max |g_ch - 1|
    noise_std     std of the additive Gaussian noise          tries       candidate geometries per image (1..16)
    seed, rank    generator seed; rank (default: the torch.distributed rank, else 0) is folded into it
    """

    def __init__(self, rotate: float = 0., scale=(1., 1.), translate: float = 0., brightness: float = 0., contrast=(1., 1.),
                 channel_gain: float = 0., noise_std: float = 0., tries: int = 4, seed: int = 0, rank: Optional[int] = None):
        self.rotate = _amount("rotate", rotate)
        self.translate = _amount("translate", translate)
        self.brightness = _amount("brightness", brightness)
        self.channel_gain = _amount("channel_gain", channel_gain)
        self.noise_std = _amount("noise_std", noise_std)
        self.scale = _range("scale", scale)
        if self.scale[0] <= 0:
            raise ValueError(f"KeypointAugment: scale must be > 0, got {self.scale}")
        self.contrast = _range("contrast", contrast)
        if self.contrast[0] < 0:
            raise ValueError(f"KeypointAugment: contrast must be >= 0, got {self.contrast}")
        if int(tries) != tries or not 1 <= tries <= AUGMENT_MAX_TRIES:
            raise ValueError(f"KeypointAugment: tries must be an integer in 1..{AUGMENT_MAX_TRIES}, got {tries}")
        self.tries = int(tries)
        if rank is None:
            import torch.distributed as dist
            rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        self.seed, self.rank = int(seed), int(rank)
        self._gen = torch.Generator().manual_seed((self.seed + self.rank * _RANK_STRIDE) % (1 << 64))
        self.calls = 0
        self.last_pick: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ parameters
    def _sample(self, B: int, H: int, W: int) -> AugmentParams:
        """Consume the generator for one call of batch B at H x W."""
        g, T = self._gen, self.tries
        u = torch.rand(B, T, 4, dtype=torch.float64, generator=g).numpy()
        v = torch.rand(B, 5, dtype=torch.float64, generator=g).numpy()
        k = torch.randint(0, 1 << 32, (2,), dtype=torch.int64, generator=g).tolist()
        theta = np.deg2rad(self.rotate * (2.0 * u[..., 0] - 1.0))
        s = self.scale[0] + (self.scale[1] - self.scale[0]) * u[..., 1]
        t = np.stack([self.translate * W * (2.0 * u[..., 2] - 1.0), self.translate * H * (2.0 * u[..., 3] - 1.0)], -1)
        ctr = np.array([(W - 1) / 2.0, (H - 1) / 2.0])
        co, si = np.cos(theta), np.sin(theta)
        rot = np.stack([np.stack([co, -si], -1), np.stack([si, co], -1)], -2)            # (B, T, 2, 2)
        m = s[..., None, None] * rot
        fwd = np.concatenate([m, (ctr + t - np.einsum("btij,j->bti", m, ctr))[..., None]], -1)
        minv = np.swapaxes(rot, -1, -2) / s[..., None, None]                              # (s R)^-1 = R^T / s
        inv = np.concatenate([minv, (ctr - np.einsum("btij,btj->bti", minv, ctr + t))[..., None]], -1)
        photo = np.empty((B, 5))
        photo[:, 0] = self.contrast[0] + (self.contrast[1] - self.contrast[0]) * v[:, 0]
        photo[:, 1] = self.brightness * (2.0 * v[:, 1] - 1.0)
        photo[:, 2:] = 1.0 + self.channel_gain * (2.0 * v[:, 2:] - 1.0)
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))   # noqa: E731
        return AugmentParams(f32(fwd), f32(inv), f32(photo), int(k[0]) | (int(k[1]) << 32))

    def draw(self, B: int, H: int, W: int) -> AugmentParams:
        """The parameter tables the next call on a (B,3,H,W) batch will use, without consuming them."""
        state = self._gen.get_state()
        try:
            return self._sample(B, H, W)
        finally:
            self._gen.set_state(state)

    # ------------------------------------------------------------------ the call
    def __call__(self, img: torch.Tensor, uv: torch.Tensor, out: Optional[torch.Tensor] = None,
                 uv_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """img (B,3,H,W) fp32 CUDA, uv (B,K,2) CUDA -> (img_aug, uv_aug), written into out / uv_out when given (neither may overlap
        its input).  Two launches on the current stream; no host synchronisation."""
        if img.dim() != 4 or img.shape[1] != 3 or not img.is_cuda:
            raise ValueError(f"KeypointAugment: img must be a (B,3,H,W) CUDA tensor, got {tuple(img.shape)} on {img.device}")
        B, _, H, W = img.shape
        if uv.dim() != 3 or uv.shape[0] != B or uv.shape[2] != 2 or not uv.is_cuda:
            raise ValueError(f"KeypointAugment: uv must be a (B,K,2) CUDA tensor with B = {B}, got {tuple(uv.shape)} on {uv.device}")
        if img.dtype != torch.float32:
            raise ValueError(f"KeypointAugment: img must be float32, got {img.dtype}")
        img = img.contiguous()
        uv = uv.to(torch.float32).contiguous()
        if (out is not None and ops._overlap(img, out)) or (uv_out is not None and ops._overlap(uv, uv_out)):
            raise ValueError("KeypointAugment: out / uv_out must not overlap img / uv (no in-place augmentation)")
        p = self._sample(B, H, W)
        tables = [p.fwd.view(-1), p.inv.view(-1), p.photo.view(-1)]
        host = torch.empty(sum(t.numel() for t in tables), dtype=torch.float32, pin_memory=True)
        torch.cat(tables, out=host)
        dev = torch.empty_like(host, device=img.device).copy_(host, non_blocking=True)
        n = p.fwd.numel()
        fwd, inv, photo = dev[:n].view(p.fwd.shape), dev[n:2 * n].view(p.inv.shape), dev[2 * n:].view(p.photo.shape)
        uv_out, pick = ops.augment_pick(fwd, uv, H, W, uv_out=uv_out)
        out = ops.augment_images(img, inv, pick, photo, self.noise_std, p.key, out=out)
        self.last_pick = pick
        self.calls += 1
        return out, uv_out

    # ------------------------------------------------------------------ checkpointing
    def state_dict(self) -> dict:
        """Generator state and call count: a run restored from it continues with the same augmentation sequence."""
        return {"generator": self._gen.get_state(), "calls": self.calls}

    def load_state_dict(self, state: dict) -> None:
        self._gen.set_state(state["generator"].clone())
        self.calls = int(state["calls"])

    def __repr__(self) -> str:
        return (f"KeypointAugment(rotate={self.rotate}, scale={self.scale}, translate={self.translate}, brightness={self.brightness}, "
                f"contrast={self.contrast}, channel_gain={self.channel_gain}, noise_std={self.noise_std}, tries={self.tries}, "
                f"seed={self.seed}, rank={self.rank})")
