"""Synthetic keypoint data + a deterministic fit loop on the B200 training engine.

The reference trains on rope images with K labelled keypoints (README.md:18-38); there is no dataset here, so the parity fixtures,
`smoke()` and the benches use the stand-in SURVEY.md §8c defines for the trained fixture "F-trn": a noisy dark image with one
coloured radius-6 disc per keypoint, labels = disc centres as (x, y), targets = the reference's Gaussians (dataset.py:36-44).
Everything random comes from a seeded CPU `torch.Generator`, the engine's kernels are bit-reproducible (fixed-order reductions,
no atomics) and the optimiser is `FusedAdam`, so `fit_synthetic` gives the same state dict on every run and every B200
(`tests/test_gpu_model.py` pins its SHA-256).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch

_SATURATED = ((1.0, 0.1, 0.1), (0.1, 1.0, 0.1), (0.1, 0.1, 1.0), (1.0, 1.0, 0.1), (0.1, 1.0, 1.0), (1.0, 0.1, 1.0), (1.0, 1.0, 1.0))
DISC_RADIUS = 6


def disc_palette(K: int) -> torch.Tensor:
    """(K, 2, 3): inner (r <= 3) and outer (3 < r <= 6) colour of keypoint k's disc.  K <= 7: uniform saturated colours (the first
    four are SURVEY.md's red / green / blue / yellow); beyond that two-tone discs, 49 distinguishable combinations."""
    if not 1 <= K <= 49:
        raise ValueError("disc_palette supports 1..49 keypoints")
    cols = torch.tensor(_SATURATED)
    if K <= 7:
        return torch.stack([cols[:K], cols[:K]], 1)
    idx = [(k % 7, (k // 7 + k) % 7) for k in range(K)]
    return torch.stack([torch.stack([cols[i], cols[j]]) for i, j in idx])


def disc_batch(gen: torch.Generator, B: int, H: int, W: int, K: int = 4, on_lattice: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (img (B,3,H,W) fp32 in [0,1] on the CPU, uv (B,K,2) fp32 = (x, y) disc centres).
    on_lattice: centres sit on the pixels the stride-8 logit lattice maps to under the align_corners=True upsample
    (x = round(j*(W-1)/(W/8-1))), so the fp32 heatmap has ONE best lattice node per keypoint with a wide margin -- a centre half-way
    between two nodes makes the two nodes tie and no finite-precision scheme can then pin the argmax to one of them."""
    if on_lattice:
        h8, w8 = H // 8, W // 8
        # distinct nodes of the odd sub-lattice (16 px apart: the radius-6 discs of one image never overlap)
        ny, nx = (h8 - 2) // 2, (w8 - 2) // 2
        if ny * nx < K:
            raise ValueError("image too small for K non-overlapping lattice discs")
        pick = torch.stack([torch.randperm(ny * nx, generator=gen)[:K] for _ in range(B)])
        jy, jx = 1 + 2 * (pick // nx), 1 + 2 * (pick % nx)
        ux = torch.round(jx.double() * (W - 1) / (w8 - 1))
        uy = torch.round(jy.double() * (H - 1) / (h8 - 1))
        uv = torch.stack([ux, uy], -1).float()
    else:
        uv = torch.stack([torch.randint(8, W - 8, (B, K), generator=gen), torch.randint(8, H - 8, (B, K), generator=gen)], -1).float()
    img = 0.2 * torch.rand(B, 3, H, W, generator=gen)
    pal = disc_palette(K)
    r = DISC_RADIUS
    d = torch.arange(-r, r + 1).float()
    rr = d.view(-1, 1) ** 2 + d.view(1, -1) ** 2                      # (13,13) squared distance to the centre
    outer = (rr <= r * r).float()
    inner = (rr <= 9).float()
    for b in range(B):
        for k in range(K):
            cx, cy = int(uv[b, k, 0]), int(uv[b, k, 1])
            y0, y1, x0, x1 = max(cy - r, 0), min(cy + r + 1, H), max(cx - r, 0), min(cx + r + 1, W)
            mo = outer[y0 - (cy - r): y1 - (cy - r), x0 - (cx - r): x1 - (cx - r)]
            mi = inner[y0 - (cy - r): y1 - (cy - r), x0 - (cx - r): x1 - (cx - r)]
            colour = pal[k, 1].view(3, 1, 1) * (mo - mi) + pal[k, 0].view(3, 1, 1) * mi
            win = img[b, :, y0:y1, x0:x1]
            img[b, :, y0:y1, x0:x1] = win * (1 - mo) + mo * (0.2 * win) + 0.8 * colour
    return img, uv


def fit_synthetic(model, steps: int, B: int, H: int, W: int, lr: float = 1e-3, weight_decay: float = 1e-4, sigma: float = 8.0,
                  data_seed: int = 42, optimizer=None, decay_after: float = 1.0) -> List[float]:
    """`steps` iterations of reference train.py:33-36 (zero_grad, forward, backward, Adam step) on disc batches through the B200
    training engine (`train_ops.train_step`, backend "hk") with `FusedAdam`.  Deterministic.  Returns the per-step losses
    (one device sync per step, like the reference's `loss.item()` at train.py:37).  After `decay_after * steps` steps the learning
    rate drops to lr / 10, so the fit settles and the BatchNorm running statistics match the final weights."""
    from . import train_ops
    from .optim import FusedAdam

    K = int(model.num_keypoints)
    dev = next(model.parameters()).device
    if dev.type != "cuda":
        raise RuntimeError("fit_synthetic needs the model on the GPU (no CPU path)")
    model.train()
    opt = optimizer if optimizer is not None else FusedAdam(model.parameters(), lr=lr, weight_decay=weight_decay)
    gen = torch.Generator().manual_seed(data_seed)
    losses = []
    for step in range(steps):
        if step == int(decay_after * steps):
            for g in opt.param_groups:
                g["lr"] = lr / 10
        img, uv = disc_batch(gen, B, H, W, K)
        losses.append(float(train_ops.train_step(model, opt, img.to(dev), uv.to(dev), sigma=sigma).item()))
    return losses


# The trained fixtures ("F-trn", SURVEY.md §8c) of the parity tests, smoke() and tools/pin_ftrn.py.  Hyper-parameters follow config.py /
# train.py where they exist (batch 4, sigma 8, weight decay 1e-4) except the learning rate (1e-3 instead of 1e-4: the fixture has to
# converge in a few hundred steps, SURVEY.md App. B); the last 40 % of the steps run at lr/10 so the fit settles (without that the
# eval-mode heatmaps -- BatchNorm on running statistics -- swing from checkpoint to checkpoint: tools/diag_ftrn_quality.py).
FIXTURES = {
    # BASELINE configs[1]/[3] shape: K=4 at config.py resolution
    "k4_480x640": dict(K=4, B=4, H=480, W=640, steps=400, decay_after=0.6, lr=1e-3, weight_decay=1e-4, sigma=8.0, model_seed=0, data_seed=42),
    # BASELINE configs[4] (960x1280, K up to 32): trained at 240x320 (the net is fully convolutional; discs keep their pixel size)
    "k32_240x320": dict(K=32, B=4, H=240, W=320, steps=1200, decay_after=0.6, lr=1e-3, weight_decay=1e-4, sigma=8.0, model_seed=0, data_seed=43),
    # smoke()-sized
    "k4_128x160": dict(K=4, B=4, H=128, W=160, steps=300, decay_after=0.6, lr=1e-3, weight_decay=1e-4, sigma=8.0, model_seed=0, data_seed=44),
}


def train_fixture(name: str):
    """Train fixture `name` from its seeds on cuda (current device) -> (state_dict on the CPU, per-step losses).  Bit-reproducible."""
    from .model import KeypointsGauss

    cfg = FIXTURES[name]
    torch.manual_seed(cfg["model_seed"])
    model = KeypointsGauss(cfg["K"], img_height=cfg["H"], img_width=cfg["W"]).cuda()
    losses = fit_synthetic(model, cfg["steps"], cfg["B"], cfg["H"], cfg["W"], lr=cfg["lr"], weight_decay=cfg["weight_decay"],
                           sigma=cfg["sigma"], data_seed=cfg["data_seed"], decay_after=cfg.get("decay_after", 1.0))
    torch.cuda.synchronize()
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    return sd, losses


def state_dict_sha256(sd) -> str:
    import hashlib

    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()
