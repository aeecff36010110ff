"""CPU oracle for the hulk-keypoints hot path.  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A functional restatement (torch CPU fp32 / numpy) of the reference's KeypointsGauss path.  The
reference's arithmetic lives in the third-party `torch` wheel (pinned torch==1.1.0,
`docker/Dockerfile:29`; here torch 2.11 executes the same call sites), so the restatement is
written against `torch.nn.functional` for the network and plain numpy for the small kernels.
Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of
`bench.py` may import this module; the product package (`hulk_keypoints_b200/`) never does.

Parity status: the reference ships no tests or golden vectors (SURVEY.md §4), so the oracle is
pinned against OUTPUTS OF THE REFERENCE ITSELF, imported unmodified in the build container
(`oracle/reference_loader.py`) -- see `oracle/make_golden.py` and `tests/test_oracle_golden.py`.
Every function cites the reference lines it restates (paths relative to the reference root).
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, List, NamedTuple, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = 1e-5  # torch default used by nn.BatchNorm2d at src/resnet.py:46,49,139,187
BN_MOMENTUM = 0.1
NUM_CLASSES = 1000  # src/resnet_dilated.py:6 -- KeypointsGauss never overrides it (src/model.py:17)
PREFIX = "resnet.resnet34_8s."  # KeypointsGauss.resnet (model.py:17) . Resnet34_8s.resnet34_8s (resnet_dilated.py:17)
# torch CPU threads of tests/golden/golden_v1.*: oneDNN blocks its fp32 convolutions (and so orders their sums) by the thread count,
# so the bit-equal golden cases reproduce only at the count they were recorded with, whatever the host's core count
GOLDEN_CPU_THREADS = 8


class ConvSpec(NamedTuple):
    name: str        # state_dict stem, e.g. "layer3.0.conv1"
    bn: Optional[str]  # matching BatchNorm stem or None (fc)
    cin: int
    cout: int
    k: int
    stride: int
    pad: int
    dil: int


class BlockSpec(NamedTuple):
    conv1: ConvSpec
    conv2: ConvSpec
    down: Optional[ConvSpec]


def network_spec() -> Tuple[ConvSpec, List[BlockSpec], ConvSpec]:
    """Shapes of the 37 convolutions of Resnet34_8s.

    Restates `ResNet.__init__` / `_make_layer` (src/resnet.py:117-196) for
    `resnet34(fully_conv=True, output_stride=8, remove_avg_pool_layer=True)`
    (src/resnet_dilated.py:10-13): blocks [3,4,6,3]; once the running stride reaches 8 every
    further stride-2 stage multiplies the dilation instead (resnet.py:170-175) and that dilation is
    handed to EVERY block of the stage including block 0 (resnet.py:191-194); conv3x3 pads by its
    dilation (resnet.py:23-37); the 1x1 downsample is never dilated (resnet.py:184-188).
    """
    stem = ConvSpec("conv1", "bn1", 3, 64, 7, 2, 3, 1)
    blocks: List[BlockSpec] = []
    inplanes, cur_stride, cur_dil, out_stride = 64, 4, 1, 8
    for li, (planes, nblocks, stride) in enumerate(((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)), start=1):
        down = None
        if stride != 1 or inplanes != planes:
            if cur_stride == out_stride:
                cur_dil *= stride
                stride = 1
            else:
                cur_stride *= stride
            down = ConvSpec(f"layer{li}.0.downsample.0", f"layer{li}.0.downsample.1", inplanes, planes, 1, stride, 0, 1)
        for bi in range(nblocks):
            s = stride if bi == 0 else 1
            cin = inplanes if bi == 0 else planes
            c1 = ConvSpec(f"layer{li}.{bi}.conv1", f"layer{li}.{bi}.bn1", cin, planes, 3, s, cur_dil, cur_dil)
            c2 = ConvSpec(f"layer{li}.{bi}.conv2", f"layer{li}.{bi}.bn2", planes, planes, 3, 1, cur_dil, cur_dil)
            blocks.append(BlockSpec(c1, c2, down if bi == 0 else None))
        inplanes = planes
    fc = ConvSpec("fc", None, 512, NUM_CLASSES, 1, 1, 0, 1)
    return stem, blocks, fc


def _default_conv_init_draws(cout: int, cin: int, k: int, bias: bool) -> None:
    """Consume the RNG exactly as nn.Conv2d/nn.Linear.reset_parameters would (values discarded).

    The reference builds every layer with torch's default init first (resnet.py:137,36,185,149,153;
    resnet_dilated.py:16) and only then overwrites it, so the default draws shift the RNG stream
    that the kept `normal_` draws come from.
    """
    w = torch.empty(cout, cin, k, k)
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    if bias:
        torch.empty(cout).uniform_(-1.0, 1.0)


def init_state_dict(seed: int) -> "OrderedDict[str, torch.Tensor]":
    """Seeded random-init weights, bit-identical to constructing the reference model after
    `torch.manual_seed(seed)` with the pretrained download stubbed out.

    Restates the init order of `ResNet.__init__` (resnet.py:137-161) followed by
    `Resnet34_8s.__init__` (resnet_dilated.py:16-22): conv `N(0, sqrt(2/(k*k*cout)))`, BN gamma=1
    beta=0, then a fresh 1x1 `fc` conv drawn `N(0, 0.01)` with zero bias.  Key order follows
    module registration order so `list(sd)` equals the reference `state_dict()` key list.
    """
    stem, blocks, fc = network_spec()
    torch.manual_seed(seed)
    # --- construction-time default inits (RNG consumed, values discarded) ---
    _default_conv_init_draws(stem.cout, stem.cin, stem.k, bias=False)
    for b in blocks:
        if b.down is not None:  # _make_layer builds the downsample before the blocks (resnet.py:184-191)
            _default_conv_init_draws(b.down.cout, b.down.cin, 1, bias=False)
        _default_conv_init_draws(b.conv1.cout, b.conv1.cin, 3, bias=False)
        _default_conv_init_draws(b.conv2.cout, b.conv2.cin, 3, bias=False)
    for _ in range(2):  # nn.Linear(512, 1000) is built twice when fully_conv (resnet.py:149,153)
        _default_conv_init_draws(NUM_CLASSES, 512, 1, bias=True)

    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()

    def put_conv(c: ConvSpec):
        n = c.k * c.k * c.cout
        sd[PREFIX + c.name + ".weight"] = torch.empty(c.cout, c.cin, c.k, c.k).normal_(0, math.sqrt(2.0 / n))

    def put_bn(stem_name: str, ch: int):
        sd[PREFIX + stem_name + ".weight"] = torch.ones(ch)
        sd[PREFIX + stem_name + ".bias"] = torch.zeros(ch)
        sd[PREFIX + stem_name + ".running_mean"] = torch.zeros(ch)
        sd[PREFIX + stem_name + ".running_var"] = torch.ones(ch)
        sd[PREFIX + stem_name + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)

    # --- the kept init: `for m in self.modules()` order (resnet.py:155-161) ---
    put_conv(stem)
    put_bn(stem.bn, stem.cout)
    for b in blocks:
        put_conv(b.conv1)
        put_bn(b.conv1.bn, b.conv1.cout)
        put_conv(b.conv2)
        put_bn(b.conv2.bn, b.conv2.cout)
        if b.down is not None:
            put_conv(b.down)
            put_bn(b.down.bn, b.down.cout)
    # --- scoring layer (resnet_dilated.py:16-22) ---
    _default_conv_init_draws(NUM_CLASSES, 512, 1, bias=True)
    sd[PREFIX + "fc.weight"] = torch.empty(NUM_CLASSES, 512, 1, 1).normal_(0, 0.01)
    sd[PREFIX + "fc.bias"] = torch.zeros(NUM_CLASSES)
    return sd


# --------------------------------------------------------------------------------------------
# forward
# --------------------------------------------------------------------------------------------

def _conv(sd, c: ConvSpec, x: torch.Tensor) -> torch.Tensor:
    return F.conv2d(x, sd[PREFIX + c.name + ".weight"], None, c.stride, c.pad, c.dil)


def _bn(sd, name: str, x: torch.Tensor, train: bool, new_stats: Optional[dict]) -> torch.Tensor:
    w, b = sd[PREFIX + name + ".weight"], sd[PREFIX + name + ".bias"]
    rm, rv = sd[PREFIX + name + ".running_mean"], sd[PREFIX + name + ".running_var"]
    if not train:
        return F.batch_norm(x, rm, rv, w, b, False, BN_MOMENTUM, BN_EPS)
    rm2, rv2 = rm.clone(), rv.clone()
    y = F.batch_norm(x, rm2, rv2, w, b, True, BN_MOMENTUM, BN_EPS)
    if new_stats is not None:
        new_stats[PREFIX + name + ".running_mean"] = rm2
        new_stats[PREFIX + name + ".running_var"] = rv2
    return y


def backbone_features(sd, x: torch.Tensor, train: bool = False, new_stats: Optional[dict] = None) -> torch.Tensor:
    """`ResNet.forward` up to (not including) `fc` (resnet.py:198-213, avgpool removed).

    Stem conv-BN-ReLU-maxpool(3,2,1) (resnet.py:199-202) then 16 BasicBlocks
    `relu(bn2(conv2(relu(bn1(conv1(x))))) + shortcut)` (resnet.py:53-69).
    """
    stem, blocks, _ = network_spec()
    x = F.relu(_bn(sd, stem.bn, _conv(sd, stem, x), train, new_stats))
    x = F.max_pool2d(x, 3, 2, 1)
    for b in blocks:
        out = F.relu(_bn(sd, b.conv1.bn, _conv(sd, b.conv1, x), train, new_stats))
        out = _bn(sd, b.conv2.bn, _conv(sd, b.conv2, out), train, new_stats)
        res = x if b.down is None else _bn(sd, b.down.bn, _conv(sd, b.down, x), train, new_stats)
        x = F.relu(out + res)
    return x


def logits_lowres(sd, feat: torch.Tensor, num_keypoints: int) -> torch.Tensor:
    """The live rows of the 1x1 scoring conv (resnet.py:215 / resnet_dilated.py:16).

    The reference computes all 1000 channels, upsamples them and only then slices `[:, :K]`
    (model.py:21).  A 1x1 conv and bilinear interpolation act per output channel, so slicing the
    weight rows first is bit-identical on the kept channels (checked in tests/test_oracle_golden).
    """
    w = sd[PREFIX + "fc.weight"][:num_keypoints]
    b = sd[PREFIX + "fc.bias"][:num_keypoints]
    return F.conv2d(feat, w, b)


def heatmaps_from_logits(logits: torch.Tensor, size: Tuple[int, int]) -> torch.Tensor:
    """`upsample_bilinear(size=input HxW)` (resnet_dilated.py:27, == align_corners=True) then sigmoid (model.py:21)."""
    up = F.interpolate(logits, size=size, mode="bilinear", align_corners=True)
    return torch.sigmoid(up)


def forward(sd, x: torch.Tensor, num_keypoints: int = 4, train: bool = False,
            new_stats: Optional[dict] = None, as_written: bool = False) -> torch.Tensor:
    """`KeypointsGauss.forward` (model.py:19-22): (B,3,H,W) f32 -> (B,K,H,W) f32 heatmaps.

    `train=False` is the eval()/no_grad oracle used for inference parity (BN folded at inference is
    the north-star semantics; the reference scripts never call .eval(), SURVEY.md §0.2).
    `as_written=True` keeps the literal op order (1000-channel fc and upsample, then slice); it is
    bit-equal to the reference module on CPU.  The default slices the fc rows first, which is the
    same arithmetic per kept channel but lets oneDNN pick another conv kernel (observed |d| <= 1e-6).
    """
    with torch.no_grad():
        feat = backbone_features(sd, x, train, new_stats)
        if as_written:
            full = F.conv2d(feat, sd[PREFIX + "fc.weight"], sd[PREFIX + "fc.bias"])
            up = F.interpolate(full, size=x.shape[2:], mode="bilinear", align_corners=True)
            return torch.sigmoid(up[:, :num_keypoints])
        return heatmaps_from_logits(logits_lowres(sd, feat, num_keypoints), x.shape[2:])


def train_step_loss_and_grads(sd, x: torch.Tensor, uv: np.ndarray, num_keypoints: int = 4, sigma: float = 8.0):
    """One training step's loss and parameter gradients as reference train.py:18-26,35 computes them: train-mode forward
    (batch-statistic BatchNorm, running stats advanced), `pred.double()`, `nn.BCELoss()(pred, gt_gauss)` with the float64 Gaussian
    targets of dataset.py:36-44, `loss.backward()` -- torch CPU autograd over the functional restatement above.

    Returns (loss float, grads {state_dict key: tensor} for every parameter, new_stats {running_mean/var key: tensor}).  The head is
    evaluated on the K live fc rows only (per-channel ops: identical values); the 996 dead rows receive exactly zero gradient, as in
    the reference where the `[:, :K]` slice (model.py:21) cuts them off."""
    work = OrderedDict()
    params = {}
    for k, v in sd.items():
        if v.dtype.is_floating_point and "running_" not in k:
            params[k] = v.detach().clone().requires_grad_(True)
            work[k] = params[k]
        else:
            work[k] = v.detach().clone()
    stats: dict = {}
    feat = backbone_features(work, x, True, stats)
    heat = heatmaps_from_logits(logits_lowres(work, feat, num_keypoints), x.shape[2:])
    gt = torch.from_numpy(gauss_targets(np.asarray(uv), x.shape[2], x.shape[3], sigma))
    loss = F.binary_cross_entropy(heat.double(), gt)          # == nn.BCELoss()(pred.double(), gt)
    loss.backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in params.items()}
    return float(loss.item()), grads, stats


def forward_as_written(sd, x: torch.Tensor, num_keypoints: int = 4) -> torch.Tensor:
    return forward(sd, x, num_keypoints, as_written=True)


def calibrate_bn(sd, batches: List[torch.Tensor]) -> "OrderedDict[str, torch.Tensor]":
    """F-cal fixture (SURVEY.md §8c): populate BN running stats with train-mode passes using a
    cumulative moving average (momentum=None semantics), then return a new state dict."""
    out = OrderedDict((k, v.clone()) for k, v in sd.items())
    sums: Dict[str, torch.Tensor] = {}
    for x in batches:
        fresh = OrderedDict((k, v.clone()) for k, v in sd.items())
        # momentum 1.0 via zeroed stats: run with rm=0, rv=0 and read back momentum*stat
        stats: dict = {}
        with torch.no_grad():
            backbone_features(fresh, x, True, stats)
        for k, v in stats.items():
            base = sd[k]
            stat = (v - (1 - BN_MOMENTUM) * base) / BN_MOMENTUM  # undo the 0.1 blend
            sums[k] = sums.get(k, 0) + stat
    for k, v in sums.items():
        out[k] = (v / len(batches)).to(torch.float32)
    return out


# --------------------------------------------------------------------------------------------
# small kernels (numpy)
# --------------------------------------------------------------------------------------------

def argmax_decode(heat: np.ndarray) -> np.ndarray:
    """Per-keypoint peak of a (B,K,H,W) f32 heatmap -> (B,K,2) int64 as (y, x).

    `np.unravel_index(h.argmax(), h.shape)` (prediction.py:46): first flat index wins ties.  The
    reference decodes batch element 0 only (prediction.py:44); the oracle decodes every element.
    """
    heat = np.asarray(heat)
    B, K, H, W = heat.shape
    flat = heat.reshape(B, K, H * W).argmax(axis=2)
    return np.stack([flat // W, flat % W], axis=-1).astype(np.int64)


def soft_expectation(d: np.ndarray) -> List[int]:
    """Soft-argmax of one (H, W) map exactly as written in reference src/prediction.py:26-38: softmax over the map, flattened in
    the order of `d.T.ravel()` (column-major), against x = i % W and y = i // W with W = d.shape[1] -- the index arrays assume
    row-major order, so for H != W the "expectation" mixes rows and columns; the quirk is part of the reference's result and is
    kept.  Truncated to int like the reference."""
    d = np.asarray(d)
    width, height = d.T.shape
    flat = d.T.ravel()
    e = np.exp(flat - np.max(flat))
    p = e / e.sum()
    idx = np.arange(width * height)
    return [int(np.dot(p, idx % width)), int(np.dot(p, idx // width))]


def soft_expectation_raw(d: np.ndarray) -> np.ndarray:
    """`soft_expectation` before the int() truncation: float64 (E[x'], E[y']) with the reference's arithmetic (prediction.py:26-38:
    softmax in the map's dtype, dot with int64 index arrays in float64)."""
    d = np.asarray(d)
    width, height = d.T.shape
    flat = d.T.ravel()
    e = np.exp(flat - np.max(flat))
    p = e / e.sum()
    idx = np.arange(width * height)
    return np.array([np.dot(p, idx % width), np.dot(p, idx // width)], dtype=np.float64)


def clip_labels(label_xy: np.ndarray, height: int, width: int) -> np.ndarray:
    """Label handling of reference src/dataset.py:63-66: (K,2) = (x, y); x clipped to [0, W-1], y to [0, H-1]."""
    lab = np.array(label_xy, dtype=np.float64).reshape(-1, 2)
    lab[:, 0] = np.clip(lab[:, 0], 0, width - 1)
    lab[:, 1] = np.clip(lab[:, 1], 0, height - 1)
    return lab


def l1_normalize_dim1(g: np.ndarray) -> np.ndarray:
    """`normalize` of reference src/dataset.py:33-34 (F.normalize(x, p=1): L1 over dim 1, eps 1e-12) on a (K,H,W) float32 array,
    widened to float64 like dataset.py:44."""
    g = np.asarray(g, dtype=np.float32)
    denom = np.maximum(np.abs(g).sum(axis=1, keepdims=True, dtype=np.float32), np.float32(1e-12))
    return (g / denom).astype(np.float64)


def gauss_targets(uv: np.ndarray, height: int, width: int, sigma: float) -> np.ndarray:
    """`gauss_2d_batch` (dataset.py:36-44) for a batch: uv (B,K,2)=(x,y) -> (B,K,H,W) float64.

    The reference evaluates `exp(-((X-U)^2+(Y-V)^2)/(2.0*sigma**2))` in FLOAT32 (X, Y are
    `arange(0.)` float32 grids, U/V are `.float()`), then widens with `.double()` (dataset.py:41,44).
    Restated with numpy float32 scalars op by op so the rounding sequence is the same.
    """
    uv = np.asarray(uv)
    B, K, _ = uv.shape
    X = np.arange(width, dtype=np.float32)[None, None, None, :]
    Y = np.arange(height, dtype=np.float32)[None, None, :, None]
    U = uv[..., 0].astype(np.float32)[:, :, None, None]
    V = uv[..., 1].astype(np.float32)[:, :, None, None]
    dx = (X - U).astype(np.float32)
    dy = (Y - V).astype(np.float32)
    d2 = (dx * dx).astype(np.float32) + (dy * dy).astype(np.float32)
    denom = np.float32(2.0 * float(sigma) ** 2)
    # torch's float32 exp is used as the arbiter (tests compare against torch.exp); numpy's expf
    # may differ by an ulp, so go through torch here.
    arg = torch.from_numpy((-d2).astype(np.float32)) / float(denom)
    g = torch.exp(arg)
    return g.double().numpy()


def bce_loss(pred_f32: np.ndarray, target_f64: np.ndarray) -> float:
    """`nn.BCELoss()(pred.double(), gt)` (train.py:21,25): mean over all elements, logs clamped at -100."""
    p = np.asarray(pred_f32, dtype=np.float32).astype(np.float64)
    t = np.asarray(target_f64, dtype=np.float64)
    with np.errstate(divide="ignore"):
        lp = np.maximum(np.log(p), -100.0)
        l1p = np.maximum(np.log(1.0 - p), -100.0)
    return float(np.mean(-(t * lp + (1.0 - t) * l1p)))


def bce_grad_logits(pred_f32: np.ndarray, target_f64: np.ndarray) -> np.ndarray:
    """d loss / d logit that autograd produces for train.py:21-25 + model.py:21.

    BCELoss backward in f64: `g_p = (p - t) / max(p*(1-p), 1e-12) / N`; `.double()` backward casts
    to f32; sigmoid backward multiplies by `p*(1-p)` evaluated in f32.
    """
    p32 = np.asarray(pred_f32, dtype=np.float32)
    p = p32.astype(np.float64)
    t = np.asarray(target_f64, dtype=np.float64)
    n = p.size
    # ATen binary_cross_entropy_backward: grad * (input - target) / max((1 - input) * input, 1e-12)
    # with grad = 1/N for reduction='mean'.
    gp = (1.0 / n) * (p - t) / np.maximum((1.0 - p) * p, 1e-12)
    gp32 = gp.astype(np.float32)
    # ATen sigmoid_backward: grad * (1 - y) * y, evaluated left to right in f32.
    return ((gp32 * (np.float32(1.0) - p32)).astype(np.float32) * p32).astype(np.float32)


def bilinear_upsample_ac(src: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """Independent numpy restatement of align_corners=True bilinear (ATen upsample_bilinear2d):
    `src_idx = dst_idx * (in-1)/(out-1)`, weights computed in float32."""
    src = np.asarray(src, dtype=np.float32)
    h, w = src.shape[-2:]
    sy = np.float32((h - 1) / (out_h - 1)) if out_h > 1 else np.float32(0)
    sx = np.float32((w - 1) / (out_w - 1)) if out_w > 1 else np.float32(0)
    fy = (sy * np.arange(out_h, dtype=np.float32)).astype(np.float32)
    fx = (sx * np.arange(out_w, dtype=np.float32)).astype(np.float32)
    y0 = np.minimum(fy.astype(np.int64), h - 1)
    x0 = np.minimum(fx.astype(np.int64), w - 1)
    y1 = np.minimum(y0 + 1, h - 1)
    x1 = np.minimum(x0 + 1, w - 1)
    ly = (fy - y0.astype(np.float32)).astype(np.float32)
    lx = (fx - x0.astype(np.float32)).astype(np.float32)
    hy, hx = np.float32(1) - ly, np.float32(1) - lx
    a = src[..., y0[:, None], x0[None, :]]
    b = src[..., y0[:, None], x1[None, :]]
    c = src[..., y1[:, None], x0[None, :]]
    d = src[..., y1[:, None], x1[None, :]]
    return (hy[:, None] * (hx[None, :] * a + lx[None, :] * b) + ly[:, None] * (hx[None, :] * c + lx[None, :] * d)).astype(np.float32)


def conv_flops_per_image(height: int, width: int, num_keypoints: int) -> float:
    """Algorithmic conv FLOPs per image (2*M*N*K summed over the 37 convs, fc restricted to K rows).
    480x640, K=4 -> 211.91 GF (SURVEY.md §2.1)."""
    stem, blocks, fc = network_spec()

    def out_hw(h, w, c: ConvSpec):
        eff = c.dil * (c.k - 1) + 1
        return (h + 2 * c.pad - eff) // c.stride + 1, (w + 2 * c.pad - eff) // c.stride + 1

    total = 0.0
    h, w = out_hw(height, width, stem)
    total += 2.0 * h * w * stem.cout * stem.cin * stem.k * stem.k
    h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
    for b in blocks:
        h1, w1 = out_hw(h, w, b.conv1)
        total += 2.0 * h1 * w1 * b.conv1.cout * b.conv1.cin * 9
        total += 2.0 * h1 * w1 * b.conv2.cout * b.conv2.cin * 9
        if b.down is not None:
            total += 2.0 * h1 * w1 * b.down.cout * b.down.cin
        h, w = h1, w1
    total += 2.0 * h * w * num_keypoints * fc.cin
    return total
