"""KeypointsGauss -- host-side mirror of the reference's model API (reference src/model.py:10-22).

Same constructor, attributes, `forward` signature and 218-key `state_dict` (prefix
`resnet.resnet34_8s.`, fc kept at (1000,512,1,1)) as the reference, so `train.py` / `analysis.py`
can import it unchanged (see INTEGRATION.md).  Underneath:

  * eval() mode  -> the B200 engine (`engine.InferenceEngine`): hand-written sm_100a kernels through
                    the C ABI; BatchNorm folded; only the K live fc rows are computed.  CUDA only.
  * train() mode -> the B200 training engine (`train_engine.TrainEngine`: bf16 tcgen05 forward, dgrad, wgrad,
                    batch-stat BatchNorm, K-row head).  `train_backend = "autograd"` selects, explicitly, the
                    torch-autograd graph over the same parameters (the fp32 checker of the parity tests);
                    nothing falls back to it silently.

The network definition restates reference src/resnet.py:117-196 + src/resnet_dilated.py:10-22
(ResNet-34, output stride 8: layer3 dilation 2, layer4 dilation 4 on EVERY block incl. block 0).
"""
from __future__ import annotations

import math
import os
from typing import List, NamedTuple, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

NUM_CLASSES = 1000  # the reference never overrides Resnet34_8s(num_classes=1000) (src/model.py:17)
_STAGES = ((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2))  # planes, blocks, nominal stride
_OUTPUT_STRIDE = 8


class _ConvShape(NamedTuple):
    cin: int
    cout: int
    k: int
    stride: int
    pad: int
    dil: int


class _BasicBlock(nn.Module):
    """conv-bn-relu-conv-bn (+shortcut) relu; parameter holder + torch forward for train mode
    (reference src/resnet.py:40-69)."""

    def __init__(self, cin: int, planes: int, stride: int, dil: int, downsample: Optional[nn.Module]):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, planes, 3, stride, dil, dil, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, dil, dil, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample

    def forward(self, x):
        out = F.relu(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        shortcut = x if self.downsample is None else self.downsample(x)
        return F.relu(out + shortcut)


class _DilatedResNet34(nn.Module):
    """Backbone + 1x1 scoring conv `fc`; child names equal the reference's so state_dict keys match."""

    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 64, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        inplanes, cur_stride, cur_dil = 64, 4, 1
        for li, (planes, nblocks, stride) in enumerate(_STAGES, start=1):
            down = None
            if stride != 1 or inplanes != planes:
                if cur_stride == _OUTPUT_STRIDE:  # stride budget spent: dilate instead (resnet.py:170-175)
                    cur_dil *= stride
                    stride = 1
                else:
                    cur_stride *= stride
                down = nn.Sequential(nn.Conv2d(inplanes, planes, 1, stride, bias=False), nn.BatchNorm2d(planes))
            blocks: List[nn.Module] = [_BasicBlock(inplanes, planes, stride, cur_dil, down)]
            blocks += [_BasicBlock(planes, planes, 1, cur_dil, None) for _ in range(1, nblocks)]
            setattr(self, f"layer{li}", nn.Sequential(*blocks))
            inplanes = planes
        self.fc = nn.Conv2d(512, NUM_CLASSES, 1)

    def blocks(self):
        for li in range(1, 5):
            yield from getattr(self, f"layer{li}")

    def features(self, x):
        x = F.max_pool2d(F.relu(self.bn1(self.conv1(x))), 3, 2, 1)
        for blk in self.blocks():
            x = blk(x)
        return x


class _Resnet34_8s(nn.Module):
    def __init__(self):
        super().__init__()
        self.resnet34_8s = _DilatedResNet34()


def _reference_seeded_init(net: _DilatedResNet34) -> None:
    """Re-draw every parameter from the GLOBAL torch RNG in exactly the order the reference consumes it,
    so `torch.manual_seed(s); KeypointsGauss(...)` gives the same weights here and there.

    Order (reference src/resnet.py:137-161, src/resnet_dilated.py:16-22): torch's default inits at
    construction (stem; per stage downsample first, then each block's conv1, conv2; nn.Linear(512,1000)
    twice), then `normal_(0, sqrt(2/(k*k*cout)))` over modules() order, BN gamma=1/beta=0, then a fresh
    default-initialised 1x1 fc conv overwritten with N(0, 0.01) and zero bias.
    """
    def default_draw(cout, cin, k, bias):
        nn.init.kaiming_uniform_(torch.empty(cout, cin, k, k), a=math.sqrt(5))
        if bias:
            torch.empty(cout).uniform_(-1.0, 1.0)

    default_draw(64, 3, 7, False)
    for blk in net.blocks():
        if blk.downsample is not None:
            d = blk.downsample[0]
            default_draw(d.out_channels, d.in_channels, 1, False)
        default_draw(blk.conv1.out_channels, blk.conv1.in_channels, 3, False)
        default_draw(blk.conv2.out_channels, blk.conv2.in_channels, 3, False)
    default_draw(NUM_CLASSES, 512, 1, True)
    default_draw(NUM_CLASSES, 512, 1, True)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, nn.Conv2d) and m is not net.fc:
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.copy_(torch.empty(m.weight.shape).normal_(0, math.sqrt(2.0 / n)))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.fill_(1)
                m.bias.zero_()
                m.running_mean.zero_()
                m.running_var.fill_(1)
                m.num_batches_tracked.zero_()
        default_draw(NUM_CLASSES, 512, 1, True)
        net.fc.weight.copy_(torch.empty(net.fc.weight.shape).normal_(0, 0.01))
        net.fc.bias.zero_()


class KeypointsGauss(nn.Module):
    """Drop-in for reference `src/model.py:KeypointsGauss`.

    Extra keywords (additive): `precision` = "bf16" (default; tcgen05 path, heatmaps within 2e-2 of
    the fp32 reference) or "fp32" (CUDA-core correctness mode, within 1e-4 relative); the env var
    HULK_PRECISION overrides the default.  `pretrained` = path of a torchvision ResNet-34 checkpoint
    (or "auto" / env HULK_PRETRAINED): the reference's real initialisation, which needs a download there.
    """

    def __init__(self, num_keypoints, img_height=480, img_width=640, precision: Optional[str] = None,
                 pretrained: Optional[str] = None):
        super().__init__()
        self.num_keypoints = num_keypoints
        self.num_outputs = self.num_keypoints
        self.img_height = img_height
        self.img_width = img_width
        if not 1 <= num_keypoints <= NUM_CLASSES:
            raise ValueError(f"num_keypoints must be in [1, {NUM_CLASSES}]")
        self.precision = (precision or os.environ.get("HULK_PRECISION", "bf16")).lower()
        if self.precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        with torch.random.fork_rng(devices=[]):  # construction-time default inits must not disturb the stream
            self.resnet = _Resnet34_8s()
        _reference_seeded_init(self.resnet.resnet34_8s)
        self.sigmoid = nn.Sigmoid()
        self._engine = None
        self._weights_generation = 0
        # The reference ALWAYS starts from the ImageNet ResNet-34 (resnet_dilated.py:10-13, pretrained=True -> model_zoo download,
        # resnet.py:237-238).  There is no network here, so that initialisation is opt-in: `pretrained=<path>` / HULK_PRETRAINED=<path>
        # names a torchvision-format `resnet34-333f7ec4.pth`; "auto" looks in the torch hub cache.  Without it the backbone keeps the
        # seeded random init (what the reference produces when its download is stubbed out) -- INTEGRATION.md §1.
        src = pretrained if pretrained is not None else os.environ.get("HULK_PRETRAINED")
        if src:
            from .checkpoint import find_pretrained_resnet34, load_pretrained_backbone
            path = find_pretrained_resnet34() if src == "auto" else src
            if path is None:
                raise FileNotFoundError("pretrained='auto': resnet34-333f7ec4.pth is not in the torch hub cache")
            load_pretrained_backbone(self, path)

    # ---- engine plumbing ----
    def engine(self):
        from .engine import InferenceEngine

        if self._engine is None or self._engine.precision != self.precision:
            self._engine = InferenceEngine(self, self.precision)
        return self._engine

    def train_engine(self, batch: int, height: int, width: int):
        """The B200 training engine (forward in train() mode + loss + backward on libhulk_sm100 kernels) for one input shape."""
        from .train_engine import TrainEngine

        key = (batch, height, width, self.resnet.resnet34_8s.conv1.weight.device)
        engines = self.__dict__.setdefault("_train_engines", {})
        if key not in engines:
            engines[key] = TrainEngine(self, batch, height, width)
        return engines[key]

    def mark_weights_changed(self) -> None:
        """Tell the inference engine that parameters or BatchNorm buffers were written behind torch's back (raw-pointer kernels:
        FusedAdam.step, TrainEngine forwards, graph replays): the folded bf16 weights are rebuilt on the next eval-mode forward."""
        self._weights_generation = getattr(self, "_weights_generation", 0) + 1

    def set_precision(self, precision: str) -> "KeypointsGauss":
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.precision = precision
        return self

    def forward(self, x):
        if self.training:
            # B200 path: bf16 tensor-core forward now, tcgen05 dgrad/wgrad when autograd calls back (train_ops._EngineForward).
            # There is NO silent fallback: the torch-autograd graph over the same parameters runs only when asked for with
            # `model.train_backend = "autograd"` (the fp32 checker of the parity tests, and CPU tests of the host logic).
            backend = getattr(self, "train_backend", "hk")
            if backend == "autograd":
                return self._forward_autograd(x)
            if backend != "hk":
                raise ValueError("train_backend must be 'hk' or 'autograd'")
            why = self._train_engine_unsupported(x)
            if why is not None:
                raise RuntimeError(f"KeypointsGauss train-mode forward cannot run on the B200 training engine: {why}.  There is no "
                                   "silent fallback; set model.train_backend = 'autograd' to use the torch autograd graph explicitly, "
                                   "or call model.eval() for inference")
            from .train_ops import engine_forward
            return engine_forward(self, x)
        if not x.is_cuda:
            raise RuntimeError("KeypointsGauss inference runs on CUDA (B200) only: there is no CPU fallback; "
                               "move the model and the input with .cuda()")
        return self.engine().forward(x)

    def _train_engine_unsupported(self, x):
        """None when the training engine (bf16 tcgen05 forward/backward) takes this input, else the reason as text."""
        if not x.is_cuda:
            return "the input is a CPU tensor (the engine is CUDA-only)"
        if self.precision != "bf16":
            return "precision='fp32' has no training engine (fp32 training is not implemented on these kernels; see DESIGN.md §7)"
        if x.dim() != 4 or x.shape[1] != 3:
            return f"expected a (B,3,H,W) batch, got {tuple(x.shape)}"
        if x.shape[2] % 8 or x.shape[3] % 8 or min(x.shape[2:]) < 32:
            return f"H and W must be multiples of 8 and >= 32, got {tuple(x.shape[2:])}"
        if not torch.is_grad_enabled():
            return "autograd is disabled (train-mode forward under no_grad; use model.eval() for inference)"
        return self._bn_unsupported()

    def _bn_unsupported(self):
        """None when the training engine can express every BatchNorm of the backbone, else the reason as text.  The engine honours
        bn.training (eval()-mode BatchNorm inside a train()-mode model: running statistics, buffers untouched) and requires_grad; it
        has no path for cumulative averaging, batch statistics without running buffers, or a BatchNorm without gamma / beta."""
        for name, m in self.resnet.resnet34_8s.named_modules():
            if isinstance(m, nn.BatchNorm2d):
                if m.momentum is None:
                    return f"BatchNorm {name} has momentum=None (cumulative moving average), which the engine does not implement"
                if not m.track_running_stats or m.running_mean is None:
                    return f"BatchNorm {name} has track_running_stats=False, which the engine does not implement"
                if not m.affine:
                    return f"BatchNorm {name} has affine=False, which the engine does not implement"
        return None

    def forward_logits(self, x):
        """Train-mode graph up to the upsampled logits of the K live channels (additive API; the fused
        sigmoid+BCE of train_ops.sigmoid_bce_loss consumes this).  Batch-stat BN; the 996 dead fc rows receive
        zero gradient exactly as in the reference (SURVEY.md §2)."""
        net = self.resnet.resnet34_8s
        size = x.shape[2:]
        feat = net.features(x)
        k = self.num_keypoints
        logits = F.conv2d(feat, net.fc.weight[:k], net.fc.bias[:k])
        return F.interpolate(logits, size=size, mode="bilinear", align_corners=True)

    def _forward_autograd(self, x):
        return self.sigmoid(self.forward_logits(x))

    def keypoints(self, x, slot: int = 0):
        """Additive serving API: eval-mode forward + argmax decode -> (yx int32 (B,K,2) as (row, col), peak value fp32 (B,K)), without
        copying the heatmaps out.  The results are views of engine buffers, valid until the next call on the same `slot`."""
        if self.training:
            raise RuntimeError("keypoints() is an inference call; use model.eval() first")
        eng = self.engine()
        _, yx = eng.forward(x, decode=True, clone=False, slot=slot)
        B = yx.shape[0]
        H, W = (x.shape[1], x.shape[2]) if x.dtype == torch.uint8 else (x.shape[-2], x.shape[-1])
        return yx, eng.plan_for(B, H, W, slot).maxval

    def peaks(self, x, max_peaks: int = 16, threshold: float = 0.5, min_distance: int = 8, slot: int = 0):
        """Additive serving API: eval-mode forward + peak decode -> every instance of each keypoint channel, (yx int32 (B,K,N,2) as
        (row, col), score fp32 (B,K,N), count int32 (B,K)), N = max_peaks.  A peak is a pixel >= threshold that is greater than every
        earlier and at least every later pixel of its (2r+1)^2 window, r = min_distance (default: the training sigma, config.py's
        GAUSS_SIGMA = 8); the top N per map by score, unused slots (-1, -1) / -inf.  Like keypoints(): one CUDA graph, no heatmap
        copy, and the results are views of engine buffers, valid until the next call on the same `slot`."""
        if self.training:
            raise RuntimeError("peaks() is an inference call; use model.eval() first")
        from .ops import check_peak_args

        N, thr, r = check_peak_args(max_peaks, threshold, min_distance)
        _, out = self.engine().forward(x, decode=("peaks", N, thr, r), clone=False, slot=slot)
        return out

    def staging_input(self, batch: int, height: int, width: int, slot: int = 0, uint8: bool = False):
        """Device input buffer of serving slot `slot`: `buf.copy_(pinned_host_images, non_blocking=True)` then `keypoints(buf, slot)`;
        two slots give H2D / compute double buffering with no device-to-device copy."""
        if self.training:
            raise RuntimeError("staging_input() is an inference call; use model.eval() first")
        return self.engine().staging_input(batch, height, width, slot, uint8)

    def heatmaps_and_keypoints(self, x):
        """Additive API: eval-mode forward + argmax decode of every batch element -> (heat, yx int32 (B,K,2))."""
        if self.training:
            raise RuntimeError("heatmaps_and_keypoints() is an inference call; use model.eval() first")
        return self.engine().forward(x, decode=True)
