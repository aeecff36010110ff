"""InferenceEngine: the eval-mode KeypointsGauss forward as a fixed sequence of libhulk_sm100 kernels.

Per (batch, H, W) "plan": pre-allocated NHWC activation buffers in HBM, packed weights, and (optionally)
one CUDA graph that replays the ~40 launches of stem -> maxpool -> 16 BasicBlocks -> head -> decode.

Data layout in HBM (per plan, B images of H x W):
  input   (B,3,H,W)        fp32 NCHW   -- the reference's tensor (ToTensor output, dataset.py:16)
  stem    (B,H/2,W/2,64)   act dtype   -- conv7x7 s2 + BN + ReLU
  act[4]  (B,H/4,W/4,64) .. (B,H/8,W/8,512) views of four rotating buffers sized for the largest
  logits  (B,K,H/8,W/8)    fp32        -- K live rows of the scoring conv
  heat    (B,K,H,W)        fp32 NCHW   -- what KeypointsGauss.forward returns
  yx      (B,K,2)          int32       -- argmax decode
  peaks   (B,K,N,2) int32, (B,K,N) fp32, (B,K) int32 + workspace -- peak decode, allocated on the first peaks() call
act dtype is bf16 in precision="bf16" (tcgen05 convs; stem on the fp32 CUDA-core kernel with bf16 output)
and fp32 in precision="fp32" (all convs on the CUDA-core FFMA kernel).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from ._lib import HK_CONV_FFMA, HK_CONV_TCGEN05, raw_write_generation, require_device

BN_EPS_DEFAULT = 1e-5


def conv_flops_per_image(model, height: int, width: int) -> float:
    """Algorithmic conv FLOPs of one image through `model` (2*M*N*K over the stem, the 16 BasicBlocks incl. their 1x1 downsamples, and
    the K live rows of the scoring conv): 211.91 GFLOP at 480x640, K=4 (SURVEY.md §2.1 / §8d) -- the figure bench.py's roofline uses."""
    net = model.resnet.resnet34_8s

    def conv(c, h, w):
        ho, wo = ops.conv_out_hw(h, w, c.kernel_size[0], c.stride[0], c.padding[0], c.dilation[0])
        return 2.0 * ho * wo * c.out_channels * c.in_channels * c.kernel_size[0] * c.kernel_size[1], ho, wo

    total, h, w = conv(net.conv1, height, width)
    h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
    for blk in net.blocks():
        f1, ho, wo = conv(blk.conv1, h, w)
        f2, _, _ = conv(blk.conv2, ho, wo)
        total += f1 + f2
        if blk.downsample is not None:
            total += conv(blk.downsample[0], h, w)[0]
        h, w = ho, wo
    return total + 2.0 * h * w * int(model.num_keypoints) * net.fc.in_channels


class _PackedConv:
    __slots__ = ("w", "scale", "bias", "stride", "pad", "dil", "algo")

    def __init__(self, w, scale, bias, stride, pad, dil, algo):
        self.w, self.scale, self.bias = w, scale, bias
        self.stride, self.pad, self.dil, self.algo = stride, pad, dil, algo


class _Plan:
    """Buffers (and the CUDA graph) for one input shape."""

    def __init__(self, engine: "InferenceEngine", B: int, H: int, W: int):
        dev = engine.device
        adt = engine.act_dtype
        K = engine.K
        self.B, self.H, self.W = B, H, W
        h2, w2 = ops.conv_out_hw(H, W, 7, 2, 3, 1)
        h4, w4 = (h2 + 2 - 3) // 2 + 1, (w2 + 2 - 3) // 2 + 1
        h8, w8 = ops.conv_out_hw(h4, w4, 3, 2, 1, 1)
        self.h2, self.w2, self.h4, self.w4, self.h8, self.w8 = h2, w2, h4, w4, h8, w8
        self.x = torch.empty((B, 3, H, W), device=dev, dtype=torch.float32)
        self.x_u8: Optional[torch.Tensor] = None  # (B,H,W,3) uint8 staging, allocated on first uint8 call
        self.input_is_u8 = False
        self._stem: Optional[torch.Tensor] = None   # (B,H/2,W/2,64): only the two-kernel stem path (fp32 mode, odd widths) needs it
        self._stem_spec = ((B, h2, w2, 64), dev, adt)
        max_elems = max(B * h4 * w4 * 64, B * h8 * w8 * 512)
        self.pool = [torch.empty(max_elems, device=dev, dtype=adt) for _ in range(4)]
        self.logits = torch.empty((B, K, h8, w8), device=dev, dtype=torch.float32)
        self.heat = torch.empty((B, K, H, W), device=dev, dtype=torch.float32)
        self.yx = torch.empty((B, K, 2), device=dev, dtype=torch.int32)
        self.maxval = torch.empty((B, K), device=dev, dtype=torch.float32)
        self.argmax_ws = torch.empty(max(1, ops.argmax_workspace_bytes(B, K, H, W)), device=dev, dtype=torch.uint8)
        self.peaks: Optional[Tuple[torch.Tensor, ...]] = None   # (yx, score, count, ws) of the peak decode, sized for (N, r)
        self._peaks_r = 0
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.graph_decode = None   # (decode mode, input_is_u8) the graph was captured with
        self.launches = 0

    @property
    def stem(self) -> torch.Tensor:
        if self._stem is None:
            shape, dev, adt = self._stem_spec
            self._stem = torch.empty(shape, device=dev, dtype=adt)
        return self._stem

    def peak_buffers(self, N: int, r: int) -> Tuple[torch.Tensor, ...]:
        K = self.heat.shape[1]
        if self.peaks is None or self.peaks[0].shape[2] != N or self._peaks_r != r:
            dev = self.heat.device
            self.peaks = (torch.empty((self.B, K, N, 2), device=dev, dtype=torch.int32),
                          torch.empty((self.B, K, N), device=dev, dtype=torch.float32),
                          torch.empty((self.B, K), device=dev, dtype=torch.int32),
                          torch.empty(max(8, ops.peak_workspace_bytes(self.B, K, self.H, self.W, N, r)), device=dev, dtype=torch.uint8))
            self._peaks_r = r
        return self.peaks

    def view(self, i: int, h: int, w: int, c: int) -> torch.Tensor:
        return self.pool[i][: self.B * h * w * c].view(self.B, h, w, c)


class InferenceEngine:
    def __init__(self, model, precision: str = "bf16", use_cuda_graph: bool = True):
        require_device()
        self.model = model
        self.precision = precision
        self.K = int(model.num_keypoints)
        self.act_dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self.use_cuda_graph = use_cuda_graph
        # stride-2 convs (layer2.0.conv1 and its 1x1 downsample) may be routed to the CUDA-core kernel
        self.stride2_algo = HK_CONV_TCGEN05
        # fused launches; False selects the unfused sequence (what the fp32 mode and unsupported shapes run), which tests compare against
        self.fuse_stem_pool = True    # False: stem_tc_kernel + maxpool3x3s2_kernel
        self.fuse_head = True         # False: the last conv writes the feature map, head_logits_kernel reads it
        self.fuse_downsample = True   # False: conv1 and the 1x1 downsample as two launches
        self._packed: Optional[Dict[str, _PackedConv]] = None
        self._packed_key = None
        self._plans: Dict[Tuple[int, int, int, int], _Plan] = {}
        self.device = None

    # ---- weights ----
    def _weights_key(self):
        """(data_ptr, _version) of every parameter and buffer, plus the model's `_weights_generation`: kernels that write through raw
        pointers (hk_adam_step, the TrainEngine's BatchNorm running-stat updates, CUDA-graph replays) never bump `_version`, so
        FusedAdam.step and every TrainEngine forward bump the generation counter instead (KeypointsGauss.mark_weights_changed)."""
        net = self.model.resnet.resnet34_8s
        gen = (getattr(self.model, "_weights_generation", 0), raw_write_generation())
        return gen + tuple((t.data_ptr(), t._version) for t in list(net.parameters()) + list(net.buffers()))

    def _pack_one(self, conv, bn, algo) -> _PackedConv:
        wdt = torch.bfloat16 if algo == HK_CONV_TCGEN05 else torch.float32
        bnp = None if bn is None else (bn.weight, bn.bias, bn.running_mean, bn.running_var)
        eps = BN_EPS_DEFAULT if bn is None else bn.eps
        w, s, b = ops.pack_conv_weights(conv.weight, bnp, eps, wdt)
        return _PackedConv(w, s, b, conv.stride[0], conv.padding[0], conv.dilation[0], algo)

    def _ensure_packed(self):
        key = self._weights_key()
        if self._packed is not None and key == self._packed_key:
            return
        net = self.model.resnet.resnet34_8s
        dev = net.conv1.weight.device
        if dev.type != "cuda":
            raise RuntimeError("KeypointsGauss parameters must live on the GPU for inference (call .cuda())")
        if self.device is not None and dev != self.device:
            self._plans.clear()
        self.device = dev
        tc = self.precision == "bf16"
        packed: Dict[str, _PackedConv] = {"stem": self._pack_one(net.conv1, net.bn1, HK_CONV_FFMA)}
        self._stem_w_tc = ops.stem_pack_weights(net.conv1.weight) if tc else None
        for i, blk in enumerate(net.blocks()):
            def algo_for(conv):
                if not tc:
                    return HK_CONV_FFMA
                return self.stride2_algo if conv.stride[0] != 1 else HK_CONV_TCGEN05
            packed[f"b{i}.c1"] = self._pack_one(blk.conv1, blk.bn1, algo_for(blk.conv1))
            packed[f"b{i}.c2"] = self._pack_one(blk.conv2, blk.bn2, algo_for(blk.conv2))
            if blk.downsample is not None:
                packed[f"b{i}.ds"] = self._pack_one(blk.downsample[0], blk.downsample[1], algo_for(blk.downsample[0]))
        self._fc_w = net.fc.weight.detach()[: self.K, :, 0, 0].contiguous().float()
        self._fc_b = net.fc.bias.detach()[: self.K].contiguous().float()
        self._packed = packed
        self._packed_key = key
        for p in self._plans.values():  # graphs captured pointers of the old packed tensors
            p.graph = None

    # ---- launch sequence ----
    def _conv(self, pc: _PackedConv, x, out, relu, residual=None, in_is_nchw=False):
        ops.conv_bn_act(x, pc.w, pc.scale, pc.bias, stride=pc.stride, pad=pc.pad, dil=pc.dil, relu=relu, residual=residual,
                        out=out, algo=pc.algo, in_is_nchw=in_is_nchw)

    def _enqueue(self, plan: _Plan, decode) -> int:
        """Enqueue the whole forward on the current stream.  Returns the number of kernel launches.
        decode: False (heatmaps only), True (argmax into plan.yx / plan.maxval) or ("peaks", N, threshold, r) (plan.peaks)."""
        net = self.model.resnet.resnet34_8s
        P = self._packed
        n = 0
        cur = 0
        x = plan.view(cur, plan.h4, plan.w4, 64)
        src = plan.x_u8 if plan.input_is_u8 else plan.x
        if self._stem_w_tc is not None and self.fuse_stem_pool and ops.stem_pool_supported(src):
            # conv7x7 + BN + ReLU + maxpool in one row-streaming kernel: the (B,H/2,W/2,64) stem map never touches HBM
            ops.stem_pool(src, self._stem_w_tc, P["stem"].scale, P["stem"].bias, out=x); n += 1
        else:
            if self._stem_w_tc is not None:
                ops.stem(src, self._stem_w_tc, P["stem"].scale, P["stem"].bias, out=plan.stem); n += 1
            else:
                self._conv(P["stem"], plan.x, plan.stem, relu=True, in_is_nchw=True); n += 1
            ops.maxpool3x3s2(plan.stem, out=x); n += 1
        h, w = plan.h4, plan.w4
        blocks = list(net.blocks())
        nblocks, head_done = len(blocks), False
        for i, blk in enumerate(blocks):
            c1, c2 = P[f"b{i}.c1"], P[f"b{i}.c2"]
            planes = c1.w.shape[0]
            ho, wo = ops.conv_out_hw(h, w, 3, c1.stride, c1.pad, c1.dil)
            free = [j for j in range(4) if j != cur]
            t = plan.view(free[0], ho, wo, planes)
            ds = P.get(f"b{i}.ds")
            if (ds is not None and self.fuse_downsample and c1.algo == HK_CONV_TCGEN05 and ds.algo == HK_CONV_TCGEN05
                    and ds.stride == c1.stride and ops.conv_ds_supported(x, c1.w, ds.w, c1.stride, c1.pad, c1.dil)):
                # block entry: conv1+bn1+relu and the 1x1 downsample+bn of the same input in one launch (centre-tap operand shared)
                sc = plan.view(free[1], ho, wo, planes)
                ops.conv_ds(x, c1.w, c1.scale, c1.bias, ds.w, ds.scale, ds.bias, stride=c1.stride, pad=c1.pad, dil=c1.dil,
                            relu=True, out=t, out_ds=sc); n += 1
            else:
                self._conv(c1, x, t, relu=True); n += 1
                if ds is not None:
                    sc = plan.view(free[1], ho, wo, planes)
                    self._conv(ds, x, sc, relu=False); n += 1
                else:
                    sc = x
            if (i == nblocks - 1 and self.fuse_head and c2.algo == HK_CONV_TCGEN05 and ops.conv_head_supported(t, c2.w, self._fc_w, c2.stride)
                    and (ho, wo) == (plan.h8, plan.w8)):
                # last conv of the network: its rows go straight into the K scoring dot products, the feature map is never written
                ops.conv_head(t, c2.w, c2.scale, c2.bias, self._fc_w, self._fc_b, plan.logits, stride=c2.stride, pad=c2.pad, dil=c2.dil,
                              relu=True, residual=sc); n += 1          # (+ a memset node for the logits)
                ops.head_upsample(plan.logits, plan.H, plan.W, heat=plan.heat, fast=True); n += 1
                head_done = True
                break
            y = plan.view(free[2], ho, wo, planes)
            self._conv(c2, t, y, relu=True, residual=sc); n += 1
            x, cur, h, w = y, free[2], ho, wo
        if not head_done:
            ops.head(x, self._fc_w, self._fc_b, plan.H, plan.W, heat=plan.heat, logits_ws=plan.logits); n += 2
        if isinstance(decode, tuple):
            _, N, thr, r = decode
            yx, score, count, ws = plan.peak_buffers(N, r)
            ops.peak_decode(plan.heat, N, thr, r, yx=yx, score=score, count=count, ws=ws); n += 2
        elif decode:
            ops.argmax_decode(plan.heat, yx=plan.yx, maxval=plan.maxval, ws=plan.argmax_ws, want_max=True); n += 2
        return n

    def plan_for(self, B: int, H: int, W: int, slot: int = 0) -> _Plan:
        """Buffers + CUDA graph for one input shape.  `slot` selects an independent copy (own input / output buffers and graph) so a
        caller can fill slot 1's input while slot 0 computes (double-buffered serving, see KeypointsGauss.staging_input)."""
        key = (B, H, W, slot)
        p = self._plans.get(key)
        if p is None:
            if H < 32 or W < 32:
                raise ValueError("input must be at least 32x32")
            p = _Plan(self, B, H, W)
            self._plans[key] = p
        return p

    def staging_input(self, B: int, H: int, W: int, slot: int = 0, uint8: bool = False) -> torch.Tensor:
        """The plan's own input buffer ((B,3,H,W) fp32, or (B,H,W,3) uint8): copy host images straight into it and pass it to
        forward() -- no device-to-device copy on the serving path."""
        self._ensure_packed()
        plan = self.plan_for(B, H, W, slot)
        if not uint8:
            return plan.x
        if plan.x_u8 is None:
            plan.x_u8 = torch.empty((B, H, W, 3), device=self.device, dtype=torch.uint8)
        return plan.x_u8

    def run_plan(self, plan: _Plan, decode) -> None:
        """Run the forward on `plan.x` (already filled) into plan.heat and the decode's buffers (decode as for _enqueue).  The graph is
        recaptured whenever the decode mode, its peak parameters or the input dtype change."""
        if not self.use_cuda_graph:
            plan.launches = self._enqueue(plan, decode)
            return
        if plan.graph is None or plan.graph_decode != (decode, plan.input_is_u8):
            # warm-up run outside capture (function attributes, lazy module load), then capture
            plan.launches = self._enqueue(plan, decode)
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue(plan, decode)
            plan.graph, plan.graph_decode = g, (decode, plan.input_is_u8)
        plan.graph.replay()

    def forward(self, x: torch.Tensor, decode=False, clone: bool = True, slot: int = 0):
        """(B,3,H,W) / (3,H,W) fp32, or (B,H,W,3) / (H,W,3) uint8 (cv2 layout), CUDA -> heat (B,K,H,W) fp32 [, yx (B,K,2)]
        [, (yx (B,K,N,2), score (B,K,N), count (B,K)) for decode=("peaks", N, threshold, r)].
        clone=False returns views of the plan's buffers (valid until the next call on the same slot); when `x` IS the plan's own
        input buffer (staging_input) no copy is made."""
        u8 = x.dtype == torch.uint8
        if x.dim() == 3:
            x = x.unsqueeze(0)
        if x.dim() != 4 or (x.shape[3] if u8 else x.shape[1]) != 3:
            raise ValueError(f"expected (B,3,H,W) float or (B,H,W,3) uint8 input, got {tuple(x.shape)} {x.dtype}")
        self._ensure_packed()
        if x.device != self.device:
            raise RuntimeError(f"input on {x.device} but model on {self.device}")
        if u8:
            B, H, W, _ = x.shape
        else:
            B, _, H, W = x.shape
        plan = self.plan_for(B, H, W, slot)
        with torch.no_grad():
            if u8 and self._stem_w_tc is not None:
                if plan.x_u8 is None:
                    plan.x_u8 = torch.empty((B, H, W, 3), device=self.device, dtype=torch.uint8)
                if x.data_ptr() != plan.x_u8.data_ptr():
                    plan.x_u8.copy_(x)
                plan.input_is_u8 = True
            elif not u8 and x.data_ptr() == plan.x.data_ptr():
                plan.input_is_u8 = False
            else:
                # fp32 path (and the fp32 correctness mode for uint8 input: ToTensor semantics, dataset.py:16)
                # (tensor / tensor keeps IEEE division on the GPU; tensor / python-scalar would multiply by 1/255)
                plan.x.copy_(x.permute(0, 3, 1, 2).float() / torch.full((), 255.0, device=x.device) if u8 else x)
                plan.input_is_u8 = False
            self.run_plan(plan, decode)
            heat = plan.heat.clone() if clone else plan.heat
            if isinstance(decode, tuple):
                peaks = plan.peaks[:3]
                return heat, (tuple(t.clone() for t in peaks) if clone else peaks)
            if decode:
                return heat, (plan.yx.clone() if clone else plan.yx)
            return heat
