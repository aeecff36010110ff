"""TrainEngine: one KeypointsGauss training step (forward in train() mode + loss + backward) as a fixed sequence of
libhulk_sm100 kernels -- the B200-native replacement of what torch autograd executes for reference train.py:33-35
(zero_grad, forward(sample, model), loss.backward()).  SURVEY.md §8 rows a4/a9/a11/a12 and f1.

Numerics: bf16 NHWC activations and bf16 conv operands (tcgen05, fp32 accumulation in TMEM), fp32 BatchNorm statistics,
fp32 parameter gradients, fp64 loss.  BatchNorm uses the statistics of the local batch (per replica, like the reference,
which has no SyncBN) and updates running_mean / running_var / num_batches_tracked exactly as nn.BatchNorm2d does.

Per conv the forward is   y = conv(x) [raw, bf16]  ->  batch stats  ->  out = relu(gamma*xhat + beta [+ shortcut])
and the backward          d' = dout*[out>0]  ->  (dgamma, dbeta, dy)  ->  dW = wgrad(x, dy),  dx = conv(dy, W flipped).
Batch statistics and their backward sums go through exact fixed-point accumulators, the ReLU mask through 1 bit per element, and the
max-pool forward records the winning taps its backward routes through.  Weight gradients (and the per-step weight repack) run on a
second stream, the downsample branches on a third, all inside the same graph.
All 110 parameter gradients land in ONE flat fp32 buffer in the layout FusedAdam adopts (one all-reduce, one update kernel);
the 996 dead rows of the 1000-row scoring conv keep a zero gradient, as in the reference.

Data layout in HBM (per engine, batch B of H x W): input (B,3,H,W) f32; per conv a raw output and an activation,
(B,h,w,C) bf16 NHWC; (B,K,H,W) f32 upsampled logits and their gradient; scratch gradients sized by stage.
The whole step is captured in one CUDA graph (287 launches when every BatchNorm and parameter trains) and replayed.

Fine-tuning: BatchNorms in eval() mode (running statistics, buffers untouched) and parameters with requires_grad=False follow torch's
semantics; `backward_plan` decides from those flags what the backward computes and where it stops (DESIGN §3.5).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch

from . import ops
from ._lib import check, lib, ptr, require_device, stream_ptr


# ---------------------------------------------------------------------------------------------------------------- backward plan
class ConvPlan(NamedTuple):
    """What the step does for one conv + BatchNorm, from the torch flags (bn.training, p.requires_grad)."""
    frozen: bool    # BatchNorm in eval() mode: normalises with the running statistics, writes none of its buffers
    dgamma: bool    # gradients wanted for the BatchNorm's gamma / beta
    dbeta: bool
    wgrad: bool     # conv weight gradient
    dgrad: bool     # gradient of the conv's input (something below still needs a gradient)
    dy: bool        # gradient of the raw conv output (for wgrad and/or dgrad)
    bwd: bool       # the BatchNorm backward runs at all


_NO_BWD = dict(dgamma=False, dbeta=False, wgrad=False, dgrad=False, dy=False, bwd=False)


class BackwardPlan(NamedTuple):
    convs: Dict[str, ConvPlan]      # by TrainEngine conv name: "stem", "b{i}.c1", "b{i}.c2", "b{i}.ds"
    fc_weight: bool
    fc_bias: bool
    dfeat: bool                     # the head backward hands a gradient to the backbone
    grad_in: Tuple[bool, ...]       # per block: the gradient of the block's input is needed
    lo: int                         # first block the backward visits (len(blocks): none)
    stem: bool                      # max-pool + stem BatchNorm (+ stem weight gradient) backward run

    @property
    def frozen_any(self) -> bool:
        return any(p.frozen for p in self.convs.values())

    @property
    def train_bn_any(self) -> bool:
        return not all(p.frozen for p in self.convs.values())


def _data_ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _trains(m: torch.nn.Module) -> bool:
    return any(p.requires_grad for p in m.parameters())


def backward_plan(net) -> BackwardPlan:
    """The work of one training step under the current torch flags of the backbone `net` (model.resnet.resnet34_8s): which BatchNorms
    are frozen, which convs need dy / a weight gradient / a data gradient, which BatchNorms need dgamma / dbeta.  The backward runs
    from the head down to the earliest point that still needs a gradient and nothing below it.  Pure (no device work)."""
    blocks = list(net.blocks())
    nb = len(blocks)
    convs: Dict[str, ConvPlan] = {}

    def conv_plan(conv, bn, dgrad: bool, extra_bwd: bool = False) -> ConvPlan:
        dg, db, wg = bn.weight is not None and bn.weight.requires_grad, bn.bias is not None and bn.bias.requires_grad, conv.weight.requires_grad
        dy = wg or dgrad
        return ConvPlan(frozen=not bn.training, dgamma=dg, dbeta=db, wgrad=wg, dgrad=dgrad, dy=dy, bwd=dy or dg or db or extra_bwd)

    below = _trains(net.conv1) or _trains(net.bn1)
    grad_in = []
    for blk in blocks:
        grad_in.append(below)
        below = below or _trains(blk)
    dfeat = below
    lo = next((bi for bi in range(nb) if grad_in[bi] or _trains(blocks[bi])), nb)
    for bi, blk in enumerate(blocks):
        ds = blk.downsample
        if bi < lo:
            for name, bn in ((f"b{bi}.c1", blk.bn1), (f"b{bi}.c2", blk.bn2)) + (((f"b{bi}.ds", ds[1]),) if ds is not None else ()):
                convs[name] = ConvPlan(frozen=not bn.training, **_NO_BWD)
            continue
        p1 = conv_plan(blk.conv1, blk.bn1, dgrad=grad_in[bi])
        pd = conv_plan(ds[0], ds[1], dgrad=grad_in[bi]) if ds is not None else None
        # conv2's BatchNorm backward also forms d' = dout*[out>0], the gradient of the shortcut branch
        p2 = conv_plan(blk.conv2, blk.bn2, dgrad=p1.bwd, extra_bwd=pd.bwd if pd is not None else grad_in[bi])
        convs[f"b{bi}.c1"], convs[f"b{bi}.c2"] = p1, p2
        if pd is not None:
            convs[f"b{bi}.ds"] = pd
    st = conv_plan(net.conv1, net.bn1, dgrad=False)
    convs["stem"] = st
    return BackwardPlan(convs=convs, fc_weight=net.fc.weight.requires_grad, fc_bias=net.fc.bias is not None and net.fc.bias.requires_grad,
                        dfeat=dfeat, grad_in=tuple(grad_in), lo=lo, stem=st.bwd)


def step_launches(net, plan: BackwardPlan) -> int:
    """Kernel launches of one TrainEngine.forward_backward step under `plan`: what `TrainEngine.launches` reports."""
    blocks = list(net.blocks())

    def fwd(name, conv) -> int:
        p = plan.convs[name]
        if p.frozen:
            return 2 if (p.dgamma or p.dbeta) else 1
        return 2 if (conv.kernel_size[0] == 3 and conv.out_channels >= 256) else 3

    def bn_bwd(name) -> int:
        return 1 if plan.convs[name].frozen else 2

    def dgrad(conv) -> int:
        return 2 if conv.stride[0] == 2 else 1

    n = 2 + (1 if plan.train_bn_any else 0) + (1 if plan.frozen_any else 0)                     # weight packs, accumulator memset, BN fold
    st = plan.convs["stem"]
    n += (2 if (st.dgamma or st.dbeta) else 1) if st.frozen else 3                                # stem conv + its BatchNorm
    n += 1                                                                                        # max-pool
    for bi, blk in enumerate(blocks):
        n += fwd(f"b{bi}.c1", blk.conv1) + fwd(f"b{bi}.c2", blk.conv2)
        if blk.downsample is not None:
            n += fwd(f"b{bi}.ds", blk.downsample[0])
    n += 2 + (1 if plan.train_bn_any else 0)                                                      # head logits, num_batches_tracked
    n += 2                                                                                        # fused loss
    # backward
    users = [name for name, p in plan.convs.items() if p.bwd and (not p.frozen or p.dgamma or p.dbeta)]
    n += 1 if users else 0                                                                        # backward accumulator memset
    if plan.dfeat or plan.fc_weight or plan.fc_bias:
        n += 5 - (not plan.dfeat) - 2 * (not plan.fc_weight) - 2 * (not plan.fc_bias)
    for bi in range(len(blocks) - 1, plan.lo - 1, -1):
        blk = blocks[bi]
        p1, p2 = plan.convs[f"b{bi}.c1"], plan.convs[f"b{bi}.c2"]
        if p2.bwd:
            n += bn_bwd(f"b{bi}.c2")
        if blk.downsample is not None:
            pd = plan.convs[f"b{bi}.ds"]
            if pd.bwd:
                n += bn_bwd(f"b{bi}.ds") + (2 if pd.wgrad else 0) + (dgrad(blk.downsample[0]) if pd.dgrad else 0)
        n += (2 if p2.wgrad else 0) + (dgrad(blk.conv2) if p2.dgrad else 0)
        if p1.bwd:
            n += bn_bwd(f"b{bi}.c1") + (2 if p1.wgrad else 0) + (dgrad(blk.conv1) if p1.dgrad else 0)
    if plan.stem:
        n += 1 + bn_bwd("stem") + (2 if st.wgrad else 0)                                          # max-pool, BatchNorm, weight gradient
    return n


class _ConvT:
    """One conv + its BatchNorm in training: parameters, packed operands, saved tensors."""

    def __init__(self, name, conv, bn, B, H, W, dev):
        self.name, self.conv, self.bn = name, conv, bn
        self.cout, self.cin, self.k, _ = conv.weight.shape
        self.stride, self.pad, self.dil = conv.stride[0], conv.padding[0], conv.dilation[0]
        self.H, self.W = H, W
        self.Ho, self.Wo = ops.conv_out_hw(H, W, self.k, self.stride, self.pad, self.dil)
        bf = torch.bfloat16
        self.w_fwd = torch.empty((self.cout, self.k, self.k, self.cin), device=dev, dtype=bf)
        self.w_dgrad = torch.empty((self.cin, self.k, self.k, self.cout), device=dev, dtype=bf)
        self.one_out = torch.empty(self.cout, device=dev)   # scale = 1 / bias = 0 of the raw forward conv (filled by the pack kernel)
        self.zero_out = torch.empty(self.cout, device=dev)
        self.one_in = torch.ones(self.cin, device=dev)      # same for the data-gradient conv (its "Cout" is cin)
        self.zero_in = torch.zeros(self.cin, device=dev)
        self.y = torch.empty((B, self.Ho, self.Wo, self.cout), device=dev, dtype=bf)   # raw conv output (saved for BN backward)
        self.mean, self.invstd, self.scale, self.shift = (torch.empty(self.cout, device=dev) for _ in range(4))
        self.relu_bits = torch.empty(self.y.numel() // 8, device=dev, dtype=torch.uint8)  # ReLU mask of the BN output, 1 bit / element
        self.dy: Optional[torch.Tensor] = None   # gradient of y, allocated by the first backward that needs it


class TrainEngine:
    def __init__(self, model, B: int, H: int, W: int, sigma: float = 8.0):
        require_device()
        if H % 8 or W % 8 or H < 32 or W < 32:
            raise ValueError("TrainEngine needs H and W to be multiples of 8 (>= 32)")
        net = model.resnet.resnet34_8s
        dev = net.conv1.weight.device
        if dev.type != "cuda":
            raise RuntimeError("TrainEngine needs the model on a CUDA device (no CPU path)")
        self.model, self.net, self.device = model, net, dev
        self.B, self.H, self.W, self.K, self.sigma = B, H, W, int(model.num_keypoints), float(sigma)
        bf = torch.bfloat16
        # first block of layer3: everything from here to the end of the parameter list (layer3, layer4, fc) is the "late" part
        self.split_block = 7
        self.all_params: List[torch.nn.Parameter] = list(model.parameters())   # the engine is bound to the model's modules, like its convs
        self.params: List[torch.nn.Parameter] = []
        self._build_grad_buffer([p for p in self.all_params if p.requires_grad])
        # ---- buffers ----
        self.x = torch.empty((B, 3, H, W), device=dev, dtype=torch.float32)
        self.uv = torch.zeros((B, self.K, 2), device=dev, dtype=torch.float32)
        self.target: Optional[torch.Tensor] = None      # (B,K,H,W) fp64/fp32 when the caller supplies targets instead of labels
        h2, w2 = ops.conv_out_hw(H, W, 7, 2, 3, 1)
        h4, w4 = (h2 + 2 - 3) // 2 + 1, (w2 + 2 - 3) // 2 + 1
        self.h2, self.w2, self.h4, self.w4 = h2, w2, h4, w4
        self.stem_w = torch.empty(int(lib().hk_stem_packed_weight_bytes()) // 2, device=dev, dtype=bf)
        self.stem = _ConvT("stem", net.conv1, net.bn1, B, H, W, dev)
        self.a0 = torch.empty((B, h2, w2, 64), device=dev, dtype=bf)
        self.p0 = torch.empty((B, h4, w4, 64), device=dev, dtype=bf)
        # the max-pool forward records the winning taps: one pass over the stem map instead of a forward pass plus an arg-max pass
        self.pool_idx = torch.empty(B * h4 * w4 * 64, device=dev, dtype=torch.uint8)
        self.blocks = []
        h, w = h4, w4
        for i, blk in enumerate(net.blocks()):
            c1 = _ConvT(f"b{i}.c1", blk.conv1, blk.bn1, B, h, w, dev)
            c2 = _ConvT(f"b{i}.c2", blk.conv2, blk.bn2, B, c1.Ho, c1.Wo, dev)
            ds = _ConvT(f"b{i}.ds", blk.downsample[0], blk.downsample[1], B, h, w, dev) if blk.downsample is not None else None
            a1 = torch.empty_like(c1.y)
            sc = torch.empty_like(c2.y) if ds is not None else None
            out = torch.empty_like(c2.y)
            self.blocks.append((c1, c2, ds, a1, sc, out))
            h, w = c1.Ho, c1.Wo
        self.h8, self.w8 = h, w
        self.convs: List[_ConvT] = [self.stem] + [c for b in self.blocks for c in (b[0], b[1], b[2]) if c is not None]
        # BatchNorm reductions through exact fixed-point accumulators (hk_bn_stats_acc / hk_bn_bwd_acc): no finalize launches, 72 fewer
        # launches per step.  One flat buffer per direction, sliced per conv in self.convs order (stem, then the blocks in order), so the
        # early part of the two-phase backward (stem + blocks < split_block) is a prefix.
        offs_acc, tot = [], 0
        for c in self.convs:
            offs_acc.append(tot)
            tot += ops.bn_acc_bytes(c.cout)
        self.acc_fwd = torch.zeros(tot, device=dev, dtype=torch.uint8)
        self.acc_bwd = torch.zeros(tot, device=dev, dtype=torch.uint8)
        for c, o in zip(self.convs, offs_acc):
            c.acc_f = self.acc_fwd[o:o + ops.bn_acc_bytes(c.cout)]
            c.acc_b = self.acc_bwd[o:o + ops.bn_acc_bytes(c.cout)]
        K = self.K
        self.logits_lr = torch.empty((B, K, h, w), device=dev, dtype=torch.float32)
        self.logits_up = torch.empty((B, K, H, W), device=dev, dtype=torch.float32)
        self.g_up = torch.empty((B, K, H, W), device=dev, dtype=torch.float32)
        self.dlogits_lr = torch.empty((B, K, h, w), device=dev, dtype=torch.float32)
        self.loss = torch.zeros((), device=dev, dtype=torch.float64)
        n = B * K * H * W
        self.bce_ws = torch.empty(int(lib().hk_bce_workspace_bytes(n)), device=dev, dtype=torch.uint8)
        wg = max(ops.conv_wgrad_workspace_bytes(B, c.H, c.W, c.cin, c.cout, c.k, c.stride, c.pad, c.dil) for c in self.convs[1:])
        self.wgrad_ws = torch.empty(max(wg, int(lib().hk_stem_wgrad_workspace_bytes())), device=dev, dtype=torch.uint8)
        self.head_ws = torch.empty(int(lib().hk_head_bwd_workspace_bytes(B, K, 512, h, w)), device=dev, dtype=torch.uint8)
        self.acc_early_bytes = offs_acc[self.convs.index(self.blocks[self.split_block][0])]   # accumulators of the stem + early blocks
        self._bwd_state = None
        self._scratch: Dict[Tuple, torch.Tensor] = {}
        self._pack_key = None
        self._pack_items: Optional[torch.Tensor] = None
        self._fold_key = None
        self._fold_items: Optional[torch.Tensor] = None
        self._flags = None
        self.sync_flags()          # flat gradient buffer, backward plan, BatchNorm counters
        self.use_cuda_graph = os.environ.get("HK_TRAIN_NO_GRAPH") is None   # eager launches for ncu launch lists
        self._graphs: Dict[str, Tuple[torch.cuda.CUDAGraph, Tuple, int]] = {}   # by entry point: (graph, _key() at capture, launches)
        # Weight gradients are leaves of the backward chain (bn_bwd -> dgrad -> bn_bwd ...): they run on a second stream inside the same
        # graph, concurrently with the data-gradient chain (each conv then keeps its own dy buffer).  Measured on one box: per-GPU batch 4
        # 5.74 -> 5.37 ms per step, batch 32 25.40 -> 24.53 ms.  All of them share wgrad_ws: the stream runs them one after another.
        self.wgrad_stream = torch.cuda.Stream(device=dev)
        self._wgrad_pending = False
        # The 1x1 downsample branch of the three stride/channel-changing blocks (conv + BN forward; BN backward + dgrad) is independent
        # of the block's main branch until the residual add: it runs on a third stream.
        self.aux_stream = torch.cuda.Stream(device=dev)
        self.launches = 0                                   # of the last forward_backward step
        self._split_launches: Dict[str, int] = {}           # of the last run of each split entry point

    # ------------------------------------------------------------------ torch flags
    def sync_flags(self) -> None:
        """Read bn.training and p.requires_grad (torch's fine-tuning switches) and, when they changed since the last step, rebuild what
        depends on them: the flat gradient buffer (trainable parameters only, the layout FusedAdam adopts), the backward plan and the list of
        BatchNorms whose num_batches_tracked advances.  The flags are part of every graph key, so no stale graph is replayed."""
        params = self.all_params
        flags = (tuple(c.bn.training for c in self.convs), tuple(p.requires_grad for p in params))
        if flags == self._flags:
            return
        why = self.model._bn_unsupported()
        if why is not None:
            raise RuntimeError(f"TrainEngine cannot run this model: {why}")
        trainable = [p for p in params if p.requires_grad]
        if [id(p) for p in trainable] != [id(p) for p in self.params]:
            self._build_grad_buffer(trainable)
        self.plan = backward_plan(self.net)
        self._bn_counters = [c.bn.num_batches_tracked for c in self.convs if c.bn.training]
        self._flags = flags

    def _build_grad_buffer(self, trainable: List[torch.nn.Parameter]) -> None:
        """Flat gradient buffer of the trainable parameters in model order, the layout FusedAdam adopts (each tensor 16-byte aligned)."""
        self.params = trainable
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4
        self.flat_grad = torch.zeros(total, device=self.device, dtype=torch.float32)
        self.grad_of: Dict[int, torch.Tensor] = {id(p): self.flat_grad[o:o + p.numel()].view_as(p) for p, o in zip(self.params, offs)}
        # the "late" part of the two-phase step (layer3, layer4, fc) starts at the first trainable parameter at or after layer3.0
        late = {id(p) for blk in list(self.net.blocks())[self.split_block:] for p in blk.parameters()}
        late |= {id(p) for p in self.net.fc.parameters()}
        self.late_offset = next((o for p, o in zip(self.params, offs) if id(p) in late), total)

    # ------------------------------------------------------------------ helpers
    def _buf(self, role: str, shape) -> torch.Tensor:
        key = (role, tuple(shape))
        t = self._scratch.get(key)
        if t is None:
            t = torch.empty(tuple(shape), device=self.device, dtype=torch.bfloat16)
            self._scratch[key] = t
        return t

    def _g(self, p) -> torch.Tensor:
        return self.grad_of[id(p)]

    def _pack_all(self) -> int:
        """Every block conv weight -> bf16 forward + data-gradient layouts in one launch (hk_pack_conv_weights_many_tiled: shared-memory
        tiles of 64 output x 32 input channels, contiguous reads and 64-byte writes; it needs cout % 64 == 0 and cin % 32 == 0, which
        every block conv of the backbone meets)."""
        import numpy as np
        key = tuple(c.conv.weight.data_ptr() for c in self.convs)
        if self._pack_items is None or key != self._pack_key:
            dt = np.dtype([("w", "<u8"), ("f", "<u8"), ("d", "<u8"), ("cout", "<i4"), ("cin", "<i4"), ("khw", "<i4"), ("r", "<i4")])
            arr = np.zeros(len(self.convs) - 1, dtype=dt)
            for i, c in enumerate(self.convs[1:]):
                arr[i] = (c.conv.weight.data_ptr(), c.w_fwd.data_ptr(), c.w_dgrad.data_ptr(), c.cout, c.cin, c.k * c.k, 0)
            self._pack_items = torch.from_numpy(arr.view(np.uint8).copy()).to(self.device)
            self._pack_key = key
            self._pack_max = max(c.cout * c.cin * c.k * c.k for c in self.convs[1:])
            self._pack_khw = max(c.k * c.k for c in self.convs[1:])
            for c in self.convs:  # scale = 1 / bias = 0 of the raw convs: constant
                c.one_out.fill_(1.0)
                c.zero_out.zero_()
        check(lib().hk_pack_conv_weights_many_tiled(ptr(self._pack_items), len(self.convs) - 1, self._pack_khw, C.c_longlong(self._pack_max),
                                                    stream_ptr()), "hk_pack_conv_weights_many_tiled")
        return 1

    def _fold_frozen(self) -> int:
        """scale / shift / invstd of every frozen BatchNorm from its running statistics and current gamma / beta, in one launch.  Inside
        the step (graph): the optimiser may change gamma / beta through raw pointers between steps."""
        frozen = [c for c in self.convs if self.plan.convs[c.name].frozen]
        if not frozen:
            return 0
        key = tuple((c.name,) + tuple(_data_ptr(t) for t in (c.bn.weight, c.bn.bias, c.bn.running_mean, c.bn.running_var)) for c in frozen)
        if self._fold_items is None or key != self._fold_key:
            items = [(c.bn.weight.data if c.bn.weight is not None else None, c.bn.bias.data if c.bn.bias is not None else None,
                      c.bn.running_mean, c.bn.running_var, c.bn.eps, c.scale, c.shift, c.invstd) for c in frozen]
            self._fold_items = ops.bn_fold_items(items).to(self.device)
            self._fold_key = key
            self._fold_n, self._fold_c = len(frozen), max(c.cout for c in frozen)
        ops.bn_fold(self._fold_items, self._fold_n, self._fold_c)
        return 1

    def _conv(self, c: _ConvT, x, scale, shift, out, relu: bool = False, residual=None) -> None:
        """The forward conv of c with a per-channel scale / shift (+ shortcut) (+ ReLU) epilogue.  The stem has a kernel of its own on
        its own packed weights (x: the fp32 NCHW input); the others run on the inference conv kernels."""
        if c is self.stem:
            ops.stem_conv(x, self.stem_w, scale, shift, relu=relu, out=out)
        else:
            ops.conv_bn_act(x, c.w_fwd, scale, shift, stride=c.stride, pad=c.pad, dil=c.dil, relu=relu, residual=residual, out=out)

    def _conv_bn_frozen(self, c: _ConvT, x, out, relu: bool, residual=None) -> int:
        """BatchNorm in eval() mode: normalise with the running statistics (folded scale / shift), buffers untouched."""
        p = self.plan.convs[c.name]
        if not (p.dgamma or p.dbeta):
            # one launch: the conv epilogue applies scale / shift (+ shortcut) (+ ReLU); the backward masks with the stored output
            self._conv(c, x, c.scale, c.shift, out, relu=relu, residual=residual)
            c.frozen_mask = out if relu else None
            return 1
        # gamma / beta trained: their gradients need the raw conv output y
        self._conv(c, x, c.one_out, c.zero_out, c.y)
        bits = c.relu_bits if relu else None
        ops.bn_apply(c.y, c.scale, c.shift, relu=relu, residual=residual, out=out, relu_bits=bits)
        c.frozen_mask = bits
        return 2

    def _conv_bn(self, c: _ConvT, x, out, relu: bool, residual=None) -> int:
        """raw conv -> batch statistics (+ running stats) -> fused normalise (+ shortcut) (+ ReLU, its mask as 1 bit per element)."""
        if self.plan.convs[c.name].frozen:
            return self._conv_bn_frozen(c, x, out, relu, residual)
        bn = c.bn
        if c.k == 3 and c.cout >= 256:
            # the conv epilogue gathers sum y / sum y^2 of the tile it stores: no statistics pass over the activation.  Only where the
            # epilogue hides under a long mainloop (3x3 convs of layers 3-4: 36 / 72 K blocks per tile); the 64/128-channel layers and
            # the 1x1 downsample convs are epilogue-bound and lose more than the stand-alone reduction costs (measured per launch)
            ops.conv_bn_stats(x, c.w_fwd, c.one_out, c.zero_out, c.acc_f, stride=c.stride, pad=c.pad, dil=c.dil, out=c.y)
            n = 2
        else:
            self._conv(c, x, c.one_out, c.zero_out, c.y)
            ops.bn_stats_acc(c.y, c.acc_f)
            n = 3
        ops.bn_apply_acc(c.y, c.acc_f, bn.weight.data, bn.bias.data, bn.running_mean, bn.running_var, bn.momentum, bn.eps, c.mean, c.invstd,
                         relu=relu, residual=residual, out=out, relu_bits=c.relu_bits if relu else None)
        return n

    def _fork_aux(self) -> torch.cuda.Stream:
        """The aux stream, made to wait for everything enqueued on the current stream so far."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.aux_stream.wait_event(ev)
        return self.aux_stream

    def _join_aux(self) -> None:
        ev = torch.cuda.Event()
        ev.record(self.aux_stream)
        torch.cuda.current_stream().wait_event(ev)

    def _bn_bwd(self, c: _ConvT, dout, relu: bool, dy, dmasked=None) -> int:
        """relu: the BN output went through a ReLU; its mask is c.relu_bits (written by the forward apply pass).  dy None: the raw
        conv output needs no gradient (only dgamma / dbeta / d' are wanted)."""
        bn = c.bn
        p = self.plan.convs[c.name]
        dg = self._g(bn.weight) if p.dgamma else None
        db = self._g(bn.bias) if p.dbeta else None
        if p.frozen:
            sums = dg is not None or db is not None
            ops.bn_frozen_bwd(dout, c.frozen_mask, c.scale, dy, dmasked=dmasked, y=c.y if sums else None, mean=bn.running_mean,
                              invstd=c.invstd, acc=c.acc_b if sums else None, dgamma=dg, dbeta=db)
            return 1
        if dy is None:   # the batch-statistics backward kernel always writes dy
            dy = self._buf("dy_unused", c.y.shape)
        ops.bn_bwd_acc(dout, c.relu_bits if relu else None, c.y, c.mean, c.invstd, bn.weight.data, c.acc_b, dg, db, dy, dmasked=dmasked)
        return 2

    def _dy_buf(self, c: _ConvT) -> torch.Tensor:
        """dL/d(raw conv output) of conv c: one buffer per conv, because its weight gradient (on the wgrad stream) may still be reading
        it while the data-gradient chain has moved on."""
        if c.dy is None:
            c.dy = torch.empty_like(c.y)
        return c.dy

    def _on_wgrad_stream(self, fn) -> None:
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())      # dy (just written on the main stream) is complete
        self.wgrad_stream.wait_event(ready)
        with torch.cuda.stream(self.wgrad_stream):
            fn()
        self._wgrad_pending = True

    def _join_wgrad_stream(self) -> None:
        if self._wgrad_pending:
            done = torch.cuda.Event()
            done.record(self.wgrad_stream)
            torch.cuda.current_stream().wait_event(done)
            self._wgrad_pending = False

    def _wgrad(self, c: _ConvT, x, dy) -> int:
        self._on_wgrad_stream(lambda: ops.conv_wgrad(x, dy, self._g(c.conv.weight), k=c.k, stride=c.stride, pad=c.pad, dil=c.dil,
                                                     ws=self.wgrad_ws))
        return 2

    def _dgrad(self, c: _ConvT, dy, dx, residual=None, scratch: str = "up") -> int:
        """dx = conv_transpose(dy, W) (+ residual) through the forward kernel on the flipped weights."""
        n = 1
        if c.stride == 2:
            up = self._buf(scratch, (self.B, c.H, c.W, c.cout))
            ops.zero_insert2x(dy, out=up)
            dy, n = up, 2
        ops.conv_bn_act(dy, c.w_dgrad, c.one_in, c.zero_in, stride=1, pad=c.dil * (c.k - 1) - c.pad, dil=c.dil, relu=False,
                        residual=residual, out=dx)
        return n

    # ------------------------------------------------------------------ the step
    def _enqueue(self) -> int:
        """pack + forward + fused loss + backward: the whole step."""
        return self._enqueue_forward() + self._enqueue_loss() + self._enqueue_backward()

    def _enqueue_forward(self) -> int:
        net, K = self.net, self.K
        # weights of this step (parameters change every optimizer step)
        check(lib().hk_stem_pack_weights(ptr(net.conv1.weight.data), ptr(self.stem_w), stream_ptr()), "hk_stem_pack_weights")
        self._on_wgrad_stream(self._pack_all)   # the block convs' weights are repacked while the stem, its BN and the maxpool run
        n = 2
        if self.plan.train_bn_any:
            self.acc_fwd.zero_()                # the forward accumulators of every BatchNorm of this step
            n += 1
        n += self._fold_frozen()                # eval()-mode BatchNorms: scale / shift from the running statistics
        # ---------------- forward (train mode) ----------------
        n += self._conv_bn(self.stem, self.x, self.a0, relu=True)
        ops.maxpool3x3s2_fwd_idx(self.a0, out=self.p0, idx=self.pool_idx)   # forward + the winning taps the backward routes through
        n += 1
        self._join_wgrad_stream()               # packed weights ready
        x = self.p0
        for (c1, c2, ds, a1, sc, out) in self.blocks:
            if ds is not None:
                with torch.cuda.stream(self._fork_aux()):
                    n += self._conv_bn(ds, x, sc, relu=False)
                n += self._conv_bn(c1, x, a1, relu=True)
                self._join_aux()
                shortcut = sc
            else:
                n += self._conv_bn(c1, x, a1, relu=True)
                shortcut = x
            n += self._conv_bn(c2, a1, out, relu=True, residual=shortcut)
            x = out
        feat = x
        if self._bn_counters:                   # train-mode BatchNorms only
            torch._foreach_add_(self._bn_counters, 1)
            n += 1
        fc_w = net.fc.weight.data[:K].view(K, 512)
        fc_b = net.fc.bias.data[:K]
        ops.head_logits(feat, fc_w, fc_b, self.H, self.W, out=self.logits_up, logits_ws=self.logits_lr)
        n += 2
        return n

    def _enqueue_loss(self) -> int:
        """sigmoid + BCE(mean) forward and d/dlogits in one pass."""
        K = self.K
        tgt = self.target
        tcode = 0 if tgt is None else ops.dtype_code(tgt.dtype)
        check(lib().hk_bce_fwd_bwd(ptr(self.logits_up), 1, ptr(tgt), tcode, None if tgt is not None else ptr(self.uv), self.B, K, self.H,
                                   self.W, C.c_float(self.sigma), ptr(self.loss), ptr(self.g_up), ptr(self.bce_ws), self.bce_ws.numel(),
                                   stream_ptr()), "hk_bce_fwd_bwd")
        return 2

    def _acc_users(self, part: str) -> bool:
        """Does a BatchNorm backward of this part fill an accumulator (train-mode BN, or frozen BN with dgamma / dbeta)?"""
        e = self.convs.index(self.blocks[self.split_block][0])
        convs = self.convs if part == "all" else self.convs[e:] if part == "late" else self.convs[:e]
        for c in convs:
            p = self.plan.convs[c.name]
            if p.bwd and (not p.frozen or p.dgamma or p.dbeta):
                return True
        return False

    def has_early_backward(self) -> bool:
        """The early part of the two-phase step (layers 2..1 + stem) has work: something there needs a gradient."""
        return self.plan.lo < self.split_block

    def _enqueue_backward(self, part: str = "all") -> int:
        """From self.g_up = dL/d(upsampled logits) to every parameter gradient.  part "late" = head + layers 4..3 (the tail of the
        flat gradient buffer, 91 % of its bytes), part "early" = layers 2..1 + stem: the data-parallel step all-reduces the tail
        while the early layers are still being differentiated.  Follows self.plan: nothing runs below the earliest point that still
        needs a gradient, frozen parameters get no kernel."""
        net, K, st, pl = self.net, self.K, self.stem, self.plan
        n = 0
        nb = len(self.blocks)
        if self._acc_users(part):   # the backward accumulators this part is going to fill
            e = self.acc_early_bytes
            (self.acc_bwd if part == "all" else self.acc_bwd[e:] if part == "late" else self.acc_bwd[:e]).zero_()
            n += 1
        if part in ("all", "late"):
            feat = self.blocks[-1][5]
            fc_w = net.fc.weight.data[:K].view(K, 512)
            d = self._buf("d0", feat.shape) if pl.dfeat else None
            dw = self._g(net.fc.weight)[:K].view(K, 512) if pl.fc_weight else None
            db = self._g(net.fc.bias)[:K] if pl.fc_bias else None
            if d is not None or dw is not None or db is not None:
                ops.head_bwd(self.g_up, feat, fc_w, d, dw, db, dlogits_ws=self.dlogits_lr, ws=self.head_ws)
                n += 5 - (d is None) - 2 * (dw is None) - 2 * (db is None)
            parity, hi = 1, nb
        else:
            d, parity, hi = self._bwd_state
        lo = max(self.split_block if part == "late" else 0, pl.lo)
        for bi in range(hi - 1, lo - 1, -1):
            c1, c2, ds, a1, sc, out = self.blocks[bi]
            p1, p2 = pl.convs[c1.name], pl.convs[c2.name]
            pd = pl.convs[ds.name] if ds is not None else None
            below = pl.grad_in[bi]
            x_in = self.blocks[bi - 1][5] if bi > 0 else self.p0
            dy2 = self._dy_buf(c2) if p2.dy else None
            dm = self._buf("dm", c2.y.shape) if (pd.bwd if pd is not None else below) else None
            if p2.bwd:
                n += self._bn_bwd(c2, d, True, dy2, dmasked=dm)        # d' = d*[out>0] also feeds the shortcut
            dxd = None
            if pd is not None and pd.bwd:                               # shortcut branch: needs only d'; joins at the residual add
                dyd = self._dy_buf(ds) if pd.dy else None
                dxd = self._buf("dxd", x_in.shape) if pd.dgrad else None
                with torch.cuda.stream(self._fork_aux()):
                    n += self._bn_bwd(ds, dm, False, dyd)
                    if pd.wgrad:
                        n += self._wgrad(ds, x_in, dyd)
                    if pd.dgrad:
                        n += self._dgrad(ds, dyd, dxd, scratch="up_aux")
            if p2.wgrad:
                n += self._wgrad(c2, a1, dy2)
            da1 = None
            if p2.dgrad:
                da1 = self._buf("da1", a1.shape)
                n += self._dgrad(c2, dy2, da1)
            dy1 = self._dy_buf(c1) if p1.dy else None
            if p1.bwd:
                n += self._bn_bwd(c1, da1, True, dy1)
            if p1.wgrad:
                n += self._wgrad(c1, x_in, dy1)
            if pd is not None and pd.bwd:
                self._join_aux()
            if not below:
                d = None
                break
            dx = self._buf(f"d{parity}", x_in.shape)
            n += self._dgrad(c1, dy1, dx, residual=dxd if ds is not None else dm)
            d, parity = dx, parity ^ 1
        if part == "late":
            if self.has_early_backward():
                # the hand-off gradient gets its own buffer: the early graph is executed more than once per capture (warm-up, capture,
                # replay) and its ping-pong scratch would otherwise overwrite its own input
                dh = self._buf("dh", d.shape)
                dh.copy_(d)
                self._bwd_state = (dh, parity, lo)
                n += 1
            self._join_wgrad_stream()
            return n
        if pl.stem:
            da0 = self._buf("da0", self.a0.shape)
            ops.maxpool3x3s2_bwd_idx(d, self.pool_idx, self.a0.shape[1], self.a0.shape[2], dx=da0)
            sp = pl.convs[st.name]
            dy0 = self._dy_buf(st) if sp.dy else None
            n += 1 + self._bn_bwd(st, da0, True, dy0)
            if sp.wgrad:
                self._on_wgrad_stream(lambda: ops.stem_wgrad(self.x, dy0, self._g(net.conv1.weight), ws=self.wgrad_ws))
                n += 2
        self._join_wgrad_stream()
        return n

    def _key(self):
        # sigma is passed by value to hk_bce_fwd_bwd, i.e. baked into a captured graph: a new sigma needs a new capture
        # the torch flags (bn.training, requires_grad) choose the kernels: a toggled flag needs a new capture
        return (tuple(p.data_ptr() for p in self.all_params), None if self.target is None else (self.target.data_ptr(), self.target.dtype),
                self.sigma, self._flags)

    def forward_backward(self, img: torch.Tensor, uv: Optional[torch.Tensor] = None, target: Optional[torch.Tensor] = None) -> torch.Tensor:
        """img (B,3,H,W) fp32 CUDA; labels uv (B,K,2) = (x,y) [Gaussian targets generated on the fly, dataset.py:36-44] or a
        (B,K,H,W) fp64/fp32 target tensor (what KeypointsDataset returns).  Returns the fp64 mean-BCE loss (0-dim, a view of an
        engine buffer); the gradients of all parameters are in `self.flat_grad` / `grad(p)`."""
        if (uv is None) == (target is None):
            raise ValueError("pass exactly one of uv / target")
        if not img.is_cuda or tuple(img.shape) != (self.B, 3, self.H, self.W):
            raise ValueError(f"expected a CUDA image batch of shape {(self.B, 3, self.H, self.W)}, got {tuple(img.shape)} on {img.device}")
        self.sync_flags()
        with torch.no_grad():
            self.x.copy_(img)
            if uv is not None:
                self.uv.copy_(uv.reshape(self.B, self.K, 2))
                self.target = None
            else:
                if tuple(target.shape) != (self.B, self.K, self.H, self.W) or target.dtype not in (torch.float64, torch.float32):
                    raise ValueError("target must be (B,K,H,W) float64 or float32")
                if self.target is None or self.target.dtype != target.dtype:
                    self.target = torch.empty_like(target, memory_format=torch.contiguous_format)
                self.target.copy_(target)
            self.launches = self._run("step", self._enqueue, forward=True)
        return self.loss

    def _run(self, name: str, fn, forward: bool = False) -> int:
        """Run `fn` (enqueues work, returns its launch count) as eager launches, or as the CUDA graph `name`: captured on first use and
        whenever _key() changes, replayed otherwise.  Returns the launch count.  forward: fn advances the BatchNorm buffers."""
        if forward:
            self.model.mark_weights_changed()   # BatchNorm running stats move (raw-pointer writes; tensor versions do not)
        if not self.use_cuda_graph:
            return fn()
        key = self._key()
        ent = self._graphs.get(name)
        if ent is None or ent[1] != key:
            # one eager run first (lazy function attributes, scratch allocation); it advances the BN buffers once more than the
            # captured replay, so restore them
            if forward:
                saved = [(c.bn.running_mean.clone(), c.bn.running_var.clone(), c.bn.num_batches_tracked.clone()) for c in self.convs]
            n = fn()
            torch.cuda.current_stream().synchronize()
            if forward:
                for c, (m, v, t) in zip(self.convs, saved):
                    c.bn.running_mean.copy_(m); c.bn.running_var.copy_(v); c.bn.num_batches_tracked.copy_(t)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            self._graphs[name] = ent = (g, key, n)
        ent[0].replay()
        return ent[2]

    # ------------------------------------------------------------------ split step: the caller owns the loss (unmodified train.py)
    def forward_heatmaps(self, img: torch.Tensor) -> torch.Tensor:
        """Train-mode forward only: (B,3,H,W) -> sigmoid heatmaps (B,K,H,W) fp32 (model.py:19-22 under model.train()); activations
        are kept for backward_from_heatmap_grad().  Returns a view of an engine buffer."""
        if not img.is_cuda or tuple(img.shape) != (self.B, 3, self.H, self.W):
            raise ValueError(f"expected a CUDA image batch of shape {(self.B, 3, self.H, self.W)}, got {tuple(img.shape)} on {img.device}")
        if "heat" not in self.__dict__:
            self.heat = torch.empty_like(self.logits_up)
            self.g_heat = torch.empty_like(self.logits_up)
        n = self.logits_up.numel()
        self.sync_flags()

        def fn():
            k = self._enqueue_forward()
            check(lib().hk_sigmoid_fwd(ptr(self.logits_up), ptr(self.heat), C.c_longlong(n), stream_ptr()), "hk_sigmoid_fwd")
            return k + 1

        with torch.no_grad():
            self.x.copy_(img)
            self._split_launches["fwd"] = self._run("fwd", fn, forward=True)
        return self.heat

    def backward_from_heatmap_grad(self, grad_heat: torch.Tensor) -> None:
        """dL/dheat (B,K,H,W) fp32 -> all parameter gradients (self.flat_grad), through sigmoid, head and backbone."""
        n = self.logits_up.numel()

        def fn():
            check(lib().hk_sigmoid_bwd(ptr(self.heat), ptr(self.g_heat), ptr(self.g_up), C.c_longlong(n), stream_ptr()), "hk_sigmoid_bwd")
            return 1 + self._enqueue_backward()

        with torch.no_grad():
            self.g_heat.copy_(grad_heat)
            self._split_launches["bwd"] = self._run("bwd", fn)

    # ------------------------------------------------------------------ two-phase step for comm/compute overlap
    def forward_backward_late(self, img: torch.Tensor, uv: torch.Tensor) -> torch.Tensor:
        """Phase 1 of the data-parallel step: forward + loss + backward of head, layer4, layer3 (gradients flat_grad[late_offset:])."""
        if not img.is_cuda or tuple(img.shape) != (self.B, 3, self.H, self.W):
            raise ValueError(f"expected a CUDA image batch of shape {(self.B, 3, self.H, self.W)}")
        self.sync_flags()

        def fn():
            return self._enqueue_forward() + self._enqueue_loss() + self._enqueue_backward("late")

        with torch.no_grad():
            self.x.copy_(img)
            self.uv.copy_(uv.reshape(self.B, self.K, 2))
            self.target = None
            self._split_launches["late"] = self._run("late", fn, forward=True)
        return self.loss

    def backward_early(self) -> None:
        """Phase 2: backward of layer2, layer1 and the stem (gradients flat_grad[:late_offset]).  Nothing to do (no launch) when
        nothing there needs a gradient."""
        if not self.has_early_backward():
            self._split_launches["bwd_early"] = 0
            return
        with torch.no_grad():
            self._split_launches["bwd_early"] = self._run("bwd_early", lambda: self._enqueue_backward("early"))

    def split_launches(self) -> int:
        """Kernel launches of the split entry points run so far (two-phase data-parallel step: "late" + "bwd_early")."""
        return sum(self._split_launches.values())

    def grad(self, p: torch.nn.Parameter) -> torch.Tensor:
        return self.grad_of[id(p)]

    def grads_into_params(self) -> None:
        """p.grad = the engine's gradient (views of the flat buffer) for every parameter."""
        for p in self.params:
            p.grad = self.grad_of[id(p)]
