"""Training-side pieces: the fused sigmoid+BCE loss as an autograd function and a fused train step.

Reference train.py:18-26 computes `nn.BCELoss()(model.forward(img).double(), gt_gauss)`: three full passes at
8 bytes/element (cast, loss, reduce) and, in backward, a 1000-channel upsample gradient.  Here the autograd
boundary is moved to the upsampled LOGITS of the K live channels: one pass of hk_bce_fwd_bwd evaluates the
sigmoid (model.py:21), the fp64 loss and the fp32 gradient w.r.t. the logits -- bit-identical to what autograd
produces for sigmoid -> .double() -> BCELoss -- optionally generating the Gaussian target on the fly from the
(B,K,2) labels so neither the heatmap nor the fp64 target tensor is ever written to HBM.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops


class _FusedSigmoidBCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, uv, sigma):
        z = logits.detach().contiguous()
        loss, grad_logits = ops.bce_fwd_bwd(z, target=target, uv=uv, sigma=sigma, want_grad=True, pred_is_logits=True)
        ctx.save_for_backward(grad_logits)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (grad_logits,) = ctx.saved_tensors
        return grad_logits * grad_out.to(grad_logits.dtype), None, None, None


def sigmoid_bce_loss(logits: torch.Tensor, target: Optional[torch.Tensor] = None, uv: Optional[torch.Tensor] = None,
                     sigma: float = 8.0) -> torch.Tensor:
    """mean BCE(sigmoid(logits), target) as a 0-dim float64 tensor, differentiable w.r.t. `logits` (fp32).
    Pass either a (B,K,H,W) fp64/fp32 `target` or the (B,K,2) labels `uv` (+ `sigma`)."""
    if (target is None) == (uv is None):
        raise ValueError("pass exactly one of target / uv")
    return _FusedSigmoidBCE.apply(logits, target, uv, float(sigma))


class _EngineStep(torch.autograd.Function):
    """forward = TrainEngine.forward_backward (loss AND all parameter gradients in one pass of our kernels); backward hands the
    stored gradients to autograd, so an unmodified `loss.backward(); optimizer.step()` (train.py:35-36) works."""

    @staticmethod
    def forward(ctx, engine, img, target, uv, *params):
        loss = engine.forward_backward(img, uv=uv, target=target)
        ctx.engine, ctx.params = engine, list(engine.params)
        return loss.clone()

    @staticmethod
    def backward(ctx, grad_out):
        eng = ctx.engine
        g = grad_out.to(torch.float32)
        return (None, None, None, None) + tuple(eng.grad(p) * g for p in ctx.params)


class _EngineForward(torch.autograd.Function):
    """KeypointsGauss.forward in train() mode on the B200 engine: returns the heatmaps; autograd hands dL/dheat back and the engine's
    backward kernels produce every parameter gradient -- so an UNMODIFIED train.py (model.forward(img).double() -> nn.BCELoss ->
    loss.backward() -> optimizer.step(), train.py:18-26,33-36) trains on tcgen05."""

    @staticmethod
    def forward(ctx, engine, img, *params):
        ctx.engine, ctx.params = engine, list(engine.params)
        return engine.forward_heatmaps(img).clone()

    @staticmethod
    def backward(ctx, grad_heat):
        eng = ctx.engine
        eng.backward_from_heatmap_grad(grad_heat.to(torch.float32).contiguous())
        return (None, None) + tuple(eng.grad(p).clone() for p in ctx.params)


def engine_forward(model, img: torch.Tensor) -> torch.Tensor:
    """Differentiable train-mode heatmaps (B,K,H,W) computed by the TrainEngine (see _EngineForward)."""
    eng = model.train_engine(img.shape[0], img.shape[2], img.shape[3])
    eng.sync_flags()   # only trainable parameters are inputs of the autograd node: frozen ones keep .grad None
    return _EngineForward.apply(eng, img.float().contiguous(), *eng.params)


def engine_loss(model, img: torch.Tensor, target: Optional[torch.Tensor] = None, uv: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Differentiable fp64 loss of one batch computed by the B200 TrainEngine (bf16 tensor-core forward/backward)."""
    eng = model.train_engine(img.shape[0], img.shape[2], img.shape[3])
    eng.sync_flags()
    return _EngineStep.apply(eng, img, target, uv, *eng.params)


def loss_from_batch(sample_batched, model, use_cuda: bool = True, backend: str = "hk") -> torch.Tensor:
    """Drop-in for reference train.py:18-26 `forward(sample_batched, model)`: (img, gt_gauss) -> float64 loss.
    backend "hk" (default): TrainEngine kernels; "autograd": torch autograd graph over the same parameters (fp32 checker)."""
    img, gt_gauss = sample_batched
    if use_cuda:
        img, gt_gauss = img.cuda(), gt_gauss.cuda()
    if backend == "hk":
        return engine_loss(model, img.float().contiguous(), target=gt_gauss.contiguous())
    return sigmoid_bce_loss(model.forward_logits(img), target=gt_gauss.contiguous())


def train_step(model, optimizer, img: torch.Tensor, uv: torch.Tensor, sigma: float = 8.0, allreduce=None,
               backend: str = "hk", exchange: bool = True, augment=None) -> torch.Tensor:
    """One step of reference train.py:33-36 (zero_grad, forward, backward, step) with targets generated from
    labels on the fly.  `optimizer` is a `hulk_keypoints_b200.optim.FusedAdam` (flat buffers: one all-reduce, one
    update kernel) or any torch optimizer; `allreduce(params)` (data-parallel exchange) runs between backward and step
    for torch optimizers, FusedAdam reduces its flat gradient buffer itself.

    `exchange=False` skips the data-parallel gradient exchange (a measurement switch: replicas then diverge).
    backend "hk" (default): the whole forward + loss + backward runs on libhulk_sm100 kernels (TrainEngine, one CUDA graph);
    with FusedAdam the engine writes the gradients straight into the optimiser's flat buffer.  backend "autograd": the
    backbone runs on torch autograd (fp32 cuDNN) -- the checker of the parity tests, not a product path.

    `augment`: a `hulk_keypoints_b200.augment.KeypointAugment` applied to (img, uv) on the device before the step.  On the engine its
    launches write the engine's input buffers (in place of the batch copy), outside the captured graph, so every step draws new
    parameters; on the autograd backend the same augmenter runs first and the torch graph sees the same batch."""
    fused = hasattr(optimizer, "flat_grad")
    if backend == "hk":
        eng = model.train_engine(img.shape[0], img.shape[2], img.shape[3])
        eng.sigma = float(sigma)
        eng.sync_flags()   # bn.training / requires_grad of this step: the flat gradient buffer holds the trainable parameters only
        if fused:
            if optimizer.flat_grad.data_ptr() != eng.flat_grad.data_ptr():
                # the engine's order is the flat layout (the two-phase split relies on it): FusedAdam reorders to it once
                optimizer.adopt_grad_buffer(eng.flat_grad, eng.params)
        import torch.distributed as dist
        if not exchange:   # measurement only (bench.py: the step with its gradient exchange switched off = the compute-only time)
            loss = eng.forward_backward(img, uv=uv, augment=augment)
            if not fused:
                eng.grads_into_params()
            optimizer.step()
            return loss.detach().clone()
        if fused and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            # data-parallel: the all-reduce of layer3/layer4/fc gradients (91 % of the bytes) overlaps the backward of layers 2..1 + stem.
            # (Also running the Adam update of that range beside the early backward was measured at 2 GPUs, batch 4: 3.957 ms against
            # 3.943 ms with one update at the end -- the update is an HBM stream that slows the backward it overlaps -- and dropped.)
            loss = eng.forward_backward_late(img, uv, augment=augment)
            w1 = optimizer.all_reduce_range_async(eng.late_offset, optimizer.numel)
            eng.backward_early()
            w0 = optimizer.all_reduce_range_async(0, eng.late_offset)
            optimizer.finish_all_reduce([w1, w0])
            optimizer.step()
            return loss.detach().clone()
        loss = eng.forward_backward(img, uv=uv, augment=augment)
        if fused:
            optimizer.all_reduce_grads()
        else:
            eng.grads_into_params()
            if allreduce is not None:
                allreduce(model.parameters())
        optimizer.step()
        return loss.detach().clone()
    if augment is not None:
        img, uv = augment(img, uv)
    if fused:
        optimizer.zero_grad()
    else:
        optimizer.zero_grad(set_to_none=True)
    loss = sigmoid_bce_loss(model.forward_logits(img), uv=uv, sigma=sigma)
    loss.backward()
    if fused:
        optimizer.all_reduce_grads()
    elif allreduce is not None:
        allreduce(model.parameters())
    optimizer.step()
    return loss.detach()


FREEZE_PRESETS = ("none", "bn", "torchvision", "head", "mixed")


def freeze_preset(model, preset: str) -> None:
    """Put `model` in train() mode and set the standard fine-tuning flags (torch's own switches, which the training engine honours):
      none        every BatchNorm in train mode, every parameter trained (the default configuration)
      bn          every BatchNorm in eval() mode (running statistics, buffers untouched); gamma / beta and all weights trained
      torchvision every BatchNorm in eval() mode with gamma / beta frozen, and conv1 + layer1 frozen (torchvision's detection and
                  keypoint models at trainable_backbone_layers=3)
      head        only the scoring conv `fc` trained; every BatchNorm in eval() mode
      mixed       BatchNorms of the stem and layers 1-2 in eval() mode, layers 3-4 in train mode; every parameter trained
    Build the optimiser after freezing, as in torch: FusedAdam lays out the trainable parameters only (when unfreezing later, hand the
    newly trainable parameters to `optimizer.add_param_group`)."""
    if preset not in FREEZE_PRESETS:
        raise ValueError(f"freeze preset must be one of {FREEZE_PRESETS}")
    net = model.resnet.resnet34_8s
    model.train()
    for p in model.parameters():
        p.requires_grad_(True)
    bns = [m for m in net.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    if preset in ("bn", "torchvision", "head"):
        for bn in bns:
            bn.eval()
    if preset == "torchvision":
        for bn in bns:
            for p in bn.parameters():
                p.requires_grad_(False)
        for m in (net.conv1, net.bn1, net.layer1):
            for p in m.parameters():
                p.requires_grad_(False)
    elif preset == "head":
        for p in model.parameters():
            p.requires_grad_(False)
        for p in net.fc.parameters():
            p.requires_grad_(True)
    elif preset == "mixed":
        for m in (net.bn1, net.layer1, net.layer2):
            for bn in m.modules():
                if isinstance(bn, torch.nn.BatchNorm2d):
                    bn.eval()
