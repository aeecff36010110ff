#!/usr/bin/env python
"""bench_train.py -- BASELINE.json configs[3]: one KeypointsGauss training step per iteration.

    python bench_train.py [--steps K] [--warmup W] [--batch 4] [--freeze {none,bn,torchvision,head}]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench_train.py --gpus N

step = Gaussian targets from (B,K,2) labels (generated on the fly inside the fused loss kernel) + forward (train-mode
BN, per-replica statistics) + fused sigmoid/BCE forward+backward (hk_bce_fwd_bwd) + backbone backward + gradient
all-reduce (NCCL, bucketed) + Adam(lr 1e-4, wd 1e-4) -- the sequence of reference train.py:33-36.
--backend hk (default): the whole step runs on libhulk_sm100 kernels (TrainEngine: tcgen05 forward / dgrad / wgrad, train-mode
BN kernels, fused loss, FusedAdam; one CUDA graph).  --backend autograd: the backbone runs on torch autograd / cuDNN fp32 (the
same-box competitor).  --freeze: fine-tuning presets (train_ops.freeze_preset): "bn" every BatchNorm in eval() mode with
gamma / beta trained, "torchvision" every BatchNorm frozen with gamma / beta plus conv1 + layer1 frozen, "head" only fc trained.
Secondary benchmark: the headline metric is bench.py (inference images/s).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4, help="per-GPU batch (config.py: 4)")
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"], help="FusedAdam (hk_adam_step) or torch.optim.Adam")
    ap.add_argument("--reference-loss", action="store_true", help="use torch's .double()+BCELoss on fp64 targets (train.py:21-25)")
    ap.add_argument("--backend", default="hk", choices=["hk", "autograd"],
                    help="hk: whole step on libhulk_sm100 kernels (TrainEngine, bf16 tcgen05, one CUDA graph); "
                         "autograd: backbone on torch autograd / cuDNN fp32 (the same-box competitor and the parity checker)")
    ap.add_argument("--freeze", default="none", choices=["none", "bn", "torchvision", "head"],
                    help="fine-tuning preset: frozen BatchNorms (eval() mode) and frozen parameters (requires_grad=False)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import hulk_keypoints_b200 as hk
    from hulk_keypoints_b200 import ops, parallel, train_ops

    torch.manual_seed(0)
    model = hk.KeypointsGauss(4, img_height=args.height, img_width=args.width).to(dev).train()
    parallel.broadcast_model(model)
    if args.freeze != "none":
        train_ops.freeze_preset(model, args.freeze)   # before the optimiser is built, as in torch
    if args.optimizer == "fused" and not args.reference_loss:
        from hulk_keypoints_b200.optim import FusedAdam
        opt = FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-4)
    else:
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-4, fused=True)
    B, H, W = args.batch, args.height, args.width
    g = torch.Generator().manual_seed(2000 + rank)
    img = torch.rand(B, 3, H, W, generator=g).to(dev)
    uv = torch.stack([torch.randint(0, W, (B, 4), generator=g), torch.randint(0, H, (B, 4), generator=g)], -1).float().to(dev)
    allreduce = (lambda params: parallel.allreduce_gradients(params)) if world > 1 else None

    def step():
        if args.reference_loss:
            opt.zero_grad(set_to_none=True)
            gt = ops.gauss_targets(uv, H, W, 8.0)                       # fp64 targets, as dataset.py returns them
            loss = torch.nn.BCELoss()(model(img).double(), gt)          # train.py:21,25
            loss.backward()
            if allreduce:
                allreduce(model.parameters())
            opt.step()
            return loss.detach()
        return train_ops.train_step(model, opt, img, uv, sigma=8.0, allreduce=allreduce, backend=args.backend)

    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record(); e1.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    if rank == 0:
        print(json.dumps({
            "metric": "train_steps_per_sec", "value": args.steps / (ms * 1e-3), "unit": "steps/s",
            "images_per_sec": world * B * args.steps / (ms * 1e-3), "n_gpus": world, "steps": args.steps,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "dtype": ("bf16 operands / f32 accumulate (tcgen05), f32 BN stats + grads, f64 loss" if args.backend == "hk" and not args.reference_loss
                      else "f32 (backbone, torch autograd / cuDNN) + f64 loss"),
            "backend": "autograd" if args.reference_loss else args.backend,
            "gpu_launches_per_step": (model.train_engine(B, H, W).launches + 1) if args.backend == "hk" and not args.reference_loss else None,
            "data": "synthetic", "loss": float(loss.item()),
            "config": {"workload": f"train step, per-GPU batch {B}, {H}x{W}, K=4, Adam lr 1e-4 wd 1e-4 (BASELINE.json configs[3])",
                       "loss_path": "torch BCELoss on fp64 targets" if args.reference_loss else "fused hk_bce_fwd_bwd, targets on the fly",
                       "optimizer": type(opt).__name__, "freeze": args.freeze,
                       "parallelism": f"data-parallel x{world}, NCCL all-reduce of the gradients"}}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
