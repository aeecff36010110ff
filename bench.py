#!/usr/bin/env python
"""bench.py -- KeypointsGauss heatmap inference images/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 64] [--precision bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic images: stem -> 16 BasicBlocks -> head ->
argmax decode for `--batch` (64) images of 480x640 (BASELINE.json configs[1]).  Rank 0 prints ONE JSON line.

  value      images/s, all ranks, inputs resident in HBM (CUDA-graph replay of the whole step), CUDA events,
             barrier + synchronize on both sides, max over ranks.
  e2e        same metric through the public API with HOST buffers: pinned-host fp32 images are copied to the
             device, Prediction-equivalent forward + decode runs, keypoints (B,K,2) + peak values come back to the
             host -- every step, inside the timed region (copies double-buffered against compute).
  roofline   the dominant kernel (tcgen05 implicit-GEMM conv): algorithmic FLOPs of its launches in one step /
             their CUDA-event time, against MEASURED_PEAKS.json's dense bf16 peak.
  cpu_baseline / --impl reference: the reference's own CPU path on the host cores -- the unmodified reference classes staged in
             oracle/_ref/ by build() (kind "reference"), else the oracle port (kind "port").
  roofline_hbm_kernels / train_step: informational extras -- the memory-bound kernels against the measured copy bandwidth, and
             (N=1, default workload) ms per training step at per-GPU batch 4 / 32 (BASELINE configs[3]; bench_train.py is the full tool).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

import torch  # noqa: E402

METRIC = "heatmap_inference_images_per_sec"
UNIT = "images/s"
K_KEYPOINTS = 4


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"],
                    help="ours: libhulk_sm100 kernels; reference: the reference's CPU path (oracle port) on the host cores; torch_gpu: the "
                         "same network through torch/cuDNN on this GPU (same-box competitor, SURVEY.md §8d; informational)")
    ap.add_argument("--torch-dtype", default="fp32", choices=["fp32", "bf16"], help="torch_gpu arm: fp32 (TF32 off) or bf16 autocast + channels_last")
    ap.add_argument("--as-written-head", action="store_true", help="torch_gpu arm: evaluate and upsample all 1000 fc channels, then slice (model.py:21)")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--keypoints", type=int, default=4, help="K (config.py: 4; BASELINE config 5 also quotes 16 and 32)")
    ap.add_argument("--cpu-images", type=int, default=0, help="images in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-step", action="store_true",
                    help="skip the secondary measurement (BASELINE configs[3]: one training step per iteration, per-GPU batch 4 and 32, N=1 only)")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 3 s sustained loop")
    ap.add_argument("--no-config3", action="store_true", help="skip the BASELINE configs[2] extra (4096 images split across the ranks)")
    ap.add_argument("--breakdown", default="", help="write the per-launch timing table to this JSON file")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay (profiling)")
    ap.add_argument("--profile-mode", action="store_true",
                    help="device-resident loop only: no e2e loop, no per-launch breakdown, no CPU baseline (for ncu runs)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) to DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def conv_flops_per_image(h, w, k):
    """Algorithmic conv FLOPs per image from the product package's own module graph (no oracle on the product arm)."""
    import hulk_keypoints_b200 as hk
    from hulk_keypoints_b200.engine import conv_flops_per_image as f
    return f(hk.KeypointsGauss(k, img_height=h, img_width=w), h, w)


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- CPU arm
class CpuReference:
    """The reference's CPU path, B=1 per call as analysis.py does, all host threads.  Weights and inputs are prepared once, outside
    any timed region.  kind "reference": the UNMODIFIED reference classes (src/model.py KeypointsGauss + src/prediction.py
    Prediction.predict + the numpy argmax of prediction.py:46) from oracle/_ref/, staged there by __graft_entry__.build() in the
    build container (git-ignored; it travels to the GPU box with the snapshot), eval() + no_grad (BASELINE configs[0]).
    kind "port": oracle/keypoints_oracle.py in the reference's as-written op order, when oracle/_ref/ is absent."""

    def __init__(self, height: int, width: int):
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        g = torch.Generator().manual_seed(1000)
        self.imgs = [torch.rand(1, 3, height, width, generator=g) for _ in range(2)]
        ref_root = os.path.join(ROOT, "oracle", "_ref")
        self.kind = "port"
        if os.path.isfile(os.path.join(ref_root, "src", "model.py")):
            try:
                os.environ["HULK_REFERENCE_ROOT"] = ref_root
                from oracle import reference_loader as RL
                model = RL.build_reference_model(0, K_KEYPOINTS, height, width).eval()
                _, pr = RL.reference_modules()
                self.pred = pr.Prediction(model, K_KEYPOINTS, height, width, False)
                self.kind = "reference"
            except Exception as exc:  # noqa: BLE001 -- fall back to the port, say why
                print(f"[bench] oracle/_ref present but not importable ({type(exc).__name__}: {exc}); timing the oracle port", file=sys.stderr)
        if self.kind == "port":
            from oracle import keypoints_oracle as O
            self.O = O
            self.sd = O.init_state_dict(0)

    def run(self, n_images: int) -> float:
        """Process n_images; returns elapsed seconds."""
        import numpy as np
        t0 = time.perf_counter()
        for i in range(n_images):
            if self.kind == "reference":
                with torch.no_grad():
                    heat = self.pred.predict(self.imgs[i % 2][0]).detach().cpu().numpy()       # analysis.py:40-41
                for k in range(K_KEYPOINTS):
                    np.unravel_index(heat[0][k].argmax(), heat[0][k].shape)                    # prediction.py:46
            else:
                # as_written=True: the reference's literal op order (1000-channel fc and upsample, then slice, model.py:21)
                self.O.argmax_decode(self.O.forward(self.sd, self.imgs[i % 2], K_KEYPOINTS, as_written=True).numpy())
        return time.perf_counter() - t0


def run_reference_arm(args, rank):
    if rank != 0:
        return
    ref = CpuReference(args.height, args.width)
    # bounded sample: ~0.2-0.5 s per image on the host cores; keep the whole run within a few minutes whatever --steps is
    n_per_step = 4 if args.steps <= 30 else (2 if args.steps <= 100 else 1)
    for _ in range(max(args.warmup, 1)):
        ref.run(1)
    dt = 0.0
    for _ in range(args.steps):
        dt += ref.run(n_per_step)
    total = n_per_step * args.steps
    cores = ref.cores
    value = total / dt
    sample = f"{n_per_step} images of {args.height}x{args.width} per step, B=1 per call (analysis.py style), {args.steps} steps"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"KeypointsGauss eval forward + argmax decode, {args.height}x{args.width}, K={K_KEYPOINTS}, "
                               + ("the unmodified reference classes (oracle/_ref)" if ref.kind == "reference" else
                                  "oracle port of the reference (as-written op order: 1000-channel head)") + " on host CPU (bounded sample)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": ref.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- same-box torch/cuDNN arm
def run_torch_gpu(args, rank, world, local_rank):
    """The same network evaluated by torch (cuDNN convs, ATen upsample/sigmoid, torch argmax) on this GPU: eval-mode BN, no_grad.
    Uses the parameters of our KeypointsGauss through its torch graph (the one the parity tests check against) -- none of our kernels."""
    import torch.nn.functional as F

    import hulk_keypoints_b200 as hk

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    B, H, W, K = args.batch, args.height, args.width, K_KEYPOINTS
    torch.manual_seed(0)
    model = hk.KeypointsGauss(K, img_height=H, img_width=W).to(dev).eval()
    net = model.resnet.resnet34_8s
    bf16 = args.torch_dtype == "bf16"
    if bf16:
        net = net.to(memory_format=torch.channels_last)
    x = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(1000 + rank)).to(dev)
    if bf16:
        x = x.contiguous(memory_format=torch.channels_last)

    def step():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            feat = net.features(x)
            if args.as_written_head:
                up = F.interpolate(net.fc(feat), size=(H, W), mode="bilinear", align_corners=True)   # all 1000 channels
                heat = torch.sigmoid(up[:, :K])
            else:
                heat = torch.sigmoid(F.interpolate(F.conv2d(feat, net.fc.weight[:K], net.fc.bias[:K]), size=(H, W), mode="bilinear",
                                                   align_corners=True))
            flat = heat.float().reshape(B, K, -1).argmax(-1)
            return torch.stack([flat // W, flat % W], -1)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record(); e1.synchronize()
    ms = e0.elapsed_time(e1)
    if rank == 0:
        print(json.dumps({"impl": "torch_gpu", "metric": METRIC, "value": world * B * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
                          "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                          "dtype": "bf16 autocast, channels_last" if bf16 else "f32 (TF32 off)", "data": "synthetic",
                          "config": {"workload": f"torch/cuDNN eval forward + torch argmax, batch {B}, {H}x{W}, K={K}, "
                                                 f"{'1000-channel head as written' if args.as_written_head else 'K-row head'}"}}), flush=True)


# --------------------------------------------------------------------------------------------- our arm
def per_launch_breakdown(engine, plan, decode=True):
    """Eager (no graph) pass with a CUDA event pair around every launch group; returns [(name, ms, flops)]."""
    from hulk_keypoints_b200 import ops

    net = engine.model.resnet.resnet34_8s
    P = engine._packed
    rows = []
    stream = torch.cuda.current_stream()

    def timed(name, flops, fn, reps=5):
        fn()
        # MEAN launch duration: `reps` back-to-back launches of the same kernel inside ONE event pair (the gaps between an event
        # record and a lone launch would otherwise be charged to the kernel); the single-launch minimum is kept for reference only
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream); b.synchronize()
        mean = a.elapsed_time(b) / reps
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); fn(); b.record(stream); b.synchronize()
            ts.append(a.elapsed_time(b))
        rows.append({"name": name, "ms": mean, "ms_min": min(ts), "flops": flops, "algo": None, "bytes": 0.0})

    B = plan.B
    cur = 0
    x = plan.view(cur, plan.h4, plan.w4, 64)
    in_bytes = 3.0 * plan.H * plan.W * (1 if plan.input_is_u8 else 4)
    if engine._stem_w_tc is not None and engine.fuse_stem_pool and ops.stem_pool_supported(plan.x):
        timed("stem_pool", 2.0 * B * plan.h2 * plan.w2 * 64 * 147,
              lambda: ops.stem_pool(plan.x, engine._stem_w_tc, P["stem"].scale, P["stem"].bias, out=x))
        rows[-1]["bytes"] = B * (in_bytes + plan.h4 * plan.w4 * 64 * 2)          # input read + pooled bf16 output write
    else:
        if engine._stem_w_tc is not None:
            timed("stem", 2.0 * B * plan.h2 * plan.w2 * 64 * 147,
                  lambda: ops.stem(plan.x, engine._stem_w_tc, P["stem"].scale, P["stem"].bias, out=plan.stem))
        else:
            timed("stem", 2.0 * B * plan.h2 * plan.w2 * 64 * 147,
                  lambda: engine._conv(P["stem"], plan.x, plan.stem, relu=True, in_is_nchw=True))
        rows[-1]["bytes"] = B * (in_bytes + plan.h2 * plan.w2 * 64 * 2)           # input read + bf16 output write
        timed("maxpool", 0.0, lambda: ops.maxpool3x3s2(plan.stem, out=x))
        rows[-1]["bytes"] = B * 64.0 * 2 * (plan.h2 * plan.w2 + plan.h4 * plan.w4)
    h, w = plan.h4, plan.w4
    blocks = list(net.blocks())
    nblocks, head_done = len(blocks), False
    for i, blk in enumerate(blocks):
        c1, c2 = P[f"b{i}.c1"], P[f"b{i}.c2"]
        planes, cin = c1.w.shape[0], c1.w.shape[3]
        ho, wo = ops.conv_out_hw(h, w, 3, c1.stride, c1.pad, c1.dil)
        free = [j for j in range(4) if j != cur]
        t = plan.view(free[0], ho, wo, planes)
        xin = x
        ds = P.get(f"b{i}.ds")
        if (ds is not None and engine.fuse_downsample and c1.algo == ds.algo == 0 and ds.stride == c1.stride
                and ops.conv_ds_supported(xin, c1.w, ds.w, c1.stride, c1.pad, c1.dil)):
            sc = plan.view(free[1], ho, wo, planes)      # block entry: conv1 + the 1x1 downsample conv in one launch (engine._enqueue)
            timed(f"b{i}.c1+ds", 2.0 * B * ho * wo * planes * cin * 10,
                  lambda: ops.conv_ds(xin, c1.w, c1.scale, c1.bias, ds.w, ds.scale, ds.bias, stride=c1.stride, pad=c1.pad, dil=c1.dil,
                                      relu=True, out=t, out_ds=sc))
            rows[-1]["algo"] = c1.algo
        elif blk.downsample is not None:
            timed(f"b{i}.c1", 2.0 * B * ho * wo * planes * cin * 9, lambda: engine._conv(c1, xin, t, relu=True))
            rows[-1]["algo"] = c1.algo
            sc = plan.view(free[1], ho, wo, planes)
            timed(f"b{i}.ds", 2.0 * B * ho * wo * planes * cin, lambda: engine._conv(P[f"b{i}.ds"], xin, sc, relu=False))
            rows[-1]["algo"] = P[f"b{i}.ds"].algo
        else:
            timed(f"b{i}.c1", 2.0 * B * ho * wo * planes * cin * 9, lambda: engine._conv(c1, xin, t, relu=True))
            rows[-1]["algo"] = c1.algo
            sc = x
        if (i == nblocks - 1 and engine.fuse_head and c2.algo == 0 and ops.conv_head_supported(t, c2.w, engine._fc_w, c2.stride)
                and (ho, wo) == (plan.h8, plan.w8)):
            # last conv + the K scoring rows in one launch (engine._enqueue); the feature map is never written
            timed(f"b{i}.c2+fc", 2.0 * B * ho * wo * planes * (planes * 9 + engine.K),
                  lambda: ops.conv_head(t, c2.w, c2.scale, c2.bias, engine._fc_w, engine._fc_b, plan.logits, stride=c2.stride, pad=c2.pad,
                                        dil=c2.dil, relu=True, residual=sc))
            rows[-1]["algo"] = c2.algo
            timed("upsample", 0.0, lambda: ops.head_upsample(plan.logits, plan.H, plan.W, heat=plan.heat, fast=True))
            rows[-1]["bytes"] = B * engine.K * (plan.H * plan.W + ho * wo) * 4.0      # fp32 logits read + fp32 heatmaps written
            head_done = True
            break
        y = plan.view(free[2], ho, wo, planes)
        timed(f"b{i}.c2", 2.0 * B * ho * wo * planes * planes * 9, lambda: engine._conv(c2, t, y, relu=True, residual=sc))
        rows[-1]["algo"] = c2.algo
        x, cur, h, w = y, free[2], ho, wo
    xf = x
    if not head_done:
        timed("head", 2.0 * B * h * w * engine.K * 512,
              lambda: ops.head(xf, engine._fc_w, engine._fc_b, plan.H, plan.W, heat=plan.heat, logits_ws=plan.logits))
        rows[-1]["bytes"] = B * (512.0 * h * w * 2 + engine.K * plan.H * plan.W * 4.0)   # SURVEY §8d: bf16 features read + fp32 heatmaps written
    if decode:
        timed("decode", 0.0, lambda: ops.argmax_decode(plan.heat, yx=plan.yx, maxval=plan.maxval, ws=plan.argmax_ws, want_max=True))
        rows[-1]["bytes"] = B * engine.K * plan.H * plan.W * 4.0
    return rows


HEAT_DUMP_VALUES = 1 << 23   # 32 MB of fp32: the dump stays well under 64 MB at any workload


def dump_outputs(out_dir, plan):
    """--dump-outputs: what a caller of the timed path receives (KeypointsGauss.heatmaps_and_keypoints / .keypoints), as the timed
    loop's last step left it in the plan's buffers.  heatmaps.npy: the (B,K,H,W) fp32 heatmaps; above HEAT_DUMP_VALUES values, the
    1-D sample at a fixed seeded set of sorted flat indices instead (the same set on every run of a workload).  keypoints_yx.npy:
    (B,K,2) (row, col) as float64 (exact).  peak_values.npy: (B,K) fp32 heatmap value at each keypoint."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    heat = plan.heat
    if heat.numel() > HEAT_DUMP_VALUES:
        idx = np.sort(np.random.default_rng(0).integers(0, heat.numel(), HEAT_DUMP_VALUES))
        idx = idx[np.diff(idx, prepend=-1) > 0]                       # drop repeats (np.unique is far slower at this size)
        heat = heat.reshape(-1)[torch.from_numpy(idx).to(heat.device)]
    arrays = {"heatmaps": heat.cpu().numpy(), "keypoints_yx": plan.yx.cpu().numpy().astype(np.float64),
              "peak_values": plan.maxval.cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist

    import hulk_keypoints_b200 as hk
    from hulk_keypoints_b200._lib import HK_CONV_TCGEN05

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, H, W = args.batch, args.height, args.width
    torch.manual_seed(0)
    model = hk.KeypointsGauss(K_KEYPOINTS, img_height=H, img_width=W, precision=args.precision).to(dev).eval()
    engine = model.engine()
    engine.use_cuda_graph = not args.no_graph
    gen = torch.Generator().manual_seed(1000 + rank)
    host_imgs = [torch.rand(B, 3, H, W, generator=gen).pin_memory() for _ in range(2)]
    x_dev = host_imgs[0].to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident throughput (value) ----------------
    engine._ensure_packed()
    plan = engine.plan_for(B, H, W)
    plan.x.copy_(x_dev)
    for _ in range(max(args.warmup, 3)):
        engine.run_plan(plan, decode=True)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for _ in range(args.steps):
        engine.run_plan(plan, decode=True)
    stop.record()
    stop.synchronize()
    barrier()
    dev_ms = max_over_ranks(start.elapsed_time(stop))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, plan)
    value = world * B * args.steps / (dev_ms * 1e-3)
    launches_per_step = plan.launches
    if args.profile_mode:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                              "ms_per_step": dev_ms / args.steps, "profile_mode": True, "clocks": clocks,
                              "gpu_launches_per_step": launches_per_step}), flush=True)
        return

    # ---------------- sustained: the same loop for >= 3 s (thermal / power steady state) ----------------
    sustained = None
    if not args.no_sustained:
        n_sus = max(args.steps, int(3.2e3 / max(dev_ms / args.steps, 1e-3)) + 1)
        sampler2 = ClockSampler(local_rank)
        barrier()
        if rank == 0:
            sampler2.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(n_sus):
            engine.run_plan(plan, decode=True)
        s1.record()
        s1.synchronize()
        barrier()
        sus_ms = max_over_ranks(s0.elapsed_time(s1))
        sustained = {"value": world * B * n_sus / (sus_ms * 1e-3), "unit": UNIT, "steps": n_sus, "seconds": sus_ms * 1e-3,
                     "ms_per_step": sus_ms / n_sus, "clocks": sampler2.stop() if rank == 0 else None}

    # ---------------- end to end through the public API, host buffers ----------------
    copy_stream = torch.cuda.Stream(device=dev)
    compute = torch.cuda.current_stream()
    host_yx = [torch.empty((B, K_KEYPOINTS, 2), dtype=torch.int32).pin_memory() for _ in range(2)]
    host_mv = [torch.empty((B, K_KEYPOINTS), dtype=torch.float32).pin_memory() for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]

    def measure_e2e(host_in):
        """host_in: two pinned host batches (fp32 (B,3,H,W) as ToTensor yields, or (B,H,W,3) uint8 as cv2 yields).  Public serving API:
        model.staging_input(slot) <- H2D copy; model.keypoints(buf, slot) -> (yx, peak) -> D2H.  Two slots: the copy of step i+1 runs
        on the copy stream while step i computes."""
        u8 = host_in[0].dtype == torch.uint8
        dev_in = [model.staging_input(B, H, W, slot=j, uint8=u8) for j in range(2)]

        def loop(steps):
            for j in range(2):
                in_free[j].record(compute)
            for i in range(steps):
                j = i & 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(in_free[j])
                    dev_in[j].copy_(host_in[j], non_blocking=True)       # H2D of this step's images
                    in_ready[j].record(copy_stream)
                compute.wait_event(in_ready[j])
                yx, peak = model.keypoints(dev_in[j], slot=j)             # public API (engine forward + decode)
                in_free[j].record(compute)
                host_yx[j].copy_(yx, non_blocking=True)                   # D2H of the step's result
                host_mv[j].copy_(peak, non_blocking=True)
            compute.synchronize()

        loop(max(2, args.warmup))
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s2.record()
        loop(args.steps)
        e2.record()
        e2.synchronize()
        barrier()
        ms = max_over_ranks(max(s2.elapsed_time(e2), 0.0))
        wall = (time.perf_counter() - t0) * 1e3
        return ms, wall, host_in[0].numel() * host_in[0].element_size()

    e2e_ms, wall_ms, h2d = measure_e2e(host_imgs)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)
    d2h = B * K_KEYPOINTS * 2 * 4 + B * K_KEYPOINTS * 4
    e2e_u8 = None
    if args.precision == "bf16":
        gen8 = torch.Generator().manual_seed(3000 + rank)
        host_u8 = [torch.randint(0, 256, (B, H, W, 3), generator=gen8, dtype=torch.uint8).pin_memory() for _ in range(2)]
        u8_ms, u8_wall, u8_h2d = measure_e2e(host_u8)
        e2e_u8 = {"value": world * B * args.steps / (u8_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": u8_h2d,
                  "d2h_bytes_per_step": d2h, "ms_per_step": u8_ms / args.steps,
                  "note": "same loop fed (B,H,W,3) uint8 host images (cv2 layout); /255 fused into the stem load"}

    # ---------------- roofline of the dominant kernel (live CUDA-event timing per launch) ----------------
    rows = per_launch_breakdown(engine, plan)
    tc = [r for r in rows if r["algo"] == HK_CONV_TCGEN05]
    peaks = load_peaks()
    traffic, traffic_note = ncu_conv_traffic_per_step(B, H, W, K_KEYPOINTS, args.precision, launches_per_step, len(tc))
    if tc:
        tc_flops, tc_ms = sum(r["flops"] for r in tc), sum(r["ms"] for r in tc)
        achieved = tc_flops / (tc_ms * 1e-3) / 1e12
        peak = peaks["bf16_tflops"]
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 implicit GEMM, all launches of one step)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_note": traffic_note,
                "peak_source": f"{peaks['source']} burst bf16 ({peak}); sustained {peaks['bf16_tflops_sustained']}",
                "launches": len(tc), "ms_in_step": tc_ms, "ms_in_step_min_of_reps": sum(r["ms_min"] for r in tc),
                "timing": "mean launch duration: 5 back-to-back launches per CUDA event pair (eager); ms_in_step_min_of_reps = sum of single-launch minima",
                "share_of_step": tc_ms / sum(r["ms"] for r in rows)}
    else:
        ff = [r for r in rows if r["flops"] > 0]
        f, ms = sum(r["flops"] for r in ff), sum(r["ms"] for r in ff)
        roof = {"bound": "tensor", "kernel": "conv_ffma_kernel (fp32 correctness mode, CUDA cores)", "achieved": f / (ms * 1e-3) / 1e12,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": f / (ms * 1e-3) / 1e12 / peaks["bf16_tflops"], "traffic": None}
    # the HBM-bound kernels of the step against the measured copy bandwidth (informational; the headline roofline is the conv one)
    hbm_rows = [{"kernel": r["name"], "bound": "hbm", "achieved": r["bytes"] / (r["ms"] * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "frac": r["bytes"] / (r["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": r["bytes"], "ms": r["ms"]}
                for r in rows if r.get("bytes", 0) > 0]
    if args.breakdown and rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.breakdown)), exist_ok=True)
        with open(args.breakdown, "w") as f:
            json.dump({"batch": B, "rows": rows}, f, indent=1)

    default_workload = args.precision == "bf16" and (B, H, W, K_KEYPOINTS) == (64, 480, 640, 4)
    config3 = measure_config3(model, dev, rank, world, barrier, max_over_ranks) if (default_workload and not args.no_config3) else None
    train = None
    if default_workload and not args.no_train_step:
        del engine, plan
        model._engine = None
        torch.cuda.empty_cache()
        train = measure_train_step(dev, H, W, rank, world, barrier, max_over_ranks)
    if rank != 0:
        return
    gf_img = conv_flops_per_image(H, W, K_KEYPOINTS) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": f"KeypointsGauss (ResnetDilated-34, OS8) eval forward + argmax decode, batch {B} per GPU, "
                               f"{H}x{W}, K={K_KEYPOINTS}, random-init weights (BASELINE.json {'configs[1]' if (B, H, W) == (64, 480, 640) else 'configs[4]' if (H, W) == (960, 1280) else 'configs[1] at another shape'})",
                   "batch_per_gpu": B, "height": H, "width": W, "precision": args.precision,
                   "l2": f"per-step activations {B * 4.9:.0f}+ MB exceed the 126 MB L2 (no explicit flush)",
                   "parallelism": f"batch-sharded x{world}, no collective", "cuda_graph": not args.no_graph},
        "algorithmic_gflop_per_image": gf_img,
        "achieved_tflops_whole_step": gf_img * value / world / 1e3,
        "frac_of_bf16_peak_whole_step": gf_img * value / world / 1e3 / peaks["bf16_tflops"],
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps, "wall_ms_per_step": wall_ms / args.steps,
                "note": "pinned-host fp32 images -> device (model.staging_input), model.keypoints: forward + decode, keypoints + peak "
                        "values -> host; H2D double-buffered over two serving slots on a copy stream"},
        "e2e_uint8_input": e2e_u8,
        "sustained": sustained,
        "config3_4096_images": config3,
        "gpu_launches": launches_per_step * args.steps * (3 if e2e_u8 else 2),  # timed regions: device-resident loop + e2e loop(s)
        "gpu_launches_per_step": launches_per_step,
        "roofline": roof,
        "roofline_hbm_kernels": hbm_rows,
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1:   # rank 0 at N=1 only (the reference arm covers N>1)
        ref = CpuReference(H, W)
        ref.run(2)
        n = args.cpu_images or 120
        secs = ref.run(n)
        v, cores = n / secs, ref.cores
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": ref.kind,
                                "sample": f"{n} images {H}x{W}, B=1 per call, " + ("unmodified reference classes from oracle/_ref" if ref.kind == "reference"
                                          else "oracle port in the reference's as-written op order") + f" (torch CPU), {secs:.1f} s"}
    if train is not None:
        line["train_step"] = train
    print(json.dumps(line), flush=True)


def measure_config3(model, dev, rank, world, barrier, max_over_ranks):
    """BASELINE.json configs[2] as SURVEY.md §8d specifies it: 4096 synthetic 480x640 images in 64-image batches, split contiguously
    across the ranks (strong scaling), each replica loops over its shard through the public serving call (model.keypoints), no
    collective on the data path; wall time = max over ranks.  Images are generated on the device (a 4096-image fp32 set is 15 GB:
    resident in HBM, H2D excluded as in configs[1])."""
    from hulk_keypoints_b200.parallel import shard_range
    total, bs = 4096, 64
    b0, b1 = shard_range(total // bs, world, rank)          # contiguous range of 64-image batches owned by this rank
    n_local = b1 - b0
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    shard = torch.rand((max(n_local, 1) * bs, 3, 480, 640), device=dev, generator=gen)
    out = torch.empty((max(n_local, 1) * bs, K_KEYPOINTS, 2), device=dev, dtype=torch.int32)
    model.keypoints(shard[:bs])                               # plan + graph for this shape
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_local):
        yx, _ = model.keypoints(shard[i * bs:(i + 1) * bs])
        out[i * bs:(i + 1) * bs].copy_(yx)
    e1.record()
    e1.synchronize()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    checksum = int(out[: n_local * bs].to(torch.int64).sum().item())
    del shard
    torch.cuda.empty_cache()
    return {"images": total, "batch": bs, "batches_on_rank0": n_local, "seconds": ms * 1e-3, "value": total / (ms * 1e-3), "unit": UNIT,
            "scaling": "strong", "keypoint_checksum_rank0": checksum,
            "note": "4096 images split contiguously over the ranks, device-resident, model.keypoints per 64-image batch, max over ranks"}


def measure_train_step(dev, H, W, rank=0, world=1, barrier=None, max_over_ranks=None):
    """Secondary metric (BASELINE.json configs[3]; bench_train.py is the full tool): ms per training step -- Gaussian targets from labels +
    train-mode forward + BCE + backward + gradient exchange (NCCL, world > 1) + fused Adam on libhulk_sm100 kernels -- at per-GPU batch
    4 (config.py) and 32, every rank, max over ranks.  For world > 1 also: the same step with the exchange switched off (compute only),
    and the all-reduce of the flat gradient buffer timed alone, so the share of the step inside NCCL and the exposed part are measured.
    Never fails the headline line: errors are reported as text."""
    out = {"config": f"BASELINE configs[3], {world} GPU(s), per-GPU batch 4 and 32, 480x640, K=4, Adam lr 1e-4 wd 1e-4, synthetic images and labels",
           "unit": "ms/step", "n_gpus": world}
    barrier = barrier or (lambda: torch.cuda.synchronize())
    max_over_ranks = max_over_ranks or (lambda ms: ms)
    try:
        import torch.distributed as dist

        import hulk_keypoints_b200 as hk
        from hulk_keypoints_b200 import parallel, train_ops
        from hulk_keypoints_b200.optim import FusedAdam

        def timed(fn, steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                r = fn()
            e1.record(); e1.synchronize()
            barrier()
            return max_over_ranks(e0.elapsed_time(e1)) / steps, r

        for bsz in (4, 32):
            torch.manual_seed(0)
            model = hk.KeypointsGauss(4, img_height=H, img_width=W).to(dev).train()
            parallel.broadcast_model(model)
            opt = FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-4)
            g = torch.Generator().manual_seed(2000 + rank)
            img = torch.rand(bsz, 3, H, W, generator=g).to(dev)
            uv = torch.stack([torch.randint(0, W, (bsz, 4), generator=g), torch.randint(0, H, (bsz, 4), generator=g)], -1).float().to(dev)
            for _ in range(3):
                train_ops.train_step(model, opt, img, uv, sigma=8.0)
            steps = 20
            ms, loss = timed(lambda: train_ops.train_step(model, opt, img, uv, sigma=8.0), steps)
            row = {"ms_per_step": ms, "images_per_sec": world * bsz / (ms * 1e-3), "loss": float(loss.item()),
                   "gpu_launches_per_step": (model.train_engine(bsz, H, W).split_launches() if world > 1 else model.train_engine(bsz, H, W).launches) + 1}
            if world > 1:
                for _ in range(2):
                    train_ops.train_step(model, opt, img, uv, sigma=8.0, exchange=False)
                ms_local, _ = timed(lambda: train_ops.train_step(model, opt, img, uv, sigma=8.0, exchange=False), steps)
                ms_ar, _ = timed(lambda: dist.all_reduce(opt.flat_grad, op=dist.ReduceOp.SUM), steps)
                row.update({"ms_per_step_no_exchange": ms_local, "allreduce_ms_alone": ms_ar, "allreduce_bytes": opt.flat_grad.numel() * 4,
                            "pct_of_step_in_nccl": 100.0 * ms_ar / ms, "pct_of_step_exposed": 100.0 * max(ms - ms_local, 0.0) / ms})
            out[f"batch{bsz}"] = row
            del model, opt
            torch.cuda.empty_cache()
    except Exception as exc:  # noqa: BLE001 -- reported, never raised: this block is informational
        out["error"] = f"{type(exc).__name__}: {exc}"
    return out


def ncu_conv_traffic_per_step(B, H, W, K, precision, launches_per_step, conv_launches):
    """DRAM bytes (read + write) of the tcgen05 conv launches of ONE step from the newest committed per-launch ncu capture
    (profiles/*_step_per_launch_dram.json: `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` over bench.py's default
    workload, tools/gpu_profile_r2.sh).  The capture is matched to the running workload: its launch list must be a whole number of
    steps of `launches_per_step` launches with `conv_launches` conv launches each.  Returns (bytes or None, note)."""
    import glob
    if (B, H, W, K, precision) != (64, 480, 640, 4, "bf16"):
        return None, "no ncu capture committed for this workload"
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_step_per_launch_dram.json")), reverse=True):
        with open(p) as f:
            data = json.load(f)
        rows = data["rows"] if isinstance(data, dict) else data
        conv = [r for r in rows if "conv_tc" in r["kernel"]]
        if launches_per_step <= 0 or len(rows) % launches_per_step or not conv:
            continue
        n_steps = len(rows) // launches_per_step
        if len(conv) != conv_launches * n_steps:
            continue
        total = float(sum(r["dram__bytes_read.sum"] + r["dram__bytes_write.sum"] for r in conv)) / n_steps
        return total, (f"DRAM bytes read+written by the {conv_launches} conv launches of one step (ncu, profiles/{os.path.basename(p)}, "
                       f"{n_steps} step(s) captured); algorithmic activation traffic of those launches: in+out+residual of every conv")
    return None, "no committed per-launch ncu capture matches this build's launch sequence"


def main():
    global K_KEYPOINTS
    args = parse_args()
    K_KEYPOINTS = args.keypoints
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    if args.impl == "torch_gpu":
        run_torch_gpu(args, rank, 1, local_rank)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
