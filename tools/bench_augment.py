"""The training-batch augmentation kernels alone, and the train step with and without an augmenter, timed with CUDA events.

    python tools/bench_augment.py [--iters 200] [--rounds 3] [--steps 50]

Kernels: `hk_augment_pick` + `hk_augment_images` (one augmenter call's device work, parameter tables already on the device) at
B = 4, 32 and 64 x 480x640, for four configurations: "full" (rotation, scale, translation, contrast, brightness, gain, noise),
"photometric" (identity geometry, no noise: the pure streaming case), "warp" (geometry only) and "noise" (noise only).  Each timing is
`iters` launch pairs between two CUDA events, 20 warm-up pairs first; successive launches rotate over several input/output buffer pairs totalling more than 3x the 126 MB L2, so
every launch reads its input from HBM.  GB/s counts the 24 B per pixel floor (12 B read + 12 B written), so gather overfetch under
rotation shows as a lower rate.  "host ms" is a whole `KeypointAugment.__call__` (parameter draw on the CPU, pinned copy, both
launches) measured on the host clock over `iters` calls followed by one synchronise.
Train step: `train_ops.train_step` with FusedAdam at B = 4 and 32 x 480x640, `augment=None` and the full augmenter alternated in
one process, `steps` steps per timing, `rounds` rounds; ms per step from CUDA events.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hulk_keypoints_b200 as hk  # noqa: E402
from hulk_keypoints_b200 import ops, train_ops  # noqa: E402
from hulk_keypoints_b200.augment import KeypointAugment  # noqa: E402
from hulk_keypoints_b200.optim import FusedAdam  # noqa: E402

H, W, K = 480, 640, 4
L2_BYTES = 126 * 2 ** 20
CONFIGS = {
    "full": dict(rotate=30.0, scale=(0.8, 1.2), translate=0.1, brightness=0.2, contrast=(0.7, 1.3), channel_gain=0.15, noise_std=0.03),
    "photometric": dict(brightness=0.2, contrast=(0.7, 1.3), channel_gain=0.15),
    "warp": dict(rotate=30.0, scale=(0.8, 1.2), translate=0.1),
    "noise": dict(noise_std=0.03),
}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] + " | " + out[1 + torch.cuda.current_device()] if len(out) > 1 else "power limit unknown"
    except (OSError, subprocess.SubprocessError):
        return "power limit unknown"


def bench_kernels(B, name, iters, rounds):
    dev = torch.device("cuda")
    bytes_img = B * 3 * H * W * 4
    pairs = max(2, -(-3 * L2_BYTES // (2 * bytes_img)))
    g = torch.Generator(device="cuda").manual_seed(B)
    ins = [torch.rand(B, 3, H, W, device=dev, generator=g) for _ in range(pairs)]
    outs = [torch.empty_like(ins[0]) for _ in range(pairs)]
    uv = torch.stack([torch.rand(B, K, device=dev, generator=g) * (W - 1), torch.rand(B, K, device=dev, generator=g) * (H - 1)], -1)
    uv_out = torch.empty_like(uv)
    aug = KeypointAugment(**CONFIGS[name], seed=1)
    p = aug.draw(B, H, W)
    fwd, inv, photo = p.fwd.to(dev), p.inv.to(dev), p.photo.to(dev)
    pick = torch.empty(B, device=dev, dtype=torch.int32)

    def launch(i):
        ops.augment_pick(fwd, uv, H, W, uv_out=uv_out, pick=pick)
        ops.augment_images(ins[i % pairs], inv, pick, photo, aug.noise_std, p.key, out=outs[i % pairs])

    for i in range(20):
        launch(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(rounds):
        e0.record()
        for i in range(iters):
            launch(i)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / iters)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(iters):
        aug(ins[i % pairs], uv, out=outs[i % pairs], uv_out=uv_out)
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - t0) * 1e3 / iters
    best = min(ms)
    return {"case": "kernels", "config": name, "B": B, "ms_per_call": [round(t, 4) for t in ms],
            "GBps_best_vs_24B_per_px": round(24 * B * H * W / (best * 1e-3) / 1e9, 1), "picked_fraction": float((pick >= 0).float().mean()),
            "host_ms_per_call": round(host_ms, 4), "buffer_pairs": pairs, "rotated_bytes_MB": round(2 * pairs * bytes_img / 2 ** 20)}


def bench_train(B, steps, rounds):
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = hk.KeypointsGauss(K, img_height=H, img_width=W).to(dev).train()
    opt = FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-4)
    g = torch.Generator().manual_seed(2000)
    img = torch.rand(B, 3, H, W, generator=g).to(dev)
    uv = torch.stack([torch.randint(40, W - 40, (B, K), generator=g), torch.randint(40, H - 40, (B, K), generator=g)], -1).float().to(dev)
    aug = KeypointAugment(**CONFIGS["full"], seed=3)
    arms = {"augment=None": None, "augment=full": aug}
    for a in arms.values():
        for _ in range(5):
            train_ops.train_step(model, opt, img, uv, sigma=8.0, augment=a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, a in arms.items():
            e0.record()
            for _ in range(steps):
                train_ops.train_step(model, opt, img, uv, sigma=8.0, augment=a)
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / steps)
    base = min(ms["augment=None"])
    return [{"case": "train_step", "B": B, "arm": k, "ms_per_step": [round(t, 4) for t in v],
             "best_over_augment_none": round(min(v) / base, 4)} for k, v in ms.items()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_augment.py needs a CUDA device")
    print(f"GPU: {torch.cuda.get_device_name()} | {gpu_info()}")
    print(f"kernels: {args.iters} launch pairs per timing, {args.rounds} timings; inputs rotate over buffer pairs totalling > 3x the "
          f"126 MB L2 (read from HBM); GB/s against the 24 B/pixel floor", flush=True)
    for B in (4, 32, 64):
        for name in CONFIGS:
            print(json.dumps(bench_kernels(B, name, args.iters, args.rounds)), flush=True)
    for B in (4, 32):
        for row in bench_train(B, args.steps, args.rounds):
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
