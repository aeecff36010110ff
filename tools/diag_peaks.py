"""Stand-alone timing of hk_peak_decode against hk_argmax_decode and a torch formulation (max_pool2d(2r+1, stride 1, padding r)
equality mask + threshold, then topk over H*W), in one process.  CUDA events around `iters` calls rotating over two heatmap buffers
(each larger than the 126 MB L2); GB/s = heatmap bytes / mean call time.  Two kinds of maps: uniform noise (every tile holds
candidates: the worst case) and sigmoid-like maps (the max of 6 Gaussian blobs of sigma 8 per channel, what a trained model emits:
most tiles hold no pixel above the threshold).  Before timing, each configuration is checked bit for bit against the numpy reference
(tests/peaks_ref.py) on a spread of maps.  Prints the card name and power limit.
    python tools/diag_peaks.py [--iters 20]"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from hulk_keypoints_b200 import ops  # noqa: E402
from peaks_ref import peak_decode_ref  # noqa: E402

SHAPES = [(64, 4, 480, 640), (16, 32, 960, 1280)]
RS, NS, THR = (1, 4, 16), (16, 256), 0.5


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] + " | " + out[1 + torch.cuda.current_device()] if len(out) > 1 else "power limit unknown"
    except (OSError, subprocess.SubprocessError):
        return "power limit unknown"


def blobs(B, K, H, W, seed, n=6):
    g = torch.Generator().manual_seed(seed)
    heat = torch.zeros((B, K, H, W), device="cuda")
    for _ in range(n):
        uv = torch.stack([torch.rand(B, K, generator=g) * (W - 1), torch.rand(B, K, generator=g) * (H - 1)], -1).cuda()
        torch.maximum(heat, ops.gauss_targets(uv, H, W, 8.0, out_dtype=torch.float32), out=heat)
    return heat


def torch_peaks(heat, N, thr, r):
    B, K, H, W = heat.shape
    mx = F.max_pool2d(heat, 2 * r + 1, stride=1, padding=r)
    cand = torch.where((heat == mx) & (heat >= thr), heat, torch.full((), -float("inf"), device=heat.device))
    return cand.view(B * K, H * W).topk(N, dim=1)


def timed(fn, heats, iters):
    for k in range(4):
        fn(heats[k & 1])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(iters):
        fn(heats[k & 1])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3   # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    print(f"{torch.cuda.get_device_name()} | {gpu_info()}")
    print(f"{'shape':>18} {'maps':>6} {'r':>3} {'N':>4} {'peaks us':>9} {'GB/s':>6} {'argmax us':>9} {'GB/s':>6} {'x argmax':>8} "
          f"{'torch us':>9} {'x torch':>7} {'mean count':>10}")
    for B, K, H, W in SHAPES:
        nbytes = B * K * H * W * 4
        for kind in ("noise", "blobs"):
            if kind == "noise":
                heats = [torch.rand((B, K, H, W), device="cuda", generator=torch.Generator(device="cuda").manual_seed(s)) for s in (1, 2)]
            else:
                heats = [blobs(B, K, H, W, s) for s in (1, 2)]
            yx = torch.empty((B, K, 2), device="cuda", dtype=torch.int32)
            mv = torch.empty((B, K), device="cuda")
            aws = torch.empty(ops.argmax_workspace_bytes(B, K, H, W), device="cuda", dtype=torch.uint8)
            t_arg = timed(lambda h: ops.argmax_decode(h, yx, mv, aws), heats, args.iters)
            sel = np.unique(np.linspace(0, B * K - 1, 6).astype(np.int64))
            for r in RS:
                for N in NS:
                    bufs = (torch.empty((B, K, N, 2), device="cuda", dtype=torch.int32), torch.empty((B, K, N), device="cuda"),
                            torch.empty((B, K), device="cuda", dtype=torch.int32),
                            torch.empty(ops.peak_workspace_bytes(B, K, H, W, N, r), device="cuda", dtype=torch.uint8))

                    def run(h):
                        return ops.peak_decode(h, N, THR, r, *bufs)

                    pyx, pscore, pcount = run(heats[0])
                    ref = peak_decode_ref(heats[0].view(B * K, H, W)[torch.as_tensor(sel, device="cuda")].cpu().numpy(), N, THR, r)
                    got = (pyx.view(B * K, N, 2).cpu().numpy()[sel], pscore.view(B * K, N).cpu().numpy()[sel],
                           pcount.view(-1).cpu().numpy()[sel])
                    assert all(np.array_equal(a, b) for a, b in zip(got, ref)), f"mismatch {kind} {(B, K, H, W)} r={r} N={N}"
                    mean_count = float(pcount.float().mean())
                    t_pk = timed(run, heats, args.iters)
                    t_torch = timed(lambda h: torch_peaks(h, N, THR, r), heats, max(4, args.iters // 4))
                    print(f"{kind:>5} {B}x{K}x{H}x{W:<5} {B * K:6d} {r:3d} {N:4d} {t_pk:9.1f} {nbytes / t_pk / 1e3:6.0f} {t_arg:9.1f} "
                          f"{nbytes / t_arg / 1e3:6.0f} {t_pk / t_arg:8.2f} {t_torch:9.1f} {t_torch / t_pk:7.1f} {mean_count:10.1f}",
                          flush=True)
            del heats
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
