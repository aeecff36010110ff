"""The fused Adam update alone: hk_adam_step against hk_adam_step_segments at the model's size, timed with CUDA events.

    python tools/bench_adam.py [--lib PATH ...] [--iters 200] [--rounds 3]

Buffers are the 21 797 672 parameters of KeypointsGauss(4) laid out as FusedAdam lays them out (each tensor on a 16-byte boundary), four
fp32 buffers of 87 MB each (349 MB, well past the 126 MB L2, so every launch streams from HBM).  Cases:
  hk_adam_step          the single-hyperparameter entry point
  segments=1            one segment (FusedAdam with one parameter group)
  segments=3            the backbone up to layer2 / layer3+layer4 / fc at three learning rates
  segments=110          one segment per parameter tensor (groups alternating along the model, e.g. no decay on BatchNorm)
Each case: 20 warm-up launches, then `iters` launches between two CUDA events, repeated `rounds` times alternating the cases (and the
libraries, when several `--lib` are given, e.g. another build for an A/B; a library without hk_adam_step_segments is timed on
hk_adam_step only).  GB/s counts the algorithmic 28 B per parameter (16 B read + 12 B written): 0.61 GB per launch."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hulk_keypoints_b200 as hk  # noqa: E402
from hulk_keypoints_b200 import _lib  # noqa: E402
from hulk_keypoints_b200.optim import build_segments, flat_offsets  # noqa: E402


def load(path):
    h = C.CDLL(path)
    h.hk_adam_step.restype = C.c_int
    h.hk_adam_step.argtypes = [C.c_void_p] * 4 + [C.c_longlong] + [C.c_float] * 5 + [C.c_int, C.c_void_p]
    has_seg = hasattr(h, "hk_adam_step_segments")
    if has_seg:
        h.hk_adam_step_segments.restype = C.c_int
        h.hk_adam_step_segments.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.POINTER(_lib.HkAdamSegment), C.c_int, C.c_void_p]
    return h, has_seg


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="library to time (repeatable; default: the in-tree build)")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_adam.py needs a CUDA device")
    libs = args.lib or [_lib.LIB_PATH]
    numels = [p.numel() for p in hk.KeypointsGauss(4).parameters()]
    offs, n = flat_offsets(numels)
    run4 = [(o // 4, (o + (k + 3) // 4 * 4) // 4) for o, k in zip(offs, numels)]
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    p, gr, m = (torch.randn(n, device=dev, generator=g) * 0.01 for _ in range(3))
    v = torch.rand(n, device=dev, generator=g) * 1e-4
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    adam = (1e-4, 0.9, 0.999, 1e-8, 1e-4, False)
    # three groups: up to layer2, layer3 + layer4, fc (the last two tensors)
    names = [k for k, _ in hk.KeypointsGauss(4).named_parameters()]
    first_l3 = next(i for i, k in enumerate(names) if ".layer3." in k)
    split3 = [0 if i < first_l3 else (2 if i >= len(names) - 2 else 1) for i in range(len(names))]
    tables = {
        1: build_segments([(0, n // 4, 0, 1)], [adam]),
        3: build_segments([(a, b, split3[i], 1) for i, (a, b) in enumerate(run4)], [adam, (3e-4,) + adam[1:], (1e-3,) + adam[1:]]),
        len(run4): build_segments([(a, b, i % 2, 1) for i, (a, b) in enumerate(run4)], [adam, adam[:4] + (0.0, False)]),
    }
    handles = [(path, *load(path)) for path in libs]
    cases = []
    for path, h, has_seg in handles:
        cases.append((path, "hk_adam_step", lambda h=h: h.hk_adam_step(p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), n,
                                                                        1e-4, 0.9, 0.999, 1e-8, 1e-4, 1, stream)))
        if has_seg:
            for k, rows in tables.items():
                tab = (_lib.HkAdamSegment * len(rows))(*(_lib.HkAdamSegment(*r) for r in rows))
                cases.append((path, f"segments={len(rows)}",
                              lambda h=h, tab=tab, k=len(rows): h.hk_adam_step_segments(p.data_ptr(), gr.data_ptr(), m.data_ptr(),
                                                                                        v.data_ptr(), n, tab, k, stream)))
    info = gpu_info()
    print(f"GPU: {info}")
    print(f"n = {n} floats ({len(numels)} tensors), {28 * n / 1e9:.3f} GB algorithmic traffic per launch, {args.iters} launches per timing")
    times = {(c[0], c[1]): [] for c in cases}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for path, name, fn in cases:
            for _ in range(20):
                assert fn() == 0, name
            e0.record()
            for _ in range(args.iters):
                fn()
            e1.record()
            e1.synchronize()
            times[(path, name)].append(e0.elapsed_time(e1) / args.iters)
    for (path, name), ts in times.items():
        best = min(ts)
        row = {"lib": path, "case": name, "ms_per_launch": [round(t, 5) for t in ts], "GBps_best": round(28 * n / (best * 1e-3) / 1e9, 1),
               "gpu": info}
        print(json.dumps(row))


if __name__ == "__main__":
    main()
