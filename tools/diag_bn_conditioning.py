"""Conditioning of the train-mode BatchNorm inputs of the trained fixture: r = |mean| / std per channel.

    python tools/diag_bn_conditioning.py [fixture]        (default k4_480x640; trains the fixture on cuda:0)

The BatchNorm kernels form their variance as E[y^2] - mean^2 from fp32 partial sums, so their relative error grows as (1 + r^2) * 2^-24
per added row.  This trains F-trn (synth.train_fixture), then runs the CPU oracle's train-mode forward at the fixture's batch and
resolution on disc images and on uniform-noise images with oracle.keypoints_oracle._bn hooked, and prints the largest r of every
BatchNorm input.  tests/test_gpu_bn_reference.py sizes its "realistic" conditioning range from the largest value printed here."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hulk_keypoints_b200 import synth  # noqa: E402
from oracle import keypoints_oracle as O  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "k4_480x640"
cfg = synth.FIXTURES[name]
sd, losses = synth.train_fixture(name)
print(f"{name}: trained, loss {losses[0]:.4f} -> {losses[-1]:.5f}", flush=True)

rows = {}
orig = O._bn


def hooked(sd_, bn_name, x, train, new_stats):
    x64 = x.double()
    m = x64.mean((0, 2, 3))
    s = x64.var((0, 2, 3), unbiased=False).sqrt()
    r = m.abs() / s.clamp_min(1e-30)
    rows.setdefault(bn_name, []).append((x.shape[1], float(r.median()), float(r.max()), int((s < 1e-6).sum())))
    return orig(sd_, bn_name, x, train, new_stats)


O._bn = hooked
B, H, W, K = cfg["B"], cfg["H"], cfg["W"], cfg["K"]
images = {"discs": synth.disc_batch(torch.Generator().manual_seed(7), B, H, W, K)[0].float(),
          "uniform": torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(8))}
worst = 0.0
for kind, x in images.items():
    rows.clear()
    O.forward(sd, x, K, train=True, new_stats={})
    print(f"--- {kind} images, {B}x{H}x{W}")
    for bn_name, recs in rows.items():
        for c, med, mx, zero in recs:
            print(f"{bn_name:26s} C={c:4d}  median r {med:6.3f}  max r {mx:7.3f}  zero-variance channels {zero}")
            worst = max(worst, mx)
print(f"largest r over every BatchNorm input: {worst:.3f}")
