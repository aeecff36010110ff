"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

    python oracle/make_golden.py

Imports the reference through `oracle/reference_loader.py`, runs its own classes / call sites on
seeded inputs and writes small fixtures.  Weights are never stored (87 MB): they are the seeded
random init of `src/resnet.py:155-161`, which `oracle.keypoints_oracle.init_state_dict` reproduces
bit for bit; a SHA-256 of every tensor is stored so a box whose torch RNG differs is detected.
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import keypoints_oracle as O  # noqa: E402
from oracle import reference_loader as RL  # noqa: E402

warnings.filterwarnings("ignore")
OUT = os.path.join(ROOT, "tests", "golden")


def digest(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def rand_img(seed, b, h, w):
    return torch.rand(b, 3, h, w, generator=torch.Generator().manual_seed(seed))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(O.GOLDEN_CPU_THREADS)
    meta = {"torch": torch.__version__, "reference": "vainaviv/hulk-keypoints", "cases": {}}
    arrays = {}

    # ---- weights: digest of the reference's seeded init ----
    for seed in (0, 1):
        m = RL.build_reference_model(seed)
        meta[f"weights_sha256_seed{seed}"] = digest(m.state_dict())

    model = RL.build_reference_model(0)

    # ---- case raw_small: F-raw, eval(), 1x3x64x96 ----
    model.eval()
    x = rand_img(5, 1, 64, 96)
    with torch.no_grad():
        y = model(x)
    arrays["raw_small_heat"] = y.numpy()
    meta["cases"]["raw_small"] = {"weights_seed": 0, "input_seed": 5, "shape": [1, 3, 64, 96], "mode": "eval"}

    # ---- case raw_train: F-raw, train-mode BN (as the reference scripts literally run), 2x3x64x96 ----
    model = RL.build_reference_model(0)
    model.train()
    x = rand_img(6, 2, 64, 96)
    with torch.no_grad():
        y = model(x)
    arrays["raw_train_heat"] = y.numpy()
    rs = model.state_dict()
    arrays["raw_train_bn1_running_mean"] = rs[O.PREFIX + "bn1.running_mean"].numpy()
    arrays["raw_train_l4_running_var"] = rs[O.PREFIX + "layer4.2.bn2.running_var"].numpy()
    meta["cases"]["raw_train"] = {"weights_seed": 0, "input_seed": 6, "shape": [2, 3, 64, 96], "mode": "train"}

    # ---- case cal_small: F-cal weights loaded INTO the reference model, eval(), 1x3x96x128 ----
    sd0 = O.init_state_dict(0)
    sd_cal = O.calibrate_bn(sd0, [rand_img(100 + i, 2, 96, 128) for i in range(2)])
    model = RL.build_reference_model(0)
    model.load_state_dict(sd_cal)
    model.eval()
    x = rand_img(7, 1, 96, 128)
    with torch.no_grad():
        y = model(x)
    arrays["cal_small_heat"] = y.numpy()
    meta["cases"]["cal_small"] = {"weights_seed": 0, "calib_seeds": [100, 101], "calib_shape": [2, 3, 96, 128],
                                  "input_seed": 7, "shape": [1, 3, 96, 128], "mode": "eval"}
    meta["weights_sha256_cal"] = digest(sd_cal)

    # ---- case raw_full: config.py resolution, eval, subsampled heatmap + decode + checksums ----
    model = RL.build_reference_model(0)
    model.eval()
    x = rand_img(1000, 1, 480, 640)
    with torch.no_grad():
        y = model(x).numpy()
    arrays["raw_full_heat_sub8"] = y[:, :, ::8, ::8].copy()
    arrays["raw_full_heat_rows"] = y[:, :, [0, 239, 479], :].copy()
    arrays["raw_full_argmax_yx"] = np.array(
        [[np.unravel_index(y[0][k].argmax(), y[0][k].shape) for k in range(4)]], dtype=np.int64)
    arrays["raw_full_sum_f64"] = y.astype(np.float64).sum(axis=(2, 3))
    meta["cases"]["raw_full"] = {"weights_seed": 0, "input_seed": 1000, "shape": [1, 3, 480, 640], "mode": "eval"}

    # ---- gaussian targets from the reference's gauss_2d_batch (dataset.py:36-44) ----
    ds, _ = RL.reference_modules()
    labels = np.array([[10.0, 20.0], [320.5, 240.25], [0.0, 0.0], [639.0, 479.0]], dtype=np.float64)
    g = ds.gauss_2d_batch(640, 480, 8, torch.from_numpy(labels[:, 0].copy()), torch.from_numpy(labels[:, 1].copy()))
    g = g.numpy()
    assert g.dtype == np.float64
    arrays["gauss_labels"] = labels
    arrays["gauss_full_sub4"] = g[:, ::4, ::4].copy()
    arrays["gauss_full_rows"] = g[:, [0, 20, 240, 479], :].copy()
    arrays["gauss_full_sum"] = g.sum(axis=(1, 2))
    arrays["gauss_full_nnz"] = (g != 0).sum(axis=(1, 2))
    labels_s = np.array([[3.0, 5.0], [31.5, 20.25], [0.0, 0.0], [63.0, 47.0]], dtype=np.float64)
    gs = ds.gauss_2d_batch(64, 48, 3, torch.from_numpy(labels_s[:, 0].copy()), torch.from_numpy(labels_s[:, 1].copy())).numpy()
    arrays["gauss_small_labels"] = labels_s
    arrays["gauss_small"] = gs

    # ---- BCE forward/backward at the reference's call site (train.py:21,25,35) ----
    gen = torch.Generator().manual_seed(11)
    z = (torch.randn(2, 4, 48, 64, generator=gen) * 6.0)
    z[0, 0, 0, 0] = 40.0   # sigmoid saturates to exactly 1.0f
    z[0, 0, 0, 1] = -120.0  # sigmoid underflows to 0
    z.requires_grad_(True)
    t = torch.from_numpy(np.stack([gs, gs[::-1].copy()]))
    p = torch.sigmoid(z)
    loss = torch.nn.BCELoss()(p.double(), t)
    loss.backward()
    arrays["bce_logits"] = z.detach().numpy()
    arrays["bce_pred"] = p.detach().numpy()
    arrays["bce_target"] = t.numpy()
    arrays["bce_loss"] = np.array(loss.item(), dtype=np.float64)
    arrays["bce_grad_logits"] = z.grad.numpy()

    np.savez_compressed(os.path.join(OUT, "golden_v1.npz"), **arrays)
    with open(os.path.join(OUT, "golden_v1.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    sz = os.path.getsize(os.path.join(OUT, "golden_v1.npz"))
    print(f"wrote {len(arrays)} arrays, {sz/1e6:.2f} MB")


if __name__ == "__main__":
    main()
