"""CPU: pin the oracle (oracle/keypoints_oracle.py) against golden vectors produced by the UNMODIFIED
reference (oracle/make_golden.py, run in the build container) and against known-answer cases (SURVEY.md §8c)."""
import warnings

import numpy as np
import pytest
import torch

from conftest import rand_img, sd_digest
from oracle import keypoints_oracle as O

warnings.filterwarnings("ignore")


@pytest.fixture(autouse=True)
def golden_cpu_threads():
    """Run each case on the CPU thread count the goldens were recorded with (see O.GOLDEN_CPU_THREADS)."""
    n = torch.get_num_threads()
    torch.set_num_threads(O.GOLDEN_CPU_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="module")
def sd0(golden):
    _, meta = golden
    sd = O.init_state_dict(0)
    if sd_digest(sd) != meta["weights_sha256_seed0"]:
        pytest.skip("torch CPU RNG on this host does not reproduce the golden weights (different ISA path)")
    return sd


def test_seeded_init_matches_reference_digest(golden):
    _, meta = golden
    for seed in (0, 1):
        sd = O.init_state_dict(seed)
        assert len(sd) == 218
        assert sd[O.PREFIX + "fc.weight"].shape == (1000, 512, 1, 1)
        assert sd_digest(sd) == meta[f"weights_sha256_seed{seed}"]


def test_network_spec_dilations():
    stem, blocks, fc = O.network_spec()
    assert len(blocks) == 16 and (stem.k, stem.stride, stem.pad) == (7, 2, 3)
    by_name = {b.conv1.name: b for b in blocks}
    assert by_name["layer2.0.conv1"].conv1.stride == 2 and by_name["layer2.0.conv1"].conv1.dil == 1
    # dilation applies to block 0 of the stage too (differs from torchvision)
    assert by_name["layer3.0.conv1"].conv1.dil == 2 and by_name["layer3.0.conv1"].conv1.pad == 2
    assert by_name["layer4.0.conv1"].conv1.dil == 4 and by_name["layer4.0.conv1"].conv1.stride == 1
    assert by_name["layer4.0.conv1"].down.dil == 1 and by_name["layer4.0.conv1"].down.k == 1
    assert abs(O.conv_flops_per_image(480, 640, 4) / 1e9 - 211.91) < 0.01
    assert abs(O.conv_flops_per_image(960, 1280, 4) / 1e9 - 847.66) < 0.01


def test_eval_forward_small_bit_equal(golden, sd0):
    arrays, meta = golden
    c = meta["cases"]["raw_small"]
    x = rand_img(c["input_seed"], *[c["shape"][0], c["shape"][2], c["shape"][3]])
    y = O.forward(sd0, x, 4, as_written=True).numpy()
    assert np.array_equal(y, arrays["raw_small_heat"])
    y2 = O.forward(sd0, x, 4).numpy()  # fc rows sliced first: same arithmetic, other oneDNN kernel
    assert np.abs(y2 - arrays["raw_small_heat"]).max() < 2e-6


def test_train_mode_forward_and_running_stats(golden, sd0):
    arrays, meta = golden
    c = meta["cases"]["raw_train"]
    x = rand_img(c["input_seed"], c["shape"][0], c["shape"][2], c["shape"][3])
    stats = {}
    y = O.forward(sd0, x, 4, train=True, new_stats=stats, as_written=True).numpy()
    assert np.abs(y - arrays["raw_train_heat"]).max() < 1e-6
    assert np.array_equal(stats[O.PREFIX + "bn1.running_mean"].numpy(), arrays["raw_train_bn1_running_mean"])
    assert np.array_equal(stats[O.PREFIX + "layer4.2.bn2.running_var"].numpy(), arrays["raw_train_l4_running_var"])


def test_calibrated_fixture(golden, sd0):
    arrays, meta = golden
    c = meta["cases"]["cal_small"]
    b, _, h, w = c["calib_shape"]
    sd_cal = O.calibrate_bn(sd0, [rand_img(s, b, h, w) for s in c["calib_seeds"]])
    assert sd_digest(sd_cal) == meta["weights_sha256_cal"]
    x = rand_img(c["input_seed"], c["shape"][0], c["shape"][2], c["shape"][3])
    y = O.forward(sd_cal, x, 4, as_written=True).numpy()
    assert np.array_equal(y, arrays["cal_small_heat"])
    assert 0.05 < y.min() and y.max() < 0.95  # un-saturated heatmaps: meaningful parity case


def test_full_resolution_case(golden, sd0):
    arrays, meta = golden
    c = meta["cases"]["raw_full"]
    x = rand_img(c["input_seed"], 1, 480, 640)
    y = O.forward(sd0, x, 4).numpy()
    assert y.shape == (1, 4, 480, 640)
    ref_sub = arrays["raw_full_heat_sub8"]
    rel = np.abs(y[:, :, ::8, ::8] - ref_sub) / np.maximum(np.abs(ref_sub), 1e-30)
    assert rel.max() < 1e-4
    assert np.abs(y[:, :, [0, 239, 479], :] - arrays["raw_full_heat_rows"]).max() < 1e-5
    assert np.allclose(y.astype(np.float64).sum(axis=(2, 3)), arrays["raw_full_sum_f64"], rtol=1e-6)


def test_gauss_targets_bit_equal(golden):
    arrays, _ = golden
    g = O.gauss_targets(arrays["gauss_small_labels"][None], 48, 64, 3)[0]
    assert g.dtype == np.float64 and np.array_equal(g, arrays["gauss_small"])
    gf = O.gauss_targets(arrays["gauss_labels"][None], 480, 640, 8)[0]
    assert np.array_equal(gf[:, ::4, ::4], arrays["gauss_full_sub4"])
    assert np.array_equal(gf[:, [0, 20, 240, 479], :], arrays["gauss_full_rows"])
    assert np.array_equal((gf != 0).sum(axis=(1, 2)), arrays["gauss_full_nnz"])
    assert np.allclose(gf.sum(axis=(1, 2)), arrays["gauss_full_sum"], rtol=1e-14)


def test_gauss_known_answers():
    g = O.gauss_targets(np.array([[[100.0, 50.0], [320.5, 240.25]]]), 480, 640, 8)[0]
    assert g[0, 50, 100] == 1.0
    assert g[0, 50, 108] == float(np.float32(np.exp(np.float32(-0.5))))
    assert abs(g[1].max() - 0.99756) < 1e-5  # fractional label never reaches 1
    assert g[0, 400, 600] == 0.0  # fp32 exp underflows far from the keypoint


def test_bce_matches_reference_call_site(golden):
    arrays, _ = golden
    loss = O.bce_loss(arrays["bce_pred"], arrays["bce_target"])
    assert abs(loss - float(arrays["bce_loss"])) <= 1e-14 * abs(float(arrays["bce_loss"]))
    g = O.bce_grad_logits(arrays["bce_pred"], arrays["bce_target"])
    assert np.array_equal(g, arrays["bce_grad_logits"])


def test_bce_known_answers():
    p = np.array([1.0, 0.5, 0.0, 0.25], dtype=np.float32)
    t = np.array([0.25, 0.5, 0.0, 1.0], dtype=np.float64)
    # p == 1, t < 1 -> 100*(1-t);  p == t == .5 -> ln 2;  p == 0, t == 0 -> 0;  p=.25,t=1 -> -ln .25
    expect = (100 * 0.75 + np.log(2.0) + 0.0 - np.log(0.25)) / 4
    assert abs(O.bce_loss(p, t) - expect) < 1e-12
    g = O.bce_grad_logits(p, t)
    assert g[0] == 0.0 and g[1] == 0.0 and g[2] == 0.0  # saturated / matched elements carry no gradient


def test_argmax_decode_semantics(golden):
    arrays, _ = golden
    h = np.zeros((2, 3, 5, 7), dtype=np.float32)
    assert (O.argmax_decode(h) == 0).all()  # constant map -> (0, 0)
    h[0, 1, 2, 3] = h[0, 1, 4, 1] = 2.0     # two equal maxima -> lower flat index
    h[1, 2, 4, 6] = np.nan                  # NaN wins (numpy semantics)
    d = O.argmax_decode(h)
    assert tuple(d[0, 1]) == (2, 3) and tuple(d[1, 2]) == (4, 6)
    sub = arrays["raw_small_heat"]
    for k in range(4):
        assert tuple(O.argmax_decode(sub)[0, k]) == np.unravel_index(sub[0, k].argmax(), sub[0, k].shape)


def test_bilinear_restatement_corners():
    lo = torch.randn(1, 2, 6, 8, generator=torch.Generator().manual_seed(3))
    up = torch.nn.functional.interpolate(lo, size=(48, 64), mode="bilinear", align_corners=True).numpy()
    mine = O.bilinear_upsample_ac(lo.numpy(), 48, 64)
    assert np.abs(up - mine).max() < 1e-6
    assert mine[0, 0, 0, 0] == lo[0, 0, 0, 0] and mine[0, 1, 47, 63] == lo[0, 1, 5, 7]


def _prediction_golden_maps():
    """The seeded maps of oracle/make_golden_prediction.py (same generator, same order)."""
    rng = np.random.RandomState(7)
    out = []
    for h, w in ((5, 7), (12, 12), (48, 64), (33, 17)):
        d = rng.rand(h, w).astype(np.float32)
        d[rng.randint(h), rng.randint(w)] += 6.0
        out.append(d)
    out.append((np.eye(9, 13, dtype=np.float32) * 3).astype(np.float32))
    return out


def test_soft_expectation_matches_reference_golden():
    """oracle.soft_expectation and the product's Prediction.expectation / softmax against outputs of the unmodified reference class
    (tests/golden/prediction_v1.json; reference src/prediction.py:26-38, transposed-ravel quirk included)."""
    import json
    import os

    import hulk_keypoints_b200 as hk

    with open(os.path.join(os.path.dirname(__file__), "golden", "prediction_v1.json")) as f:
        cases = json.load(f)["cases"]
    pred = hk.Prediction(hk.KeypointsGauss(4), 4, 480, 640, use_cuda=False)
    maps = _prediction_golden_maps()
    assert len(maps) == len(cases)
    for d, c in zip(maps, cases):
        assert list(d.shape) == c["shape"]
        assert O.soft_expectation(d) == c["expectation"]
        assert pred.expectation(d) == c["expectation"]
        sm = pred.softmax(d.ravel().astype(np.float64))
        assert abs(sm.max() - c["softmax_max"]) < 1e-15 and abs(sm.sum() - c["softmax_sum"]) < 1e-15


def test_round2_goldens_dataset_normalize_expectation(golden2):
    """Oracle restatements against outputs of the unmodified reference (tests/golden/golden_v2.npz, oracle/make_golden_v2.py):
    KeypointsDataset's label clipping and Gaussians (dataset.py:63-66,72-76), normalize_dist (dataset.py:33-34,42-44) and
    Prediction.expectation before its int() (prediction.py:26-38)."""
    g = golden2
    for i in range(2):
        clipped = O.clip_labels(g[f"ds_raw_label_{i}"], 48, 64)
        assert np.array_equal(clipped, g[f"ds_clipped_label_{i}"])
        assert np.array_equal(O.gauss_targets(clipped[None].astype(np.float32), 48, 64, 3.0)[0], g[f"ds_gauss_{i}"])
        img = g[f"ds_img_{i}"]
        assert img.dtype == np.float32 and img.shape == (3, 48, 64) and 0.0 <= img.min() and img.max() <= 1.0
    gn = O.l1_normalize_dim1(O.gauss_targets(g["gauss_norm_uv"][None].astype(np.float32), 48, 64, 3.0)[0].astype(np.float32))
    assert np.allclose(gn, g["gauss_norm"], rtol=2e-6, atol=1e-12)
    colsum = g["gauss_norm"].sum(axis=1)
    assert np.allclose(colsum[:, 5:16][0], 1.0, atol=1e-5)                   # (k, :, w) columns near a keypoint sum to one
    for i in range(6):
        raw = O.soft_expectation_raw(g[f"exp_map_{i}"])
        assert np.array_equal(raw, g[f"exp_raw_{i}"])
        assert O.soft_expectation(g[f"exp_map_{i}"]) == list(g[f"exp_int_{i}"])


def test_train_step_loss_and_grads_match_reference_golden(golden2, sd0):
    """oracle.train_step_loss_and_grads (the checker of the GPU TrainEngine tests) against autograd through the UNMODIFIED reference
    modules (train.py:18-26,35; golden_v2.npz): loss bit-equal, gradients to 1e-5 of each tensor's scale, dead fc rows exactly 0."""
    g = golden2
    x = torch.rand(2, 3, 64, 96, generator=torch.Generator().manual_seed(3))
    loss, grads, stats = O.train_step_loss_and_grads(sd0, x, g["step_uv"], 4, 8.0)
    assert abs(loss - float(g["step_loss"])) <= 1e-12 * abs(loss)
    for key in g:
        if not key.startswith("step_grad_") or key.endswith("_sum") or key.endswith("_live") or key.endswith("_sub"):
            continue
        ref = g[key]
        got = grads[O.PREFIX + key[len("step_grad_"):]].numpy()
        assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max() + 1e-12, key
    fcw = grads[O.PREFIX + "fc.weight"].numpy()
    assert np.abs(fcw[:4] - g["step_grad_fc.weight_live"]).max() <= 1e-5 * np.abs(g["step_grad_fc.weight_live"]).max()
    assert np.abs(fcw[4:]).sum() == 0.0 == float(g["step_grad_fc.weight_dead_abs_sum"])
    l4 = grads[O.PREFIX + "layer4.2.conv2.weight"].numpy()[::16, ::16]
    assert np.abs(l4 - g["step_grad_l4_conv2_sub"]).max() <= 1e-5 * np.abs(g["step_grad_l4_conv2_sub"]).max()
    assert len(stats) == 72      # running_mean + running_var of the 36 BatchNorms
