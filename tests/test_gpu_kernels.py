"""GPU parity tests, kernel by kernel, through the C ABI (hulk_keypoints_b200.ops -> libhulk_sm100.so).
Every expected value comes from the CPU oracle (oracle/keypoints_oracle.py) or the committed goldens."""
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from hulk_keypoints_b200 import _lib, ops
from oracle import keypoints_oracle as O

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def test_device_is_b200():
    _lib.require_device()
    assert torch.cuda.get_device_capability(0) == (10, 0)


# ------------------------------------------------------------------ argmax decode (bit-exact)
def test_argmax_decode_matches_numpy():
    g = torch.Generator().manual_seed(0)
    for shape in [(2, 4, 48, 64), (1, 3, 37, 53), (3, 1, 480, 640), (1, 2, 5, 3)]:
        h = torch.rand(shape, generator=g)
        yx = ops.argmax_decode(h.to(dev())).cpu().numpy()
        assert np.array_equal(yx.astype(np.int64), O.argmax_decode(h.numpy())), shape


def test_argmax_decode_ties_constant_nan():
    h = torch.zeros(2, 3, 40, 56)
    h[0, 1, 20, 30] = h[0, 1, 39, 1] = h[0, 1, 20, 31] = 2.0
    h[1, 0] = 1.0                      # saturated map (sigmoid == 1.0f everywhere) -> (0, 0)
    h[1, 2, 33, 7] = float("nan")
    h[0, 2] = -3.0
    h[0, 2, 39, 55] = -0.0 - 2.5       # max at the very last element
    yx, mv = ops.argmax_decode(h.to(dev()), want_max=True)
    assert np.array_equal(yx.cpu().numpy().astype(np.int64), O.argmax_decode(h.numpy()))
    assert mv[0, 1].item() == 2.0 and np.isnan(mv[1, 2].item())


def test_argmax_decode_full_size_planted_peaks():
    # BASELINE config 2 size: 64 x 4 maps of 480x640; property: a planted unique maximum is always found
    B, K, H, W = 64, 4, 480, 640
    h = torch.rand(B, K, H, W, device=dev()) * 0.5
    rs = np.random.RandomState(1)
    ys, xs = rs.randint(0, H, (B, K)), rs.randint(0, W, (B, K))
    bi, ki = np.meshgrid(np.arange(B), np.arange(K), indexing="ij")
    h[torch.from_numpy(bi), torch.from_numpy(ki), torch.from_numpy(ys), torch.from_numpy(xs)] = 0.75
    yx = ops.argmax_decode(h).cpu().numpy()
    assert np.array_equal(yx[..., 0], ys) and np.array_equal(yx[..., 1], xs)


# ------------------------------------------------------------------ Gaussian targets
def _ulp_close(a, b, ulps=4):
    a32, b32 = a.astype(np.float32), b.astype(np.float32)
    tol = ulps * np.spacing(np.maximum(np.abs(a32), np.abs(b32))).astype(np.float64) + 1e-38
    return np.all(np.abs(a.astype(np.float64) - b.astype(np.float64)) <= tol)


def test_gauss_targets_vs_oracle_and_golden(golden):
    arrays, _ = golden
    uv = torch.from_numpy(arrays["gauss_small_labels"]).float()[None].to(dev())
    g = ops.gauss_targets(uv, 48, 64, 3.0)
    assert g.dtype == torch.float64 and g.shape == (1, 4, 48, 64)
    assert _ulp_close(g.cpu().numpy()[0], arrays["gauss_small"])
    uvf = torch.from_numpy(arrays["gauss_labels"]).float()[None].to(dev())
    gf = ops.gauss_targets(uvf, 480, 640, 8.0).cpu().numpy()[0]
    assert _ulp_close(gf[:, ::4, ::4], arrays["gauss_full_sub4"])
    assert _ulp_close(gf[:, [0, 20, 240, 479], :], arrays["gauss_full_rows"])
    assert gf[0, 20, 10] == 1.0 and gf[2, 0, 0] == 1.0 and gf[3, 479, 639] == 1.0
    assert np.allclose(gf.sum(axis=(1, 2)), arrays["gauss_full_sum"], rtol=1e-6)
    g32 = ops.gauss_targets(uvf, 480, 640, 8.0, torch.float32).cpu().numpy()[0]
    assert np.array_equal(g32.astype(np.float64), gf)  # f64 output is the widened f32 value


def test_gauss_targets_batched_ragged_width():
    uv = torch.tensor([[[3.0, 2.0], [0.0, 0.0]], [[8.5, 4.25], [10.0, 6.0]]])
    g = ops.gauss_targets(uv.to(dev()), 7, 11, 2.0).cpu().numpy()   # W not a multiple of 4
    assert _ulp_close(g, O.gauss_targets(uv.numpy(), 7, 11, 2.0))
    g = ops.gauss_targets(uv.to(dev()), 9, 10, 2.0).cpu().numpy()   # even W, not a multiple of 4, map smaller than one warp run of 128
    assert _ulp_close(g, O.gauss_targets(uv.numpy(), 9, 10, 2.0))
    g = ops.gauss_targets(uv.to(dev()), 33, 26, 2.0).cpu().numpy()  # pairs of one warp run fall into different rows
    assert _ulp_close(g, O.gauss_targets(uv.numpy(), 33, 26, 2.0))


def test_dropin_gauss_2d_batch(golden):
    import hulk_keypoints_b200 as hk
    arrays, _ = golden
    lab = arrays["gauss_small_labels"]
    g = hk.gauss_2d_batch(64, 48, 3, torch.from_numpy(lab[:, 0].copy()), torch.from_numpy(lab[:, 1].copy()))
    assert g.is_cuda and g.dtype == torch.float64 and g.shape == (4, 48, 64)
    assert _ulp_close(g.cpu().numpy(), arrays["gauss_small"])


def test_gauss_normalize_dist_vs_reference_golden(golden2):
    """gauss_2d_batch(normalize_dist=True) (dataset.py:33-34,42-44) on the hk_l1_normalize_dim1 kernel vs the reference's output."""
    import hulk_keypoints_b200 as hk
    uv = golden2["gauss_norm_uv"]
    g = hk.gauss_2d_batch(64, 48, 3, torch.from_numpy(uv[:, 0].copy()), torch.from_numpy(uv[:, 1].copy()), normalize_dist=True)
    assert g.is_cuda and g.dtype == torch.float64 and g.shape == (4, 48, 64)
    assert np.allclose(g.cpu().numpy(), golden2["gauss_norm"], rtol=4e-6, atol=1e-12)


# ------------------------------------------------------------------ soft-argmax (Prediction.expectation)
def test_soft_argmax_vs_reference_golden_and_oracle(golden2):
    """hk_soft_argmax vs the reference's Prediction.expectation (golden, before and after its int()) and the oracle; the
    transposed-ravel quirk (prediction.py:32: d.T.ravel() against row-major index arrays) is part of the expected result."""
    import hulk_keypoints_b200 as hk
    pred = hk.Prediction(hk.KeypointsGauss(4), 4, 48, 64, use_cuda=True)
    for i in range(6):
        d = golden2[f"exp_map_{i}"]
        t = torch.from_numpy(d).to(dev())
        raw, ints = ops.soft_argmax(t)
        assert raw.shape == (2,) and raw.dtype == torch.float64 and ints.dtype == torch.int32
        ref = golden2[f"exp_raw_{i}"]
        assert np.allclose(raw.cpu().numpy(), ref, rtol=1e-6, atol=1e-6), (i, raw.cpu().numpy(), ref)
        if np.all(np.abs(ref - np.round(ref)) > 1e-4):            # away from an integer boundary the truncation agrees too
            assert ints.cpu().tolist() == list(golden2[f"exp_int_{i}"])
            assert pred.expectation(t) == list(golden2[f"exp_int_{i}"])          # CUDA tensor -> kernel
        assert pred.expectation(d) == list(golden2[f"exp_int_{i}"])              # numpy -> the reference's host formula


def test_soft_argmax_batched_full_resolution():
    """(B,K,480,640) in one launch pair vs the oracle map by map; saturated / constant maps; ragged width (scalar path)."""
    g = torch.Generator().manual_seed(5)
    heat = torch.rand(2, 4, 480, 640, generator=g) * 0.2
    heat[0, 0, 100, 200] = 0.95
    heat[0, 1] = 1.0                       # constant map: uniform softmax
    heat[1, 2, 479, 639] = 1.0
    heat[1, 3] *= 50.0                     # wide dynamic range: exp underflows away from the maximum
    import hulk_keypoints_b200 as hk
    pred = hk.Prediction(hk.KeypointsGauss(4), 4, 480, 640, use_cuda=True)
    raw, ints = pred.expectation_batch(heat.to(dev()))
    assert raw.shape == (2, 4, 2)
    for b in range(2):
        for k in range(4):
            ref = O.soft_expectation_raw(heat[b, k].numpy())
            assert np.allclose(raw[b, k].cpu().numpy(), ref, rtol=2e-6, atol=1e-4), (b, k, raw[b, k].tolist(), ref)
    assert torch.equal(ints.cpu(), raw.cpu().to(torch.int32))
    odd = torch.rand(3, 37, 53, generator=g)
    raw_odd, _ = ops.soft_argmax(odd.to(dev()))
    for j in range(3):
        assert np.allclose(raw_odd[j].cpu().numpy(), O.soft_expectation_raw(odd[j].numpy()), rtol=2e-6, atol=1e-5)


# ------------------------------------------------------------------ KeypointsDataset (reference src/dataset.py:52-79)
def test_keypoints_dataset_roundtrip_vs_reference_golden(golden2, tmp_path):
    """A temporary folder of `%05d.jpg` + `%05d.npy` files through hk.KeypointsDataset against what the unmodified reference class
    returned for the same files (oracle/make_golden_v2.py): label clipping, (x, y) order, labels on the GPU, the fp32 host image
    tensor (3,H,W) = ToTensor(cv2.imread), the fp64 CUDA Gaussians (K,H,W)."""
    import hulk_keypoints_b200 as hk
    img_dir, lab_dir = tmp_path / "images", tmp_path / "keypoints"
    img_dir.mkdir(); lab_dir.mkdir()
    for i in range(2):
        np.save(str(lab_dir / ("%05d.npy" % i)), golden2[f"ds_raw_label_{i}"])
        (img_dir / ("%05d.jpg" % i)).write_bytes(golden2[f"ds_jpeg_{i}"].tobytes())
    ds = hk.KeypointsDataset(str(img_dir), str(lab_dir), 4, 48, 64, hk.transform, gauss_sigma=3)
    assert len(ds) == 2
    for i in range(2):
        assert ds.labels[i].is_cuda and ds.labels[i].dtype == torch.float64
        assert np.array_equal(ds.labels[i].cpu().numpy(), golden2[f"ds_clipped_label_{i}"])
        img, gauss = ds[i]
        assert not img.is_cuda and img.dtype == torch.float32 and tuple(img.shape) == (3, 48, 64)
        assert np.array_equal(img.numpy(), golden2[f"ds_img_{i}"])               # same cv2 build decodes the same JPEG bytes
        assert gauss.is_cuda and gauss.dtype == torch.float64 and tuple(gauss.shape) == (4, 48, 64)
        assert _ulp_close(gauss.cpu().numpy(), golden2[f"ds_gauss_{i}"])
    # the DataLoader of train.py:63 (shuffle, num_workers=0) collates (img CPU fp32, gauss CUDA fp64) batches
    loader = torch.utils.data.DataLoader(ds, batch_size=2, shuffle=False, num_workers=0)
    imgs, gausses = next(iter(loader))
    assert tuple(imgs.shape) == (2, 3, 48, 64) and tuple(gausses.shape) == (2, 4, 48, 64) and gausses.is_cuda


# ------------------------------------------------------------------ BCE
def test_bce_vs_golden_bit_exact_grad(golden):
    arrays, _ = golden
    p = torch.from_numpy(arrays["bce_pred"]).to(dev())
    t = torch.from_numpy(arrays["bce_target"]).to(dev())
    loss, grad = ops.bce_fwd_bwd(p, target=t)
    ref = float(arrays["bce_loss"])
    assert abs(loss.item() - ref) <= 1e-12 * abs(ref)
    assert np.array_equal(grad.cpu().numpy(), arrays["bce_grad_logits"])
    loss32, _ = ops.bce_fwd_bwd(p, target=t.float(), want_grad=False)
    assert abs(loss32.item() - O.bce_loss(arrays["bce_pred"], arrays["bce_target"].astype(np.float32).astype(np.float64))) < 1e-12


def test_bce_from_labels_and_logits(golden):
    arrays, _ = golden
    B, K, H, W = 2, 4, 48, 64
    uv = torch.from_numpy(np.stack([arrays["gauss_small_labels"], arrays["gauss_small_labels"][::-1].copy()])).float()
    z = torch.from_numpy(arrays["bce_logits"])
    t = O.gauss_targets(uv.numpy(), H, W, 3.0)
    p = torch.sigmoid(z)
    loss, grad = ops.bce_fwd_bwd(z.to(dev()), uv=uv.to(dev()), sigma=3.0, pred_is_logits=True)
    ref = O.bce_loss(p.numpy(), t)
    assert abs(loss.item() - ref) <= 1e-6 * abs(ref)
    gref = O.bce_grad_logits(p.numpy(), t)
    assert np.abs(grad.cpu().numpy() - gref).max() <= 1e-6 * np.abs(gref).max()
    # saturated elements: exact zeros, like the reference autograd
    assert grad[0, 0, 0, 0].item() == 0.0


def test_bce_known_answers():
    p = torch.tensor([1.0, 0.5, 0.0, 0.25] * 4).view(1, 1, 4, 4).to(dev())
    t = torch.tensor([0.25, 0.5, 0.0, 1.0] * 4, dtype=torch.float64).view(1, 1, 4, 4).to(dev())
    loss, g = ops.bce_fwd_bwd(p, target=t)
    expect = (100 * 0.75 + np.log(2.0) + 0.0 - np.log(0.25)) / 4
    assert abs(loss.item() - expect) < 1e-12
    gc = g.cpu().view(-1)
    assert gc[0] == 0 and gc[1] == 0 and gc[2] == 0


def test_fused_loss_autograd_matches_torch():
    from hulk_keypoints_b200 import train_ops
    torch.manual_seed(0)
    z = (torch.randn(2, 4, 32, 48, device=dev()) * 3).requires_grad_(True)
    uv = torch.tensor([[[5., 6.], [40., 20.], [0., 0.], [47., 31.]]] * 2, device=dev())
    loss = train_ops.sigmoid_bce_loss(z, uv=uv, sigma=4.0)
    loss.backward()
    z2 = z.detach().clone().requires_grad_(True)
    t = ops.gauss_targets(uv, 32, 48, 4.0)
    ref = torch.nn.BCELoss()(torch.sigmoid(z2).double(), t)
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-9
    assert (z.grad - z2.grad).abs().max().item() <= 1e-6 * z2.grad.abs().max().item()


# ------------------------------------------------------------------ head
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_head_vs_oracle(dtype):
    g = torch.Generator().manual_seed(2)
    B, h, w, C, K, H, W = 2, 8, 12, 512, 4, 64, 96
    feat = (torch.randn(B, C, h, w, generator=g) * 2).to(dtype).float()
    wfc = torch.randn(K, C, generator=g) * 0.05
    bfc = torch.randn(K, generator=g) * 0.1
    logits = F.conv2d(feat, wfc.view(K, C, 1, 1), bfc)
    ref = O.heatmaps_from_logits(logits, (H, W)).numpy()
    got = ops.head(feat.permute(0, 2, 3, 1).contiguous().to(dtype).to(dev()), wfc.to(dev()), bfc.to(dev()), H, W).cpu().numpy()
    assert got.shape == (B, K, H, W)
    assert np.abs(got - ref).max() < 2e-5
    # corners of align_corners=True map exactly to the low-res logits
    assert abs(got[0, 0, 0, 0] - torch.sigmoid(logits[0, 0, 0, 0]).item()) < 2e-6
    assert abs(got[1, 3, H - 1, W - 1] - torch.sigmoid(logits[1, 3, h - 1, w - 1]).item()) < 2e-6


def test_head_more_keypoints_and_saturation():
    g = torch.Generator().manual_seed(3)
    B, h, w, C, K, H, W = 1, 15, 20, 512, 16, 120, 160
    feat = torch.randn(B, C, h, w, generator=g) * 30     # logits of +-60: sigmoid saturates to exactly 1.0f / ~0
    wfc = torch.randn(K, C, generator=g) * 0.1
    bfc = torch.zeros(K)
    ref = O.heatmaps_from_logits(F.conv2d(feat, wfc.view(K, C, 1, 1), bfc), (H, W)).numpy()
    got = ops.head(feat.permute(0, 2, 3, 1).contiguous().to(dev()), wfc.to(dev()), bfc.to(dev()), H, W).cpu().numpy()
    assert np.abs(got - ref).max() < 1e-4
    assert (got == 1.0).sum() > 0 and got.min() >= 0.0


# ------------------------------------------------------------------ maxpool / pack
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_maxpool_exact(dtype):
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 64, 31, 46, generator=g).to(dtype)
    ref = F.max_pool2d(x.float(), 3, 2, 1)
    got = ops.maxpool3x3s2(x.permute(0, 2, 3, 1).contiguous().to(dev())).float().cpu().permute(0, 3, 1, 2)
    assert torch.equal(got, ref)


def test_pack_weights_and_bn_fold():
    g = torch.Generator().manual_seed(5)
    w = torch.randn(128, 64, 3, 3, generator=g)
    gamma, beta = torch.rand(128, generator=g) + 0.5, torch.randn(128, generator=g)
    mean, var = torch.randn(128, generator=g), torch.rand(128, generator=g) + 0.1
    wp, s, b = ops.pack_conv_weights(w.to(dev()), tuple(t.to(dev()) for t in (gamma, beta, mean, var)), 1e-5, torch.bfloat16)
    assert torch.equal(wp.cpu(), w.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))
    s_ref = gamma / torch.sqrt(var + 1e-5)
    assert torch.allclose(s.cpu(), s_ref, rtol=1e-6) and torch.allclose(b.cpu(), beta - mean * s_ref, rtol=1e-5, atol=1e-6)
    wp32, s1, b0 = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.float32)
    assert torch.equal(wp32.cpu(), w.permute(0, 2, 3, 1).contiguous()) and (s1 == 1).all() and (b0 == 0).all()


# ------------------------------------------------------------------ convolutions
def _conv_case(B, H, W, cin, cout, k, stride, dil, residual, relu, seed, scale_in=1.0):
    g = torch.Generator().manual_seed(seed)
    pad = dil * (k - 1) // 2
    x = torch.randn(B, cin, H, W, generator=g) * scale_in
    w = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (k * k * cin)) ** 0.5
    s = torch.rand(cout, generator=g) + 0.5
    b = torch.randn(cout, generator=g) * 0.1
    Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
    res = torch.randn(B, cout, Ho, Wo, generator=g) if residual else None
    return x, w, s, b, res, pad


def _conv_ref(x, w, s, b, res, stride, pad, dil, relu):
    y = F.conv2d(x.double(), w.double(), None, stride, pad, dil) * s.double().view(1, -1, 1, 1) + b.double().view(1, -1, 1, 1)
    if res is not None:
        y = y + res.double()
    return (F.relu(y) if relu else y)


FFMA_CASES = [
    # B, H, W, cin, cout, k, stride, dil, residual, relu
    (1, 20, 28, 64, 64, 3, 1, 1, True, True),
    (2, 15, 20, 64, 128, 3, 2, 1, False, True),
    (2, 15, 20, 64, 128, 1, 2, 1, False, False),
    (1, 15, 20, 128, 256, 3, 1, 2, True, True),
    (1, 15, 20, 256, 512, 3, 1, 4, False, True),
    (3, 9, 7, 64, 68, 3, 1, 1, True, False),   # ragged M and N tiles
]


@pytest.mark.parametrize("case", FFMA_CASES)
def test_conv_ffma_fp32_vs_oracle(case):
    B, H, W, cin, cout, k, stride, dil, residual, relu = case
    x, w, s, b, res, pad = _conv_case(*case, seed=11)
    ref = _conv_ref(x, w, s, b, res, stride, pad, dil, relu)
    wp, _, _ = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.float32)
    y = ops.conv_bn_act(x.permute(0, 2, 3, 1).contiguous().to(dev()), wp, s.to(dev()), b.to(dev()), stride=stride, pad=pad,
                        dil=dil, relu=relu, residual=None if res is None else res.permute(0, 2, 3, 1).contiguous().to(dev()),
                        algo=_lib.HK_CONV_FFMA)
    got = y.cpu().permute(0, 3, 1, 2).double()
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 2e-5 * max(1.0, ref.abs().max().item())


def test_conv_ffma_stem_nchw_input():
    g = torch.Generator().manual_seed(12)
    x = torch.rand(2, 3, 64, 96, generator=g)
    w = torch.randn(64, 3, 7, 7, generator=g) * 0.05
    s, b = torch.rand(64, generator=g) + 0.5, torch.randn(64, generator=g) * 0.1
    ref = _conv_ref(x, w, s, b, None, 2, 3, 1, True)
    wp, _, _ = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.float32)
    for odt, tol in ((torch.float32, 2e-6), (torch.bfloat16, 8e-3)):
        y = ops.conv_bn_act(x.to(dev()), wp, s.to(dev()), b.to(dev()), stride=2, pad=3, dil=1, relu=True, out_dtype=odt,
                            algo=_lib.HK_CONV_FFMA, in_is_nchw=True)
        got = y.float().cpu().permute(0, 3, 1, 2).double()
        assert (got - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())


TC_CASES = [
    # B, H, W, cin, cout, k, stride, dil, residual, relu
    (1, 4, 16, 64, 64, 1, 1, 1, False, False),     # one box, one K block: the bare GEMM
    (1, 8, 16, 64, 64, 1, 1, 1, False, False),     # one full M tile
    (2, 8, 32, 128, 128, 1, 1, 1, False, True),    # two K blocks
    (1, 12, 20, 64, 64, 3, 1, 1, True, True),      # ragged spatial tiles, 9 taps, halo zero fill
    (2, 15, 20, 128, 256, 3, 1, 2, True, True),    # dilation 2, N=256
    (1, 60, 80, 256, 512, 3, 1, 4, True, True),    # layer4 shape: dilation 4, 2 N tiles, 36+ K blocks
    (4, 60, 80, 64, 128, 1, 1, 1, False, False),   # 150 M tiles > 148 SMs: persistence + TMEM double buffer
    (2, 30, 40, 64, 128, 3, 2, 1, False, True),    # stride 2 via TMA element strides
    (2, 30, 40, 64, 128, 1, 2, 1, False, False),   # 1x1 stride-2 downsample
    (3, 15, 20, 512, 512, 3, 1, 4, True, True),    # odd number of boxes -> padding box
]


@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tcgen05_single_cta_kernel(case):
    """The generic 1-CTA kernel on every shape (the default route sends Cout>=128 to the CTA-pair kernel)."""
    test_conv_tcgen05_vs_oracle(case, algo=_lib.HK_CONV_TCGEN05_1CTA)


@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tcgen05_vs_oracle(case, algo=_lib.HK_CONV_TCGEN05):
    B, H, W, cin, cout, k, stride, dil, residual, relu = case
    x, w, s, b, res, pad = _conv_case(*case, seed=21)
    xb, wb = x.to(torch.bfloat16), w.to(torch.bfloat16)
    resb = None if res is None else res.to(torch.bfloat16)
    # oracle: same bf16-rounded operands, exact (f64) accumulation
    ref = _conv_ref(xb.float(), wb.float(), s, b, None if resb is None else resb.float(), stride, pad, dil, relu)
    wp, _, _ = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.bfloat16)
    y = ops.conv_bn_act(xb.permute(0, 2, 3, 1).contiguous().to(dev()), wp, s.to(dev()), b.to(dev()), stride=stride, pad=pad,
                        dil=dil, relu=relu, residual=None if resb is None else resb.permute(0, 2, 3, 1).contiguous().to(dev()),
                        algo=algo)
    torch.cuda.synchronize()
    got = y.float().cpu().permute(0, 3, 1, 2).double()
    assert got.shape == ref.shape
    err = (got - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 1e-3 * max(1.0, ref.abs().max().item())   # one bf16 rounding of the output
    bad = (err > tol).sum().item()
    assert bad == 0, f"{bad} / {err.numel()} outputs off; max err {err.max().item():.4g}, ref max {ref.abs().max().item():.4g}"


@pytest.mark.parametrize("shape", [(2, 64, 96), (1, 480, 640), (3, 50, 70)])
def test_stem_tcgen05_vs_oracle(shape):
    B, H, W = shape
    g = torch.Generator().manual_seed(31)
    x = torch.rand(B, 3, H, W, generator=g)
    w = torch.randn(64, 3, 7, 7, generator=g) * (2.0 / (49 * 64)) ** 0.5
    s, b = torch.rand(64, generator=g) + 0.5, torch.randn(64, generator=g) * 0.1
    ref = _conv_ref(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), s, b, None, 2, 3, 1, True)
    y = ops.stem(x.to(dev()), ops.stem_pack_weights(w.to(dev())), s.to(dev()), b.to(dev()))
    torch.cuda.synchronize()
    got = y.float().cpu().permute(0, 3, 1, 2).double()
    assert got.shape == ref.shape
    err = (got - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 1e-3 * max(1.0, ref.abs().max().item())
    assert (err > tol).sum().item() == 0, f"max err {err.max().item():.4g}"


C64_CASES = [
    # B, H, W, dil, residual, relu   (3x3, 64 -> 64, stride 1: the layer1 specialisation)
    (1, 8, 16, 1, False, False),      # exactly one tile
    (2, 120, 160, 1, True, True),     # layer1 shape: 300 tiles > 148 SMs
    (3, 20, 28, 1, True, True),       # ragged tiles in both directions
    (1, 24, 32, 2, False, True),      # dilation 2 (taller halo box)
]


@pytest.mark.parametrize("case", C64_CASES)
def test_conv_tcgen05_c64_specialisation(case):
    B, H, W, dil, residual, relu = case
    test_conv_tcgen05_vs_oracle((B, H, W, 64, 64, 3, 1, dil, residual, relu))


@pytest.mark.parametrize("shape", [(2, 480, 640), (1, 96, 128), (3, 64, 96), (1, 100, 132), (2, 72, 1040), (1, 330, 36)],
                         ids=lambda s: "x".join(map(str, s)))
def test_stem_pool_fused_bit_identical_to_two_kernels(shape):
    """hk_stem_pool_fwd (row-streaming stem + max-pool, no-swizzle overlapping-core-matrix A operand straight from the input ring)
    against hk_stem_fwd + hk_maxpool3x3s2_fwd: BIT-identical, incl. ragged strips (W/4 not a multiple of 63), odd stem heights,
    widths over several strips, bands with carry rows."""
    B, H, W = shape
    g = torch.Generator().manual_seed(H * 7 + W)
    x = torch.rand(B, 3, H, W, generator=g).to(dev())
    w = (torch.randn(64, 3, 7, 7, generator=g) * 0.1).to(dev())
    scale = (torch.rand(64, generator=g) + 0.5).to(dev())
    bias = (torch.randn(64, generator=g) * 0.2).to(dev())
    wp = ops.stem_pack_weights(w)
    ref = ops.maxpool3x3s2(ops.stem(x, wp, scale, bias))
    got = ops.stem_pool(x, wp, scale, bias)
    assert got.shape == ref.shape and got.dtype == torch.bfloat16
    assert torch.equal(got, ref), (got.float() - ref.float()).abs().max().item()
    if W % 16 == 0:
        u8 = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).to(dev())
        ref8 = ops.maxpool3x3s2(ops.stem(u8, wp, scale, bias))
        got8 = ops.stem_pool(u8, wp, scale, bias)
        assert torch.equal(got8, ref8), (got8.float() - ref8.float()).abs().max().item()


def test_stem_pool_rejects_unaligned_width():
    x = torch.rand(1, 3, 64, 98).to(dev())
    assert not ops.stem_pool_supported(x)
    with pytest.raises(ValueError):
        ops.stem_pool(x, torch.empty(64 * 256, device=dev(), dtype=torch.bfloat16), torch.ones(64, device=dev()), torch.zeros(64, device=dev()))


def test_stem_uint8_input_matches_float_path():
    """(B,H,W,3) uint8 input with /255 fused into the load == the fp32 NCHW path fed ToTensor(img) (dataset.py:16)."""
    g = torch.Generator().manual_seed(33)
    img = torch.randint(0, 256, (2, 70, 90, 3), generator=g, dtype=torch.uint8)
    w = torch.randn(64, 3, 7, 7, generator=g) * 0.05
    s, b = torch.rand(64, generator=g) + 0.5, torch.randn(64, generator=g) * 0.1
    wp = ops.stem_pack_weights(w.to(dev()))
    y8 = ops.stem(img.to(dev()), wp, s.to(dev()), b.to(dev()))
    xf = img.permute(0, 3, 1, 2).float().div(255).contiguous()
    yf = ops.stem(xf.to(dev()), wp, s.to(dev()), b.to(dev()))
    assert torch.equal(y8, yf)


def test_fused_adam_matches_torch_adam():
    from hulk_keypoints_b200.optim import FusedAdam
    torch.manual_seed(0)
    shapes = [(64, 3, 7, 7), (64,), (128, 64, 3, 3), (1000, 512, 1, 1), (5,), (3, 3)]
    ref_params = [torch.nn.Parameter(torch.randn(s, device=dev())) for s in shapes]
    our_params = [torch.nn.Parameter(p.detach().clone()) for p in ref_params]
    ref = torch.optim.Adam(ref_params, lr=1e-3, weight_decay=1e-4)
    ours = FusedAdam(our_params, lr=1e-3, weight_decay=1e-4)
    for step in range(5):
        grads = [torch.randn(s, device=dev()) * (0.0 if (i == 3 and step % 2) else 1.0) for i, s in enumerate(shapes)]
        ref.zero_grad(); ours.zero_grad()
        for p, q, g in zip(ref_params, our_params, grads):
            p.grad = g.clone()
            q.grad.copy_(g)          # gradient views into the flat buffer stay attached
        ref.step(); ours.step()
    for p, q in zip(ref_params, our_params):
        assert torch.allclose(p, q, rtol=2e-6, atol=2e-7), (p - q).abs().max().item()
    assert our_params[0].grad.data_ptr() == ours.flat_grad.data_ptr()


HALO_CASES = [
    (2, 60, 80, 128, 128, 3, 1, 1, True, True),     # layer2 shape, height 60: half-empty last patch row
    (2, 60, 80, 128, 128, 3, 1, 1, False, False),
    (1, 64, 80, 256, 256, 3, 1, 2, True, True),     # layer3-like, dilation 2, height multiple of 8
    (2, 60, 80, 128, 256, 3, 1, 2, False, True),    # layer3.0.conv1
    (1, 60, 80, 512, 512, 3, 1, 4, True, True),     # layer4 shape, dilation 4, 2 N tiles: stays on the plain CTA-pair kernel
    (3, 21, 37, 128, 128, 3, 1, 1, True, True),     # ragged patches in both directions, odd patch count -> padding patch
    (5, 120, 160, 128, 128, 3, 1, 1, False, True),  # more tiles than clusters: ring wrap-around over many tiles
]


STRIP_CASES = [
    # heights 1..4 rows past a multiple of 8: the bottom rows are covered by 4x32 strip patches (conv_tc2h.cu)
    (2, 60, 80, 128, 128, 3, 1, 1, True, True),     # layer2 shape: 7 patch rows + a strip row, 80 = 2.5 strips wide
    (1, 60, 80, 256, 256, 3, 1, 2, True, True),     # layer3 shape, dilation 2 (32 KB strip boxes)
    (3, 12, 37, 128, 128, 3, 1, 1, True, False),    # odd number of 8x16 patches -> padded boundary; ragged strips
    (2, 9, 70, 128, 256, 3, 1, 2, False, True),     # one remainder row only: strips clipped to a single row
    (5, 20, 48, 128, 128, 3, 1, 1, False, True),    # strips with odd count per batch
]


@pytest.mark.parametrize("case", STRIP_CASES)
def test_conv_tcgen05_strip_patches(case):
    """Strip patches against the oracle, and bit-identical to the all-8x16 schedule (same accumulation order per output element).
    The all-8x16 result comes from the same conv on the input (and residual) zero-extended at the bottom to a multiple of 8 rows:
    output rows < H read only zeros below the input in both runs, so their first H rows must be equal."""
    test_conv_tcgen05_vs_oracle(case)
    B, H, W, cin, cout, k, stride, dil, residual, relu = case
    He = -(-H // 8) * 8
    assert H > 8 and 1 <= H % 8 <= 4 and He % 8 == 0   # strips here, none in the extended map
    x, w, s, b, res, pad = _conv_case(*case, seed=21)
    xd = x.to(torch.bfloat16).permute(0, 2, 3, 1).contiguous().to(dev())
    rd = None if res is None else res.to(torch.bfloat16).permute(0, 2, 3, 1).contiguous().to(dev())
    extend = lambda t: None if t is None else F.pad(t, (0, 0, 0, 0, 0, He - H))
    wp, _, _ = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.bfloat16)
    run = lambda xx, rr: ops.conv_bn_act(xx, wp, s.to(dev()), b.to(dev()), stride=stride, pad=pad, dil=dil, relu=relu, residual=rr)
    y_strips = run(xd, rd)
    y_plain = run(extend(xd), extend(rd))
    assert y_plain.shape[1] == He
    assert torch.equal(y_strips, y_plain[:, :H])


@pytest.mark.parametrize("case", HALO_CASES)
def test_conv_tcgen05_haloed_operand_kernel(case):
    """The shapes of the haloed-operand kernel (conv_tc2h, one haloed activation box per horizontal tap) against the oracle, and the
    dilation-4 layer4 shape, which the default route keeps on conv_tc2."""
    test_conv_tcgen05_vs_oracle(case)


# ------------------------------------------------------------------ block entry: conv1 + 1x1 downsample in one launch (src/resnet.py:56-58,64-65,184-188)
DS_CASES = [
    # B, H, W, cin, cout, stride, dil
    (2, 30, 40, 64, 128, 2, 1),      # layer2.0: 3x3 stride 2 + 1x1 stride 2
    (1, 60, 80, 128, 256, 1, 2),     # layer3.0: dilation 2
    (1, 60, 80, 256, 512, 1, 4),     # layer4.0: dilation 4, two N tiles of 256
    (3, 21, 27, 128, 256, 1, 2),     # ragged boxes in both directions, odd tile count
    (5, 120, 160, 64, 128, 2, 1),    # more work items than CTA pairs (several accumulator turns per cluster)
    (1, 8, 16, 64, 128, 1, 1),       # a single 256-pixel tile, half of it out of range
]


@pytest.mark.parametrize("case", DS_CASES)
def test_conv_ds_block_entry(case):
    """hk_conv_ds_fwd: both outputs bit-identical to two hk_conv_bn_act_fwd launches, and within one bf16 rounding of the fp64 conv on
    the same bf16 operands."""
    B, H, W, cin, cout, stride, dil = case
    g = torch.Generator().manual_seed(77)
    x = (torch.randn(B, cin, H, W, generator=g)).to(torch.bfloat16)
    w = torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5
    wd = torch.randn(cout, cin, 1, 1, generator=g) * (1.0 / cin) ** 0.5
    s, b = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.1
    sd, bd = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.1
    xd = x.permute(0, 2, 3, 1).contiguous().to(dev())
    wp, _, _ = ops.pack_conv_weights(w.to(dev()), None, 1e-5, torch.bfloat16)
    wdp, _, _ = ops.pack_conv_weights(wd.to(dev()), None, 1e-5, torch.bfloat16)
    sD, bD, sdD, bdD = s.to(dev()), b.to(dev()), sd.to(dev()), bd.to(dev())
    assert ops.conv_ds_supported(xd, wp, wdp, stride, dil, dil)
    y, yds = ops.conv_ds(xd, wp, sD, bD, wdp, sdD, bdD, stride=stride, pad=dil, dil=dil, relu=True)
    torch.cuda.synchronize()
    # the two-launch path with its default routing (dilation <= 2, stride 1 runs on the haloed kernel: hk_conv_ds_fwd then accumulates
    # its K blocks in that kernel's order, so the comparison is exact either way)
    y2 = ops.conv_bn_act(xd, wp, sD, bD, stride=stride, pad=dil, dil=dil, relu=True)
    yds2 = ops.conv_bn_act(xd, wdp, sdD, bdD, stride=stride, pad=0, dil=1, relu=False)
    torch.cuda.synchronize()
    assert torch.equal(y, y2), f"conv1 output differs from the separate launch: {(y.float() - y2.float()).abs().max().item()}"
    assert torch.equal(yds, yds2), f"downsample output differs from the separate launch: {(yds.float() - yds2.float()).abs().max().item()}"
    for got_t, ww, ss, bb, pad_, dil_, relu_ in ((y, w, s, b, dil, dil, True), (yds, wd, sd, bd, 0, 1, False)):
        ref = _conv_ref(x.float(), ww.to(torch.bfloat16).float(), ss, bb, None, stride, pad_, dil_, relu_)
        got = got_t.float().cpu().permute(0, 3, 1, 2).double()
        err = (got - ref).abs()
        tol = 2.0 ** -8 * ref.abs() + 1e-3 * max(1.0, ref.abs().max().item())
        assert (err > tol).sum().item() == 0, f"max err {err.max().item():.4g}"


def test_conv_ds_rejects_bad_shapes():
    x = torch.zeros(1, 16, 16, 64, device=dev(), dtype=torch.bfloat16)
    wp = torch.zeros(128, 3, 3, 64, device=dev(), dtype=torch.bfloat16)
    wd = torch.zeros(128, 1, 1, 64, device=dev(), dtype=torch.bfloat16)
    v = torch.zeros(128, device=dev())
    with pytest.raises(ValueError):
        ops.conv_ds(x, wp, v, v, wd, v, v, stride=1, pad=0, dil=1)       # pad != dil*(k/2): the 1x1 is not the centre tap
    with pytest.raises(ValueError):
        ops.conv_ds(x.float(), wp, v, v, wd, v, v, stride=1, pad=1, dil=1)  # fp32 activations: tcgen05 path only


# ------------------------------------------------------------------ last conv + scoring rows in one launch (src/resnet.py:60-67,215; src/model.py:21)
HEAD_CASES = [
    # B, H, W, cin, K, dil, residual
    (1, 16, 16, 512, 4, 4, True),      # one 256-pixel tile per N tile
    (2, 60, 80, 512, 4, 4, True),      # layer4[2].conv2 at config.py resolution (feature map 60x80)
    (3, 21, 27, 256, 8, 2, True),      # ragged boxes, K = 8, another dilation / Cin
    (1, 13, 9, 512, 1, 1, False),      # K = 1, no shortcut, a single partial tile
    (5, 60, 80, 512, 3, 4, True),      # more work items than CTA pairs
]


@pytest.mark.parametrize("case", HEAD_CASES)
def test_conv_head_fused_logits(case):
    """hk_conv_head_fwd against hk_conv_bn_act_fwd followed by the fc rows applied (in fp64) to the bf16 feature map it stores: the fused
    epilogue rounds each row to bf16 exactly as the feature map would have held it, so only the fp32 summation order differs.  Also
    bit-reproducible run to run (two commutative contributions per logit) and equal, to fp32 rounding, to hk_head_fwd's logits."""
    B, H, W, cin, K, dil, residual = case
    g = torch.Generator().manual_seed(100 + cin + K)
    x = torch.randn(B, H, W, cin, generator=g).to(dev()).to(torch.bfloat16)
    w = (torch.randn(512, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5).to(dev())
    s, b = (torch.rand(512, generator=g) + 0.5).to(dev()), (torch.randn(512, generator=g) * 0.1).to(dev())
    res = torch.randn(B, H, W, 512, generator=g).to(dev()).to(torch.bfloat16) if residual else None
    w_fc = (torch.randn(K, 512, generator=g) * 0.05).to(dev())
    b_fc = (torch.randn(K, generator=g) * 0.1).to(dev())
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, torch.bfloat16)
    assert ops.conv_head_supported(x, wp, w_fc, 1)
    # the reference feature map from a kernel with the fused one's K-block order, (r, s, channel block): the haloed kernel, the default
    # route at dilation 1 and 2, accumulates in another order, which moves a few bf16 roundings of the feature map by one ulp
    feat = ops.conv_bn_act(x, wp, s, b, stride=1, pad=dil, dil=dil, relu=True, residual=res, algo=_lib.HK_CONV_TCGEN05_1CTA)
    torch.cuda.synchronize()
    ref = torch.einsum("bhwc,kc->bkhw", feat.double(), w_fc.double()) + b_fc.double().view(1, K, 1, 1)
    logits = torch.full((B, K, H, W), float("nan"), device=dev())
    ops.conv_head(x, wp, s, b, w_fc, b_fc, logits, stride=1, pad=dil, dil=dil, relu=True, residual=res)
    torch.cuda.synchronize()
    first = logits.clone()
    ops.conv_head(x, wp, s, b, w_fc, b_fc, logits, stride=1, pad=dil, dil=dil, relu=True, residual=res)
    torch.cuda.synchronize()
    assert torch.equal(first, logits)
    err = (logits.double() - ref).abs()
    bound = 1e-5 * (feat.double().abs().unsqueeze(1) * w_fc.double().abs().view(1, K, 1, 1, 512)).sum(-1) + 1e-6   # fp32 accumulation of 512 terms
    assert (err <= bound).all(), f"max err {err.max().item():.3g} (bound {bound.max().item():.3g})"
    # and the two-kernel head produces the same heatmaps to fp32 rounding of the logits
    heat2 = ops.head(feat, w_fc, b_fc, 8 * (H - 1) + 8, 8 * (W - 1) + 8)
    heat1 = ops.head_upsample(logits, 8 * (H - 1) + 8, 8 * (W - 1) + 8)
    assert (heat1 - heat2).abs().max().item() < 2e-6


def test_conv_head_rejects_unsupported():
    x = torch.zeros(1, 16, 16, 64, device=dev(), dtype=torch.bfloat16)
    wp = torch.zeros(512, 3, 3, 64, device=dev(), dtype=torch.bfloat16)
    v = torch.zeros(512, device=dev())
    with pytest.raises(ValueError):   # nine scoring rows: beyond the fused epilogue's register budget
        ops.conv_head(x, wp, v, v, torch.zeros(9, 512, device=dev()), torch.zeros(9, device=dev()), torch.zeros(1, 9, 16, 16, device=dev()),
                      stride=1, pad=1, dil=1)
    wp256 = torch.zeros(256, 3, 3, 64, device=dev(), dtype=torch.bfloat16)
    assert not ops.conv_head_supported(x, wp256, torch.zeros(4, 512, device=dev()), 1)
