"""GPU parity tests of the training-side kernels (SURVEY.md §8 f1), through the C ABI.

The checker for each kernel is the torch fp32/fp64 op the reference's train step executes at that point (nn.BatchNorm2d in
train() mode, autograd of nn.Conv2d / MaxPool2d / upsample_bilinear / the 1x1 scoring conv), evaluated on the SAME
bf16-rounded operands, so the only differences are accumulation order and the final bf16 rounding of activations."""
import warnings

import pytest
import torch
import torch.nn.functional as F

from hulk_keypoints_b200 import ops

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu
DEV = "cuda:0"
torch.backends.cudnn.allow_tf32 = False        # the checker must be true fp32 (SURVEY.md §8c)
torch.backends.cuda.matmul.allow_tf32 = False


def bf(x):
    return x.to(torch.bfloat16)


def nhwc(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous()


def nchw(x_nhwc):
    return x_nhwc.permute(0, 3, 1, 2).contiguous()


def rel_err(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


# ------------------------------------------------------------------ BatchNorm (train) forward
@pytest.mark.parametrize("C_,shape", [(64, (2, 24, 40)), (128, (3, 15, 20)), (256, (1, 15, 20)), (512, (2, 8, 16))])
def test_bn_train_forward_matches_torch(C_, shape):
    torch.manual_seed(C_)
    B, H, W = shape
    y = bf(torch.randn(B, H, W, C_, device=DEV) * 2.0 + 0.7)
    res = bf(torch.randn(B, H, W, C_, device=DEV))
    gamma = torch.rand(C_, device=DEV) + 0.5
    beta = torch.randn(C_, device=DEV) * 0.1
    rm, rv = torch.randn(C_, device=DEV) * 0.1, torch.rand(C_, device=DEV) + 0.5
    rm_ref, rv_ref = rm.clone(), rv.clone()
    mean, invstd, scale, shift = (torch.empty(C_, device=DEV) for _ in range(4))
    ws = ops.bn_workspace(C_, DEV)
    ops.bn_train_stats(y, gamma, beta, rm, rv, 0.1, 1e-5, mean, invstd, scale, shift, ws)
    out = ops.bn_apply(y, scale, shift, relu=True, residual=res)
    y32 = nchw(y.float())
    ref = F.relu(F.batch_norm(y32, rm_ref, rv_ref, gamma, beta, training=True, momentum=0.1, eps=1e-5) + nchw(res.float()))
    assert torch.allclose(mean, y32.mean(dim=(0, 2, 3)), atol=1e-5, rtol=1e-5)
    assert torch.allclose(invstd, 1.0 / torch.sqrt(y32.var(dim=(0, 2, 3), unbiased=False) + 1e-5), rtol=1e-4)
    assert torch.allclose(rm, rm_ref, atol=1e-5, rtol=1e-5) and torch.allclose(rv, rv_ref, atol=1e-5, rtol=1e-4)
    got = nchw(out.float())
    assert torch.allclose(got, ref, atol=2e-2, rtol=1e-2)          # one bf16 rounding of the output
    assert rel_err(got, ref) < 4e-3


# ------------------------------------------------------------------ BatchNorm (train) + ReLU backward
@pytest.mark.parametrize("C_,with_relu", [(64, True), (128, False), (512, True)])
def test_bn_train_backward_matches_autograd(C_, with_relu):
    torch.manual_seed(7 + C_)
    B, H, W = 2, 12, 20
    y = bf(torch.randn(B, H, W, C_, device=DEV) * 1.5 + 0.3)
    res = bf(torch.randn(B, H, W, C_, device=DEV))
    dout = bf(torch.randn(B, H, W, C_, device=DEV) * 1e-3)
    gamma = torch.rand(C_, device=DEV) + 0.5
    beta = torch.randn(C_, device=DEV) * 0.1
    mean, invstd, scale, shift = (torch.empty(C_, device=DEV) for _ in range(4))
    ws = ops.bn_workspace(C_, DEV)
    ops.bn_train_stats(y, gamma, beta, None, None, 0.1, 1e-5, mean, invstd, scale, shift, ws)
    bits = torch.zeros(y.numel() // 8, device=DEV, dtype=torch.uint8)
    out = ops.bn_apply(y, scale, shift, relu=with_relu, residual=res, relu_bits=bits)
    dgamma, dbeta = torch.empty(C_, device=DEV), torch.empty(C_, device=DEV)
    dy, dmasked = torch.empty_like(y), torch.empty_like(y)
    ops.bn_train_bwd(dout, out if with_relu else None, y, mean, invstd, gamma, dgamma, dbeta, dy, ws, dmasked=dmasked)
    if with_relu:
        # the 1-bit-per-element ReLU mask written by the forward apply pass == [out > 0], and the backward fed with it is bit-identical
        expect = ((out.reshape(-1, 8) > 0).to(torch.int32) << torch.arange(8, device=DEV, dtype=torch.int32)).sum(1).to(torch.uint8)
        assert torch.equal(bits, expect)
        dg2, db2, dy2, dm2 = torch.empty_like(dgamma), torch.empty_like(dbeta), torch.empty_like(y), torch.empty_like(y)
        ops.bn_train_bwd(dout, bits, y, mean, invstd, gamma, dg2, db2, dy2, ws, dmasked=dm2)
        assert torch.equal(dy2, dy) and torch.equal(dm2, dmasked) and torch.equal(dg2, dgamma) and torch.equal(db2, dbeta)
    # autograd on the same operands; the ReLU mask is taken from OUR post-ReLU output (what the next layer saw)
    y32 = nchw(y.float()).requires_grad_(True)
    g32, b32 = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    r32 = nchw(res.float()).requires_grad_(True)
    pre = F.batch_norm(y32, None, None, g32, b32, training=True, eps=1e-5) + r32
    mask = (nchw(out.float()) > 0).float() if with_relu else torch.ones_like(pre)
    (pre * mask * nchw(dout.float())).sum().backward()
    assert rel_err(nchw(dy.float()), y32.grad) < 1e-2
    assert rel_err(nchw(dmasked.float()), r32.grad) < 1e-6        # d' is exactly dout*mask (both bf16)
    assert rel_err(dgamma, g32.grad) < 1e-3 and rel_err(dbeta, b32.grad) < 1e-3


# ------------------------------------------------------------------ BatchNorm through exact fixed-point accumulators (no finalize launch)
@pytest.mark.parametrize("C_,shape,relu", [(64, (2, 24, 40), True), (128, (3, 15, 20), False), (512, (2, 8, 16), True), (64, (4, 120, 160), True)])
def test_bn_accumulator_path_matches_three_launch_path(C_, shape, relu):
    """hk_bn_stats_acc + hk_bn_apply_fwd_acc and hk_bn_bwd_acc against hk_bn_train_stats / hk_bn_apply_fwd / hk_bn_train_bwd on the same
    operands: statistics to fp32 rounding (the accumulators add the block partials exactly, the three-launch path adds them in fp32 and
    double), outputs to one bf16 ulp where a coefficient moved, ReLU masks and d' exactly; and bit-reproducible run to run."""
    torch.manual_seed(3 * C_ + shape[0])
    B, H, W = shape
    y = bf(torch.randn(B, H, W, C_, device=DEV) * 2.0 + 0.7)
    res = bf(torch.randn(B, H, W, C_, device=DEV))
    dout = bf(torch.randn(B, H, W, C_, device=DEV) * 1e-3)
    gamma, beta = torch.rand(C_, device=DEV) + 0.5, torch.randn(C_, device=DEV) * 0.1
    rm0, rv0 = torch.randn(C_, device=DEV) * 0.1, torch.rand(C_, device=DEV) + 0.5
    ws = ops.bn_workspace(C_, DEV)
    # three-launch path
    rm, rv = rm0.clone(), rv0.clone()
    mean, invstd, scale, shift = (torch.empty(C_, device=DEV) for _ in range(4))
    ops.bn_train_stats(y, gamma, beta, rm, rv, 0.1, 1e-5, mean, invstd, scale, shift, ws)
    bits = torch.zeros(y.numel() // 8, device=DEV, dtype=torch.uint8)
    out = ops.bn_apply(y, scale, shift, relu=relu, residual=res, relu_bits=bits if relu else None)
    dg, db, dy, dm = torch.empty(C_, device=DEV), torch.empty(C_, device=DEV), torch.empty_like(y), torch.empty_like(y)
    ops.bn_train_bwd(dout, bits if relu else None, y, mean, invstd, gamma, dg, db, dy, ws, dmasked=dm)

    def acc_path():
        rm2, rv2 = rm0.clone(), rv0.clone()
        mean2, invstd2 = torch.empty(C_, device=DEV), torch.empty(C_, device=DEV)
        acc_f = torch.zeros(ops.bn_acc_bytes(C_), device=DEV, dtype=torch.uint8)
        acc_b = torch.zeros(ops.bn_acc_bytes(C_), device=DEV, dtype=torch.uint8)
        ops.bn_stats_acc(y, acc_f)
        bits2 = torch.zeros(y.numel() // 8, device=DEV, dtype=torch.uint8)
        out2 = ops.bn_apply_acc(y, acc_f, gamma, beta, rm2, rv2, 0.1, 1e-5, mean2, invstd2, relu=relu, residual=res,
                                relu_bits=bits2 if relu else None)
        dg2, db2, dy2, dm2 = torch.empty(C_, device=DEV), torch.empty(C_, device=DEV), torch.empty_like(y), torch.empty_like(y)
        ops.bn_bwd_acc(dout, bits2 if relu else None, y, mean2, invstd2, gamma, acc_b, dg2, db2, dy2, dmasked=dm2)
        torch.cuda.synchronize()
        return rm2, rv2, mean2, invstd2, bits2, out2, dg2, db2, dy2, dm2

    a = acc_path()
    b = acc_path()
    for t1, t2 in zip(a, b):
        assert torch.equal(t1, t2)                                     # atomics, yet bit-reproducible
    rm2, rv2, mean2, invstd2, bits2, out2, dg2, db2, dy2, dm2 = a
    assert torch.allclose(mean2, mean, rtol=2e-6, atol=1e-6) and torch.allclose(invstd2, invstd, rtol=2e-6)
    assert torch.allclose(rm2, rm, rtol=2e-6, atol=1e-6) and torch.allclose(rv2, rv, rtol=2e-6)
    d_out = (out2.float() - out.float()).abs()
    assert (d_out <= 2.0 ** -7 * out.float().abs() + 1e-6).all()          # at most one bf16 ulp
    assert (d_out > 0).float().mean().item() < 0.02
    if relu:
        assert (bits2 != bits).float().mean().item() < 1e-3
    else:
        assert torch.equal(dm2, dm)
    assert rel_err(dg2, dg) < 1e-4 and rel_err(db2, db) < 1e-4 and rel_err(dy2.float(), dy.float()) < 2e-3


def test_bn_accumulator_poison_and_exactness():
    """Inf/NaN anywhere in a channel reads back as NaN statistics for that channel only; a channel of exactly representable values gives
    the exact mean (the integer accumulators add the block partials without rounding)."""
    C_ = 64
    y = torch.zeros(2, 16, 16, C_, device=DEV)
    y[..., 1] = 3.0
    y[0, 3, 5, 2] = float("inf")
    y[..., 4] = torch.arange(512, device=DEV, dtype=torch.float32).view(2, 16, 16) - 200.0
    y = bf(y)
    acc = torch.zeros(ops.bn_acc_bytes(C_), device=DEV, dtype=torch.uint8)
    ops.bn_stats_acc(y, acc)
    mean, invstd = torch.empty(C_, device=DEV), torch.empty(C_, device=DEV)
    ops.bn_apply_acc(y, acc, None, None, None, None, 0.1, 1e-5, mean, invstd, relu=False)
    torch.cuda.synchronize()
    assert mean[0].item() == 0.0 and mean[1].item() == 3.0 and torch.isnan(mean[2]).item()
    assert mean[4].item() == y[..., 4].double().mean().item()
    assert not torch.isnan(mean[3]).item() and abs(invstd[1].item() - 1.0 / (1e-5 ** 0.5)) / (1.0 / (1e-5 ** 0.5)) < 1e-6


# ------------------------------------------------------------------ conv data gradient = forward kernel on repacked weights
@pytest.mark.parametrize("cin,cout,k,dil,hw", [(64, 64, 3, 1, (24, 32)), (128, 128, 3, 1, (16, 32)), (128, 256, 3, 2, (16, 32)),
                                               (256, 256, 3, 2, (12, 16)), (512, 512, 3, 4, (12, 16)), (256, 512, 1, 1, (12, 16))])
def test_conv_dgrad_matches_autograd(cin, cout, k, dil, hw):
    torch.manual_seed(cin + cout + k)
    B, (H, W) = 2, hw
    pad = dil * (k - 1) // 2
    w = torch.randn(cout, cin, k, k, device=DEV) * (2.0 / (k * k * cout)) ** 0.5
    dy = bf(torch.randn(B, H, W, cout, device=DEV))
    extra = bf(torch.randn(B, H, W, cin, device=DEV))
    wd = ops.pack_conv_weights_dgrad(w)
    one, zero = torch.ones(cin, device=DEV), torch.zeros(cin, device=DEV)
    dx = ops.conv_bn_act(dy, wd, one, zero, stride=1, pad=pad, dil=dil, relu=False, residual=extra)
    w_b = bf(w).float()
    ref = torch.nn.grad.conv2d_input((B, cin, H, W), w_b, nchw(dy.float()), stride=1, padding=pad, dilation=dil) + nchw(extra.float())
    got = nchw(dx.float())
    assert rel_err(got, ref) < 5e-3, rel_err(got, ref)


@pytest.mark.parametrize("k", [3, 1])
def test_conv_dgrad_stride2_via_zero_insertion(k):
    torch.manual_seed(k)
    B, H, W, cin, cout = 2, 24, 32, 64, 128
    pad = (k - 1) // 2
    w = torch.randn(cout, cin, k, k, device=DEV) * 0.05
    Ho, Wo = ops.conv_out_hw(H, W, k, 2, pad, 1)
    dy = bf(torch.randn(B, Ho, Wo, cout, device=DEV))
    up = ops.zero_insert2x(dy)
    assert tuple(up.shape) == (B, H, W, cout)
    wd = ops.pack_conv_weights_dgrad(w)
    one, zero = torch.ones(cin, device=DEV), torch.zeros(cin, device=DEV)
    dx = ops.conv_bn_act(up, wd, one, zero, stride=1, pad=k - 1 - pad, dil=1, relu=False)
    ref = torch.nn.grad.conv2d_input((B, cin, H, W), bf(w).float(), nchw(dy.float()), stride=2, padding=pad)
    assert rel_err(nchw(dx.float()), ref) < 5e-3


# ------------------------------------------------------------------ conv weight gradient (tcgen05, MN-major operands)
@pytest.mark.parametrize("cin,cout,k,stride,dil,B,hw", [
    (64, 64, 3, 1, 1, 2, (24, 32)),      # layer1 shape (Cout = 64: two taps per unit, the shift on dY)
    (64, 64, 3, 1, 1, 3, (21, 27)),      # the same with ragged tiles: zero-filled dY boxes on every side
    (64, 64, 3, 1, 2, 2, (24, 32)),      # ... and dilation 2
    (64, 128, 3, 2, 1, 2, (24, 32)),     # layer2.0.conv1 (stride 2 through the tensor map's element strides)
    (64, 128, 1, 2, 1, 2, (24, 32)),     # layer2.0.downsample
    (128, 128, 3, 1, 1, 3, (12, 16)),
    (128, 256, 3, 1, 2, 2, (12, 16)),    # layer3.0.conv1, dilation 2
    (256, 256, 3, 1, 2, 2, (12, 32)),
    (256, 512, 1, 1, 1, 2, (12, 16)),    # layer4.0.downsample
    (512, 512, 3, 1, 4, 1, (12, 16)),    # layer4, dilation 4
    (128, 128, 3, 1, 1, 1, (10, 21)),    # ragged tiles (zero-filled boxes)
])
def test_conv_wgrad_matches_autograd(cin, cout, k, stride, dil, B, hw):
    torch.manual_seed(cin * 3 + cout + k + stride)
    H, W = hw
    pad = dil * (k - 1) // 2
    Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
    x = bf(torch.randn(B, H, W, cin, device=DEV))
    dy = bf(torch.randn(B, Ho, Wo, cout, device=DEV))
    dw = torch.full((cout, cin, k, k), 7.0, device=DEV)            # must be overwritten, not accumulated into
    ops.conv_wgrad(x, dy, dw, k=k, stride=stride, pad=pad, dil=dil)
    ref = torch.nn.grad.conv2d_weight(nchw(x.float()).double(), (cout, cin, k, k), nchw(dy.float()).double(), stride=stride, padding=pad,
                                      dilation=dil)
    assert rel_err(dw, ref) < 1e-5, rel_err(dw, ref)              # exact products of bf16 operands, fp32 accumulation
    dw2 = dw.clone()
    ops.conv_wgrad(x, dy, dw2, k=k, stride=stride, pad=pad, dil=dil, accumulate=True)
    assert rel_err(dw2, 2 * ref) < 1e-5


@pytest.mark.parametrize("B,H,W", [(2, 64, 96), (3, 72, 104), (1, 480, 640)])
def test_stem_wgrad_matches_autograd(B, H, W):
    """tcgen05 stem weight gradient (MN-major operands, accumulator resident in TMEM over all tiles of a CTA) vs fp64 autograd on
    the same operands (x rounded to bf16 as in the forward stem, dy bf16); ragged tiles (Ho % 8, Wo % 16 != 0) and accumulate."""
    torch.manual_seed(3)
    x = torch.rand(B, 3, H, W, device=DEV)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    dy = bf(torch.randn(B, Ho, Wo, 64, device=DEV))
    dw = torch.empty(64, 3, 7, 7, device=DEV)
    ops.stem_wgrad(x, dy, dw)
    ref = torch.nn.grad.conv2d_weight(bf(x).double(), (64, 3, 7, 7), nchw(dy.float()).double(), stride=2, padding=3)
    assert rel_err(dw, ref) < 2e-5
    dw1 = dw.clone()
    ops.stem_wgrad(x, dy, dw, accumulate=True)
    assert rel_err(dw, 2 * ref) < 2e-5
    ops.stem_wgrad(x, dy, dw)                      # deterministic: fixed-order reduction of the per-CTA partials
    assert torch.equal(dw, dw1)


# ------------------------------------------------------------------ maxpool backward (first-maximum routing, ties from ReLU zeros)
@pytest.mark.parametrize("H,W", [(24, 40), (23, 37), (6, 5)])
def test_maxpool_backward_matches_autograd_with_ties(H, W):
    torch.manual_seed(5)
    B, C_ = 2, 64
    x = bf(F.relu(torch.randn(B, H, W, C_, device=DEV)))           # ~half zeros: many tied windows
    Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
    dout = bf(torch.randn(B, Ho, Wo, C_, device=DEV))
    dx = ops.maxpool3x3s2_bwd(dout, x)
    x32 = nchw(x.float()).requires_grad_(True)
    F.max_pool2d(x32, 3, 2, 1).backward(nchw(dout.float()))
    got, ref = nchw(dx.float()), x32.grad
    # sums of up to 4 bf16 gradients are rounded to bf16 once
    assert torch.allclose(got, ref, atol=2e-2, rtol=1e-2)
    assert torch.equal(got != 0, bf(ref).float() != 0) or rel_err(got, ref) < 5e-3
    # the training step's split form: forward with recorded indices (== the forward max-pool, bit for bit) + gather (== the call above)
    y_idx, idx = ops.maxpool3x3s2_fwd_idx(x)
    assert torch.equal(y_idx, ops.maxpool3x3s2(x))
    assert torch.equal(ops.maxpool3x3s2_bwd_idx(dout, idx, H, W), dx)


# ------------------------------------------------------------------ head (training): logits forward and backward
@pytest.mark.parametrize("K", [4, 7])
def test_head_logits_forward_and_backward_match_autograd(K):
    torch.manual_seed(K)
    B, h, w, C_, H, W = 2, 8, 12, 512, 64, 96
    feat = bf(torch.randn(B, h, w, C_, device=DEV))
    w_fc = torch.randn(K, C_, device=DEV) * 0.05
    b_fc = torch.randn(K, device=DEV) * 0.1
    up = ops.head_logits(feat, w_fc, b_fc, H, W)
    f32 = nchw(feat.float()).requires_grad_(True)
    w32, b32 = w_fc.clone().requires_grad_(True), b_fc.clone().requires_grad_(True)
    ref = F.interpolate(F.conv2d(f32, w32.view(K, C_, 1, 1), b32), size=(H, W), mode="bilinear", align_corners=True)
    assert torch.allclose(up, ref, atol=2e-5, rtol=1e-5)
    g = torch.randn(B, K, H, W, device=DEV) * 1e-4
    ref.backward(g)
    dfeat = torch.empty_like(feat)
    dw, db = torch.empty(K, C_, device=DEV), torch.empty(K, device=DEV)
    ops.head_bwd(g, feat, w_fc, dfeat, dw, db)
    assert rel_err(dw, w32.grad) < 1e-4 and rel_err(db, b32.grad) < 1e-4
    assert rel_err(nchw(dfeat.float()), f32.grad) < 5e-3         # bf16 rounding of dfeat


# ------------------------------------------------------------------ conv + BatchNorm statistics in one launch (epilogue-gathered sums)
CONV_STATS_CASES = [
    # B, H, W, cin, cout, k, stride, dil     -> kernel
    (2, 24, 32, 64, 64, 3, 1, 1),      # conv_tc_c64 (layer1)
    (3, 21, 27, 64, 64, 3, 1, 1),      # conv_tc_c64, ragged tiles in both directions
    (2, 30, 40, 64, 128, 3, 2, 1),     # conv_tc2<128> (layer2.0 conv1, stride 2)
    (2, 30, 40, 64, 128, 1, 2, 1),     # conv_tc2<128> (1x1 downsample)
    (2, 60, 80, 128, 128, 3, 1, 1),    # conv_tc2h<128> with strip patches (60 rows)
    (1, 27, 21, 128, 256, 3, 1, 2),    # conv_tc2h, ragged
    (2, 60, 80, 256, 256, 3, 1, 2),    # conv_tc2h<256>
    (1, 60, 80, 256, 512, 3, 1, 4),    # conv_tc2<256>, two N tiles
    (4, 60, 80, 512, 512, 3, 1, 4),    # conv_tc2, more tiles than CTA pairs
    (1, 16, 16, 256, 512, 1, 1, 1),    # 1x1 downsample of layer4
]


@pytest.mark.parametrize("case", CONV_STATS_CASES)
def test_conv_epilogue_statistics_match_standalone_reduction(case):
    """hk_conv_bn_stats_fwd: the conv output is bit-identical to hk_conv_bn_act_fwd and the accumulated (sum y, sum y^2) equal what
    hk_bn_stats_acc computes from that output -- read back through hk_bn_apply_fwd_acc as (mean, invstd) -- to fp32 rounding of the
    partial sums (different partition of the pixels into partial sums); bit-reproducible run to run."""
    B, H, W, cin, cout, k, stride, dil = case
    g = torch.Generator().manual_seed(5 + cin + cout)
    pad = dil * (k - 1) // 2
    x = bf((torch.randn(B, H, W, cin, generator=g) + 0.3).to(DEV))
    w = (torch.randn(cout, cin, k, k, generator=g) * (2.0 / (k * k * cin)) ** 0.5).to(DEV)
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, torch.bfloat16)
    one, zero = torch.ones(cout, device=DEV), torch.zeros(cout, device=DEV)
    y_ref = ops.conv_bn_act(x, wp, one, zero, stride=stride, pad=pad, dil=dil, relu=False)
    acc_ref = torch.zeros(ops.bn_acc_bytes(cout), device=DEV, dtype=torch.uint8)
    ops.bn_stats_acc(y_ref, acc_ref)

    def fused():
        acc = torch.zeros(ops.bn_acc_bytes(cout), device=DEV, dtype=torch.uint8)
        y = ops.conv_bn_stats(x, wp, one, zero, acc, stride=stride, pad=pad, dil=dil)
        torch.cuda.synchronize()
        return y, acc

    y1, acc1 = fused()
    y2, acc2 = fused()
    assert torch.equal(y1, y_ref) and torch.equal(y1, y2)
    assert torch.equal(acc1, acc2)                                   # deterministic
    stats = []
    for acc in (acc_ref, acc1):
        mean, invstd = torch.empty(cout, device=DEV), torch.empty(cout, device=DEV)
        ops.bn_apply_acc(y_ref, acc, None, None, None, None, 0.1, 1e-5, mean, invstd, relu=False)
        stats.append((mean.clone(), invstd.clone()))
    y32 = y_ref.float().reshape(-1, cout)
    assert torch.allclose(stats[1][0], y32.double().mean(0).float(), rtol=1e-5, atol=1e-6)
    assert torch.allclose(stats[1][0], stats[0][0], rtol=2e-6, atol=1e-6) and torch.allclose(stats[1][1], stats[0][1], rtol=1e-5)


# ------------------------------------------------------------------ all conv weights repacked in one launch (training repacks every step)
def test_pack_weights_many_tiled_equals_elementwise():
    """hk_pack_conv_weights_many_tiled (shared-memory tiles) against hk_pack_conv_weights_many (element-wise gather) and against the
    single-conv packers: identical bf16 bytes in the forward (cout,kh,kw,cin) and the data-gradient (cin,kh,kw flipped,cout) layouts."""
    _check_pack_weights_many_tiled(DEV)


def test_pack_weights_many_tiled_on_a_second_device():
    """The same on cuda:0 and then on cuda:1 in one process: the shared-memory opt-in of the tiled packer is per device, so its first
    launch on the second device must set it again."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    for dev in ("cuda:0", "cuda:1"):
        _check_pack_weights_many_tiled(dev)


def _check_pack_weights_many_tiled(dev):
    with torch.cuda.device(dev):   # tensors, current stream and launch all on `dev`
        import ctypes as C
        import numpy as np
        from hulk_keypoints_b200._lib import lib, ptr, check, stream_ptr
        shapes = [(64, 64, 3), (128, 64, 3), (128, 64, 1), (256, 128, 3), (512, 256, 1), (512, 512, 3)]
        g = torch.Generator().manual_seed(9)
        ws = [torch.randn(co, ci, k, k, generator=g).to(dev) for co, ci, k in shapes]
        outs = {}
        for tiled in (False, True):
            f = [torch.zeros(co, k, k, ci, device=dev, dtype=torch.bfloat16) for co, ci, k in shapes]
            d = [torch.zeros(ci, k, k, co, device=dev, dtype=torch.bfloat16) for co, ci, k in shapes]
            dt = np.dtype([("w", "<u8"), ("f", "<u8"), ("d", "<u8"), ("cout", "<i4"), ("cin", "<i4"), ("khw", "<i4"), ("r", "<i4")])
            arr = np.zeros(len(shapes), dtype=dt)
            for i, (co, ci, k) in enumerate(shapes):
                arr[i] = (ws[i].data_ptr(), f[i].data_ptr(), d[i].data_ptr(), co, ci, k * k, 0)
            items = torch.from_numpy(arr.view(np.uint8).copy()).to(dev)
            mx = max(co * ci * k * k for co, ci, k in shapes)
            if tiled:
                check(lib().hk_pack_conv_weights_many_tiled(ptr(items), len(shapes), 9, C.c_longlong(mx), stream_ptr()), "tiled")
            else:
                check(lib().hk_pack_conv_weights_many(ptr(items), len(shapes), C.c_longlong(mx), stream_ptr()), "elementwise")
            torch.cuda.synchronize()
            outs[tiled] = (f, d)
        for i, (co, ci, k) in enumerate(shapes):
            assert torch.equal(outs[True][0][i], outs[False][0][i]) and torch.equal(outs[True][1][i], outs[False][1][i]), shapes[i]
            wp, _, _ = ops.pack_conv_weights(ws[i], None, 1e-5, torch.bfloat16)
            assert torch.equal(outs[True][0][i], wp)
            assert torch.equal(outs[True][1][i], ops.pack_conv_weights_dgrad(ws[i]))
