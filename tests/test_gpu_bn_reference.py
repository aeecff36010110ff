"""Train-mode BatchNorm kernels against exact integer sums and fp64 references, at the BatchNorm shapes of the train step.

Independent of (and stricter than) the BatchNorm tests of test_gpu_train_kernels.py, which compare the two kernel paths with each other
and with autograd on zero-mean gradients.  Here:

  A. Exact sums.  Data on the grid k/8 with P*K^2 < 2^24 makes every fp32 partial sum exact in any order, so the 128-bit fixed-point
     accumulators (hk_bn_acc.cuh, unit 2^-50) must hold exactly sum(k) * 2^47 and sum(k^2) * 2^44, and both paths must return the
     exact mean, dbeta = sum d' and dgamma = sum d'*y -- no tolerance.  The conv-epilogue statistics use centre-tap weights so that
     y = x[..., co % cin] + bias[co] exactly, with a non-zero bias: a counted out-of-image (ragged or phantom-box) row changes a sum.
  B. Semantics against fp64 at the benchmark shapes, on both paths (three-launch: bn_train_stats / bn_apply / bn_train_bwd;
     accumulator: bn_stats_acc / bn_apply_acc / bn_bwd_acc).  The backward uses reduction-dominated gradients
     d' = alpha_c + beta_c*xhat + 0.01*noise, so an error of relative size 1/P in dbeta/N or dgamma/N shows in dy.
  C. Conditioning: both paths form var = E[y^2] - mean^2 from fp32 partial sums and the accumulator backward forms
     sum d'*y - mean*sum d' in fp32, so their error grows as (1 + r^2) * 2^-24 per added row, r = |mean|/std of a channel.  The envelope
     (1 + r^2) * 64 * 2^-24 is asserted at every r of the sweep (which includes R_REALISTIC = 4x the largest r of the trained fixture) and
     the errors printed; the tight bars of B are asserted where they were measured to hold (forward r <= R_TIGHT, backward r <= R_REALISTIC).

Run with -s to see the measured errors.  The whole file takes about 7 s on a B200."""
import math

import numpy as np
import pytest
import torch

from hulk_keypoints_b200 import ops
from oracle import keypoints_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U24 = 2.0 ** -24
EPS, MOM = 1e-5, 0.1
# Largest |mean|/std of any BatchNorm input of the trained fixture F-trn (k4_480x640) in a train-mode forward at 4x480x640, disc and
# uniform-noise images (tools/diag_bn_conditioning.py): 7.0, layer4.1.bn1 on disc images.  The issue-level target is the tight bars up to
# R_REALISTIC = four times that; measured on a B200 they hold up to R_TIGHT = 16 and the accumulator path's invstd exceeds BAR_INVSTD at
# r = 28 (1.09e-5; three-launch 9.1e-6) -- see test_conditioning_forward_statistics and DESIGN 3.5.
R_FTRN = 7.0
R_REALISTIC = 4 * R_FTRN
R_TIGHT = 16
# Tight bars (B, and C up to R_REALISTIC): |mean - mean64| / sqrt(var64 + eps) and |invstd / invstd64 - 1|; dbeta, dgamma relative to
# sum |d'| and sum |d'|*(1 + |xhat|).  Worst measured on a B200: 2.7e-6 (B), 5.0e-6 (B: 4.1e-6; sweep at r = 16: 5.0e-6), 2.3e-7.
BAR_MEAN, BAR_INVSTD, BAR_DPARAM = 5e-6, 1e-5, 1e-5
# Empirical envelope factor of the conditioning model (1 + r^2) * ENVELOPE * 2^-24.  Not a summation depth: a partial passes through
# about 2 000 fp32 additions (a thread's rows, the block's rows, the 8 CTAs of a cluster) before the exact or double stage, but rounding
# errors of random sign grow like sqrt(depth); 64 bounds every measured error with a wide margin and catches a worse summation.
ENVELOPE = 64


# ------------------------------------------------------------------ the train step's BatchNorm shapes, from the network itself
def train_step_bn_shapes(H=480, W=640, batches=(1, 4, 32)):
    stem, blocks, _ = O.network_spec()
    shapes = set()
    for B in batches:
        h, w = ops.conv_out_hw(H, W, stem.k, stem.stride, stem.pad, stem.dil)
        shapes.add((B * h * w, stem.cout))
        h, w = ops.conv_out_hw(h, w, 3, 2, 1, 1)                         # max-pool 3x3 s2 p1
        for blk in blocks:
            h1, w1 = ops.conv_out_hw(h, w, blk.conv1.k, blk.conv1.stride, blk.conv1.pad, blk.conv1.dil)
            shapes.add((B * h1 * w1, blk.conv1.cout))
            h2, w2 = ops.conv_out_hw(h1, w1, blk.conv2.k, blk.conv2.stride, blk.conv2.pad, blk.conv2.dil)
            shapes.add((B * h2 * w2, blk.conv2.cout))
            if blk.down is not None:
                hd, wd = ops.conv_out_hw(h, w, blk.down.k, blk.down.stride, blk.down.pad, blk.down.dil)
                shapes.add((B * hd * wd, blk.down.cout))
            h, w = h2, w2
    return sorted(shapes)


NET_SHAPES = train_step_bn_shapes()


def _rows(C):
    return 256 // (C // 8)                                              # rows of one reduce block pass (256 threads, 8 channels each)


# edges: P smaller than one chunk (whole clusters idle), one chunk +- 1 (chunk = rows x rows-in-flight: 4 in the statistics kernel, 2 in
# the backward reduce), rows x 4 x 1184 +- 1 (1184 = BN_ACC_MAX_BLOCKS, the cap of the reduce grid: a tail chunk at a few hundred
# thousand rows; the grid itself comes from the occupancy API, so this is not a grid-multiple boundary), and the admitted channel counts
# outside the network
EDGE_SHAPES = sorted({(1, 64), (2, 64), (3, 512), (7, 64), (7, 2048),
                      (_rows(64) * 4 - 1, 64), (_rows(64) * 4 + 1, 64), (_rows(64) * 2 - 1, 64), (_rows(64) * 2 + 1, 64),
                      (_rows(512) * 4 - 1, 512), (_rows(512) * 4 + 1, 512),
                      (_rows(64) * 4 * 1184 - 1, 64), (_rows(64) * 4 * 1184 + 1, 64), (_rows(256) * 4 * 1184 + 1, 256),
                      (4801, 8), (19, 8), (4801, 16), (4801, 32), (4801, 1024), (4801, 2048)})
ALL_SHAPES = NET_SHAPES + [s for s in EDGE_SHAPES if s not in NET_SHAPES]


def shape_id(s):
    return f"P{s[0]}-C{s[1]}"


def test_shape_list_covers_the_train_step():
    """The derived list holds the stem, layer-1 and 60x80 shapes of B = 32 (and nothing the kernels do not admit)."""
    assert (32 * 240 * 320, 64) in NET_SHAPES and (32 * 120 * 160, 64) in NET_SHAPES
    assert {(32 * 60 * 80, c) for c in (128, 256, 512)} <= set(NET_SHAPES)
    assert len(NET_SHAPES) == 14                          # B = 1 and B = 4 share the stem / layer-1 P of 76 800 and 19 200
    for P, C in ALL_SHAPES:
        assert P > 0 and 8 <= C <= 2048 and 256 % (C // 8) == 0


# ------------------------------------------------------------------ helpers
def gpu_gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def grid_ints(P, C, K, gen):
    """(P, C) int32 with |k| <= K and a distribution per channel: symmetric, mostly negative, constant (the sum counts the rows), mostly
    positive, strictly negative (large negative totals: the high word and the two's-complement carries of the accumulators)."""
    c = torch.arange(C, device=DEV)
    mode = c % 5
    q = K // 4
    lo = torch.full((C,), -K, device=DEV, dtype=torch.int64)
    hi = torch.full((C,), K, device=DEV, dtype=torch.int64)
    hi[mode == 1] = q
    lo[mode == 3] = -q
    hi[mode == 4] = -1
    const = torch.where(c % 2 == 0, torch.full_like(c, -K), torch.full_like(c, (K + 1) // 2))
    lo = torch.where(mode == 2, const, lo)
    hi = torch.where(mode == 2, const, hi)
    u = torch.rand(P, C, generator=gen, device=DEV)
    k = lo + torch.floor(u * (hi - lo + 1).float()).long()
    return torch.minimum(k, hi).to(torch.int32)


def grid_bound(P):
    """Largest K with P*K^2 < 2^24 (every fp32 partial sum of k/8 and (k/8)^2 exact) and k/8 exact in bf16."""
    K = min(256, math.isqrt((2 ** 24 - 1) // P))
    assert K >= 1 and P * K * K < 2 ** 24
    return K


def acc_ints(acc, C):
    """The 2C accumulators as Python ints (128-bit two's complement, unit 2^-50); asserts that none is poisoned."""
    a = acc.cpu().numpy().view(np.uint64).reshape(2 * C, 4)
    assert not a[:, 2].any(), "poisoned accumulator"
    out = []
    for lo, hi in zip(a[:, 0].tolist(), a[:, 1].tolist()):
        v = (int(hi) << 64) | int(lo)
        out.append(v - (1 << 128) if hi >> 63 else v)
    return out


def assert_acc_exact(acc, C, sums, squares, what):
    """acc holds exactly sums[c] / 8 and squares[c] / 64 (sums, squares: integer tensors of the k grid)."""
    got = acc_ints(acc, C)
    want = [int(s) << 47 for s in sums.tolist()] + [int(q) << 44 for q in squares.tolist()]
    bad = [i for i in range(2 * C) if got[i] != want[i]]
    assert not bad, f"{what}: {len(bad)} accumulators differ, first [{bad[0]}] {got[bad[0]]} != {want[bad[0]]}"


def pack_bits(mask):
    """bool (..., C) -> one bit per element, 8 consecutive elements per byte (the layout of relu_bits)."""
    m = mask.reshape(-1, 8).to(torch.int32) << torch.arange(8, device=mask.device, dtype=torch.int32)
    return m.sum(1).to(torch.uint8)


def bf16_ulp(x):
    """one bf16 ulp at |x| (x fp64), 0 where x == 0"""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - 8))


def new_acc(C):
    return torch.zeros(ops.bn_acc_bytes(C), device=DEV, dtype=torch.uint8)


def forward(path, y, gamma, beta, rm, rv, residual=None, relu=True, bits=None):
    """-> (mean, invstd, out) of one train-mode BatchNorm forward on `path` ("three": 3 launches, "acc": the accumulator pair)"""
    C = y.shape[-1]
    mean, invstd = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    if path == "three":
        scale, shift = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        ops.bn_train_stats(y, gamma, beta, rm, rv, MOM, EPS, mean, invstd, scale, shift, ops.bn_workspace(C, DEV))
        out = ops.bn_apply(y, scale, shift, relu=relu, residual=residual, relu_bits=bits)
    else:
        acc = new_acc(C)
        ops.bn_stats_acc(y, acc)
        out = ops.bn_apply_acc(y, acc, gamma, beta, rm, rv, MOM, EPS, mean, invstd, relu=relu, residual=residual, relu_bits=bits)
    return mean, invstd, out


def backward(path, dout, mask, y, mean, invstd, gamma, dgamma, dbeta, dy, dmasked=None, accumulate=False):
    if path == "three":
        ops.bn_train_bwd(dout, mask, y, mean, invstd, gamma, dgamma, dbeta, dy, ops.bn_workspace(y.shape[-1], DEV), dmasked=dmasked,
                         accumulate=accumulate)
    else:
        ops.bn_bwd_acc(dout, mask, y, mean, invstd, gamma, new_acc(y.shape[-1]), dgamma, dbeta, dy, dmasked=dmasked, accumulate=accumulate)


def channel_data(P, C, r_values, seed):
    """bf16 y (P, C) with per-channel |mean|/std = r (drawn from r_values when it is a pair (lo, hi), else that value for every channel),
    random sign and scale."""
    g = torch.Generator().manual_seed(seed)
    sd = torch.exp(torch.empty(C).uniform_(-1.5, 1.5, generator=g))
    if isinstance(r_values, tuple):
        r = torch.empty(C).uniform_(*r_values, generator=g)
    else:
        r = torch.full((C,), float(r_values))
    sign = torch.where(torch.rand(C, generator=g) < 0.5, -1.0, 1.0)
    mu = (sign * r * sd).to(DEV)
    y = (mu + sd.to(DEV) * torch.randn(P, C, generator=gpu_gen(seed), device=DEV)).to(torch.bfloat16)
    return y, g


def ref_stats(y):
    y64 = y.double()
    m = y64.mean(0)
    v = (y64 - m).square_().mean(0)
    return y64, m, v


def fwd_errors(mean, invstd, m64, v64):
    s = torch.sqrt(v64 + EPS)
    e_mean = (mean.double() - m64).abs() / s
    e_inv = (invstd.double() * s - 1.0).abs()
    # relative error of the variance the kernel used (1/invstd^2 - eps), against var64
    var_k = 1.0 / invstd.double().square() - EPS
    e_var = (var_k - v64).abs() / v64.clamp_min(1e-30)
    return e_mean, e_inv, e_var


# ================================================================== A. exact sums
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=shape_id)
def test_statistics_exact_on_integer_grid(shape):
    """bn_stats_acc: the accumulators hold exactly sum(k) * 2^47 and sum(k^2) * 2^44 (raw bytes); bn_apply_acc and bn_train_stats both
    return mean == float(sum / P) bit for bit."""
    P, C = shape
    K = grid_bound(P)
    k = grid_ints(P, C, K, gpu_gen(P + C))
    y = (k.float() / 8).to(torch.bfloat16)
    assert torch.equal((y.float() * 8).to(torch.int32), k)
    sums, squares = k.sum(0, dtype=torch.int64), k.square().sum(0, dtype=torch.int64)
    if P >= 4800:
        assert sums.min().item() < -(2 ** 14) * 8          # some channel total below -2^14: the high word and its carries are used
    acc = new_acc(C)
    ops.bn_stats_acc(y, acc)
    assert_acc_exact(acc, C, sums, squares, "bn_stats_acc")
    want = torch.from_numpy((sums.cpu().numpy().astype(np.float64) / 8.0 / float(P)).astype(np.float32)).to(DEV)
    for path in ("acc", "three"):
        if path == "acc":
            mean, invstd = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
            ops.bn_apply_acc(y, acc, None, None, None, None, MOM, EPS, mean, invstd, relu=False)
        else:
            mean, invstd, _ = forward("three", y, None, None, None, None, relu=False)
        assert torch.equal(mean, want), (path, (mean - want).abs().max().item())


@pytest.mark.parametrize("shape", ALL_SHAPES, ids=shape_id)
def test_backward_sums_exact_on_integer_grid(shape):
    """With mean = 0, invstd = 1 and gamma = 1 (xhat = y): dbeta == sum d' and dgamma == sum d'*y over the masked elements, exactly, on
    both paths, with no mask, a bf16-output mask (> 0 keeps: 0, -0 and negatives drop) and a bit mask; d' (dmasked) exact; the backward
    accumulators exact; accumulate=True adds to what is there."""
    P, C = shape
    K = grid_bound(P)
    g = gpu_gen(7 * P + C)
    ky, kd = grid_ints(P, C, K, g), grid_ints(P, C, K, g).flip(1)
    y, dout = (ky.float() / 8).to(torch.bfloat16), (kd.float() / 8).to(torch.bfloat16)
    keep = torch.rand(P, C, generator=g, device=DEV) < 0.6
    neg = torch.randint(0, 3, (P, C), generator=g, device=DEV)
    drop = torch.where(neg == 0, 0.0, torch.where(neg == 1, -0.0, -1.5))
    masks = {"none": (None, torch.ones_like(keep)),
             "bf16": (torch.where(keep, torch.rand(P, C, generator=g, device=DEV) + 2.0 ** -20, drop).to(torch.bfloat16), keep),
             "bits": (pack_bits(keep), keep)}
    zero, one = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    for mname, (mask, keep_m) in masks.items():
        kdm = kd * keep_m
        s1, s2 = kdm.sum(0, dtype=torch.int64), (kdm * ky).sum(0, dtype=torch.int64)
        want_db = (s1.double() / 8).float()
        want_dg = (s2.double() / 64).float()
        dm_want = torch.where(keep_m, dout, torch.zeros_like(dout))
        for path in ("three", "acc"):
            dg, db, dy, dm = torch.empty(C, device=DEV), torch.empty(C, device=DEV), torch.empty_like(y), torch.empty_like(y)
            if path == "acc":
                acc = new_acc(C)
                ops.bn_bwd_acc(dout, mask, y, zero, one, one, acc, dg, db, dy, dmasked=dm)
                assert_acc_exact(acc, C, s1, s2, f"bn_bwd_acc/{mname}")        # sum d' = s1/8, sum d'*y = s2/64
            else:
                backward("three", dout, mask, y, zero, one, one, dg, db, dy, dmasked=dm)
            assert torch.equal(db, want_db), (path, mname, (db - want_db).abs().max().item())
            assert torch.equal(dg, want_dg), (path, mname, (dg - want_dg).abs().max().item())
            assert torch.equal(dm, dm_want), (path, mname)
            backward(path, dout, mask, y, zero, one, one, dg, db, dy, accumulate=True)
            assert torch.equal(db, 2 * want_db) and torch.equal(dg, 2 * want_dg), (path, mname, "accumulate")


# conv + statistics in one launch, on the kernels the engine uses for the train step's convolutions
CONV_CASES = [
    # B, H, W, cin, cout, k, stride, dil     -> kernel
    (1, 120, 160, 64, 64, 3, 1, 1),    # conv_tc_c64 (layer1, B = 1)
    (3, 21, 27, 64, 64, 3, 1, 1),      # conv_tc_c64, ragged tiles in both directions
    (1, 120, 160, 64, 128, 3, 2, 1),   # conv_tc2<128>, stride 2 (layer2.0.conv1, B = 1): 60x80 = 75 boxes, odd -> a phantom box
    (1, 120, 160, 64, 128, 1, 2, 1),   # conv_tc2<128>, 1x1 stride 2 (layer2.0.downsample): odd box count
    (2, 29, 37, 64, 128, 3, 2, 1),     # conv_tc2<128>, stride 2, ragged
    (1, 60, 80, 128, 128, 3, 1, 1),    # conv_tc2h<128> (layer2, B = 1)
    (3, 60, 80, 128, 128, 3, 1, 1),    # conv_tc2h<128>, three images
    (1, 27, 21, 128, 256, 3, 1, 2),    # conv_tc2h, ragged
    (1, 60, 80, 256, 256, 3, 1, 2),    # conv_tc2h<256> (layer3)
    (1, 60, 80, 256, 512, 3, 1, 4),    # conv_tc2<256>, two N tiles, 75 boxes (layer4.0.conv1, B = 1)
    (1, 60, 80, 256, 512, 1, 1, 1),    # conv_tc2<256>, 1x1 (layer4.0.downsample), odd box count
    (4, 60, 80, 512, 512, 3, 1, 4),    # conv_tc2<256>, more tiles than CTA pairs
]


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv_epilogue_statistics_exact(case):
    """hk_conv_bn_stats_fwd with centre-tap weights w[co, co % cin] = 1 and a non-zero bias on the grid: y == x[..., co % cin] + bias
    exactly (every pad, dilation and stride), and the accumulators hold exactly the sums of y and y^2 over the image.  Every 8th channel
    has zero weights and bias +-1/8, so its sum is exactly +-P/8: a counted ragged or phantom-box row (which stages the bias) shows.
    Every case reaches a specialised epilogue kernel under the default dispatch (hk_conv_bn_stats_fwd falls back to conv + hk_bn_stats_acc only
    outside them)."""
    B, H, W, cin, cout, k, stride, dil = case
    pad = dil * (k - 1) // 2
    Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
    P = B * Ho * Wo
    Kmax = grid_bound(P)
    Kb = max(1, Kmax // 4)
    Kx = max(1, Kmax - Kb)
    g = gpu_gen(cin + cout + H)
    kx = grid_ints(B * H * W, cin, Kx, g).view(B, H, W, cin)
    x = (kx.float() / 8).to(torch.bfloat16)
    co = torch.arange(cout, device=DEV)
    dead = co % 8 == 5
    kb = torch.randint(-Kb, Kb + 1, (cout,), generator=g, device=DEV)
    kb = torch.where(kb == 0, torch.ones_like(kb), kb)
    kb = torch.where(dead, torch.where(co % 16 == 5, 1, -1), kb)
    w = torch.zeros(cout, cin, k, k, device=DEV)
    live = (~dead).nonzero().flatten()
    w[live, live % cin, k // 2, k // 2] = 1.0
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, torch.bfloat16)
    bias = kb.float() / 8
    acc = new_acc(cout)
    y = ops.conv_bn_stats(x, wp, torch.ones(cout, device=DEV), bias, acc, stride=stride, pad=pad, dil=dil)
    xs = kx[:, : Ho * stride: stride, : Wo * stride: stride, :]
    ky = torch.where(dead, 0, xs[..., co % cin]) + kb
    assert ky.abs().max().item() <= Kmax
    assert torch.equal(y, (ky.float() / 8).to(torch.bfloat16)), "conv output"
    kyf = ky.reshape(P, cout).to(torch.int64)
    assert_acc_exact(acc, cout, kyf.sum(0), kyf.square().sum(0), "conv epilogue")


# ================================================================== B. semantics against fp64 at the benchmark shapes
@pytest.mark.parametrize("path", ["three", "acc"])
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=shape_id)
def test_forward_matches_fp64(shape, path):
    """Statistics, running statistics and relu(gamma*xhat + beta + residual) with relu_bits against two-pass fp64 statistics of the same
    bf16 y, at |mean|/std <= 4: mean within BAR_MEAN*std, invstd within BAR_INVSTD, every output within one bf16 ulp of the fp64 value
    (plus 2^-18 of the fp32 terms, for outputs near zero), at least 99 % of the positive ones the correctly rounded fp64 value.
    Measured (B200, all shapes, both paths): mean 2.7e-6 std, invstd 4.1e-6, outputs <= 0.50 ulp beyond the fp32 term, >= 99.97 %
    correctly rounded."""
    P, C = shape
    y, g = channel_data(P, C, (0.0, 4.0), seed=P + C)
    res = (0.5 * torch.randn(P, C, generator=gpu_gen(P + C + 1), device=DEV)).to(torch.bfloat16)
    gamma = (torch.rand(C, generator=g) + 0.5) * torch.where(torch.rand(C, generator=g) < 0.1, -1.0, 1.0)
    beta = 0.3 * torch.randn(C, generator=g)
    rm0, rv0 = 0.1 * torch.randn(C, generator=g), torch.rand(C, generator=g) + 0.5
    gamma, beta, rm0, rv0 = (t.to(DEV) for t in (gamma, beta, rm0, rv0))
    rm, rv = rm0.clone(), rv0.clone()
    bits = torch.zeros(P * C // 8, device=DEV, dtype=torch.uint8)
    mean, invstd, out = forward(path, y, gamma, beta, rm, rv, residual=res, relu=True, bits=bits)
    y64, m64, v64 = ref_stats(y)
    e_mean, e_inv, _ = fwd_errors(mean, invstd, m64, v64)
    # the mean is returned in fp32: half an fp32 ulp of |mean| comes on top of the bar
    assert (e_mean <= BAR_MEAN + U24 * m64.abs() / torch.sqrt(v64 + EPS)).all() and e_inv.max().item() <= BAR_INVSTD, (e_mean.max().item(), e_inv.max().item())
    # running statistics: momentum, unbiased n/(n-1) (n = 1: the biased value, 0)
    s = torch.sqrt(v64 + EPS)
    unb = v64 * P / (P - 1) if P > 1 else v64
    rm_want = (1 - MOM) * rm0.double() + MOM * m64
    rv_want = (1 - MOM) * rv0.double() + MOM * unb
    assert ((rm.double() - rm_want).abs() <= 4 * U24 * (rm0.double().abs() + m64.abs()) + MOM * BAR_MEAN * s).all()
    assert ((rv.double() - rv_want).abs() <= 4 * U24 * (rv0.double() + unb) + MOM * 3 * BAR_INVSTD * unb).all()
    # output
    is64 = 1.0 / s
    sc, sh = gamma.double() * is64, beta.double() - m64 * gamma.double() * is64
    r64 = res.double()
    pre = y64 * sc + sh + r64
    ref = pre.clamp_min(0.0)
    got = out.double()
    slack = 2.0 ** -18 * ((y64 * sc).abs() + sh.abs() + r64.abs())
    err = (got - ref).abs()
    assert (err <= bf16_ulp(ref) + slack).all(), ((err - bf16_ulp(ref) - slack).max().item())
    live = ref > 0                                                   # outputs the ReLU clamps to 0 would match trivially
    exact = (out == ref.float().to(torch.bfloat16))[live].double().mean().item()
    assert exact >= 0.99 or P * C < 2 ** 14, exact                  # (a fraction of a handful of outputs says nothing)
    assert torch.equal(bits, pack_bits(out > 0))
    print(f"\n[fwd {path} P={P} C={C}] measured: mean {e_mean.max().item():.2e} std, invstd {e_inv.max().item():.2e}, "
          f"out correctly rounded {100 * exact:.3f} %, worst {((err - slack).clamp_min(0) / bf16_ulp(ref).clamp_min(1e-300)).max().item():.3f} ulp")


@pytest.mark.parametrize("path", ["three", "acc"])
def test_forward_without_gamma_or_beta(path):
    """gamma=None / beta=None are gamma = 1 / beta = 0, bit for bit, with no running statistics."""
    P, C = 4801, 256
    y, _ = channel_data(P, C, (0.0, 4.0), seed=11)
    one, zero = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)
    ref = forward(path, y, one, zero, None, None, relu=False)
    for gm, bt in ((None, zero), (one, None), (None, None)):
        got = forward(path, y, gm, bt, None, None, relu=False)
        for a, b in zip(got, ref):
            assert torch.equal(a, b)


def grad_case(P, C, path, r_values, seed):
    """A real forward (beta 2..3, so ~99 % of the ReLU mask is set) and reduction-dominated gradients
    d' = bf16(alpha_c + beta_c*xhat + 0.01*noise): most of d' cancels against sum d'/N and xhat*sum d'*xhat/N.  Returns both ReLU
    masks of the forward: relu_bits and the bf16 output."""
    y, g = channel_data(P, C, r_values, seed)
    gamma = ((torch.rand(C, generator=g) + 0.5) * torch.where(torch.rand(C, generator=g) < 0.1, -1.0, 1.0)).to(DEV)
    beta = (2.0 + torch.rand(C, generator=g)).to(DEV)
    res = (0.5 * torch.randn(P, C, generator=gpu_gen(seed + 1), device=DEV)).to(torch.bfloat16)
    bits = torch.zeros(P * C // 8, device=DEV, dtype=torch.uint8)
    mean, invstd, out = forward(path, y, gamma, beta, None, None, residual=res, relu=True, bits=bits)
    alpha, slope = torch.randn(C, generator=g).to(DEV).double(), torch.randn(C, generator=g).to(DEV).double()
    y64 = y.double()
    xhat = (y64 - mean.double()) * invstd.double()
    dout = (alpha + slope * xhat + 0.01 * torch.randn(P, C, generator=gpu_gen(seed + 2), device=DEV, dtype=torch.float64))
    dout = dout.to(torch.bfloat16)
    dprime = torch.where(out > 0, dout.double(), torch.zeros_like(y64))
    return y, y64, gamma, mean, invstd, xhat, dout, bits, out, dprime


def bwd_reference(P, gamma, mean, invstd, xhat, dprime):
    s1, s2 = dprime.sum(0), (dprime * xhat).sum(0)
    a = gamma.double() * invstd.double()
    dy = a * (dprime - s1 / P - xhat * (s2 / P))
    return s1, s2, dy


@pytest.mark.parametrize("path", ["three", "acc"])
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=shape_id)
def test_backward_matches_fp64(shape, path):
    """Reduction-dominated gradients against fp64 on the kernel's own fp32 mean / invstd: dbeta within BAR_DPARAM of sum |d'|, dgamma
    within BAR_DPARAM of sum |d'|*(1 + |xhat|); dy within one bf16 ulp plus the fp32 cancellation term of dy = k0*d' + k1*y + k2, at
    least 99 % correctly rounded; the bf16-output mask gives the same as the bit mask; accumulate=True adds; gamma=None is gamma = 1.
    Measured (B200, all shapes, both paths): dbeta 9.9e-8, dgamma 2.3e-7, dy <= 0.50 ulp beyond the cancellation term, >= 99.6 %
    correctly rounded."""
    P, C = shape
    y, y64, gamma, mean, invstd, xhat, dout, bits, out, dprime = grad_case(P, C, path, (0.0, 4.0), seed=3 * P + C)
    s1, s2, dy_ref = bwd_reference(P, gamma, mean, invstd, xhat, dprime)
    dg, db, dy, dm = torch.empty(C, device=DEV), torch.empty(C, device=DEV), torch.empty_like(y), torch.empty_like(y)
    backward(path, dout, bits, y, mean, invstd, gamma, dg, db, dy, dmasked=dm)
    assert torch.equal(dm.double(), dprime)
    e_db = ((db.double() - s1).abs() / dprime.abs().sum(0).clamp_min(1e-30)).max().item()
    e_dg = ((dg.double() - s2).abs() / (dprime.abs() * (1 + xhat.abs())).sum(0).clamp_min(1e-30)).max().item()
    assert e_db <= BAR_DPARAM and e_dg <= BAR_DPARAM, (e_db, e_dg)
    # the kernel's dy = k0*d' + (k1*y + k2), k0 = gamma*invstd, k1 = -k0*c2*invstd, k2 = -k0*c1 - k1*mean (c1 = dbeta/N, c2 = dgamma/N):
    # fp32 rounding of its terms, plus what the kernel's own (separately checked) dbeta / dgamma errors move c1 and c2 by
    k0 = (gamma.double() * invstd.double()).abs()
    k1 = k0 * (s2 / P).abs() * invstd.double()
    k2 = k0 * (s1 / P).abs() + k1 * mean.double().abs()
    d1, d2 = (db.double() - s1).abs() / P, (dg.double() - s2).abs() / P
    cancel = 2.0 ** -21 * ((k0 * dprime).abs() + k1 * y64.abs() + k2) + k0 * (d1 + xhat.abs() * d2)
    err = (dy.double() - dy_ref).abs()
    ulp = bf16_ulp(dy_ref)
    assert (err <= ulp + cancel).all(), ((err - ulp - cancel).max().item())
    exact = (dy == dy_ref.float().to(torch.bfloat16)).double().mean().item()
    assert exact >= 0.99 or P * C < 2 ** 14, exact
    # the bf16-output mask is the same mask
    dg2, db2, dy2 = torch.empty_like(dg), torch.empty_like(db), torch.empty_like(dy)
    backward(path, dout, out, y, mean, invstd, gamma, dg2, db2, dy2)
    assert torch.equal(dg2, dg) and torch.equal(db2, db) and torch.equal(dy2, dy)
    # accumulate=True adds the same values to what is there; gamma=None is gamma = 1
    backward(path, dout, bits, y, mean, invstd, gamma, dg2, db2, dy2, accumulate=True)
    assert torch.equal(db2, 2 * db) and torch.equal(dg2, 2 * dg) and torch.equal(dy2, dy)
    one = torch.ones(C, device=DEV)
    dy_a, dy_b = torch.empty_like(dy), torch.empty_like(dy)
    backward(path, dout, bits, y, mean, invstd, None, dg2, db2, dy_a)
    backward(path, dout, bits, y, mean, invstd, one, dg2, db2, dy_b)
    assert torch.equal(dy_a, dy_b)
    worst = ((err - cancel).clamp_min(0) / ulp.clamp_min(1e-300)).max().item()
    print(f"\n[bwd {path} P={P} C={C}] measured: dbeta {e_db:.2e}, dgamma {e_dg:.2e}, dy correctly rounded {100 * exact:.3f} %, "
          f"worst {worst:.3f} ulp beyond the cancellation term")


# ================================================================== C. conditioning sweep
COND_SHAPE = (32 * 60 * 80, 128)        # layer2 of the B = 32 step
R_SWEEP = [0, 1, 4, 16, int(R_REALISTIC), 64, 256]


def _model(r):
    """(1 + r^2) * 64 * 2^-24, and never below (1 + r) * 64 * 2^-24 (the mean's bound, larger for r < 1)"""
    return torch.maximum(1.0 + r * r, 1.0 + r) * ENVELOPE * U24


@pytest.mark.parametrize("path", ["three", "acc"])
@pytest.mark.parametrize("r", R_SWEEP)
def test_conditioning_forward_statistics(r, path):
    """Forward statistics at |mean|/std = r for every channel.  Every r: per channel |dmean| <= (1 + r^2) * 64 * 2^-24 * std (plus half
    an fp32 ulp of the returned mean) and |dvar| / var <= (1 + r^2) * 64 * 2^-24, the fp32 E[y^2] - mean^2 envelope.  r <= R_TIGHT: the
    tight bars of B.  Measured (B200; three-launch / accumulator): invstd 3.5e-6 / 5.0e-6 at r = 16, 9.1e-6 / 1.09e-5 at r = 28 (= 4x the
    largest r of F-trn: the accumulator path is above BAR_INVSTD there), 3.5e-5 / 6.8e-5 at r = 64; variance 6.7e-4 / 1.5e-3 at r = 256
    against an envelope of 0.23."""
    P, C = COND_SHAPE
    y, _ = channel_data(P, C, r, seed=100 + r)
    mean, invstd, _ = forward(path, y, None, None, None, None, relu=False)
    _, m64, v64 = ref_stats(y)
    sd = v64.sqrt()
    r_c = m64.abs() / sd
    e_mean, e_inv, e_var = fwd_errors(mean, invstd, m64, v64)
    print(f"\n[cond fwd {path} r={r}] measured (max r {r_c.max().item():.1f}): mean {e_mean.max().item():.2e} std, "
          f"invstd {e_inv.max().item():.2e}, var {e_var.max().item():.2e} (envelope {_model(r_c.max()).item():.2e})")
    assert (e_mean <= _model(r_c) + U24 * r_c).all()
    assert (e_var <= _model(r_c) + 4 * U24).all()
    if r <= R_TIGHT:
        assert (e_mean <= BAR_MEAN + U24 * r_c).all() and e_inv.max().item() <= BAR_INVSTD


@pytest.mark.parametrize("path", ["three", "acc"])
@pytest.mark.parametrize("r", R_SWEEP)
def test_conditioning_backward_reduce(r, path):
    """dbeta / dgamma of reduction-dominated gradients at |mean|/std = r: the tight bar of B up to R_REALISTIC; at every r dgamma within
    (1 + r^2) * 64 * 2^-24 of sum |d'|*(1 + |xhat|) (the accumulator backward's raw moment sum d'*y - mean*sum d').
    Measured (B200): dbeta <= 5.9e-8 and dgamma <= 4.0e-8 at every r on both paths, except the accumulator's dgamma at r = 256: 1.2e-7."""
    P, C = COND_SHAPE
    y, y64, gamma, mean, invstd, xhat, dout, bits, _, dprime = grad_case(P, C, path, r, seed=200 + r)
    s1, s2, _ = bwd_reference(P, gamma, mean, invstd, xhat, dprime)
    dg, db, dy = torch.empty(C, device=DEV), torch.empty(C, device=DEV), torch.empty_like(y)
    backward(path, dout, bits, y, mean, invstd, gamma, dg, db, dy)
    r_c = (y64.mean(0).abs() / y64.std(0, unbiased=False))
    e_db = (db.double() - s1).abs() / dprime.abs().sum(0)
    e_dg = (dg.double() - s2).abs() / (dprime.abs() * (1 + xhat.abs())).sum(0)
    print(f"\n[cond bwd {path} r={r}] measured (max r {r_c.max().item():.1f}): dbeta {e_db.max().item():.2e}, dgamma {e_dg.max().item():.2e} "
          f"(model {_model(r_c.max()).item():.2e})")
    assert (e_db <= ENVELOPE * U24).all()
    assert (e_dg <= _model(r_c)).all()
    if r <= R_REALISTIC:
        assert e_db.max().item() <= BAR_DPARAM and e_dg.max().item() <= BAR_DPARAM
