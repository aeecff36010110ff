"""Convolution kernels bit-exact against fp64 references on integer-grid data, at the train step's and the benchmark's shapes.

Exactness.  Activations, gradients and weights are ternary ({-1, 0, 1}, exact in bf16), so every product is exact and every partial sum
is an integer.  The premises K*max|x|*max|w| < 2^22 (forward, data gradient; K = taps * input channels) and P*max|x|*max|dy| < 2^22
(weight gradient; P = output pixels) are asserted per case: every fp32 partial sum -- in TMEM, in any MMA order, in a K split, in the
fixed-order split reduce -- is then an exact integer well below 2^24, and the tensor core's alignment of addends to the largest one
loses nothing.  The epilogues add exactly representable values (scale in {-1/2, 1/2, 1, 2}, shift on the 1/4 grid, an integer bf16
residual), so every output must equal the exact result rounded ONCE (through fp32, to bf16): bit for bit, no tolerance.  A missing,
duplicated or mis-addressed product moves an output by at least 1/2, which bf16 shows wherever |y| <= 256; at least 99 % of the
reference outputs of every forward and data-gradient case are in that range (asserted).  The fp64 references (F.conv2d,
torch.nn.grad.conv2d_input / conv2d_weight on the GPU) are asserted integral before they are rounded.  Data is drawn per channel:
symmetric, one-signed, all-zero and constant-1 channels; a constant channel makes the zero fill of out-of-image taps visible (a border
output differs from an interior one only through it).  A failure reports the mismatch count and the first (b, y, x, c) positions with
their tile coordinates (y // 8, x // 16): an addressing bug is confined to tiles, rows or splits.

Cases.  NET_CASES: every distinct conv shape of the train step at 480x640 for B = 1, 4, 32, derived from
oracle.keypoints_oracle.network_spec() -- the stem, layer1, 2.0.conv1, 2.0.downsample, 2.x.conv2, 3.0.conv1, 3.0.downsample, 3.x.conv2,
4.0.conv1, 4.0.downsample, 4.x.conv2 (11 per batch).  FWD_EDGE: output heights 1..7 mod 8 (strip patches for 1..4, ceil tiles for
5..7), widths not a multiple of 16, odd patch counts, on every forward route.  WGRAD_EDGE: a tap-pair shape whose splits start
mid-image and whose last split is ragged, a shape with fewer than 4 boxes (one split), the Cout = 64 path without tap pairs (stride 2;
input grid != output grid).  Inference launches at B = 1 and 64 (the bench.py workload): conv_ds for the three block entries,
conv_head for layer4.2.conv2 with K = 4 scoring rows, stem_pool.

What each case asserts, calling the ops exactly as TrainEngine and InferenceEngine do:
  A. train forward: conv_bn_act (ones / zeros, no ReLU) bit-exact; for the 3x3 Cout >= 256 convs conv_bn_stats too, equal to it, with
     sum y read back from the 128-bit accumulators exact and sum y^2 within the fp32 rounding of the per-CTA partials; stem_conv with
     x in {0, 1} bit-exact.
  B. folded epilogue (frozen BatchNorm, inference): per-channel scale / shift, integer residual, ReLU: bit-exact.
  C. data gradient as TrainEngine._dgrad runs it (flipped weights, zero insertion for stride 2, pad = dil*(k-1) - pad, residual).
  D. weight gradient (conv_wgrad, stem_wgrad): dw exact in fp32; accumulate=True onto an integer dw adds exactly; a second run is
     bit-identical.
  E. conv_ds (both outputs), conv_head (fc rows on the 1/8 grid: the fp32 logits are exact, equal to the fp64 dot products of the
     bf16-rounded feature map), stem_pool (max-pool of the exact stem) at B = 1, 64: bit-exact.
  Route coverage: torch.profiler records the kernels one pass over the case list launches; every tcgen05 conv instance of the default
  routes must appear.

Run with -s to see the per-case timings.  The whole file takes about 9 s on a B200 (1000 W power limit)."""
import math
import re
import zlib

import pytest
import torch
import torch.nn.functional as F

from hulk_keypoints_b200 import ops
from oracle import keypoints_oracle as O

DEV = "cuda:0"
BF = torch.bfloat16
LIMIT = 2 ** 22


# ------------------------------------------------------------------ cases, from the network itself
def train_step_conv_cases(H=480, W=640, batches=(1, 4, 32)):
    """(name, B, H, W, cin, cout, k, stride, pad, dil) of every distinct conv shape of the train step (H, W: the conv's input grid)."""
    stem, blocks, _ = O.network_spec()
    cases = []
    for B in batches:
        cases.append((stem.name, B, H, W, stem.cin, stem.cout, stem.k, stem.stride, stem.pad, stem.dil))
        h, w = ops.conv_out_hw(H, W, stem.k, stem.stride, stem.pad, stem.dil)
        h, w = ops.conv_out_hw(h, w, 3, 2, 1, 1)                          # max-pool 3x3 s2 p1
        seen = set()
        for blk in blocks:
            h1, w1 = ops.conv_out_hw(h, w, blk.conv1.k, blk.conv1.stride, blk.conv1.pad, blk.conv1.dil)
            for c, hi, wi in ((blk.conv1, h, w), (blk.down, h, w), (blk.conv2, h1, w1)):
                if c is None:
                    continue
                key = (hi, wi, c.cin, c.cout, c.k, c.stride, c.pad, c.dil)
                if key not in seen:
                    seen.add(key)
                    cases.append((c.name, B) + key)
            h, w = ops.conv_out_hw(h1, w1, blk.conv2.k, blk.conv2.stride, blk.conv2.pad, blk.conv2.dil)
    return cases


def inference_cases(H=480, W=640, batches=(1, 64)):
    """(ds, head, stem_pool) launches of InferenceEngine: conv_ds per block entry, conv_head for the last conv, stem_pool."""
    stem, blocks, _ = O.network_spec()
    h, w = ops.conv_out_hw(*ops.conv_out_hw(H, W, stem.k, stem.stride, stem.pad, stem.dil), 3, 2, 1, 1)
    ds, head = [], []
    for blk in blocks:
        h1, w1 = ops.conv_out_hw(h, w, blk.conv1.k, blk.conv1.stride, blk.conv1.pad, blk.conv1.dil)
        if blk.down is not None:
            c = blk.conv1
            ds += [(c.name, B, h, w, c.cin, c.cout, c.k, c.stride, c.pad, c.dil) for B in batches]
        h, w = h1, w1
    c = blocks[-1].conv2
    head = [(c.name, B, h, w, c.cin, c.cout, c.k, c.stride, c.pad, c.dil) for B in batches]
    pool = [("stem_pool", B, H, W, 3, 64, 7, 2, 3, 1) for B in batches]
    return ds, head, pool


NET_CASES = train_step_conv_cases()
STEM_CASES = [c for c in NET_CASES if c[0] == "conv1"]
BLOCK_CASES = [c for c in NET_CASES if c[0] != "conv1"]
DS_CASES, HEAD_CASES, POOL_CASES = inference_cases()

FWD_EDGE = [
    # name, B, H, W, cin, cout, k, stride, pad, dil   (output height mod 8; route of the forward / of the data gradient)
    ("edge-h17", 1, 17, 40, 128, 128, 3, 1, 1, 1),     # 1: tc2h strips clipped to one row; width 40
    ("edge-h26", 3, 26, 37, 128, 256, 3, 1, 2, 2),     # 2: tc2h, dilation 2, width 37
    ("edge-h35", 2, 35, 70, 256, 256, 3, 1, 1, 1),     # 3: tc2h, strips over 70 = 2.2 strips
    ("edge-h12", 1, 12, 48, 128, 128, 3, 1, 1, 1),     # 4: 3 full patches (odd) + one strip row
    ("edge-h21", 1, 21, 40, 128, 128, 3, 1, 1, 1),     # 5: ceil patch rows, 9 patches (odd)
    ("edge-h30", 3, 30, 56, 256, 256, 3, 1, 2, 2),     # 6: tc2h dilation 2, no strips
    ("edge-h15", 1, 15, 20, 64, 64, 3, 1, 1, 1),       # 7: c64, width 20
    ("edge-h13", 2, 13, 27, 256, 512, 3, 1, 4, 4),     # 5: tc2 dilation 4, odd box count
    ("edge-s2", 2, 34, 44, 64, 128, 3, 2, 1, 1),       # output 17x22: tc2 stride 2; its data gradient on conv_tc_kernel<64>
    ("edge-ds", 1, 26, 38, 128, 256, 1, 2, 0, 1),      # 1x1 stride 2, output 13x19
]
WGRAD_EDGE = [
    ("edge-pairs", 2, 28, 40, 64, 64, 3, 1, 1, 1),     # tap pairs: 42 boxes in 9 splits of 5, split 4 spans both images, last split 2 boxes
    ("edge-1split", 1, 4, 40, 128, 128, 3, 1, 1, 1),   # 3 boxes: a single K split
    ("edge-c64-s2", 2, 30, 44, 64, 64, 3, 2, 1, 1),    # Cout = 64 without tap pairs: stride 2
    ("edge-c64-p0", 3, 22, 34, 64, 64, 3, 1, 0, 1),    # ... and output grid (20x32) != input grid
]


def case_id(c):
    return f"{c[0]}-B{c[1]}-{c[2]}x{c[3]}"


def test_case_list_covers_the_network():
    """The derived list: 11 distinct conv shapes per batch, B = 32 layer1 at 120x160 and layers 2-4 at 60x80 among them."""
    assert len(NET_CASES) == 33 and all(sum(c[1] == B for c in NET_CASES) == 11 for B in (1, 4, 32))
    assert ("layer1.0.conv1", 32, 120, 160, 64, 64, 3, 1, 1, 1) in NET_CASES
    assert ("layer2.0.conv1", 32, 120, 160, 64, 128, 3, 2, 1, 1) in NET_CASES
    at60 = {c[0] for c in NET_CASES if c[1] == 32 and (c[2], c[3]) == (60, 80)}
    assert at60 == {"layer2.0.conv2", "layer3.0.conv1", "layer3.0.downsample.0", "layer3.0.conv2", "layer4.0.conv1",
                    "layer4.0.downsample.0", "layer4.0.conv2"}
    assert ("layer4.0.conv2", 32, 60, 80, 512, 512, 3, 1, 4, 4) in NET_CASES
    assert [c[0] for c in DS_CASES[::2]] == ["layer2.0.conv1", "layer3.0.conv1", "layer4.0.conv1"]
    assert HEAD_CASES[1] == ("layer4.2.conv2", 64, 60, 80, 512, 512, 3, 1, 4, 4) and len(POOL_CASES) == 2
    for c in BLOCK_CASES + FWD_EDGE + WGRAD_EDGE:
        assert c[4] % 64 == 0 and c[5] % 64 == 0 and c[7] in (1, 2)


# ------------------------------------------------------------------ data
def gen(case, salt=0):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(repr((case, salt)).encode()))


def ternary(shape, g, dtype=BF, density=0.25):
    """{-1, 0, 1}, mostly zero; by channel (last dim) c % 8: 0-3 symmetric, 4 only +1, 5 only -1, 6 all zero, 7 constant 1."""
    C = shape[-1]
    mode = torch.arange(C, device=DEV) % 8
    v = torch.where(torch.rand(shape, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    v = v * (torch.rand(shape, generator=g, device=DEV) < density)
    v = torch.where(mode == 4, v.abs(), v)
    v = torch.where(mode == 5, -v.abs(), v)
    v = torch.where(mode == 6, torch.zeros_like(v), v)
    v = torch.where(mode == 7, torch.ones_like(v), v)
    return v.to(dtype).contiguous()


def weights(cout, cin, k, g):
    """fp32 OIHW in {-1, 0, 1}: output channel co % 8 == 6 all zero, == 7 only +1, the rest symmetric (density 1/4)."""
    shape = (cout, cin, k, k)
    w = torch.where(torch.rand(shape, generator=g, device=DEV) < 0.5, -1.0, 1.0) * (torch.rand(shape, generator=g, device=DEV) < 0.25)
    mode = (torch.arange(cout, device=DEV) % 8).view(cout, 1, 1, 1)
    w = torch.where(mode == 7, w.abs(), w)
    return torch.where(mode == 6, torch.zeros_like(w), w).contiguous()


def folded(C, g):
    """scale in {-1/2, 1/2, 1, 2}, shift on the 1/4 grid in [-2, 2]"""
    scale = torch.tensor([-0.5, 0.5, 1.0, 2.0], device=DEV)[torch.randint(0, 4, (C,), generator=g, device=DEV)]
    shift = torch.randint(-8, 9, (C,), generator=g, device=DEV).float() / 4
    return scale.contiguous(), shift.contiguous()


def int_residual(shape, g):
    return torch.randint(-3, 4, shape, generator=g, device=DEV).to(BF)


# ------------------------------------------------------------------ references
def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def integral(r, what):
    err = (r - r.round()).abs().max().item() if r.numel() else 0.0
    assert err < 1e-6, f"{what}: fp64 reference not integral ({err:.3g})"
    return r.round()


def conv_ref(x, w, stride, pad, dil):
    """exact conv of NHWC x with OIHW w -> NHWC fp64"""
    return nhwc(integral(F.conv2d(nchw(x).double(), w.double(), None, stride, pad, dil), "conv2d"))


def rounded(v64):
    """the exact value rounded once: fp64 -> fp32 is exact on these grids, fp32 -> bf16 rounds to nearest even"""
    return v64.float().to(BF)


def assert_bound(K, a, b, what):
    bound = K * a.abs().max().item() * b.abs().max().item()
    assert bound < LIMIT, f"{what}: premise K*max|a|*max|b| = {bound} >= 2^22"


def assert_in_range(ref, what):
    frac = (ref.abs() <= 256).double().mean().item()
    assert frac >= 0.99, f"{what}: premise: only {100 * frac:.2f} % of the reference outputs have |y| <= 256"


def assert_exact(got, want, what):
    """got == want for (B, H, W, C) tensors; the message locates the first mismatches with their 8x16 tile coordinates"""
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    bad = got != want
    n = int(bad.sum().item())
    if n:
        first = []
        for b, y, x, c in bad.nonzero()[:6].tolist():
            first.append(f"(b{b} y{y} x{x} c{c}) tile ({y // 8},{x // 16}): {got[b, y, x, c].item()} != {want[b, y, x, c].item()}")
        rows = bad.any(3).any(0).nonzero()[:, 0].unique().tolist()
        pytest.fail(f"{what}: {n} of {bad.numel()} outputs differ; first {'; '.join(first)}; rows with mismatches {rows[:12]}")


def assert_exact_w(got, want, what):
    """dw (cout, cin, k, k) fp32 == want"""
    bad = got != want
    n = int(bad.sum().item())
    if n:
        first = [f"(co{o} ci{i} r{r} s{s}): {got[o, i, r, s].item()} != {want[o, i, r, s].item()}" for o, i, r, s in bad.nonzero()[:6].tolist()]
        taps = bad.any(1).any(0).nonzero().tolist()
        pytest.fail(f"{what}: {n} of {bad.numel()} weights differ; first {'; '.join(first)}; taps with mismatches {taps}")


def acc_values(acc, C):
    """(sum, sum of squares) per channel of bn accumulators as Python ints in units of 2^-50; asserts that none is poisoned"""
    a = acc.view(torch.int64).cpu().view(2 * C, 4).tolist()
    assert not any(r[2] for r in a), "poisoned accumulator"
    vals = []
    for lo, hi, _, _ in a:
        v = ((hi % 2 ** 64) << 64) | (lo % 2 ** 64)
        vals.append(v - (1 << 128) if v >> 127 else v)
    return vals[:C], vals[C:]


# ================================================================== A + B. forward: raw (train), epilogue statistics, folded
@pytest.mark.gpu
@pytest.mark.parametrize("case", BLOCK_CASES + FWD_EDGE, ids=case_id)
def test_forward_exact(case):
    """A: conv_bn_act with ones / zeros == the exact conv rounded once; the 3x3 Cout >= 256 convs also through conv_bn_stats (same y, sum y
    exact, sum y^2 within the fp32 rounding of the per-CTA partials).  B: the folded epilogue (scale, shift, integer residual, ReLU)."""
    name, B, H, W, cin, cout, k, stride, pad, dil = case
    g = gen(case)
    x = ternary((B, H, W, cin), g)
    w = weights(cout, cin, k, g)
    assert_bound(k * k * cin, x, w, name)
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, BF)
    one, zero = torch.ones(cout, device=DEV), torch.zeros(cout, device=DEV)
    ref = conv_ref(x, w, stride, pad, dil)
    assert_in_range(ref, name)
    want = rounded(ref)
    y = ops.conv_bn_act(x, wp, one, zero, stride=stride, pad=pad, dil=dil, relu=False)
    assert_exact(y, want, f"A conv_bn_act {name}")
    if k == 3 and cout >= 256:                                       # TrainEngine._conv_bn's epilogue-statistics convs
        acc = torch.zeros(ops.bn_acc_bytes(cout), device=DEV, dtype=torch.uint8)
        ys = ops.conv_bn_stats(x, wp, one, zero, acc, stride=stride, pad=pad, dil=dil)
        assert torch.equal(ys, y), f"A conv_bn_stats {name}: y differs from conv_bn_act"
        sums, squares = acc_values(acc, cout)
        yv = want.double().view(-1, cout)
        s_exact = [int(v) << 50 for v in yv.sum(0).long().tolist()]
        bad = [c for c in range(cout) if sums[c] != s_exact[c]]
        assert not bad, f"A conv_bn_stats {name}: sum y of {len(bad)} channels differs, first c{bad[0]}: {sums[bad[0]] / 2 ** 50} != {s_exact[bad[0]] / 2 ** 50}"
        q_exact = yv.square().sum(0).cpu()
        # every addition into a per-CTA fp32 partial rounds by at most 2^-24 of the channel total; one addition per 128-pixel chunk
        chunks = math.ceil(B * ref.shape[1] * ref.shape[2] / 128)
        q_got = torch.tensor([q / 2 ** 50 for q in squares], dtype=torch.float64)
        err = (q_got - q_exact).abs()
        assert (err <= q_exact * 2.0 ** -24 * chunks).all(), f"A conv_bn_stats {name}: sum y^2 off by {err.max().item()}"
    # B: frozen BatchNorm / inference epilogue
    scale, shift = folded(cout, g)
    res = int_residual(tuple(y.shape), g)
    yf = ops.conv_bn_act(x, wp, scale, shift, stride=stride, pad=pad, dil=dil, relu=True, residual=res)
    assert_exact(yf, rounded((ref * scale.double() + shift.double() + res.double()).clamp_min(0)), f"B folded {name}")


# ================================================================== C. data gradient, as TrainEngine._dgrad runs it
@pytest.mark.gpu
@pytest.mark.parametrize("case", BLOCK_CASES + FWD_EDGE, ids=case_id)
def test_dgrad_exact(case):
    """dx = conv(zero_insert2x(dy) or dy, flipped weights, pad = dil*(k-1) - pad) + residual == conv2d_input + residual, bit for bit."""
    name, B, H, W, cin, cout, k, stride, pad, dil = case
    g = gen(case, 1)
    Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
    dy = ternary((B, Ho, Wo, cout), g)
    w = weights(cout, cin, k, g)
    assert_bound(k * k * cout, dy, w, name)
    wd = ops.pack_conv_weights_dgrad(w)
    src = dy
    if stride == 2:
        assert (H, W) == (2 * Ho, 2 * Wo)
        src = torch.empty((B, H, W, cout), device=DEV, dtype=BF)
        ops.zero_insert2x(dy, out=src)
    res = int_residual((B, H, W, cin), g)
    one, zero = torch.ones(cin, device=DEV), torch.zeros(cin, device=DEV)
    dx = ops.conv_bn_act(src, wd, one, zero, stride=1, pad=dil * (k - 1) - pad, dil=dil, relu=False, residual=res)
    ref = torch.nn.grad.conv2d_input((B, cin, H, W), w.double(), nchw(dy).double(), stride=stride, padding=pad, dilation=dil)
    ref = nhwc(integral(ref, "conv2d_input"))
    assert_in_range(ref, name)
    assert_exact(dx, rounded(ref + res.double()), f"C dgrad {name}")


# ================================================================== D. weight gradient
def _wgrad_check(what, run, ref, g):
    """run(dw, accumulate) fills dw; exact, accumulate onto integers exact, rerun bit-identical"""
    dw = torch.full(tuple(ref.shape), float("nan"), device=DEV)          # must be overwritten
    run(dw, False)
    assert_exact_w(dw, ref, f"D {what}")
    base = torch.randint(-4, 5, tuple(ref.shape), generator=g, device=DEV).float()
    acc = base.clone()
    run(acc, True)
    assert_exact_w(acc, base + ref, f"D {what} accumulate")
    again = torch.full_like(dw, float("nan"))
    run(again, False)
    assert torch.equal(again.view(torch.int32), dw.view(torch.int32)), f"D {what}: second run not bit-identical"


@pytest.mark.gpu
@pytest.mark.parametrize("case", BLOCK_CASES + FWD_EDGE + WGRAD_EDGE, ids=case_id)
def test_wgrad_exact(case):
    """conv_wgrad (split-K tcgen05 + fixed-order reduce) == conv2d_weight exactly in fp32."""
    name, B, H, W, cin, cout, k, stride, pad, dil = case
    g = gen(case, 2)
    Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
    x = ternary((B, H, W, cin), g)
    dy = ternary((B, Ho, Wo, cout), g)
    assert_bound(B * Ho * Wo, x, dy, name)
    ref = torch.nn.grad.conv2d_weight(nchw(x).double(), (cout, cin, k, k), nchw(dy).double(), stride=stride, padding=pad, dilation=dil)
    ref = integral(ref, "conv2d_weight").float()
    ws = torch.empty(ops.conv_wgrad_workspace_bytes(B, H, W, cin, cout, k, stride, pad, dil), device=DEV, dtype=torch.uint8)
    _wgrad_check(name, lambda dw, a: ops.conv_wgrad(x, dy, dw, k=k, stride=stride, pad=pad, dil=dil, ws=ws, accumulate=a), ref, g)


# ================================================================== stem: forward (A, B), weight gradient (D), fused max-pool (E)
def stem_input(B, H, W, g):
    """fp32 NCHW in {0, 1}: channel 0 sparse, channel 1 constant 1, channel 2 dense"""
    u = torch.rand(B, 3, H, W, generator=g, device=DEV)
    x = (u < torch.tensor([0.25, 2.0, 0.5], device=DEV).view(1, 3, 1, 1)).float()
    return x.contiguous()


def stem_ref(x, w):
    return nhwc(integral(F.conv2d(x.double(), w.double(), None, 2, 3, 1), "stem conv2d"))


@pytest.mark.gpu
@pytest.mark.parametrize("case", STEM_CASES, ids=case_id)
def test_stem_conv_exact(case):
    """stem_conv raw (train forward) and with a folded epilogue + ReLU, bit-exact."""
    _, B, H, W, *_ = case
    g = gen(case)
    x = stem_input(B, H, W, g)
    w = weights(64, 3, 7, g)
    assert_bound(147, x, w, "stem")
    wp = ops.stem_pack_weights(w)
    ref = stem_ref(x, w)
    assert_in_range(ref, "stem")
    one, zero = torch.ones(64, device=DEV), torch.zeros(64, device=DEV)
    assert_exact(ops.stem_conv(x, wp, one, zero, relu=False), rounded(ref), "A stem_conv")
    scale, shift = folded(64, g)
    assert_exact(ops.stem_conv(x, wp, scale, shift, relu=True), rounded((ref * scale.double() + shift.double()).clamp_min(0)), "B stem_conv")


@pytest.mark.gpu
@pytest.mark.parametrize("case", STEM_CASES, ids=case_id)
def test_stem_wgrad_exact(case):
    _, B, H, W, *_ = case
    g = gen(case, 2)
    x = stem_input(B, H, W, g)
    Ho, Wo = ops.conv_out_hw(H, W, 7, 2, 3, 1)
    dy = ternary((B, Ho, Wo, 64), g)
    assert_bound(B * Ho * Wo, x, dy, "stem wgrad")
    ref = integral(torch.nn.grad.conv2d_weight(x.double(), (64, 3, 7, 7), nchw(dy).double(), stride=2, padding=3), "stem conv2d_weight").float()
    _wgrad_check(f"stem_wgrad B{B}", lambda dw, a: ops.stem_wgrad(x, dy, dw, accumulate=a), ref, g)


@pytest.mark.gpu
@pytest.mark.parametrize("case", POOL_CASES, ids=case_id)
def test_stem_pool_exact(case):
    """E: stem_pool == max-pool 3x3 s2 p1 of the exact stem (negative scales included: the kernel pools the pre-activation extremes)."""
    _, B, H, W, *_ = case
    g = gen(case)
    x = stem_input(B, H, W, g)
    w = weights(64, 3, 7, g)
    scale, shift = folded(64, g)
    stem = rounded((stem_ref(x, w) * scale.double() + shift.double()).clamp_min(0))
    want = nhwc(F.max_pool2d(nchw(stem).float(), 3, 2, 1)).to(BF)
    assert_exact(ops.stem_pool(x, ops.stem_pack_weights(w), scale, shift), want, "E stem_pool")


# ================================================================== E. inference launches at B = 1 and 64
@pytest.mark.gpu
@pytest.mark.parametrize("case", DS_CASES, ids=case_id)
def test_conv_ds_exact(case):
    """conv_ds: relu(scale*conv_kxk + shift) and scale_ds*conv_1x1 + shift_ds of the same input, both bit-exact."""
    name, B, H, W, cin, cout, k, stride, pad, dil = case
    g = gen(case)
    x = ternary((B, H, W, cin), g)
    w, wd = weights(cout, cin, k, g), weights(cout, cin, 1, g)
    assert_bound(k * k * cin, x, w, name)
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, BF)
    wdp, _, _ = ops.pack_conv_weights(wd, None, 1e-5, BF)
    (s, b), (sd, bd) = folded(cout, g), folded(cout, g)
    y, yds = ops.conv_ds(x, wp, s, b, wdp, sd, bd, stride=stride, pad=pad, dil=dil, relu=True)
    ref = conv_ref(x, w, stride, pad, dil)
    assert_in_range(ref, name)
    assert_exact(y, rounded((ref * s.double() + b.double()).clamp_min(0)), f"E conv_ds {name}")
    ref_ds = conv_ref(x, wd, stride, 0, 1)
    assert_exact(yds, rounded(ref_ds * sd.double() + bd.double()), f"E conv_ds downsample {name}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", HEAD_CASES, ids=case_id)
def test_conv_head_exact(case):
    """conv_head with K = 4 scoring rows on the 1/8 grid: the logits equal the fp64 dot products of the bf16-rounded feature map."""
    name, B, H, W, cin, cout, k, stride, pad, dil = case
    K = 4
    g = gen(case)
    x = ternary((B, H, W, cin), g)
    w = weights(cout, cin, k, g)
    assert_bound(k * k * cin, x, w, name)
    wp, _, _ = ops.pack_conv_weights(w, None, 1e-5, BF)
    s, b = folded(cout, g)
    res = int_residual((B, H, W, cout), g)
    w_fc = (torch.randint(-8, 9, (K, cout), generator=g, device=DEV).float() / 8).contiguous()
    b_fc = torch.randint(-8, 9, (K,), generator=g, device=DEV).float() / 8
    ref = conv_ref(x, w, stride, pad, dil)
    assert_in_range(ref, name)
    feat = rounded((ref * s.double() + b.double() + res.double()).clamp_min(0)).double()
    # premise: on the 1/32 grid every fp32 partial of the dot products stays below 2^24 * 2^-5
    worst = torch.einsum("bhwc,kc->bkhw", feat.abs(), w_fc.double().abs()).max().item() + 1
    assert worst * 32 < 2 ** 24, f"premise: dot products up to {worst}"
    want = torch.einsum("bhwc,kc->bkhw", feat, w_fc.double()) + b_fc.double().view(1, K, 1, 1)
    logits = torch.full((B, K, H, W), float("nan"), device=DEV)
    ops.conv_head(x, wp, s, b, w_fc, b_fc, logits, stride=stride, pad=pad, dil=dil, relu=True, residual=res)
    assert_exact(logits.double().permute(0, 2, 3, 1), want.permute(0, 2, 3, 1), f"E conv_head {name}")


# ================================================================== route coverage
_KERNEL_RE = re.compile(r"(conv_tc2h_kernel|conv_tc2_kernel|conv_tc_c64_kernel|conv_tc_kernel|conv_wgrad_kernel|stem_tc_kernel|"
                        r"stem_wgrad_tc_kernel|stem_pool_kernel)(?:<([^>]*)>)?")


def kernel_instance(name):
    """'void hk::conv_tc2_kernel<256, false, true, false>(...)' or '...<(int)256, (bool)0, ...>' -> ('conv_tc2_kernel', ('256', 'false', ...))"""
    m = _KERNEL_RE.search(name)
    if m is None:
        return None
    args = (m.group(2) or "").replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true")
    return m.group(1), tuple(a.strip() for a in args.split(",") if a.strip())


def _launch_all():
    """one launch of every op at every case, on zero data"""
    z = lambda *s: torch.zeros(s, device=DEV, dtype=BF)
    for name, B, H, W, cin, cout, k, stride, pad, dil in BLOCK_CASES + FWD_EDGE:
        Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
        w = torch.zeros(cout, cin, k, k, device=DEV)
        wp, one, zero = ops.pack_conv_weights(w, None, 1e-5, BF)
        ops.conv_bn_act(z(B, H, W, cin), wp, one, zero, stride=stride, pad=pad, dil=dil, relu=False)
        if k == 3 and cout >= 256:
            ops.conv_bn_stats(z(B, H, W, cin), wp, one, zero, torch.zeros(ops.bn_acc_bytes(cout), device=DEV, dtype=torch.uint8),
                              stride=stride, pad=pad, dil=dil)
        ones_in, zeros_in = torch.ones(cin, device=DEV), torch.zeros(cin, device=DEV)
        ops.conv_bn_act(z(B, H, W, cout), ops.pack_conv_weights_dgrad(w), ones_in, zeros_in, stride=1, pad=dil * (k - 1) - pad, dil=dil,
                        relu=False)
    for name, B, H, W, cin, cout, k, stride, pad, dil in BLOCK_CASES + FWD_EDGE + WGRAD_EDGE:
        Ho, Wo = ops.conv_out_hw(H, W, k, stride, pad, dil)
        ops.conv_wgrad(z(B, H, W, cin), z(B, Ho, Wo, cout), torch.empty(cout, cin, k, k, device=DEV), k=k, stride=stride, pad=pad, dil=dil)
    w7 = ops.stem_pack_weights(torch.zeros(64, 3, 7, 7, device=DEV))
    one, zero = torch.ones(64, device=DEV), torch.zeros(64, device=DEV)
    for _, B, H, W, *_ in STEM_CASES:
        x = torch.zeros(B, 3, H, W, device=DEV)
        ops.stem_conv(x, w7, one, zero, relu=False)
        ops.stem_wgrad(x, z(B, (H + 1) // 2, (W + 1) // 2, 64), torch.empty(64, 3, 7, 7, device=DEV))
    for _, B, H, W, *_ in POOL_CASES:
        ops.stem_pool(torch.zeros(B, 3, H, W, device=DEV), w7, one, zero)
    for name, B, H, W, cin, cout, k, stride, pad, dil in DS_CASES:
        wp = torch.zeros(cout, k, k, cin, device=DEV, dtype=BF)
        v = torch.zeros(cout, device=DEV)
        ops.conv_ds(z(B, H, W, cin), wp, v, v, torch.zeros(cout, 1, 1, cin, device=DEV, dtype=BF), v, v, stride=stride, pad=pad, dil=dil)
    for name, B, H, W, cin, cout, k, stride, pad, dil in HEAD_CASES:
        v = torch.zeros(cout, device=DEV)
        ops.conv_head(z(B, H, W, cin), torch.zeros(cout, k, k, cin, device=DEV, dtype=BF), v, v, torch.zeros(4, cout, device=DEV),
                      torch.zeros(4, device=DEV), torch.empty(B, 4, H, W, device=DEV), stride=stride, pad=pad, dil=dil, residual=z(B, H, W, cout))


@pytest.mark.gpu
def test_cases_reach_every_default_route():
    """Every tcgen05 conv instance the default routes use is launched by the case list: conv_tc_c64, conv_tc2h at both BLOCK_N, conv_tc2
    at both BLOCK_N plus its block-entry (DS) and head instances, conv_tc_kernel<64> (the 64-channel data gradients of layer2.0),
    conv_wgrad at 64 / 128 / 256 input-channel tiles, and the stem kernels."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _launch_all()
        torch.cuda.synchronize()
    seen = {kernel_instance(e.key) for e in prof.key_averages()} - {None}
    names = sorted(f"{n}<{', '.join(a)}>" for n, a in seen)
    print("\n[routes] " + "\n[routes] ".join(names))

    def has(kernel, **want):
        pos = {"bn": 0, "ds": 1, "stats": 2, "head": 3} if kernel == "conv_tc2_kernel" else {"bn": 0, "stats": 1}
        for n, a in seen:
            if n == kernel and all(a[pos[key]] == str(v).lower() for key, v in want.items()):
                return True
        return False

    missing = [what for what, ok in [
        ("conv_tc_c64_kernel", has("conv_tc_c64_kernel")),
        ("conv_tc2h_kernel<128>", has("conv_tc2h_kernel", bn=128)), ("conv_tc2h_kernel<256>", has("conv_tc2h_kernel", bn=256)),
        ("conv_tc2_kernel<128>", has("conv_tc2_kernel", bn=128, ds=False, head=False)),
        ("conv_tc2_kernel<256>", has("conv_tc2_kernel", bn=256, ds=False, head=False)),
        ("conv_tc2_kernel DS", has("conv_tc2_kernel", ds=True)), ("conv_tc2_kernel HEAD", has("conv_tc2_kernel", head=True)),
        ("conv_tc_kernel<64>", has("conv_tc_kernel", bn=64)),
        ("conv_wgrad_kernel<64>", has("conv_wgrad_kernel", bn=64)), ("conv_wgrad_kernel<128>", has("conv_wgrad_kernel", bn=128)),
        ("conv_wgrad_kernel<256>", has("conv_wgrad_kernel", bn=256)),
        ("stem_tc_kernel", has("stem_tc_kernel")), ("stem_wgrad_tc_kernel", has("stem_wgrad_tc_kernel")),
        ("stem_pool_kernel", has("stem_pool_kernel")),
    ] if not ok]
    assert not missing, f"not launched by the case list: {missing}; launched: {names}"
