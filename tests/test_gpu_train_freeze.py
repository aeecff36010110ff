"""Fine-tuning configurations of the training engine: BatchNorm modules in eval() mode inside a train()-mode model ("frozen BN":
running statistics, buffers untouched) and parameters with requires_grad=False (no gradient, no kernel, pruned backward).

Checks the frozen-BatchNorm kernels against fp64 on exact inputs, and whole steps against torch autograd with the same flags on the
trained fixture, at the presets of bench_train.py --freeze."""
import warnings

import pytest
import torch

import hulk_keypoints_b200 as hk
from hulk_keypoints_b200 import ops, synth, train_ops
from hulk_keypoints_b200.train_engine import backward_plan, step_launches

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

B, H, W = 4, 128, 160


def apply_preset(model, preset: str) -> None:
    """The presets of bench_train.py --freeze (model left in train() mode)."""
    train_ops.freeze_preset(model, preset)


def cosine(a, b):
    a, b = a.flatten().double(), b.flatten().double()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-300))


# ---------------------------------------------------------------------------------------------------------------- kernel vs fp64
def _bits(out):
    w = torch.tensor([1 << j for j in range(8)], device=out.device, dtype=torch.int32)
    return ((out.float() > 0).view(-1, 8).int() * w).sum(1).to(torch.uint8)


@pytest.mark.parametrize("C", [64, 512])
@pytest.mark.parametrize("P_kind", ["1", "7", "chunk_edge"])
@pytest.mark.parametrize("mask_kind", ["bits", "bf16", "none"])
def test_frozen_bwd_kernel_against_fp64(C, P_kind, mask_kind):
    P = {"1": 1, "7": 7, "chunk_edge": 1024 * 8 // C + 1}[P_kind]
    g = torch.Generator().manual_seed(C * 1000 + P)
    dev = "cuda"
    # integer grid (k/8): every fp32 partial and accumulator sum is exact
    dout = (torch.randint(-64, 65, (P, C), generator=g).float() / 8).to(dev).bfloat16()
    y = (torch.randint(-64, 65, (P, C), generator=g).float() / 8).to(dev).bfloat16()
    out = (torch.randint(-4, 5, (P, C), generator=g).float() / 8).to(dev).bfloat16()   # stands in for the post-ReLU output
    gamma = (torch.rand(C, generator=g) + 0.5).to(dev)
    beta = (torch.rand(C, generator=g) - 0.5).to(dev)
    rmean = (torch.randn(C, generator=g)).to(dev)
    rvar = (torch.rand(C, generator=g) + 0.25).to(dev)
    eps = 1e-5
    scale, shift, invstd = (torch.empty(C, device=dev) for _ in range(3))
    items = ops.bn_fold_items([(gamma, beta, rmean, rvar, eps, scale, shift, invstd)]).to(dev)
    ops.bn_fold(items, 1, C)
    inv64 = 1.0 / torch.sqrt(rvar.double() + eps)
    assert torch.allclose(invstd.double(), inv64, rtol=1e-6, atol=0)
    assert torch.allclose(scale.double(), gamma.double() * inv64, rtol=1e-6, atol=0)
    assert torch.allclose(shift.double(), beta.double() - rmean.double() * gamma.double() * inv64, rtol=1e-6, atol=1e-6)

    mask = {"bits": _bits(out), "bf16": out, "none": None}[mask_kind]
    dprime = dout.double() * ((out.double() > 0) if mask is not None else 1.0)
    ref_dy = scale.double() * dprime
    ref_db = dprime.sum(0)
    xhat = (y.double() - rmean.double()) * invstd.double()
    ref_dg = (dprime * xhat).sum(0)
    dg_bar = (dprime * xhat).abs().sum(0)

    def bf16_ok(got, ref):   # within one bf16 rounding of the fp64 value
        return bool(((got.double() - ref).abs() <= ref.abs() * 2.0 ** -8 + 1e-30).all())

    acc = torch.zeros(ops.bn_acc_bytes(C), device=dev, dtype=torch.uint8)
    for want_dy in (True, False):
        for want_dm in (True, False):
            acc.zero_()
            dy = torch.empty_like(dout) if want_dy else None
            dm = torch.empty_like(dout) if want_dm else None
            dgam, dbet = torch.full((C,), 3.0, device=dev), torch.full((C,), -2.0, device=dev)
            ops.bn_frozen_bwd(dout, mask, scale, dy, dmasked=dm, y=y, mean=rmean, invstd=invstd, acc=acc, dgamma=dgam, dbeta=dbet)
            torch.cuda.synchronize()
            if want_dy:
                assert bf16_ok(dy, ref_dy)
            if want_dm:
                assert torch.equal(dm.double(), dprime)
            assert torch.equal(dbet.double(), ref_db), (dbet.double() - ref_db).abs().max()
            assert bool(((dgam.double() - ref_dg).abs() <= 1e-5 * dg_bar + 1e-12).all()), ((dgam.double() - ref_dg).abs() / dg_bar).max()
            # accumulate adds exactly onto what is there
            acc.zero_()
            ops.bn_frozen_bwd(dout, mask, scale, dy, dmasked=dm, y=y, mean=rmean, invstd=invstd, acc=acc, dgamma=dgam, dbeta=dbet,
                              accumulate=True)
            assert torch.equal(dbet.double(), 2 * ref_db)
            assert bool(((dgam.double() - 2 * ref_dg).abs() <= 2e-5 * dg_bar + 1e-12).all())
    # no sums: dy (and d') only, y / accumulator not needed
    dy = torch.empty_like(dout)
    ops.bn_frozen_bwd(dout, mask, scale, dy)
    assert bf16_ok(dy, ref_dy)
    # only the sums (frozen conv weight under a trained BatchNorm): dy is NULL
    acc.zero_()
    dbet = torch.empty(C, device=dev)
    ops.bn_frozen_bwd(dout, mask, scale, None, y=y, mean=rmean, invstd=invstd, acc=acc, dbeta=dbet)
    assert torch.equal(dbet.double(), ref_db)


# ---------------------------------------------------------------------------------------------------------------- whole steps
@pytest.fixture(scope="module")
def fixture_sd():
    sd, _ = synth.train_fixture("k4_128x160")
    return sd


def _model(sd, preset):
    m = hk.KeypointsGauss(4, img_height=H, img_width=W).cuda().train()
    m.load_state_dict(sd)
    apply_preset(m, preset)
    return m


def _batch(seed):
    img, uv = synth.disc_batch(torch.Generator().manual_seed(seed), B, H, W, 4)
    return img.cuda(), uv.cuda()


def _bn_buffers(m):
    return {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches_tracked" in k}


@pytest.mark.parametrize("preset", ["bn", "torchvision", "head", "mixed"])
def test_step_matches_autograd_with_the_same_flags(fixture_sd, preset):
    m, ref = _model(fixture_sd, preset), _model(fixture_sd, preset)
    img, uv = _batch(7)
    before = _bn_buffers(m)
    eng = m.train_engine(B, H, W)
    loss = eng.forward_backward(img, uv=uv).item()
    loss_ref = train_ops.sigmoid_bce_loss(ref.forward_logits(img), uv=uv, sigma=8.0)
    loss_ref.backward()
    assert abs(loss - loss_ref.item()) < 1e-3 * abs(loss_ref.item()), (loss, loss_ref.item())
    rows = []
    for (name, p), (_, q) in zip(ref.named_parameters(), m.named_parameters()):
        assert p.requires_grad == q.requires_grad
        if not q.requires_grad:
            assert p.grad is None
            continue
        if p.grad.norm() == 0:
            assert eng.grad(q).norm() == 0, name
            continue
        rows.append((cosine(eng.grad(q), p.grad), float(eng.grad(q).norm() / p.grad.norm()), name))
    rows.sort()
    assert rows, "no trainable parameter"
    assert rows[0][0] >= 0.98, rows[:5]
    assert sum(c for c, _, _ in rows) / len(rows) >= 0.997
    assert all(0.95 <= ratio <= 1.05 for _, ratio, _ in rows), [r for r in rows if not 0.95 <= r[1] <= 1.05][:5]
    # BatchNorm buffers: frozen ones bit-unchanged, train-mode ones as torch moved them
    after, sr = _bn_buffers(m), ref.state_dict()
    bn_mode = {n: mod.training for n, mod in m.named_modules() if isinstance(mod, torch.nn.BatchNorm2d)}
    for k, v in after.items():
        if not bn_mode[k.rsplit(".", 1)[0]]:
            assert torch.equal(v, before[k]), k
        elif k.endswith("num_batches_tracked"):
            assert int(v) == int(sr[k]) == int(before[k]) + 1, k
        else:
            assert torch.allclose(v, sr[k], rtol=2e-2, atol=2e-3), (k, (v - sr[k]).abs().max().item())


def test_frozen_parameters_get_no_grad_and_stay_put(fixture_sd):
    from hulk_keypoints_b200.optim import FusedAdam
    img, uv = _batch(8)
    gt = torch.stack([hk.gauss_2d_batch(W, H, 8, uv[b, :, 0], uv[b, :, 1]) for b in range(B)])
    # drop-in path: model.forward(img).double() -> BCELoss -> backward()
    m = _model(fixture_sd, "torchvision")
    loss = torch.nn.BCELoss()(m.forward(img).double(), gt)
    loss.backward()
    for n, p in m.named_parameters():
        assert (p.grad is None) == (not p.requires_grad), n
    # several optimiser steps: frozen parameters and frozen BatchNorm buffers bit-unchanged
    for make_opt in (lambda ps: FusedAdam(ps, lr=1e-3, weight_decay=1e-4), lambda ps: torch.optim.Adam(ps, lr=1e-3, weight_decay=1e-4)):
        m = _model(fixture_sd, "torchvision")
        frozen = {n: p.detach().clone() for n, p in m.named_parameters() if not p.requires_grad}
        buffers = _bn_buffers(m)
        opt = make_opt(m.parameters())
        for s in range(3):
            train_ops.train_step(m, opt, *_batch(20 + s), sigma=8.0)
        torch.cuda.synchronize()
        for n, p in m.named_parameters():
            if n in frozen:
                assert torch.equal(p.detach(), frozen[n]), n
                assert p.grad is None, n
        assert all(torch.equal(v, buffers[k]) for k, v in _bn_buffers(m).items())
        trained = m.resnet.resnet34_8s.layer4[2].conv2.weight
        assert trained.requires_grad


def test_backward_is_pruned_and_launches_match_the_plan(fixture_sd):
    img, uv = _batch(9)
    counts = {}
    for preset in ("none", "bn", "torchvision", "head", "mixed"):
        m = _model(fixture_sd, preset)
        eng = m.train_engine(B, H, W)
        eng.forward_backward(img, uv=uv)
        counts[preset] = eng.launches
        assert eng.launches == step_launches(m.resnet.resnet34_8s, backward_plan(m.resnet.resnet34_8s)), preset
    assert counts["torchvision"] < counts["none"] and counts["head"] < counts["none"], counts


def test_graph_replay_equals_eager_and_toggling_equals_fresh(fixture_sd):
    img, uv = _batch(10)
    m = _model(fixture_sd, "torchvision")
    eng = m.train_engine(B, H, W)
    l1 = eng.forward_backward(img, uv=uv).item()
    g1 = eng.flat_grad.clone()
    eng.use_cuda_graph = False
    l2 = eng.forward_backward(img, uv=uv).item()
    eng.use_cuda_graph = True
    assert l1 == l2 and torch.equal(g1, eng.flat_grad)
    # toggle: "none" step, then "torchvision" / "head" on the same engine == a fresh model with that preset from the same state
    m = _model(fixture_sd, "none")
    eng = m.train_engine(B, H, W)
    eng.forward_backward(img, uv=uv)
    for preset in ("torchvision", "head", "bn"):
        state = {k: v.clone() for k, v in m.state_dict().items()}
        apply_preset(m, preset)
        loss = eng.forward_backward(img, uv=uv).item()
        fresh = _model(state, preset)
        feng = fresh.train_engine(B, H, W)
        assert loss == feng.forward_backward(img, uv=uv).item(), preset
        assert torch.equal(eng.flat_grad, feng.flat_grad), preset
        m.load_state_dict(state)   # the next preset starts from the same weights / buffers for both


@pytest.mark.parametrize("preset", ["torchvision", "head"])
def test_two_phase_step_equals_single_phase(fixture_sd, preset):
    img, uv = _batch(11)
    m = _model(fixture_sd, preset)
    eng = m.train_engine(B, H, W)
    loss = eng.forward_backward(img, uv=uv).item()
    ref = eng.flat_grad.clone()
    eng.flat_grad.zero_()
    late = eng.forward_backward_late(img, uv).item()
    eng.backward_early()
    assert late == loss and torch.equal(eng.flat_grad, ref)
    if preset == "head":
        assert eng.late_offset == 0 and not eng.has_early_backward()


@pytest.mark.parametrize("what", ["momentum", "track_running_stats", "affine"])
def test_unsupported_batchnorm_is_rejected(what):
    m = hk.KeypointsGauss(4, img_height=64, img_width=96).cuda().train()
    net = m.resnet.resnet34_8s
    if what == "momentum":
        net.layer2[0].bn1.momentum = None
    elif what == "track_running_stats":
        net.layer2[0].bn1 = torch.nn.BatchNorm2d(128, track_running_stats=False).cuda()
    else:
        net.layer2[0].bn1 = torch.nn.BatchNorm2d(128, affine=False).cuda()
    img = torch.rand(2, 3, 64, 96, device="cuda")
    with pytest.raises(RuntimeError, match=what if what != "momentum" else "momentum=None"):
        m.forward(img)
