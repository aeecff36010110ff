"""GPU: the augmentation kernels (csrc/augment.cu) against the host restatements of tests/augment_ref.py, and the training step with an
augmenter against the same step on a batch augmented beforehand."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import hulk_keypoints_b200 as hk
from augment_ref import noise_normals, photometric_ref, pick_and_move, warp_ref
from hulk_keypoints_b200 import _lib, ops, synth, train_ops
from hulk_keypoints_b200.augment import KeypointAugment
from hulk_keypoints_b200.optim import FusedAdam

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

# the training shape (float4 stores) and an odd width (scalar tail: 150 = 37 groups of 4 + 2)
SHAPES = [(4, 480, 640), (2, 100, 150)]
GEOM = dict(rotate=30.0, scale=(0.8, 1.2), translate=0.1)
FULL = dict(GEOM, brightness=0.2, contrast=(0.7, 1.3), channel_gain=0.15, noise_std=0.03)


def batch(seed, B, H, W, K=5, margin=0.0):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 3, H, W, generator=g)
    uv = torch.stack([margin + torch.rand(B, K, generator=g) * (W - 1 - 2 * margin),
                      margin + torch.rand(B, K, generator=g) * (H - 1 - 2 * margin)], -1)
    return img.cuda(), uv.cuda()


@pytest.mark.parametrize("shape", SHAPES)
def test_identity_is_bit_exact(shape):
    B, H, W = shape
    img, uv = batch(1, B, H, W)
    a = KeypointAugment(seed=3)
    out, uv2 = a(img, uv)
    assert torch.equal(out, img) and torch.equal(uv2, uv)
    assert a.last_pick.dtype == torch.int32 and (a.last_pick == 0).all() and a.calls == 1


@pytest.mark.parametrize("shape", SHAPES)
def test_pick_and_labels_match_restatement(shape):
    B, H, W = shape
    img, uv = batch(2, B, H, W, K=6)
    a = KeypointAugment(rotate=40.0, scale=(0.7, 1.4), translate=0.2, seed=11)
    for _ in range(3):
        p = a.draw(B, H, W)
        _, uv2 = a(img, uv)
        pick, want = pick_and_move(p.fwd.numpy(), uv.cpu().numpy(), H, W)
        got = uv2.cpu().numpy()
        assert np.array_equal(a.last_pick.cpu().numpy(), pick)
        assert np.abs(got - want).max() <= 1e-4
        x, y = got[pick >= 0, :, 0], got[pick >= 0, :, 1]
        assert (x >= 0).all() and (x <= W - 1).all() and (y >= 0).all() and (y <= H - 1).all()
    # scale 4 with labels near the corners: no candidate fits -> identity geometry, labels and (neutral photometry) image unchanged
    corners = torch.tensor([[2.0, 2.0], [W - 3.0, 2.0], [2.0, H - 3.0], [W - 3.0, H - 3.0]]).expand(B, 4, 2).contiguous().cuda()
    f = KeypointAugment(scale=(4.0, 4.0), rotate=10.0, seed=1)
    out, uv3 = f(img, corners)
    assert (f.last_pick == -1).all() and torch.equal(uv3, corners) and torch.equal(out, img)


@pytest.mark.parametrize("shape", SHAPES)
def test_warp_matches_grid_sample_fp64(shape):
    B, H, W = shape
    img, uv = batch(3, B, H, W, margin=0.3 * min(H, W))
    a = KeypointAugment(**GEOM, seed=5)
    p = a.draw(B, H, W)
    out, _ = a(img, uv)
    pick = a.last_pick.cpu()
    assert (pick >= 0).all()
    ref = warp_ref(img, p.inv, pick)
    assert (out.cpu().double() - ref).abs().max().item() <= 2e-6
    assert (out.cpu() == 0).float().mean() > 0.01           # some of the frame comes from outside the image (zero fill)


@pytest.mark.parametrize("shape", SHAPES)
def test_photometric_matches_fp64(shape):
    B, H, W = shape
    img, uv = batch(4, B, H, W)
    img = img * 1.2 - 0.1                                    # values outside [0, 1] too: the clamp is exercised
    a = KeypointAugment(brightness=0.2, contrast=(0.7, 1.3), channel_gain=0.15, seed=6)
    p = a.draw(B, H, W)
    out, uv2 = a(img, uv)
    assert torch.equal(uv2, uv)
    assert (out.cpu().double() - photometric_ref(img, p.photo)).abs().max().item() <= 1e-6


@pytest.mark.parametrize("shape", SHAPES)
def test_noise_matches_philox_box_muller(shape):
    B, H, W = shape
    img, uv = batch(5, B, H, W)
    a = KeypointAugment(noise_std=0.05, seed=7)
    p = a.draw(B, H, W)
    out, _ = a(img, uv)
    ref = photometric_ref(img, p.photo, 0.05, noise_normals(p.key, B, H, W))
    assert (out.cpu().double() - ref).abs().max().item() <= 1e-5


def test_noise_moments():
    sigma = 0.05                                             # 0.5 +- 5.8 sigma stays inside [0, 1]: the clamp is inactive
    img = torch.full((32, 3, 480, 640), 0.5, device="cuda")
    uv = torch.full((32, 4, 2), 100.0, device="cuda")
    out, _ = KeypointAugment(noise_std=sigma, seed=8)(img, uv)
    d = out.double() - 0.5
    assert 0 < out.min().item() and out.max().item() < 1
    assert abs(d.mean().item()) < 1e-3 and abs(d.std().item() - sigma) < 1e-3
    n = d / float(np.float32(sigma))                         # the normals themselves (29.5 M of them)
    assert abs(n.mean().item()) < 1e-3 and abs(n.std().item() - 1.0) < 1e-3


def test_labels_follow_the_discs():
    """Geometry only, on disc images: the colour centroid of every disc in the warped image is within 0.5 px of its moved label."""
    B, H, W, K = 8, 240, 320, 4
    img, uv = synth.disc_batch(torch.Generator().manual_seed(9), B, H, W, K, on_lattice=True)
    a = KeypointAugment(**GEOM, seed=12)
    out, uv2 = a(img.cuda(), uv.cuda())
    out, uv2 = out.cpu().double(), uv2.cpu().double()
    on = synth.disc_palette(K)[:, 0] > 0.5                   # (K, 3): the channels each disc colour saturates
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    checked = 0
    for b in range(B):
        for k in range(K):
            x, y = uv2[b, k].tolist()
            if not (12 <= x <= W - 13 and 12 <= y <= H - 13):    # a disc cut by the frame has a biased centroid
                continue
            lo_on = out[b, on[k]].min(0).values
            hi_off = out[b, ~on[k]].max(0).values
            w = (lo_on - hi_off - 0.3).clamp_min(0)
            cx, cy = float((w * xx).sum() / w.sum()), float((w * yy).sum() / w.sum())
            assert abs(cx - x) <= 0.5 and abs(cy - y) <= 0.5, (b, k, (cx, cy), (x, y))
            checked += 1
    assert (a.last_pick >= 0).sum() >= B // 2 and checked >= B * K // 2


def test_same_seed_same_batch_different_seed_different_batch():
    img, uv = batch(10, 4, 480, 640)
    runs = []
    for seed in (21, 21, 22):
        a = KeypointAugment(**FULL, seed=seed)
        runs.append([t.clone() for _ in range(2) for t in (*a(img, uv), a.last_pick)])
    assert all(torch.equal(x, y) for x, y in zip(runs[0], runs[1]))
    assert not torch.equal(runs[0][0], runs[2][0]) and not torch.equal(runs[0][0], runs[0][3])   # other seed / next call


def test_rejects_aliasing_bad_shapes_and_targets():
    B, H, W = 2, 64, 96
    img, uv = batch(11, B, H, W, K=4)
    a = KeypointAugment(**FULL)
    with pytest.raises(ValueError):
        a(img, uv, out=img)                                  # in-place warp
    buf = torch.empty(img.numel() + 16, device="cuda")
    src = buf[:img.numel()].view_as(img).copy_(img)
    with pytest.raises(ValueError):
        a(src, uv, out=buf[16:].view_as(img))                # partial overlap
    with pytest.raises(ValueError):
        a(img, uv, uv_out=uv)
    with pytest.raises(ValueError):
        a(img[:, :2], uv)
    with pytest.raises(ValueError):
        a(img.double(), uv)
    with pytest.raises(ValueError):
        a(img, uv[:1])
    with pytest.raises(ValueError):
        a(img.cpu(), uv.cpu())
    p = a.draw(B, H, W)
    pick = torch.zeros(B, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        ops.augment_images(img, p.inv.cuda(), pick.long(), p.photo.cuda(), 0.0, 0)
    with pytest.raises(ValueError):
        ops.augment_pick(p.fwd.cuda().double(), uv, H, W)
    # the C ABI refuses in-place and overlapping buffers itself
    lib = _lib.lib()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.hk_augment_images(img.data_ptr(), img.data_ptr(), B, H, W, p.inv.cuda().data_ptr(), 4, pick.data_ptr(),
                               p.photo.cuda().data_ptr(), 0.0, 0, s)
    assert rc == -1 and b"overlaps" in lib.hk_last_error()
    rc = lib.hk_augment_pick(p.fwd.cuda().data_ptr(), B, 4, 4, H, W, uv.data_ptr(), uv.data_ptr() + 8, pick.data_ptr(), s)
    assert rc == -1
    # labels are what the augmenter moves: a target tensor cannot go with it
    torch.manual_seed(0)
    m = hk.KeypointsGauss(4).cuda().train()
    eng = m.train_engine(B, H, W)
    with pytest.raises(ValueError, match="augment"):
        eng.forward_backward(img, target=torch.zeros(B, 4, H, W, device="cuda", dtype=torch.float64), augment=a)


def _train(mode: str, graph: bool, steps: int = 3, B: int = 4, H: int = 128, W: int = 160):
    """Three seeded train_step calls: mode "engine" (augment= on the step), "pre" (a clone of the augmenter applied first, the step
    without augment=) or "none".  Returns per step (loss, flat gradient, parameters)."""
    torch.manual_seed(0)
    m = hk.KeypointsGauss(4).cuda().train()
    m.train_engine(B, H, W).use_cuda_graph = graph
    opt = FusedAdam(m.parameters(), lr=1e-3, weight_decay=1e-4)
    aug = KeypointAugment(**FULL, seed=31)
    if mode == "pre":
        clone = KeypointAugment(**FULL, seed=0)
        clone.load_state_dict(aug.state_dict())
        aug = clone
    gen = torch.Generator().manual_seed(5)
    rec = []
    for _ in range(steps):
        img, uv = synth.disc_batch(gen, B, H, W, 4)
        img, uv = img.cuda(), uv.cuda()
        if mode == "engine":
            loss = train_ops.train_step(m, opt, img, uv, augment=aug)
        else:
            if mode == "pre":
                img, uv = aug(img, uv)
            loss = train_ops.train_step(m, opt, img, uv)
        rec.append((loss.clone(), m.train_engine(B, H, W).flat_grad.clone(), [p.detach().clone() for p in m.parameters()]))
    torch.cuda.synchronize()
    return rec


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "eager"])
def test_train_step_with_augmenter_equals_pre_augmented_batch(graph):
    eng, pre, none = _train("engine", graph), _train("pre", graph), _train("none", graph)
    for (l0, g0, p0), (l1, g1, p1), (l2, _, _) in zip(eng, pre, none):
        assert torch.equal(l0, l1) and torch.equal(g0, g1) and all(torch.equal(a, b) for a, b in zip(p0, p1))
        assert not torch.equal(l0, l2)
    assert len({float(r[0]) for r in eng}) == 3


def test_autograd_backend_sees_the_same_batch():
    torch.backends.cudnn.deterministic = True
    B, H, W = 2, 64, 96
    losses = []
    for mode in ("engine", "pre"):
        torch.manual_seed(0)
        m = hk.KeypointsGauss(4).cuda().train()
        opt = torch.optim.SGD(m.parameters(), lr=0.0)
        aug = KeypointAugment(**FULL, seed=41)
        img, uv = batch(12, B, H, W, K=4, margin=10)
        if mode == "engine":
            losses.append(train_ops.train_step(m, opt, img, uv, backend="autograd", augment=aug))
        else:
            a_img, a_uv = aug(img, uv)
            losses.append(train_ops.train_step(m, opt, a_img, a_uv, backend="autograd"))
    assert torch.equal(losses[0], losses[1])
