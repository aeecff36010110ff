"""CPU: KeypointAugment's configuration checks and parameter draws, and the numpy restatements (tests/augment_ref.py) the GPU tests
compare the augmentation kernels against (no kernels run)."""
import math

import numpy as np
import pytest
import torch

from augment_ref import noise_normals, philox4x32_10, pick_and_move
from hulk_keypoints_b200.augment import KeypointAugment

FULL = dict(rotate=30.0, scale=(0.8, 1.2), translate=0.1, brightness=0.2, contrast=(0.7, 1.3), channel_gain=0.15, noise_std=0.02)


@pytest.mark.parametrize("kw", [dict(rotate=-1.0), dict(translate=-0.1), dict(brightness=-0.1), dict(channel_gain=-0.1),
                                dict(noise_std=-0.01), dict(scale=(0.0, 1.0)), dict(scale=(-1.0, 1.0)), dict(scale=(1.2, 0.8)),
                                dict(contrast=(1.3, 0.7)), dict(contrast=(-0.5, 1.0)), dict(tries=0), dict(tries=17),
                                dict(rotate=float("nan")), dict(scale=(1.0, float("inf")))])
def test_config_validation(kw):
    with pytest.raises(ValueError):
        KeypointAugment(**kw)


def test_limits_accepted():
    KeypointAugment(tries=1)
    KeypointAugment(tries=16, scale=(0.5, 0.5), contrast=(0.0, 0.0))


def _geometry(p, H, W):
    """theta (deg), s, tx, ty recovered in float64 from the fp32 forward table."""
    f = p.fwd.double()
    s = torch.hypot(f[..., 0, 0], f[..., 1, 0])
    theta = torch.rad2deg(torch.atan2(f[..., 1, 0], f[..., 0, 0]))
    ctr = torch.tensor([(W - 1) / 2, (H - 1) / 2], dtype=torch.float64)
    t = f[..., :, 2] - (ctr - torch.einsum("btij,j->bti", f[..., :, :2], ctr))
    return theta, s, t[..., 0], t[..., 1]


def test_draws_deterministic_distinct_and_in_range():
    B, H, W = 64, 480, 640
    a, b = KeypointAugment(**FULL, seed=5), KeypointAugment(**FULL, seed=5)
    p0 = a.draw(B, H, W)
    assert all(torch.equal(x, y) for x, y in zip(p0[:3], a.draw(B, H, W)[:3])) and p0.key == a.draw(B, H, W).key   # draw consumes nothing
    q0 = b.draw(B, H, W)
    assert all(torch.equal(x, y) for x, y in zip(p0[:3], q0[:3])) and p0.key == q0.key                             # same seed
    a._sample(B, H, W)
    p1 = a.draw(B, H, W)
    assert not torch.equal(p0.fwd, p1.fwd) and not torch.equal(p0.photo, p1.photo) and p0.key != p1.key              # next call differs
    assert p0.fwd.shape == (B, 4, 2, 3) and p0.inv.shape == (B, 4, 2, 3) and p0.photo.shape == (B, 5)
    assert all(t.dtype == torch.float32 for t in p0[:3]) and 0 <= p0.key < 2 ** 64
    theta, s, tx, ty = _geometry(p0, H, W)
    eps = 1e-4
    assert theta.abs().max() <= 30 + eps and theta.abs().max() > 25
    assert s.min() >= 0.8 - eps and s.max() <= 1.2 + eps and s.max() - s.min() > 0.3
    assert tx.abs().max() <= 0.1 * W + 1e-2 and ty.abs().max() <= 0.1 * H + 1e-2 and tx.abs().max() > 0.08 * W
    c, beta, g = p0.photo[:, 0], p0.photo[:, 1], p0.photo[:, 2:]
    assert c.min() >= 0.7 and c.max() <= 1.3 and beta.abs().max() <= 0.2 and (g - 1).abs().max() <= 0.15 + 1e-7
    # the inverse table inverts the forward one (both rounded once from fp64)
    ones = torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64).expand(B, 4, 1, 3)
    fwd, inv = torch.cat([p0.fwd.double(), ones], -2), torch.cat([p0.inv.double(), ones], -2)
    assert (inv @ fwd - torch.eye(3, dtype=torch.float64)).abs().max() < 1e-4     # px: offsets up to ~300 carry fp32 ulps of 3e-5


def test_neutral_tables_are_exact_identity():
    p = KeypointAugment().draw(8, 48, 64)
    eye = torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])
    assert torch.equal(p.fwd, eye.expand_as(p.fwd)) and torch.equal(p.inv, eye.expand_as(p.inv))
    assert torch.equal(p.photo, torch.tensor([1.0, 0.0, 1.0, 1.0, 1.0]).expand_as(p.photo))


def test_state_dict_round_trip():
    a = KeypointAugment(**FULL, seed=3)
    for _ in range(3):
        a._sample(4, 96, 128)
        a.calls += 1
    sd = a.state_dict()
    nxt = a.draw(4, 96, 128)
    b = KeypointAugment(**FULL, seed=99)
    b.load_state_dict(sd)
    assert b.calls == 3
    got = b.draw(4, 96, 128)
    assert all(torch.equal(x, y) for x, y in zip(nxt[:3], got[:3])) and nxt.key == got.key
    a._sample(4, 96, 128)                      # the saved state is a copy: advancing `a` leaves it alone
    b.load_state_dict(sd)
    assert torch.equal(b.draw(4, 96, 128).fwd, nxt.fwd)


def test_rank_changes_the_stream():
    base = KeypointAugment(**FULL, seed=1).draw(4, 96, 128)
    assert torch.equal(KeypointAugment(**FULL, seed=1, rank=0).draw(4, 96, 128).fwd, base.fwd)   # no process group: rank 0
    r1 = KeypointAugment(**FULL, seed=1, rank=1).draw(4, 96, 128)
    r2 = KeypointAugment(**FULL, seed=1, rank=2).draw(4, 96, 128)
    assert not torch.equal(r1.fwd, base.fwd) and not torch.equal(r2.fwd, r1.fwd) and len({base.key, r1.key, r2.key}) == 3


def test_philox_known_answers():
    """Random123's known-answer vectors for philox4x32-10."""
    assert philox4x32_10([0, 0, 0, 0], [0, 0]).tolist() == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert philox4x32_10([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2).tolist() == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert (philox4x32_10([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]).tolist()
            == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])
    # broadcast over a batch of counters equals one call per counter
    ctr = np.array([[i, 7, 1, 2] for i in range(5)], dtype=np.uint32)
    batch = philox4x32_10(ctr, [123, 456])
    assert all(batch[i].tolist() == philox4x32_10(ctr[i], [123, 456]).tolist() for i in range(5))


def test_noise_normals_layout_and_moments():
    n = noise_normals(0x0123456789ABCDEF, 2, 24, 30)
    assert n.shape == (2, 3, 24, 30) and np.isfinite(n).all()
    assert abs(n.mean()) < 0.05 and abs(n.std() - 1) < 0.05
    assert np.array_equal(n[..., :28], noise_normals(0x0123456789ABCDEF, 2, 24, 28))     # per 4-pixel group: the width only cuts
    assert not np.array_equal(n, noise_normals(0x0123456789ABCDEE, 2, 24, 30))


def test_pick_restatement_in_frame_and_fallback():
    B, H, W, K = 32, 96, 128, 6
    gen = torch.Generator().manual_seed(0)
    uv = torch.stack([torch.rand(B, K, generator=gen) * (W - 1), torch.rand(B, K, generator=gen) * (H - 1)], -1).numpy()
    p = KeypointAugment(rotate=40, scale=(0.7, 1.4), translate=0.2, seed=4).draw(B, H, W)
    pick, moved = pick_and_move(p.fwd.numpy(), uv, H, W)
    inside = lambda q: ((q[..., 0] >= 0) & (q[..., 0] <= W - 1) & (q[..., 1] >= 0) & (q[..., 1] <= H - 1)).all(-1)  # noqa: E731
    assert (pick >= 0).sum() >= B // 2
    assert inside(moved).all()
    for b in range(B):
        fwd = p.fwd[b].double().numpy()
        for t in range(max(pick[b], 0) if pick[b] >= 0 else 4):                  # the candidates before the pick leave the frame
            q = uv[b] @ fwd[t, :, :2].T + fwd[t, :, 2]
            assert not inside(q + np.sign(q - [(W - 1) / 2, (H - 1) / 2]) * 1e-3)
        if pick[b] >= 0:
            want = uv[b].astype(np.float64) @ fwd[pick[b], :, :2].T + fwd[pick[b], :, 2]
            assert np.abs(moved[b] - want).max() < 1e-4
        else:
            assert np.array_equal(moved[b], uv[b])
    # scale 4 with keypoints near the corners: no candidate keeps them in the frame -> identity, labels unchanged
    corners = np.array([[[2.0, 2.0], [W - 3.0, 2.0], [2.0, H - 3.0], [W - 3.0, H - 3.0]]] * 4, dtype=np.float32)
    q = KeypointAugment(scale=(4.0, 4.0), rotate=10, seed=1).draw(4, H, W)
    pick, moved = pick_and_move(q.fwd.numpy(), corners, H, W)
    assert (pick == -1).all() and np.array_equal(moved, corners)


def test_rotation_direction_and_centre():
    """The label map fixes the image centre, and a positive angle (here the largest of 64 draws with rotate=90) turns +x towards +y."""
    H, W = 48, 64
    p = KeypointAugment(rotate=90, seed=0).draw(16, H, W)
    theta, s, _, _ = _geometry(p, H, W)
    b, t = np.unravel_index(int(theta.argmax()), theta.shape)
    f = p.fwd[b, t].double()
    ctr = torch.tensor([(W - 1) / 2, (H - 1) / 2], dtype=torch.float64)
    assert torch.allclose(f[:, :2] @ ctr + f[:, 2], ctr, atol=1e-4)
    d = f[:, :2] @ torch.tensor([1.0, 0.0], dtype=torch.float64)
    assert d[1] > 0 and math.isclose(float(d.norm()), 1.0, rel_tol=1e-5)
