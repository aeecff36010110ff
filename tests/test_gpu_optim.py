"""FusedAdam as a torch optimizer: parameter groups, learning-rate schedulers, decoupled weight decay, torch's state_dict format,
resume, progressive unfreezing and the engine-defined flat layout -- all on one hk_adam_step_segments launch per step."""
import ctypes as C
import io
import warnings

import pytest
import torch

import hulk_keypoints_b200 as hk
from hulk_keypoints_b200 import synth, train_ops
from hulk_keypoints_b200._lib import HkAdamSegment, check, lib, ptr, stream_ptr
from hulk_keypoints_b200.optim import FusedAdam, segment_row

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

SHAPES = [(64, 3, 7, 7), (64,), (128, 64, 3, 3), (1000, 512, 1, 1), (5,), (3, 3)]   # those of test_fused_adam_matches_torch_adam
RTOL, ATOL = 2e-6, 2e-7
B, H, W = 4, 128, 160


def dev():
    return torch.device("cuda")


def _params(seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.nn.Parameter(torch.randn(s, device=dev(), generator=g)) for s in SHAPES]


def _clone(params):
    return [torch.nn.Parameter(p.detach().clone()) for p in params]


def _groups(ps):
    """Three groups that differ in every option: coupled decay, decoupled decay, no decay."""
    return [dict(params=ps[0:2], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4),
            dict(params=ps[2:4], lr=3e-4, betas=(0.8, 0.99), eps=1e-6, weight_decay=1e-2, decoupled_weight_decay=True),
            dict(params=ps[4:6], lr=2e-3, betas=(0.95, 0.9999), eps=1e-7, weight_decay=0.0)]


def _grads(step):
    g = torch.Generator(device="cuda").manual_seed(100 + step)
    return [torch.randn(s, device=dev(), generator=g) * (0.0 if (i == 3 and step % 2) else 1.0) for i, s in enumerate(SHAPES)]


def _set_grads(opt, params, step):
    for p, g in zip(params, _grads(step)):
        if isinstance(opt, FusedAdam):
            p.grad.copy_(g)        # gradient views into the flat buffer stay attached
        else:
            p.grad = g.clone()


def _close(ref, ours):
    worst = 0.0
    for p, q in zip(ref, ours):
        assert torch.allclose(p, q, rtol=RTOL, atol=ATOL), (p - q).abs().max().item()
        worst = max(worst, ((p - q).abs() / (ATOL + RTOL * p.abs())).max().item())
    return worst


# ------------------------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("n", [1_000_003, 4099])
def test_one_segment_equals_hk_adam_step_bit_for_bit(n):
    g = torch.Generator(device="cuda").manual_seed(n)
    p, gr, m = (torch.randn(n, device=dev(), generator=g) for _ in range(3))
    v = torch.rand(n, device=dev(), generator=g) * 1e-2
    ref = [t.clone() for t in (p, m, v)]
    one = [t.clone() for t in (p, m, v)]
    many = [t.clone() for t in (p, m, v)]
    lr, b1, b2, eps, wd = 1e-3, 0.9, 0.999, 1e-8, 1e-4
    n4 = (n + 3) // 4
    cuts = [0, 1, 2, n4 // 3, n4 // 2, n4 - 1, n4]   # the same hyperparameters split into unmerged segments
    for step in range(1, 6):
        check(lib().hk_adam_step(ptr(ref[0]), ptr(gr), ptr(ref[1]), ptr(ref[2]), C.c_longlong(n), lr, b1, b2, eps, wd, step,
                                 stream_ptr()), "hk_adam_step")
        row = segment_row(lr, b1, b2, eps, wd, False, step)
        for bufs, bounds in ((one, [0, n4]), (many, cuts)):
            segs = [HkAdamSegment(a, b, *row) for a, b in zip(bounds, bounds[1:])]
            check(lib().hk_adam_step_segments(ptr(bufs[0]), ptr(gr), ptr(bufs[1]), ptr(bufs[2]), C.c_longlong(n),
                                              (HkAdamSegment * len(segs))(*segs), len(segs), stream_ptr()), "hk_adam_step_segments")
    for a, b, c in zip(ref, one, many):
        assert torch.equal(a, b) and torch.equal(a, c)
    # malformed tables are refused before any launch
    bad = (HkAdamSegment * 2)(HkAdamSegment(0, 5, *row), HkAdamSegment(6, n4, *row))
    assert lib().hk_adam_step_segments(ptr(p), ptr(gr), ptr(m), ptr(v), C.c_longlong(n), bad, 2, stream_ptr()) != 0
    assert b"contiguous" in lib().hk_last_error()


# -------------------------------------------------------------------------------------------------------------------------- groups
def test_groups_match_torch_adam_and_adamw():
    ref_p = _params()
    ours_p = _clone(ref_p)
    ref = torch.optim.Adam(_groups(ref_p), foreach=False)
    ours = FusedAdam(_groups(ours_p))
    for step in range(5):
        ref.zero_grad(); ours.zero_grad()
        _set_grads(ref, ref_p, step); _set_grads(ours, ours_p, step)
        ref.step(); ours.step()
    _close(ref_p, ours_p)
    # the decoupled group against torch.optim.AdamW itself
    aw_p = _clone(_params())
    aw = torch.optim.AdamW(aw_p[2:4], lr=3e-4, betas=(0.8, 0.99), eps=1e-6, weight_decay=1e-2, foreach=False)
    for step in range(5):
        for p, g in zip(aw_p[2:4], _grads(step)[2:4]):
            p.grad = g.clone()
        aw.step()
    _close(aw_p[2:4], ours_p[2:4])
    # lr 0 on one group: its parameters stay exactly where they are, the others move
    ours.param_groups[1]["lr"] = 0.0
    before = [p.detach().clone() for p in ours_p]
    _set_grads(ours, ours_p, 5)
    ours.step()
    torch.cuda.synchronize()
    assert all(torch.equal(p, b) for p, b in zip(ours_p[2:4], before[2:4]))
    assert not any(torch.equal(p, b) for p, b in zip(ours_p[0:2], before[0:2]))


@pytest.mark.parametrize("sched", ["StepLR", "CosineAnnealingLR", "OneCycleLR"])
def test_schedulers_track_torch_adam(sched):
    """20 steps under the same scheduler: every parameter within 2e-6 relative + 2e-7 absolute of torch.optim.Adam."""
    def make(opt):
        S = torch.optim.lr_scheduler
        if sched == "StepLR":
            return S.StepLR(opt, step_size=4, gamma=0.5)
        if sched == "CosineAnnealingLR":
            return S.CosineAnnealingLR(opt, T_max=20, eta_min=1e-5)
        return S.OneCycleLR(opt, max_lr=[2e-3, 1e-3, 4e-3], total_steps=20, cycle_momentum=True)
    ref_p = _params(1)
    ours_p = _clone(ref_p)
    ref = torch.optim.Adam(_groups(ref_p), foreach=False)
    ours = FusedAdam(_groups(ours_p))
    rs, os_ = make(ref), make(ours)
    for step in range(20):
        _set_grads(ref, ref_p, step); _set_grads(ours, ours_p, step)
        ref.step(); ours.step()
        rs.step(); os_.step()
        assert [g["lr"] for g in ref.param_groups] == [g["lr"] for g in ours.param_groups]
        assert [g["betas"] for g in ref.param_groups] == [g["betas"] for g in ours.param_groups]
    worst = _close(ref_p, ours_p)
    print(f"\n[{sched}] worst |torch - ours| / (2e-7 + 2e-6 |torch|) over 20 steps: {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------- state_dict
def _strip(sd):
    return {"state": {i: {k: (v.dtype, tuple(v.shape), v.device.type) for k, v in s.items()} for i, s in sd["state"].items()},
            "param_groups": sd["param_groups"]}


def test_state_dict_is_torch_adam_format_and_cross_loads():
    ref_p, ours_p = _params(2), _clone(_params(2))
    ref, ours = torch.optim.Adam(_groups(ref_p)), FusedAdam(_groups(ours_p))
    for step in range(2):
        _set_grads(ref, ref_p, step); _set_grads(ours, ours_p, step)
        ref.step(); ours.step()
    a, b = ref.state_dict(), ours.state_dict()
    assert list(a) == list(b) and _strip(a) == _strip(b)
    for s in b["state"].values():
        assert s["step"].item() == 2.0 and s["step"].dim() == 0
    assert all(list(ga) == list(gb) for ga, gb in zip(a["param_groups"], b["param_groups"]))

    def uninterrupted():
        ps = _params(3)
        opt = torch.optim.Adam(_groups(ps), foreach=False)
        for step in range(6):
            _set_grads(opt, ps, step)
            opt.step()
        return ps

    def interrupted(first, second):
        ps = _params(3)
        opt = first(_groups(ps))
        for step in range(3):
            _set_grads(opt, ps, step)
            opt.step()
        buf = io.BytesIO()
        torch.save(opt.state_dict(), buf)
        ps = _clone(ps)
        opt = second([dict(params=g["params"]) for g in _groups(ps)])   # hyperparameters come from the saved groups
        buf.seek(0)
        opt.load_state_dict(torch.load(buf, weights_only=True))
        for step in range(3, 6):
            _set_grads(opt, ps, step)
            opt.step()
        return ps

    full = uninterrupted()
    torch_adam = lambda gs: torch.optim.Adam(gs, foreach=False)   # noqa: E731
    _close(full, interrupted(FusedAdam, torch_adam))
    _close(full, interrupted(torch_adam, FusedAdam))
    # the decoupled group's state also loads into torch.optim.AdamW
    aw = torch.optim.AdamW([torch.nn.Parameter(p.detach().clone()) for p in ours_p[2:4]], lr=3e-4)
    sd = ours.state_dict()
    aw.load_state_dict({"state": {i - 2: s for i, s in sd["state"].items() if i in (2, 3)},
                        "param_groups": [dict(sd["param_groups"][1], params=[0, 1])]})
    assert aw.param_groups[0]["decoupled_weight_decay"] and aw.param_groups[0]["lr"] == 3e-4


# ------------------------------------------------------------------------------------------------------------------------- engine
def _model(seed=0):
    torch.manual_seed(seed)
    return hk.KeypointsGauss(4, img_height=H, img_width=W).cuda().train()


def _batch(step):
    img, uv = synth.disc_batch(torch.Generator().manual_seed(300 + step), B, H, W, 4)
    return img.cuda(), uv.cuda()


def _finetune_groups(m):
    net = m.resnet.resnet34_8s
    fc = list(net.fc.parameters())
    bn = [p for mod in m.modules() if isinstance(mod, torch.nn.BatchNorm2d) for p in mod.parameters()]
    skip = {id(p) for p in fc + bn}
    rest = [p for p in m.parameters() if id(p) not in skip]
    return [dict(params=fc, lr=1e-3), dict(params=rest), dict(params=bn, weight_decay=0.0)]


def test_resume_on_the_engine_is_bit_for_bit():
    def setup(seed):
        m = _model(seed)
        opt = FusedAdam(_finetune_groups(m), lr=1e-4, weight_decay=1e-4)
        return m, opt, torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)

    m, opt, sched = setup(0)
    for s in range(6):
        train_ops.train_step(m, opt, *_batch(s))
        sched.step()
    run_a = ({k: v.clone() for k, v in m.state_dict().items()}, opt.state_dict())

    m, opt, sched = setup(0)
    for s in range(3):
        train_ops.train_step(m, opt, *_batch(s))
        sched.step()
    buf = io.BytesIO()
    torch.save({"model": m.state_dict(), "optimizer": opt.state_dict(), "scheduler": sched.state_dict()}, buf)
    del m, opt, sched
    m, opt, sched = setup(1)   # fresh objects from another init: everything comes from the checkpoint
    buf.seek(0)
    ck = torch.load(buf, weights_only=True)
    m.load_state_dict(ck["model"]); opt.load_state_dict(ck["optimizer"]); sched.load_state_dict(ck["scheduler"])
    for s in range(3, 6):
        train_ops.train_step(m, opt, *_batch(s))
        sched.step()
    sd_a, osd_a = run_a
    sd_b, osd_b = m.state_dict(), opt.state_dict()
    assert all(torch.equal(sd_a[k], sd_b[k]) for k in sd_a)           # parameters and BatchNorm buffers
    assert osd_a["param_groups"] == osd_b["param_groups"] and list(osd_a["state"]) == list(osd_b["state"])
    for i, s in osd_a["state"].items():
        assert all(torch.equal(s[k], osd_b["state"][i][k]) for k in s), i


def test_flat_layout_follows_the_engine():
    plain_m = _model()
    plain = FusedAdam(plain_m.parameters(), lr=1e-3, weight_decay=1e-4)
    fc_first_m = _model()
    net = fc_first_m.resnet.resnet34_8s
    fc = list(net.fc.parameters())
    fc_first = FusedAdam([{"params": fc}, {"params": [p for p in fc_first_m.parameters() if all(p is not q for q in fc)]}],
                         lr=1e-3, weight_decay=1e-4)
    two_phase_m = _model()
    tfc = list(two_phase_m.resnet.resnet34_8s.fc.parameters())
    two_phase = FusedAdam([{"params": tfc}, {"params": [p for p in two_phase_m.parameters() if all(p is not q for q in tfc)]}],
                          lr=1e-3, weight_decay=1e-4)
    for s in range(3):
        img, uv = _batch(s)
        train_ops.train_step(plain_m, plain, img, uv)
        train_ops.train_step(fc_first_m, fc_first, img, uv)
        # the data-parallel step's two phases, by hand (train_step takes them only in a multi-rank job)
        eng = two_phase_m.train_engine(B, H, W)
        eng.sync_flags()
        if two_phase.flat_grad.data_ptr() != eng.flat_grad.data_ptr():
            two_phase.adopt_grad_buffer(eng.flat_grad, eng.params)
        eng.flat_grad.zero_()
        eng.forward_backward_late(img, uv)
        eng.backward_early()
        two_phase.step()
    assert [id(p) for p in fc_first.params] == [id(p) for p in fc_first_m.train_engine(B, H, W).params]
    for a, b, c in zip(plain_m.parameters(), fc_first_m.parameters(), two_phase_m.parameters()):
        assert torch.equal(a, b) and torch.equal(a, c)
    assert torch.equal(plain.exp_avg, fc_first.exp_avg) and torch.equal(plain.exp_avg_sq, two_phase.exp_avg_sq)
    # an optimiser that misses one trainable parameter refuses to train
    m = _model()
    w0 = m.resnet.resnet34_8s.conv1.weight.detach().clone()
    opt = FusedAdam(list(m.parameters())[1:], lr=1e-3)
    with pytest.raises(ValueError, match="gradient buffer layout mismatch"):
        train_ops.train_step(m, opt, *_batch(0))
    assert torch.equal(m.resnet.resnet34_8s.conv1.weight, w0)


def test_progressive_unfreezing_tracks_torch_adam():
    def run(make_opt, profile=False):
        m = _model(4)
        train_ops.freeze_preset(m, "torchvision")
        opt = make_opt([p for p in m.parameters() if p.requires_grad])   # torch.optim.Adam keeps frozen parameters; FusedAdam drops them
        losses = []
        for s in range(3):
            losses.append(train_ops.train_step(m, opt, *_batch(10 + s)).item())
        layer1 = list(m.resnet.resnet34_8s.layer1.parameters())
        for p in layer1:
            p.requires_grad_(True)
        before = opt.state_dict() if isinstance(opt, FusedAdam) else None
        opt.add_param_group({"params": layer1, "lr": 1e-5})
        launches = None
        if before is not None:
            after = opt.state_dict()
            n_old = sum(len(g["params"]) for g in before["param_groups"])
            assert sorted(after["state"]) == list(range(n_old))              # the new parameters start at step 0
            for i, s in before["state"].items():
                assert all(torch.equal(s[k], after["state"][i][k]) for k in s), i
            assert all(float(opt.exp_avg[o:o + p.numel()].abs().sum()) == 0 for p, o in zip(opt.params, opt._offs)
                       if any(p is q for q in layer1))
        for s in range(3, 6):
            img, uv = _batch(10 + s)
            if profile and s == 5:
                torch.cuda.synchronize()
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    losses.append(train_ops.train_step(m, opt, img, uv).item())
                launches = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "adam" in e.name]
            else:
                losses.append(train_ops.train_step(m, opt, img, uv).item())
        return m, losses, launches

    a, la, launches = run(lambda ps: FusedAdam(ps, lr=1e-4, weight_decay=1e-4), profile=True)
    b, lb, _ = run(lambda ps: torch.optim.Adam(ps, lr=1e-4, weight_decay=1e-4))
    assert len(launches) == 1 and "adam_segments_kernel" in launches[0], launches   # one update launch for three groups
    for x, y in zip(la, lb):
        assert abs(x - y) < 2e-3 * abs(y)
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        if sa[k].dtype.is_floating_point:
            # the bar of test_fused_adam_training_tracks_torch_adam, for 6 steps at lr <= 1e-4
            assert torch.allclose(sa[k], sb[k], rtol=1e-3, atol=2 * 1e-4 * 6 + 1e-5), k


# ---------------------------------------------------------------------------------------------------------------------- rejections
@pytest.mark.parametrize("option", ["amsgrad", "maximize", "capturable", "differentiable", "foreach", "fused"])
def test_unsupported_options_are_rejected(option):
    ps = _params()
    with pytest.raises(ValueError, match=f"FusedAdam does not support {option}=True"):
        FusedAdam(ps, **{option: True})
    with pytest.raises(ValueError, match=f"FusedAdam does not support {option}=True"):
        FusedAdam([{"params": ps[:2], option: True}, {"params": ps[2:]}])
    opt = FusedAdam(ps)
    opt.param_groups[0][option] = True
    with pytest.raises(ValueError, match=f"FusedAdam does not support {option}=True"):
        opt.step()


def test_cuda_lr_and_amsgrad_state_are_rejected():
    ps = _params()
    with pytest.raises(ValueError, match="lr is a tensor on cuda"):
        FusedAdam(ps, lr=torch.tensor(1e-3, device="cuda"))
    opt = FusedAdam(ps, lr=torch.tensor(1e-3))   # a CPU tensor is read without a device sync
    opt.step()
    opt.param_groups[0]["lr"] = torch.tensor(1e-3, device="cuda")
    with pytest.raises(ValueError, match="lr is a tensor on cuda"):
        opt.step()
    ref_p = _clone(ps)
    ams = torch.optim.Adam(ref_p, amsgrad=True)
    for p in ref_p:
        p.grad = torch.ones_like(p)
    ams.step()
    opt = FusedAdam(_clone(ps))
    with pytest.raises(ValueError, match="amsgrad"):
        opt.load_state_dict(ams.state_dict())
    sd = ams.state_dict()
    sd["param_groups"][0]["amsgrad"] = False
    with pytest.raises(ValueError, match="max_exp_avg_sq"):
        opt.load_state_dict(sd)
