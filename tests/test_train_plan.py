"""The training engine's backward plan (train_engine.backward_plan) under torch's fine-tuning flags, on the CPU: which convs get a
weight gradient, a data gradient and a BatchNorm backward, where the backward stops, and the launch count it predicts."""
import pytest
import torch

import hulk_keypoints_b200 as hk
from hulk_keypoints_b200 import train_ops
from hulk_keypoints_b200.train_engine import backward_plan, step_launches


@pytest.fixture(scope="module")
def model():
    return hk.KeypointsGauss(4, img_height=64, img_width=96)


def _plan(model, preset):
    train_ops.freeze_preset(model, preset)
    return backward_plan(model.resnet.resnet34_8s)


def test_default_plan_runs_everything(model):
    pl = _plan(model, "none")
    assert pl.lo == 0 and pl.stem and pl.dfeat and pl.fc_weight and pl.fc_bias
    assert not pl.frozen_any and pl.train_bn_any
    for name, p in pl.convs.items():
        assert not p.frozen and p.wgrad and p.dy and p.bwd and p.dgamma and p.dbeta, name
        assert p.dgrad == (name != "stem"), name


def test_frozen_bn_plan(model):
    pl = _plan(model, "bn")
    assert all(p.frozen and p.bwd and p.dgamma and p.dbeta for p in pl.convs.values())
    assert not pl.train_bn_any and pl.lo == 0 and pl.stem
    assert step_launches(model.resnet.resnet34_8s, pl) < step_launches(model.resnet.resnet34_8s, _plan(model, "none"))


def test_torchvision_plan_stops_above_layer1(model):
    pl = _plan(model, "torchvision")
    assert not pl.stem and pl.lo == 3          # layer1 = blocks 0..2
    for bi in range(3):
        assert not any(pl.convs[f"b{bi}.{k}"].bwd for k in ("c1", "c2")), bi
    assert not pl.grad_in[3] and pl.grad_in[4]
    b3 = pl.convs["b3.c1"]                     # layer2.0.conv1: weight gradient, no data gradient
    assert b3.wgrad and not b3.dgrad and b3.dy and b3.frozen and not b3.dgamma
    assert pl.convs["b3.ds"].wgrad and not pl.convs["b3.ds"].dgrad
    assert all(not (p.dgamma or p.dbeta) for p in pl.convs.values())


def test_head_plan_runs_only_the_head(model):
    pl = _plan(model, "head")
    assert not pl.dfeat and pl.lo == 16 and not pl.stem and pl.fc_weight and pl.fc_bias
    assert not any(p.bwd for p in pl.convs.values())
    # forward: packs, fold, stem + pool, 35 one-launch convs, head logits, loss; backward: the head without dfeat
    assert step_launches(model.resnet.resnet34_8s, pl) == 2 + 1 + 2 + 35 + 2 + 2 + 4


def test_only_stem_bn_trained(model):
    train_ops.freeze_preset(model, "head")
    net = model.resnet.resnet34_8s
    net.fc.weight.requires_grad_(False)
    net.fc.bias.requires_grad_(False)
    net.bn1.weight.requires_grad_(True)
    pl = backward_plan(net)
    assert pl.stem and pl.lo == 0 and pl.dfeat and not pl.fc_weight
    st = pl.convs["stem"]
    assert st.dgamma and not st.dbeta and not st.wgrad and not st.dy
    for bi in range(16):                        # the gradient passes through every block, no weight gradient anywhere
        p1 = pl.convs[f"b{bi}.c1"]
        assert pl.grad_in[bi] and p1.dgrad and not p1.wgrad and not p1.dgamma


def test_layer3_conv1_frozen(model):
    train_ops.freeze_preset(model, "none")
    net = model.resnet.resnet34_8s
    net.layer3[0].conv1.weight.requires_grad_(False)
    pl = backward_plan(net)
    p = pl.convs["b7.c1"]
    assert not p.wgrad and p.dgrad and p.dy and p.bwd
    assert pl.lo == 0 and pl.stem


def test_unsupported_batchnorm_is_reported(model):
    m = hk.KeypointsGauss(4, img_height=64, img_width=96)
    assert m._bn_unsupported() is None
    m.resnet.resnet34_8s.layer1[0].bn2.momentum = None
    assert "momentum=None" in m._bn_unsupported()
    m = hk.KeypointsGauss(4, img_height=64, img_width=96)
    m.resnet.resnet34_8s.bn1 = torch.nn.BatchNorm2d(64, track_running_stats=False)
    assert "track_running_stats=False" in m._bn_unsupported()
    m = hk.KeypointsGauss(4, img_height=64, img_width=96)
    m.resnet.resnet34_8s.bn1 = torch.nn.BatchNorm2d(64, affine=False)
    assert "affine=False" in m._bn_unsupported()
