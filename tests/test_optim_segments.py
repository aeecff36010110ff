"""The segment table of FusedAdam's update launch (hk_adam_step_segments), built on the host: flat offsets, merging of runs, bias
corrections, decoupled weight-decay multipliers and the table's cap.  Pure Python, no device."""
import ctypes
import math

import numpy as np
import pytest

from hulk_keypoints_b200 import _lib
from hulk_keypoints_b200.optim import build_segments, flat_offsets, segment_row

ADAM = (1e-3, 0.9, 0.999, 1e-8, 1e-4, False)


def f32(x):
    return float(np.float32(x))


def test_flat_offsets_start_every_tensor_on_16_bytes():
    offs, total = flat_offsets([5, 4, 1, 0, 7, 3])
    assert offs == [0, 8, 12, 16, 16, 24] and total == 28
    assert all(o % 4 == 0 for o in offs)
    # float4 runs of each tensor: padding belongs to the tensor before it, so a float4 never straddles two tensors
    runs = [(o // 4, (o + (n + 3) // 4 * 4) // 4) for o, n in zip(offs, [5, 4, 1, 0, 7, 3])]
    assert runs == [(0, 2), (2, 3), (3, 4), (4, 4), (4, 6), (6, 7)]
    assert all(a[1] == b[0] for a, b in zip(runs, runs[1:]))


def test_adjacent_equal_runs_merge_and_empty_runs_vanish():
    hyp = [ADAM, ADAM, (2e-3,) + ADAM[1:]]
    # groups 0 and 1 have equal hyperparameters: one segment; group 2 differs; the empty run between them does not split them
    rows = build_segments([(0, 2, 0, 1), (2, 2, 2, 1), (2, 5, 1, 1), (5, 9, 2, 1), (9, 10, 0, 1)], hyp)
    assert [(r[0], r[1]) for r in rows] == [(0, 5), (5, 9), (9, 10)]
    assert rows[0][2:] == rows[2][2:] != rows[1][2:]
    # the same group at different step counts does not merge
    rows = build_segments([(0, 2, 0, 1), (2, 4, 0, 2)], hyp)
    assert len(rows) == 2 and rows[0][2] != rows[1][2]
    # no decay vs decay: different segments
    rows = build_segments([(0, 2, 0, 3), (2, 4, 1, 3)], [ADAM, ADAM[:4] + (0.0, False)])
    assert len(rows) == 2 and (rows[0][7], rows[1][7]) == (f32(1e-4), 0.0)


@pytest.mark.parametrize("step", [1, 2, 7, 1000])
def test_bias_corrections_follow_hk_adam_step(step):
    lr, b1, b2 = 3e-4, 0.85, 0.995
    row = segment_row(lr, b1, b2, 1e-6, 0.0, False, step)
    # hk_adam_step: fp32 arguments, corrections in double, rounded to fp32 once
    lr32, b132, b232 = np.float32(lr), np.float32(b1), np.float32(b2)
    bc1 = 1.0 - math.pow(float(b132), step)
    bc2 = 1.0 - math.pow(float(b232), step)
    assert row[0] == f32(float(lr32) / bc1)
    assert row[1] == f32(1.0 / math.sqrt(bc2))
    assert row[2:6] == (float(b132), float(b232), f32(1e-6), 0.0)
    assert row[6:] == (1.0, 0)
    if step == 1:
        assert row[0] == pytest.approx(lr / (1 - b1), rel=1e-6) and row[1] == pytest.approx(1 / math.sqrt(1 - b2), rel=1e-6)


def test_decoupled_multiplier():
    lr, wd = 1e-3, 1e-2
    coupled = segment_row(lr, 0.9, 0.999, 1e-8, wd, False, 4)
    decoupled = segment_row(lr, 0.9, 0.999, 1e-8, wd, True, 4)
    assert coupled[6:] == (1.0, 0)
    # torch's param.mul_(1 - lr * weight_decay): the multiplier is formed in double and applied in fp32
    assert decoupled[6:] == (f32(1.0 - lr * wd), 1)
    assert coupled[:6] == decoupled[:6]
    # different decay modes never merge
    rows = build_segments([(0, 1, 0, 4), (1, 2, 1, 4)], [(lr, 0.9, 0.999, 1e-8, wd, False), (lr, 0.9, 0.999, 1e-8, wd, True)])
    assert len(rows) == 2


def test_table_cap():
    cap = _lib.ADAM_MAX_SEGMENTS
    hyp = [ADAM, (2e-3,) + ADAM[1:]]
    rows = build_segments([(i, i + 1, i % 2, 1) for i in range(cap)], hyp)
    assert len(rows) == cap
    with pytest.raises(RuntimeError, match=f"at most {cap}"):
        build_segments([(i, i + 1, i % 2, 1) for i in range(cap + 1)], hyp)
    # the table travels as one launch parameter: it has to stay inside the 32 KB kernel-parameter space of sm_100
    assert ctypes.sizeof(_lib.HkAdamSegment) == 48 and cap * ctypes.sizeof(_lib.HkAdamSegment) + 64 <= 32764
