"""FusedAdam: torch.optim.Adam / AdamW (reference train.py:79) as ONE kernel per step, with torch's optimizer interface.

Parameters and gradients are flattened into contiguous fp32 buffers (each `param.data` / `param.grad` becomes a view into them), so
autograd accumulates straight into the flat gradient buffer, a data-parallel all-reduce is a single collective over it, and the update is
one pass of `hk_adam_step_segments`.  Parameter groups, learning-rate schedulers, `state_dict` / `load_state_dict` and `add_param_group`
work as on `torch.optim.Adam`: every step reads the groups' hyperparameters and turns them into a table of segments -- runs of the flat
buffer that share every hyperparameter and the step count -- which the kernel takes as a launch parameter (one launch for any number
of groups, no host synchronisation).  All parameters are updated, including the 996 dead fc rows, which receive zero gradient but are
still decayed -- as in the reference.

The flat layout is the training engine's parameter order (`TrainEngine.params`: model order, trainable parameters only); `train_ops`
hands it over through `adopt_grad_buffer(flat_grad, params)`, which reorders the buffers once when the groups list the parameters in
another order.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Any, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from ._lib import ADAM_MAX_SEGMENTS, HkAdamSegment, check, lib, note_raw_parameter_write, ptr, stream_ptr

# torch.optim.Adam options without a fused path here (their defaults are all off).  foreach / fused only choose torch's implementation,
# so False is accepted too.
_UNSUPPORTED = ("amsgrad", "maximize", "capturable", "differentiable", "foreach", "fused")
_LAYOUT_MISMATCH = ("gradient buffer layout mismatch (the optimiser was built for another set of trainable parameters: build it after "
                    "setting requires_grad, or add_param_group when unfreezing, as in torch)")


def _f32(x: float) -> float:
    return float(np.float32(x))


def segment_row(lr: float, beta1: float, beta2: float, eps: float, weight_decay: float, decoupled: bool, step: int) -> Tuple:
    """The hyperparameter fields of one HkAdamSegment at 1-based `step`: (lr_over_bc1, inv_sqrt_bc2, beta1, beta2, eps, weight_decay,
    decay, decoupled), fp32 values.  The bias corrections are computed in double from the fp32-rounded lr and betas, exactly as
    hk_adam_step does, so a coupled segment updates bit for bit like it.  decay = fp32(1 - lr*wd) for decoupled decay, 1 otherwise."""
    lr32, b1, b2 = _f32(lr), _f32(beta1), _f32(beta2)
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    decay = _f32(1.0 - lr * weight_decay) if decoupled else 1.0
    return (_f32(lr32 / bc1), _f32(1.0 / math.sqrt(bc2)), b1, b2, _f32(eps), _f32(weight_decay), decay, int(bool(decoupled)))


def flat_offsets(numels: Sequence[int]) -> Tuple[List[int], int]:
    """Offsets (in floats) of tensors laid out back to back with each one starting on a 16-byte boundary, and the padded total."""
    offs, total = [], 0
    for n in numels:
        offs.append(total)
        total += (n + 3) // 4 * 4
    return offs, total


def build_segments(runs: Iterable[Tuple[int, int, int, int]], hypers: Sequence[Tuple]) -> List[Tuple]:
    """The segment table of one step.  `runs`: (begin4, end4, group, step) in flat order, contiguous, with the step this update
    performs; `hypers[group]` = (lr, beta1, beta2, eps, weight_decay, decoupled).  Adjacent runs whose fields come out equal merge
    into one segment; empty runs are dropped.  Returns (begin4, end4, *segment_row) tuples; more than ADAM_MAX_SEGMENTS raise."""
    rows: List[list] = []
    cache: Dict[Tuple[int, int], Tuple] = {}
    for b4, e4, gi, step in runs:
        if e4 <= b4:
            continue
        row = cache.get((gi, step))
        if row is None:
            row = cache[(gi, step)] = segment_row(*hypers[gi], step)
        if rows and rows[-1][1] == b4 and rows[-1][2:] == list(row):
            rows[-1][1] = e4
        else:
            rows.append([b4, e4, *row])
    if len(rows) > ADAM_MAX_SEGMENTS:
        raise RuntimeError(f"FusedAdam: the parameter groups split the flat buffer into {len(rows)} segments of distinct "
                           f"hyperparameters; one update launch takes at most {ADAM_MAX_SEGMENTS}")
    return [tuple(r) for r in rows]


def _trainable(params) -> list:
    """A group's parameters without the frozen ones (plain tensors or (name, tensor) pairs)."""
    if isinstance(params, torch.Tensor):
        params = [params]
    return [p for p in params if (p[1] if isinstance(p, tuple) else p).requires_grad]


def _scalar(v, what: str) -> float:
    if isinstance(v, torch.Tensor):
        if v.device.type != "cpu":
            raise ValueError(f"FusedAdam: {what} is a tensor on {v.device}; reading it would synchronise with the device every step "
                             "(use a Python float or a CPU tensor)")
        return float(v.item())
    return float(v)


def _group_hyper(group: Dict[str, Any]) -> Tuple:
    """(lr, beta1, beta2, eps, weight_decay, decoupled) of a parameter group, rejecting the options FusedAdam has no path for."""
    for name in _UNSUPPORTED:
        if group.get(name):
            raise ValueError(f"FusedAdam does not support {name}={group[name]!r} (use torch.optim.Adam for it)")
    b1, b2 = group["betas"]
    return (_scalar(group["lr"], "lr"), _scalar(b1, "beta1"), _scalar(b2, "beta2"), _scalar(group["eps"], "eps"),
            _scalar(group["weight_decay"], "weight_decay"), bool(group.get("decoupled_weight_decay", False)))


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam (coupled L2 weight decay) or, with `decoupled_weight_decay=True`, AdamW, over flat fp32 buffers.

    `params` is an iterable of parameters or of group dicts; every option can be set per group.  Parameters with
    `requires_grad=False` are left out, as at construction time.  `flat_param`, `flat_grad`, `exp_avg`, `exp_avg_sq` are the flat
    buffers and `numel` their length; `params` lists the parameters in flat order."""

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, *,
                 decoupled_weight_decay: bool = False, amsgrad: bool = False, maximize: bool = False, foreach: Optional[bool] = None,
                 capturable: bool = False, differentiable: bool = False, fused: Optional[bool] = None):
        if not 0.0 <= _scalar(lr, "lr"):
            raise ValueError(f"Invalid learning rate: {lr}")
        if not 0.0 <= eps:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not (0.0 <= _scalar(betas[0], "beta1") < 1.0 and 0.0 <= _scalar(betas[1], "beta2") < 1.0):
            raise ValueError(f"Invalid beta parameters: {betas}")
        if not 0.0 <= weight_decay:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad, maximize=maximize, foreach=foreach,
                        capturable=capturable, differentiable=differentiable, fused=fused, decoupled_weight_decay=decoupled_weight_decay)
        _group_hyper(defaults)
        if not isinstance(params, torch.Tensor):
            params = list(params)
            if params and isinstance(params[0], dict):
                params = [dict(g, params=_trainable(g["params"])) for g in params]
            else:
                params = [{"params": _trainable(params)}]
        self._built = False
        super().__init__(params, defaults)
        for g in self.param_groups:
            _group_hyper(g)
        order = [p for g in self.param_groups for p in g["params"]]
        if not order:
            raise ValueError("FusedAdam got no parameters")
        self._check_params(order, order[0].device)
        # data-parallel exchange of bf16-rounded gradients (half the bytes; see all_reduce_range_async); opt-in
        self.bf16_exchange = os.environ.get("HK_DP_BF16_GRADS", "0") == "1"
        self._bf16_buf = None
        self.params: List[torch.nn.Parameter] = []
        self._relayout(order, {})
        self._built = True

    @staticmethod
    def _check_params(params, dev) -> None:
        if dev.type != "cuda" or any(p.device != dev or p.dtype != torch.float32 for p in params):
            raise RuntimeError("FusedAdam needs fp32 CUDA parameters on one device (no CPU fallback)")

    # ------------------------------------------------------------------ flat layout
    def _param_steps(self) -> Dict[int, int]:
        steps = {}
        for r in self._runs:
            for p in self.params[r[4]:r[5]]:
                steps[id(p)] = r[3]
        return steps

    def _relayout(self, order: List[torch.nn.Parameter], steps: Dict[int, int], flat_grad: Optional[torch.Tensor] = None) -> None:
        """Lay `order` out in fresh flat buffers: parameters, moments and gradients of parameters already laid out are copied bit for
        bit, new ones start from their data with zero moments.  `flat_grad` (already in the new layout) replaces the gradient buffer.
        `steps` maps id(param) -> steps taken (absent = 0).  p.data / p.grad are re-pointed into the new buffers."""
        old = {id(p): o for p, o in zip(self.params, getattr(self, "_offs", []))}
        offs, total = flat_offsets([p.numel() for p in order])
        dev = order[0].device
        fp, fm, fv = (torch.zeros(total, device=dev, dtype=torch.float32) for _ in range(3))
        fg = flat_grad if flat_grad is not None else torch.zeros(total, device=dev, dtype=torch.float32)
        with torch.no_grad():
            for p, o in zip(order, offs):
                n = p.numel()
                oo = old.get(id(p))
                if oo is None:
                    fp[o:o + n].copy_(p.data.reshape(-1))
                else:
                    for dst, src in ((fp, self.flat_param), (fm, self.exp_avg), (fv, self.exp_avg_sq)) + \
                            (((fg, self.flat_grad),) if flat_grad is None else ()):
                        dst[o:o + n].copy_(src[oo:oo + n])
        self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq = fp, fg, fm, fv
        self.numel = total
        for p, o in zip(order, offs):
            p.data = fp[o:o + p.numel()].view_as(p.data)
            p.grad = fg[o:o + p.numel()].view_as(p.data)
        self.params, self._offs = order, offs
        self._rebuild_runs(steps)
        note_raw_parameter_write()   # new data pointers: eval engines refold, train engines recapture

    def _rebuild_runs(self, steps: Dict[int, int]) -> None:
        """Runs of consecutive parameters (flat order) in the same group with the same step count: [begin4, end4, group, step, i0, i1]."""
        group_of = {id(p): gi for gi, g in enumerate(self.param_groups) for p in g["params"]}
        runs: List[list] = []
        for i, (p, o) in enumerate(zip(self.params, self._offs)):
            gi, t = group_of[id(p)], steps.get(id(p), 0)
            e4 = (o + (p.numel() + 3) // 4 * 4) // 4
            if runs and runs[-1][2] == gi and runs[-1][3] == t:
                runs[-1][1], runs[-1][5] = e4, i + 1
            else:
                runs.append([o // 4, e4, gi, t, i, i + 1])
        self._runs = runs

    def add_param_group(self, param_group: Dict[str, Any]) -> None:
        """torch's add_param_group: the group's trainable parameters join with step 0.  The flat buffers are rebuilt (existing
        parameters, moments and steps copied bit for bit) and p.data / p.grad re-pointed into them."""
        if not self._built:   # torch.optim.Optimizer.__init__ adding the constructor's groups
            return super().add_param_group(param_group)
        group = dict(param_group, params=_trainable(param_group["params"]))
        super().add_param_group(group)
        new = list(self.param_groups[-1]["params"])
        try:
            _group_hyper(self.param_groups[-1])
            self._check_params(new, self.params[0].device)
        except Exception:
            self.param_groups.pop()
            raise
        self._relayout(self.params + new, self._param_steps())

    def adopt_grad_buffer(self, flat_grad: torch.Tensor, params: Optional[Sequence[torch.nn.Parameter]] = None) -> None:
        """Use an external flat gradient buffer (TrainEngine.flat_grad): the engine's kernels then write the gradients exactly where
        the all-reduce and the update read them -- no copy.  `params` is the buffer's parameter order (TrainEngine.params); it must
        be this optimiser's parameter set (checked by identity), and when its order differs the flat parameter and moment buffers
        are reordered to it once.  Without `params` the buffer is taken to be in this optimiser's order."""
        if params is not None:
            params = list(params)
            ids = {id(p) for p in params}
            if len(params) != len(self.params) or len(ids) != len(params) or any(id(p) not in ids for p in self.params):
                raise ValueError(_LAYOUT_MISMATCH)
        if flat_grad.shape != (self.numel,) or flat_grad.dtype != torch.float32 or flat_grad.device != self.flat_grad.device:
            raise ValueError(_LAYOUT_MISMATCH)
        if params is not None and any(a is not b for a, b in zip(params, self.params)):
            self._relayout(params, self._param_steps(), flat_grad=flat_grad)
            return
        self.flat_grad = flat_grad
        for p, o in zip(self.params, self._offs):
            p.grad = flat_grad[o:o + p.numel()].view_as(p.data)

    def zero_grad(self, set_to_none: bool = True) -> None:
        """Zeroes the flat gradient buffer whatever `set_to_none` says: the .grad views stay attached to it (setting them to None
        would detach the parameters from the buffer the engine, the all-reduce and the update share)."""
        self.flat_grad.zero_()

    # ------------------------------------------------------------------ torch's Adam state format
    def state_dict(self) -> Dict[str, Any]:
        """torch.optim.Adam's format: param_groups with every option and parameter indices; state {index: {"step" (fp32 0-dim CPU
        tensor), "exp_avg", "exp_avg_sq"}} for the parameters that have stepped.  The moments are copies."""
        steps = self._param_steps()
        pos = {id(p): o for p, o in zip(self.params, self._offs)}
        groups, state, idx = [], {}, 0
        for g in self.param_groups:
            packed = {k: v for k, v in g.items() if k != "params"}
            packed["params"] = list(range(idx, idx + len(g["params"])))
            for i, p in zip(packed["params"], g["params"]):
                t = steps[id(p)]
                if t > 0:
                    o, n = pos[id(p)], p.numel()
                    state[i] = {"step": torch.tensor(float(t), dtype=torch.float32),
                                "exp_avg": self.exp_avg[o:o + n].view_as(p).clone(),
                                "exp_avg_sq": self.exp_avg_sq[o:o + n].view_as(p).clone()}
            idx += len(g["params"])
            groups.append(packed)
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, state_dict: Dict[str, Any]) -> None:
        """torch's load_state_dict (group count and sizes validated, hyperparameters taken from the saved groups); the moments are
        copied into the flat buffers at the current layout and the steps restored.  amsgrad / maximize state is rejected."""
        for g in state_dict["param_groups"]:
            _group_hyper(g)
        saved_ids = [i for g in state_dict["param_groups"] for i in g["params"]]
        for i, p in zip(saved_ids, [p for g in self.param_groups for p in g["params"]]):
            s = state_dict["state"].get(i)
            if not s:
                continue
            if "max_exp_avg_sq" in s:
                raise ValueError("FusedAdam does not support amsgrad state (max_exp_avg_sq)")
            if s["exp_avg"].numel() != p.numel() or s["exp_avg_sq"].numel() != p.numel():
                raise ValueError(f"loaded Adam state has moments of {s['exp_avg'].numel()} / {s['exp_avg_sq'].numel()} elements for a "
                                 f"parameter of {p.numel()}")
        super().load_state_dict(state_dict)
        # the base class left standalone moment tensors in self.state: move them into the flat buffers
        steps = {}
        with torch.no_grad():
            for p, o in zip(self.params, self._offs):
                n = p.numel()
                st = self.state.get(p)
                if not st:
                    self.exp_avg[o:o + n].zero_()
                    self.exp_avg_sq[o:o + n].zero_()
                    continue
                self.exp_avg[o:o + n].copy_(st["exp_avg"].reshape(-1))
                self.exp_avg_sq[o:o + n].copy_(st["exp_avg_sq"].reshape(-1))
                steps[id(p)] = int(_scalar(st["step"], "step"))
        self.state.clear()
        self._rebuild_runs(steps)

    # ------------------------------------------------------------------ data-parallel exchange
    @staticmethod
    def _avg_op():
        """NCCL averages inside the collective (ReduceOp.AVG: every contribution is pre-multiplied by 1/world, exact for the 2/4/8 ranks of
        one box), which saves the separate 1/world pass over the 87 MB buffer; other backends (gloo in the CPU tests) sum and divide."""
        import torch.distributed as dist
        return dist.ReduceOp.AVG if dist.get_backend() == "nccl" else None

    def all_reduce_grads(self) -> None:
        """Data-parallel exchange: ONE averaging all-reduce over the flat gradient buffer."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            avg = self._avg_op()
            if avg is not None:
                dist.all_reduce(self.flat_grad, op=avg)
            else:
                dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)
                self.flat_grad.div_(dist.get_world_size())

    def all_reduce_range_async(self, begin: int, end: int):
        """Start the averaging all-reduce of flat_grad[begin:end] on the collective's stream (it waits for the work already enqueued on the
        current stream); returns (work, begin, end, averaged), or None outside a multi-rank job.  finish_all_reduce() waits (and divides
        where the backend could only sum)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1 or end <= begin:
            return None
        avg = self._avg_op()
        if self.bf16_exchange and avg is not None:
            # opt-in (HK_DP_BF16_GRADS=1): the range travels as bf16 (half the bytes of the exchange); every rank rounds its fp32 gradients
            # once, NCCL averages in bf16, finish_all_reduce() widens the result back into the fp32 buffer Adam reads (fp32 master
            # statistics and parameters are untouched).  Not bit-identical to the fp32 exchange -- off by default.
            if self._bf16_buf is None or self._bf16_buf.numel() != self.numel:
                self._bf16_buf = torch.empty(self.numel, device=self.flat_grad.device, dtype=torch.bfloat16)
            half = self._bf16_buf[begin:end]
            half.copy_(self.flat_grad[begin:end])
            work = dist.all_reduce(half, op=avg, async_op=True)
            return (work, begin, end, "bf16")
        work = dist.all_reduce(self.flat_grad[begin:end], op=avg if avg is not None else dist.ReduceOp.SUM, async_op=True)
        return (work, begin, end, avg is not None)

    def finish_all_reduce(self, works) -> None:
        """The current stream waits for the given exchanges; ranges a backend could only sum are divided by the world size."""
        import torch.distributed as dist
        for w in works:
            if w is None:
                continue
            work, begin, end, averaged = w
            work.wait()
            if averaged == "bf16":
                self.flat_grad[begin:end].copy_(self._bf16_buf[begin:end])
            elif not averaged:
                self.flat_grad[begin:end].div_(dist.get_world_size())

    # ------------------------------------------------------------------ the update
    @torch.no_grad()
    def step(self, closure=None):
        """One Adam step of every parameter with its group's current hyperparameters: one hk_adam_step_segments launch."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        hypers = [_group_hyper(g) for g in self.param_groups]
        rows = build_segments(((r[0], r[1], r[2], r[3] + 1) for r in self._runs), hypers)
        table = (HkAdamSegment * len(rows))(*(HkAdamSegment(*r) for r in rows))
        check(lib().hk_adam_step_segments(ptr(self.flat_param), ptr(self.flat_grad), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                          C.c_longlong(self.numel), table, len(rows), stream_ptr()), "hk_adam_step_segments")
        for r in self._runs:
            r[3] += 1
        note_raw_parameter_write()   # raw-pointer write: tensor versions do not move, eval engines must refold their weights
        return loss
