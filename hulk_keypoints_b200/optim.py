"""FusedAdam: torch.optim.Adam(lr, weight_decay) semantics (reference train.py:79) as ONE kernel per step.

Parameters and gradients are flattened into two contiguous fp32 buffers at construction (each `param.data` / `param.grad`
becomes a view into them), so autograd accumulates straight into the flat gradient buffer, a data-parallel all-reduce is
a single collective over it, and the update is one pass of `hk_adam_step`.  All 21,797,672 parameters are updated,
including the 996 dead fc rows, which receive zero gradient but are still decayed -- as in the reference.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Iterable

import torch

from ._lib import check, lib, note_raw_parameter_write, ptr, stream_ptr


class FusedAdam:
    def __init__(self, params: Iterable[torch.nn.Parameter], lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("FusedAdam got no parameters")
        dev = self.params[0].device
        if dev.type != "cuda" or any(p.device != dev or p.dtype != torch.float32 for p in self.params):
            raise RuntimeError("FusedAdam needs fp32 CUDA parameters on one device (no CPU fallback)")
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
        self.step_count = 0
        # data-parallel exchange of bf16-rounded gradients (half the bytes; see all_reduce_range_async); opt-in
        self.bf16_exchange = os.environ.get("HK_DP_BF16_GRADS", "0") == "1"
        self._bf16_buf = None
        # every tensor starts on a 16-byte boundary inside the flat buffers
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4
        self.numel = total
        self.flat_param = torch.zeros(total, device=dev, dtype=torch.float32)
        self.flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(total, device=dev, dtype=torch.float32)
        with torch.no_grad():
            for p, o in zip(self.params, offs):
                n = p.numel()
                self.flat_param[o:o + n].copy_(p.data.reshape(-1))
                p.data = self.flat_param[o:o + n].view_as(p.data)
                p.grad = self.flat_grad[o:o + n].view_as(p.data)

    def adopt_grad_buffer(self, flat_grad: torch.Tensor) -> None:
        """Use an external flat gradient buffer with this optimiser's layout (TrainEngine.flat_grad): the engine's kernels then write
        the gradients exactly where the all-reduce and hk_adam_step read them -- no copy."""
        if flat_grad.shape != self.flat_grad.shape or flat_grad.dtype != torch.float32 or flat_grad.device != self.flat_grad.device:
            raise ValueError("gradient buffer layout mismatch (the optimiser was built for another set of trainable parameters: "
                             "build it after setting requires_grad, as in torch)")
        self.flat_grad = flat_grad
        o = 0
        for p in self.params:
            n = p.numel()
            p.grad = flat_grad[o:o + n].view_as(p.data)
            o += (n + 3) // 4 * 4

    def zero_grad(self, set_to_none: bool = False) -> None:
        """Keeps the gradient views alive (set_to_none would detach them from the flat buffer)."""
        self.flat_grad.zero_()

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

    @torch.no_grad()
    def step(self) -> None:
        self.step_count += 1
        check(lib().hk_adam_step(ptr(self.flat_param), ptr(self.flat_grad), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                 C.c_longlong(self.numel), C.c_float(self.lr), C.c_float(self.betas[0]), C.c_float(self.betas[1]),
                                 C.c_float(self.eps), C.c_float(self.weight_decay), self.step_count, stream_ptr()), "hk_adam_step")
        note_raw_parameter_write()   # raw-pointer write: tensor versions do not move, eval engines must refold their weights
