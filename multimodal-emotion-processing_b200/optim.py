"""Fused gradient clipping + Adam / AdamW (SURVEY.md §8f-1): the step right after the hot path in
every reference training loop,

    nn.utils.clip_grad_norm_(model.parameters(), CLIP)     # others/realformer.py:314 etc.
    optimizer.step()                                        # optim.Adam :342 / optim.AdamW

``Adam`` / ``AdamW`` keep torch.optim's constructor arguments, ``param_groups`` (so
``ReduceLROnPlateau`` keeps working, others/realformer.py:343) and ``state_dict`` layout
(``step``, ``exp_avg``, ``exp_avg_sq``), and run the whole update as one libmmemo launch per 96
tensors.  ``step_group`` steps several of them (the k folds of a cross-validation) in the same
launches; ``step()`` is ``step_group`` of one optimizer.  Two ways to clip:

* drop-in: keep the reference's two calls, with ``clip_grad_norm_`` from this module (two launches:
  squared norm, scale; returns the total norm like torch's);
* fused: ``AdamW(..., max_grad_norm=CLIP)`` and no separate clip call — the coefficient is computed
  on the device from the squared norm and applied while the update reads the gradients (no extra
  pass over them, no host sync).

float32 CUDA parameters only (the master parameters of both precision modes are float32); there is
no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, List, Optional

import torch
from torch import Tensor

from . import ops

def _ptrs(ts: List[Tensor]):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _ns(ts: List[Tensor]):
    return (C.c_int64 * len(ts))(*[t.numel() for t in ts])


def _check(ts: Iterable[Tensor], what: str) -> None:
    for t in ts:
        if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise RuntimeError(f"mmemo_b200.optim needs contiguous float32 CUDA {what} "
                               "(no CPU fallback)")


def _arr(ctype, vals):
    return (ctype * len(vals))(*vals)


def grad_sqnorm(grads: List[Tensor]) -> Tensor:
    """Device scalar  sum_i |g_i|^2  in one launch (per 96 tensors)."""
    _check(grads, "gradients")
    out = torch.zeros(1, dtype=torch.float32, device=grads[0].device)
    ops._call("mmemo_grad_sqnorm_multi_f32", len(grads), _ptrs(grads), _ns(grads),
              _arr(C.c_int, [0] * len(grads)), out.data_ptr(), ops._stream())
    return out


def clip_grad_norm_(parameters, max_norm: float) -> Tensor:
    """Fused ``torch.nn.utils.clip_grad_norm_(parameters, max_norm)`` (L2 norm): scales the
    gradients in place by ``min(1, max_norm / (norm + 1e-6))`` and returns the total norm as a
    0-dim device tensor.  No host synchronisation."""
    if isinstance(parameters, Tensor):
        parameters = [parameters]
    grads = [p.grad for p in parameters if p.grad is not None]
    if not grads:
        return torch.zeros(())
    sq = grad_sqnorm(grads)
    ops._call("mmemo_clip_grads_f32", len(grads), _ptrs(grads), _ns(grads), sq.data_ptr(),
              float(max_norm), ops._stream())
    return sq.sqrt().reshape(())


class _FusedAdam(torch.optim.Optimizer):
    _decoupled = False

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, amsgrad: bool = False,
                 max_grad_norm: Optional[float] = None):
        if amsgrad:
            raise ValueError("amsgrad is not used by the reference and not implemented")
        if lr < 0 or eps < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameter")
        if max_grad_norm is not None and max_grad_norm <= 0:
            raise ValueError("max_grad_norm must be positive")
        self.max_grad_norm = max_grad_norm
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay,
                                      amsgrad=False))

    def _collect(self):
        """[(param_group, params with a gradient, their gradients)], state initialised."""
        groups = []
        for group in self.param_groups:
            ps = [p for p in group["params"] if p.grad is not None]
            if not ps:
                continue       # e.g. the empty second group of Ren-MME/run.py:376-379
            _check(ps, "parameters")
            gs = [p.grad for p in ps]
            _check(gs, "gradients")
            for p in ps:
                st = self.state[p]
                if not st:
                    st["step"] = torch.tensor(0.0)          # torch.optim keeps a CPU float tensor
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            groups.append((group, ps, gs))
        return groups

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        step_group([self])
        return loss


class Adam(_FusedAdam):
    """``torch.optim.Adam`` (L2 weight decay folded into the gradient); others/realformer.py:342."""
    _decoupled = False


class AdamW(_FusedAdam):
    """``torch.optim.AdamW`` (decoupled weight decay, default 1e-2); cmu-mosei/run.py:398,
    Ren-MME/run.py:379, rencecps/run.py:202, robot_demo.py:502."""
    _decoupled = True

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-2, amsgrad: bool = False,
                 max_grad_norm: Optional[float] = None):
        super().__init__(params, lr, betas, eps, weight_decay, amsgrad, max_grad_norm)


@torch.no_grad()
def step_group(optimizers) -> None:
    """``for opt in optimizers: opt.step()`` for one or several ``Adam`` / ``AdamW`` instances (the
    k folds of a cross-validation, one model each) in one launch per 96 tensors, whatever their
    number.  ``step()`` itself is ``step_group([self])``.

    Each optimizer keeps its own ``param_groups``, ``state`` and ``state_dict`` and ends up exactly
    as if it had been stepped alone: its own lr (e.g. set by its own ``ReduceLROnPlateau``), weight
    decay and per-tensor step counts (a parameter that starts receiving gradients later has its own
    bias corrections), and with ``max_grad_norm`` its gradients clipped by the norm over all of its
    param groups (one squared norm per optimizer, computed first).  That is one library call for the
    norms and one update call per combination of class, ``betas``, ``eps`` and ``max_grad_norm``."""
    opts = list(optimizers)
    for o in opts:
        if not isinstance(o, _FusedAdam):
            raise TypeError(f"step_group takes mmemo_b200.optim.Adam / AdamW, not {type(o).__name__}")
    collected = [o._collect() for o in opts]
    sq = None
    norm_g, norm_slot = [], []
    for k, (o, groups) in enumerate(zip(opts, collected)):
        if o.max_grad_norm is not None:
            for _, _, gs in groups:
                norm_g += gs
                norm_slot += [k] * len(gs)
    if norm_g:
        sq = torch.zeros(len(opts), dtype=torch.float32, device=norm_g[0].device)
        ops._call("mmemo_grad_sqnorm_multi_f32", len(norm_g), _ptrs(norm_g), _ns(norm_g),
                  _arr(C.c_int, norm_slot), sq.data_ptr(), ops._stream())
    # [(param, grad, optimizer index, param_group)] per combination of the shared hyper-parameters
    calls = {}
    for k, (o, groups) in enumerate(zip(opts, collected)):
        for group, ps, gs in groups:
            key = (o._decoupled, tuple(group["betas"]), float(group["eps"]), o.max_grad_norm)
            calls.setdefault(key, []).extend((p, g, k, group) for p, g in zip(ps, gs))
    for (decoupled, (b1, b2), eps, max_norm), items in calls.items():
        pp = [it[0] for it in items]
        st = [opts[it[2]].state[it[0]] for it in items]
        ops._call("mmemo_adam_step_multi_f32", len(items), _ptrs(pp), _ptrs([it[1] for it in items]),
                  _ptrs([s["exp_avg"] for s in st]), _ptrs([s["exp_avg_sq"] for s in st]),
                  _ns(pp), _arr(C.c_float, [float(it[3]["lr"]) for it in items]),
                  _arr(C.c_int64, [int(s["step"]) + 1 for s in st]),
                  _arr(C.c_float, [float(it[3]["weight_decay"]) for it in items]),
                  _arr(C.c_int, [it[2] for it in items]), float(b1), float(b2), eps,
                  int(decoupled), None if sq is None or max_norm is None else sq.data_ptr(),
                  float(max_norm or 0.0), ops._stream())
        for s in st:
            s["step"] += 1
        # the launch wrote the parameters through raw pointers: bump their version counters so
        # that everything keyed on them (the bf16 weight shadows of ops.shadow_bf16, autograd's
        # saved-tensor checks) sees the update like after an in-place torch op
        torch._C._increment_version(pp)

