"""torch custom ops over the C ABI of libmmemo.so (include/mmemo.h).

Every op allocates its outputs with torch (device memory + stream plumbing only), passes raw
device pointers + the current CUDA stream to an ``extern "C"`` launcher, and registers an explicit
backward (``torch.library.register_autograd``) that calls the matching ``*_bwd`` launchers, so the
reference training loops (``loss.backward()``, ``clip_grad_norm_``, ``optimizer.step()``) work
unchanged.  No op has a CPU implementation: calling one without a CUDA tensor or without the
built library raises.

Precision: activations are float32 (parity mode) or bfloat16 (``bf16=True``).  Parameters stay
float32 ("master"); in bf16 mode GEMM weights are used through bf16 shadow copies refreshed when
the parameter's version counter changes; all parameter gradients are returned in float32.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib

BF = torch.bfloat16
F32 = torch.float32
LN_EPS = 1e-5

# number of libmmemo kernel launches issued through this module (bench.py's gpu_launches)
launch_count = 0


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# Launch settings live with the STREAM in libmmemo (mmemo_stream_set_*): the first launch on a
# stream attaches a split-K scratch buffer of its own (launches of one stream are ordered and can
# share it; two streams never do), so concurrent streams - the ensemble's side streams, a capture
# stream next to the default stream - are independent.  The buffers live as long as the process:
# a captured CUDA graph keeps the pointer of the stream it was captured on.
_stream_ws: dict = {}
WORKSPACE_BYTES = 32 << 20
_PDL_OFF = os.environ.get("MMEMO_PDL", "1") == "0"     # debugging knob: fully serialised launches


def _ensure_stream(stream: int) -> None:
    key = (torch.cuda.current_device(), stream)
    if key in _stream_ws:
        return
    lib = _lib.load()
    buf = torch.empty(WORKSPACE_BYTES, dtype=torch.uint8, device=f"cuda:{key[0]}")
    _lib.check(lib.mmemo_stream_set_workspace(stream, buf.data_ptr(), buf.numel()), "stream_set_workspace")
    if _PDL_OFF:
        _lib.check(lib.mmemo_stream_set_pdl(stream, 0), "stream_set_pdl")
    _stream_ws[key] = buf


# Data-parallel overlap: while a bucket all-reduce is in flight its CTAs hold some SMs; a
# persistent (one CTA per SM) GEMM launched meanwhile would have that many CTAs serialised behind
# the others (measured: 12.9 -> 23.4 us per GEMM).  dp.GradReducer therefore lowers the SM budget of
# the next few GEMM launches of the compute stream after it issues an all-reduce; the countdown
# restores the full budget.
_budget_countdown = 0
_budget_stream = 0


def reserve_sms_for(n_launches: int, n_sms_reserved: int) -> None:
    global _budget_countdown, _budget_stream
    total = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    release_sms()
    _budget_stream = _stream()
    _lib.check(_lib.load().mmemo_stream_set_sm_budget(
        _budget_stream, max(2, (total - n_sms_reserved) // 2 * 2)), "sm_budget")
    _budget_countdown = n_launches


def release_sms() -> None:
    global _budget_countdown
    if _budget_countdown:
        _budget_countdown = 0
        _lib.check(_lib.load().mmemo_stream_set_sm_budget(_budget_stream, 0), "sm_budget")


def _call(name: str, *args) -> None:
    global launch_count, _budget_countdown
    _ensure_stream(_stream())
    launch_count += 1
    _lib.check(getattr(_lib.load(), name)(*args), name)
    if _budget_countdown and name.startswith("mmemo_linear"):
        _budget_countdown -= 1
        if _budget_countdown == 0:
            _lib.check(_lib.load().mmemo_stream_set_sm_budget(_budget_stream, 0), "sm_budget")


def _try_call(name: str, *args) -> bool:
    """Like ``_call`` for the grouped entry points: False when the library answers
    MMEMO_ERR_SHAPE (a problem of the group is outside the grouped kernel's limits; the caller then
    issues the problems one by one), raises on any other error."""
    global launch_count
    _ensure_stream(_stream())
    rc = getattr(_lib.load(), name)(*args)
    if rc == -2:
        return False
    _lib.check(rc, name)
    launch_count += 1
    return True


def _sfx(bf16: bool) -> str:
    return "bf16" if bf16 else "f32"


def _act_dtype(bf16: bool):
    return BF if bf16 else F32


def _need_cuda(*ts: Optional[Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("mmemo_b200 ops run on CUDA tensors only (no CPU fallback)")


# ------------------------------------------------------------------------------------------------
# bf16 shadow copies of float32 master weights
# ------------------------------------------------------------------------------------------------
_shadow: dict = {}
_shadow_pad: dict = {}     # zero-padded (N, K rounded up to 8) shadows of the projection weights


def clear_shadow_cache() -> None:
    """Drop all bf16 weight shadows (call before CUDA-graph capture so the casts are captured)."""
    _shadow.clear()
    _shadow_pad.clear()


def shadow_bf16(*ws: Tensor) -> Tensor:
    """bf16 copy of one weight, or of several weights concatenated along dim 0 (e.g. [Wk; Wv])."""
    key = tuple((w.data_ptr(), w._version, tuple(w.shape)) for w in ws)
    hit = _shadow.get(key)
    if hit is not None:
        return hit
    # evict stale entries of the same storage(s)
    ptrs = {k[0] for k in key}
    for k in [k for k in _shadow if any(e[0] in ptrs for e in k) and len(k) == len(key)]:
        del _shadow[k]
    rows = sum(w.shape[0] for w in ws)
    cols = ws[0].numel() // ws[0].shape[0]
    out = torch.empty(rows, cols, dtype=BF, device=ws[0].device)
    r = 0
    for w in ws:
        wd = w.detach()
        if not wd.is_contiguous():
            wd = wd.contiguous()
        _call("mmemo_cast_f32_to_bf16", wd.data_ptr(), out[r:].data_ptr(), wd.numel(), _stream())
        r += w.shape[0]
    _shadow[key] = out
    return out


def shadow_bf16_block(groups: Sequence[Sequence[Tensor]]) -> List[Tensor]:
    """bf16 shadows of several weight groups (each group = weights concatenated along dim 0) with
    ONE cast call (one launch per 64 tensors); also fills the per-group cache used by
    ``shadow_bf16``."""
    keys = [tuple((w.data_ptr(), w._version, tuple(w.shape)) for w in g) for g in groups]
    if all(k in _shadow for k in keys):
        return [_shadow[k] for k in keys]
    outs, srcs, dsts, ns = [], [], [], []
    for g, k in zip(groups, keys):
        ptrs = {e[0] for e in k}
        for old in [o for o in _shadow if any(e[0] in ptrs for e in o) and len(o) == len(k)]:
            del _shadow[old]
        rows = sum(w.shape[0] for w in g)
        out = torch.empty(rows, g[0].numel() // g[0].shape[0], dtype=BF, device=g[0].device)
        r = 0
        for w in g:
            wd = w.detach()
            wd = wd if wd.is_contiguous() else wd.contiguous()
            srcs.append(wd)
            dsts.append(out[r:].data_ptr())
            ns.append(wd.numel())
            r += w.shape[0]
        _shadow[k] = out
        outs.append(out)
    _call("mmemo_cast_f32_to_bf16_multi", len(srcs), _arr(C.c_void_p, [t.data_ptr() for t in srcs]),
          _arr(C.c_void_p, dsts), _arr(C.c_int64, ns), _stream())
    return outs


def _weight(bf16: bool, *ws: Tensor) -> Tensor:
    if bf16:
        return shadow_bf16(*ws)
    if len(ws) == 1:
        w = ws[0].detach()
        w = w.reshape(w.shape[0], -1)
        return w if w.is_contiguous() else w.contiguous()
    return torch.cat([w.detach().reshape(w.shape[0], -1) for w in ws], 0)


def _rows(x: Tensor) -> Tuple[Tensor, int, int]:
    """View (..., K) as (M, K) with unit inner stride; returns (tensor, M, ld)."""
    K = x.shape[-1]
    if x.dim() == 2 and x.stride(1) == 1:
        return x, x.shape[0], x.stride(0)
    if not x.is_contiguous():
        x = x.contiguous()
    return x, x.numel() // K, K


# ------------------------------------------------------------------------------------------------
# gradient regions: the backward of a fused block layer (group_ops) accumulates ALL parameter
# gradients of a block (weight gradients + the small "+=" outputs) into one zero-filled buffer
# ("zbuf", layout: group_ops.full_grad_unit / lite_grad_unit).  Under data parallelism the reducer
# (dp.GradReducer) gives every block a contiguous bucket region with that layout and registers it
# here, keyed by the block's first weight: the block's zbuf IS then a bucket slice, p.grad of all
# its parameters are views of the bucket, and nothing is copied or filled per block.  Only valid
# while p.grad is None at backward time (zero_grad(set_to_none=True)); the reducer disables it
# otherwise.
# ------------------------------------------------------------------------------------------------
_zbuf_dest: dict = {}
grad_dest_enabled = True
# set by dp.GradReducer.backward(): the bucket regions were zero-filled before this backward
grad_dest_zeroed = False


# A region can be WRITTEN by one op per backward: a block that is used twice (shared weights) gets
# a fresh buffer for its second gradient and autograd sums the two as usual.
_dest_claimed: set = set()


def register_zbuf_dest(key: Tensor, flat: Tensor, offset: int, total: int) -> None:
    _zbuf_dest[key.data_ptr()] = (flat, offset, total)


def begin_backward() -> None:
    """Called by dp.GradReducer.backward(): every region is writable again."""
    _dest_claimed.clear()


def clear_grad_dest() -> None:
    _zbuf_dest.clear()


def unregister_zbuf_dests(flats: Sequence[Tensor]) -> None:
    """Forget every region that lives in one of ``flats`` (a reducer that goes away must not
    leave entries keyed by parameter addresses a later model could reuse)."""
    ids = {id(f) for f in flats}
    for k in [k for k, v in _zbuf_dest.items() if id(v[0]) in ids]:
        del _zbuf_dest[k]


def claim_zbufs(keys: Sequence[Tensor], total: int) -> Optional[List[Tensor]]:
    """Bucket regions for the zero buffers of a GROUP of blocks (one grouped trunk layer): all of
    them or none (None: the caller allocates and fills its own buffer)."""
    if not (grad_dest_enabled and grad_dest_zeroed):
        return None
    zs = [_zbuf_dest.get(k.data_ptr()) for k in keys]
    if any(z is None or z[2] != total for z in zs):
        return None
    if any(k.data_ptr() in _dest_claimed for k in keys):
        return None
    _dest_claimed.update(k.data_ptr() for k in keys)
    return [z[0][z[1]:z[1] + z[2]] for z in zs]


def zbuf_region(key: Tensor) -> Tensor:
    z = _zbuf_dest[key.data_ptr()]
    return z[0][z[1]:z[1] + z[2]]


# ------------------------------------------------------------------------------------------------
# raw launch helpers (no autograd) -- shared by the fine-grained ops and the grouped ops
# ------------------------------------------------------------------------------------------------
def _linear_fwd(bf16, x, w, bias, pos, out, relu=False, accumulate=False, ldw=None, N=None, K=None):
    x, M, ldx = _rows(x)
    N = w.shape[0] if N is None else N
    K = x.shape[-1] if K is None else K
    ldw = w.stride(0) if ldw is None else ldw
    _call(f"mmemo_linear_fwd_{_sfx(bf16)}", x.data_ptr(), int(x.dtype == F32), ldx, w.data_ptr(),
          ldw, _p(bias), _p(pos), 0 if pos is None else pos.shape[0], out.data_ptr(),
          out.stride(-2), M, N, K, int(relu), int(accumulate), _stream())


def _linear_bwd_x(bf16, dy, w, dx, relu_src=None, accumulate=False, ldw=None, N=None, K=None):
    dy, M, lddy = _rows(dy)
    N = w.shape[0] if N is None else N
    K = w.shape[1] if K is None else K
    ldw = w.stride(0) if ldw is None else ldw
    _call(f"mmemo_linear_bwd_x_{_sfx(bf16)}", dy.data_ptr(), lddy, w.data_ptr(), ldw,
          dx.data_ptr(), dx.stride(-2), _p(relu_src),
          0 if relu_src is None else relu_src.stride(-2), M, N, K, int(accumulate), _stream())


def _linear_bwd_w(bf16, dy, x, dw, dbias=None, accumulate=False, N=None, K=None):
    dy, M, lddy = _rows(dy)
    x, _, ldx = _rows(x)
    N = dy.shape[-1] if N is None else N
    K = x.shape[-1] if K is None else K
    _call(f"mmemo_linear_bwd_w_{_sfx(bf16)}", dy.data_ptr(), lddy, x.data_ptr(),
          int(x.dtype == F32), ldx, dw.data_ptr(), dw.stride(0), _p(dbias), M, N, K,
          int(accumulate), _stream())


def _arr(ctype, vals):
    return (ctype * len(vals))(*vals)


MAX_GEMM_GROUP = 48     # problems per grouped tensor-core launch (csrc/gemm.h GEMM_TC_MAX_GROUP)


def _chunks(items, n=MAX_GEMM_GROUP):
    return [items[i:i + n] for i in range(0, len(items), n)]


def _linear_fwd_group(bf16, items):
    """items: [(x, w, bias, out2d, relu[, accumulate[, pos]])].  One grouped tensor-core launch (per
    48 problems) in bf16 mode; N, K and the weight's leading dimension come from ``w`` (a 2-D view,
    e.g. one half of a concat weight); ``pos`` = (L, N) position table added with period L (may be a
    column slice of a wider table: its row stride is passed along)."""
    items = [tuple(it) + (False, None)[len(it) - 5:] for it in items]
    if not bf16 or len(items) == 1:
        for x, w, b, out, relu, acc, pos in items:
            assert pos is None or pos.is_contiguous(), "a sliced position table needs the grouped path"
            _linear_fwd(bf16, x, w, b, pos, out, relu=relu, accumulate=acc, ldw=w.stride(0),
                        N=w.shape[0], K=w.shape[1])
        return
    for part in _chunks(items):
        xs = [_rows(it[0]) for it in part]
        _call("mmemo_linear_fwd_grouped_bf16", len(part),
              _arr(C.c_void_p, [x.data_ptr() for x, _, _ in xs]), _arr(C.c_int64, [ld for _, _, ld in xs]),
              _arr(C.c_void_p, [it[1].data_ptr() for it in part]),
              _arr(C.c_int64, [it[1].stride(0) for it in part]),
              _arr(C.c_void_p, [_p(it[2]) for it in part]),
              _arr(C.c_void_p, [it[3].data_ptr() for it in part]),
              _arr(C.c_int64, [it[3].stride(-2) for it in part]),
              _arr(C.c_int64, [M for _, M, _ in xs]), _arr(C.c_int64, [it[1].shape[0] for it in part]),
              _arr(C.c_int64, [it[1].shape[1] for it in part]),
              _arr(C.c_int, [int(it[4]) for it in part]), _arr(C.c_int, [int(it[5]) for it in part]),
              _arr(C.c_void_p, [_p(it[6]) for it in part]),
              _arr(C.c_int64, [0 if it[6] is None else it[6].shape[0] for it in part]),
              _arr(C.c_int64, [0 if it[6] is None else it[6].stride(0) for it in part]), _stream())


def _linear_bwd_x_group(bf16, items):
    """items: [(dy, w, dx2d, accumulate[, relu_src2d])] — outputs must not alias each other."""
    items = [it if len(it) == 5 else (*it, None) for it in items]
    if not bf16 or len(items) == 1:
        for dy, w, dx, acc, rs in items:
            _linear_bwd_x(bf16, dy, w, dx, relu_src=rs, accumulate=acc, ldw=w.stride(0),
                          N=w.shape[0], K=w.shape[1])
        return
    for part in _chunks(items):
        dys = [_rows(it[0]) for it in part]
        _call("mmemo_linear_bwd_x_grouped_bf16", len(part),
              _arr(C.c_void_p, [d.data_ptr() for d, _, _ in dys]), _arr(C.c_int64, [ld for _, _, ld in dys]),
              _arr(C.c_void_p, [it[1].data_ptr() for it in part]),
              _arr(C.c_int64, [it[1].stride(0) for it in part]),
              _arr(C.c_void_p, [it[2].data_ptr() for it in part]),
              _arr(C.c_int64, [it[2].stride(-2) for it in part]),
              _arr(C.c_void_p, [_p(it[4]) for it in part]),
              _arr(C.c_int64, [0 if it[4] is None else it[4].stride(-2) for it in part]),
              _arr(C.c_int64, [M for _, M, _ in dys]), _arr(C.c_int64, [it[1].shape[0] for it in part]),
              _arr(C.c_int64, [it[1].shape[1] for it in part]),
              _arr(C.c_int, [int(it[3]) for it in part]), _stream())


def _linear_bwd_w_group(bf16, items, zeroed=False):
    """items: [(dy, x, dw)] -> dw = dy^T x (float32), all in one grouped launch (per 48 problems) in
    bf16 mode.  ``zeroed``: every dw is already all zero (saves the split-K path its own fills)."""
    if not bf16 or len(items) == 1:
        for dy, x, dw in items:
            _linear_bwd_w(bf16, dy, x, dw)
        return
    for part in _chunks(items):
        dys = [_rows(it[0]) for it in part]
        xs = [_rows(it[1]) for it in part]
        _call("mmemo_linear_bwd_w_grouped_bf16", len(part),
              _arr(C.c_void_p, [d.data_ptr() for d, _, _ in dys]), _arr(C.c_int64, [ld for _, _, ld in dys]),
              _arr(C.c_void_p, [x.data_ptr() for x, _, _ in xs]), _arr(C.c_int64, [ld for _, _, ld in xs]),
              _arr(C.c_void_p, [it[2].data_ptr() for it in part]),
              _arr(C.c_int64, [it[2].stride(0) for it in part]),
              _arr(C.c_int64, [M for _, M, _ in dys]), _arr(C.c_int64, [d.shape[-1] for d, _, _ in dys]),
              _arr(C.c_int64, [x.shape[-1] for x, _, _ in xs]), 2 if zeroed else 0, _stream())


def _add_ln_fwd(bf16, res, x, gate, gamma, beta, relu=False):
    x2, M, ldx = _rows(x)
    d = x.shape[-1]
    if res is not None:
        res, _, ldres = _rows(res)
    else:
        ldres = 0
    y = torch.empty(x.shape, dtype=x.dtype, device=x.device)
    stat = torch.empty(2, M, dtype=F32, device=x.device)
    _call(f"mmemo_add_ln_fwd_{_sfx(bf16)}", _p(res), ldres, x2.data_ptr(), ldx, _p(gate),
          gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), d, stat[0].data_ptr(),
          stat[1].data_ptr(), M, d, LN_EPS, int(relu), _stream())
    return y, stat


def _add_ln_bwd(bf16, dy, res, x, gate, gamma, y, stat, relu, want_dres, dres_out=None, dpar=None,
                dxsum=None):
    """Returns (dres, dx, dparams) with dparams = float32 [1 + 2d] = (dgate | dgamma | dbeta);
    ``dxsum`` (float32 [d], zero-initialised by the caller) receives the column sums of dx."""
    dy, M, lddy = _rows(dy)
    x2, _, ldx = _rows(x)
    d = x.shape[-1]
    ldres = 0
    if res is not None:
        res, _, ldres = _rows(res)
    dx = torch.empty(x.shape, dtype=x.dtype, device=x.device)
    dres = None
    if want_dres:
        dres = dres_out if dres_out is not None else torch.empty(x.shape, dtype=x.dtype,
                                                                 device=x.device)
    if dpar is None:
        dpar = torch.zeros(1 + 2 * d, dtype=F32, device=x.device)
    _call(f"mmemo_add_ln_bwd_{_sfx(bf16)}", dy.data_ptr(), lddy, _p(res), ldres, x2.data_ptr(),
          ldx, _p(gate), gamma.data_ptr(), _p(y) if relu else None, d, stat[0].data_ptr(),
          stat[1].data_ptr(), _p(dres), d, dx.data_ptr(), d, dpar.data_ptr(),
          dpar[1:].data_ptr(), dpar[1 + d:].data_ptr(), _p(dxsum), M, d, int(relu), _stream())
    return dres, dx, dpar


def _rowsum(bf16_in: bool, x, out, period=1):
    x, M, ldx = _rows(x)
    _call(f"mmemo_rowsum_{_sfx(bf16_in)}", x.data_ptr(), ldx, out.data_ptr(), M, x.shape[-1],
          period, _stream())


def _bld(t: Tensor, L: int) -> int:
    """Row stride of a (B, L, d) activation whose batch stride must be L*ld."""
    assert t.dim() == 3 and t.stride(2) == 1 and (t.shape[0] == 1 or t.stride(0) == L * t.stride(1)), \
        "activation must be (B, L, d) with unit inner stride and packed batch"
    return t.stride(1)


def _mask_strides(mask: Optional[Tensor], Lq: int, Lk: int) -> Tuple[int, int]:
    if mask is None:
        return 0, 0
    if mask.dim() == 2:
        return Lk, 0
    return Lq * Lk, Lk


def _attn_fwd(bf16, q, k, v, mask, s_prev, c, H, want_s):
    B, Lq, d = q.shape
    Lk = k.shape[1]
    hd = d // H
    dt = _act_dtype(bf16)
    o = torch.empty(B, Lq, d, dtype=dt, device=q.device)
    s = torch.empty(B, H, Lq, Lk, dtype=dt, device=q.device) if want_s else None
    stat = torch.empty(B, H, Lq, 2, dtype=F32, device=q.device)
    mbs, mrs = _mask_strides(mask, Lq, Lk)
    _call(f"mmemo_resattn_fwd_{_sfx(bf16)}", q.data_ptr(), _bld(q, Lq), k.data_ptr(), _bld(k, Lk),
          v.data_ptr(), _bld(v, Lk), _p(mask), mbs, mrs, _p(s_prev),
          _p(c) if s_prev is not None else None, _p(s), o.data_ptr(), d, stat.data_ptr(), B, H, Lq,
          Lk, hd, _stream())
    return o, s, stat


def _attn_bwd(bf16, do, q, k, v, mask, s, s_prev, c, ds_next, o, stat, H, dq, dk, dv, want_dsprev,
              dc_out=None):
    B, Lq, d = q.shape
    Lk = k.shape[1]
    hd = d // H
    dt = _act_dtype(bf16)
    ds_prev = None
    dc = None
    if s_prev is not None:
        # "+=" scalar: a zero-initialised slot of the caller, or our own
        dc = dc_out if dc_out is not None else torch.zeros(1, dtype=F32, device=q.device)
        if want_dsprev:
            ds_prev = torch.empty(B, H, Lq, Lk, dtype=dt, device=q.device)
    ws = None
    if bf16 and Lk > 128 and not _lib.load().mmemo_resattn_uses_tensor_cores(Lq, Lk, hd, d):
        ws = torch.empty(B, Lq, d, dtype=F32, device=q.device)
    mbs, mrs = _mask_strides(mask, Lq, Lk)
    _call(f"mmemo_resattn_bwd_{_sfx(bf16)}", do.data_ptr(), _bld(do, Lq), q.data_ptr(),
          _bld(q, Lq), k.data_ptr(), _bld(k, Lk), v.data_ptr(), _bld(v, Lk), _p(mask), mbs, mrs,
          _p(s), _p(s_prev), _p(c) if s_prev is not None else None, _p(ds_next), o.data_ptr(),
          _bld(o, Lq), stat.data_ptr(), dq.data_ptr(), _bld(dq, Lq), dk.data_ptr(), _bld(dk, Lk),
          dv.data_ptr(), _bld(dv, Lk), _p(ds_prev), _p(dc), _p(ws), B, H, Lq, Lk, hd, _stream())
    return ds_prev, dc


# ------------------------------------------------------------------------------------------------
# grouped residual attention (bf16): the problems of a fusion-trunk layer in ONE launch
# ------------------------------------------------------------------------------------------------
def score_stride(Lk: int) -> int:
    """Row stride of the score tensors the fused trunk allocates: padded to 8 elements so that the
    kernels move S / S_prev / dS as 16-byte vectors (the returned scores are the [..., :Lk] view)."""
    return (Lk + 7) // 8 * 8


def _attn_problem(q, k, v, mask, s_prev, c, s_out, o, stat, H, lds, d_o=None, s=None, ds_next=None,
                  dq=None, dk=None, dv=None, ds_prev=None, dc=None) -> "_lib.AttnProblem":
    B, Lq, d = q.shape
    Lk = k.shape[1]
    a = _lib.AttnProblem()
    a.q, a.k, a.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    a.ldq, a.ldk, a.ldv = _bld(q, Lq), _bld(k, Lk), _bld(v, Lk)
    a.mask, a.mask_bs = _p(mask), Lk
    a.s_prev, a.c = _p(s_prev), (_p(c) if s_prev is not None else None)
    a.s_out, a.lds = _p(s_out), lds
    a.o, a.ldo, a.lse = o.data_ptr(), _bld(o, Lq), stat.data_ptr()
    a.B, a.H, a.Lq, a.Lk, a.hd = B, H, Lq, Lk, d // H
    if d_o is not None:
        a.d_o, a.lddo = d_o.data_ptr(), _bld(d_o, Lq)
        a.s, a.ds_next = _p(s), _p(ds_next)
        a.dq, a.dk, a.dv = dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
        a.lddq, a.lddk, a.lddv = _bld(dq, Lq), _bld(dk, Lk), _bld(dv, Lk)
        a.ds_prev, a.dc = _p(ds_prev), _p(dc)
    return a


def _attn_group_call(name: str, probs) -> bool:
    """One grouped launch; False when the mma kernels do not take one of the shapes."""
    arr = (_lib.AttnProblem * len(probs))(*probs)
    return _try_call(name, len(probs), C.cast(arr, C.c_void_p), _stream())


# ------------------------------------------------------------------------------------------------
# mmemo::linear  (Linear / Conv1d(k=1) with optional bias, fused position table, fused ReLU)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::linear", mutates_args=())
def linear_op(x: Tensor, w: Tensor, bias: Optional[Tensor], pos: Optional[Tensor], relu: bool,
              bf16: bool) -> Tensor:
    _need_cuda(x, w)
    N = w.shape[0]
    y = torch.empty(*x.shape[:-1], N, dtype=_act_dtype(bf16), device=x.device)
    if pos is not None:
        assert x.dim() == 3 and pos.shape[0] == x.shape[1], "position table length != seq length"
    _linear_fwd(bf16, x, _weight(bf16, w), bias, pos, y.view(-1, N), relu=relu)
    return y


@linear_op.register_fake
def _(x, w, bias, pos, relu, bf16):
    return x.new_empty(*x.shape[:-1], w.shape[0], dtype=_act_dtype(bf16))


@torch.library.custom_op("mmemo::linear_bwd", mutates_args=())
def linear_bwd_op(dy: Tensor, x: Tensor, w: Tensor, y: Optional[Tensor], has_bias: bool,
                  pos_len: int, need_dx: bool, bf16: bool) -> List[Tensor]:
    N, K = w.shape[0], w.numel() // w.shape[0]
    dev = x.device
    dy = dy.contiguous()
    if y is not None:  # fused ReLU: mask the incoming gradient once
        dy = torch.where(y > 0, dy, torch.zeros((), dtype=dy.dtype, device=dev))
    dw = torch.empty(N, K, dtype=F32, device=dev)
    dbias = torch.zeros(N, dtype=F32, device=dev) if has_bias else torch.empty(0, device=dev)
    _linear_bwd_w(bf16, dy.view(-1, N), x, dw, dbias if has_bias else None)
    dpos = torch.empty(0, device=dev)
    if pos_len > 0:
        dpos = torch.zeros(pos_len, N, dtype=F32, device=dev)
        _rowsum(bf16, dy.view(-1, N), dpos, period=pos_len)
    dx = torch.empty(0, device=dev)
    if need_dx:
        dxa = torch.empty(x.shape, dtype=_act_dtype(bf16), device=dev)
        _linear_bwd_x(bf16, dy.view(-1, N), _weight(bf16, w), dxa.view(-1, K))
        dx = dxa if dxa.dtype == x.dtype else dxa.to(x.dtype)
    return [dx, dw.view(w.shape), dbias, dpos]


def _linear_setup(ctx, inputs, output):
    x, w, bias, pos, relu, bf16 = inputs
    ctx.save_for_backward(x, w, output if relu else None)
    ctx.has_bias = bias is not None
    ctx.pos_len = 0 if pos is None else pos.shape[0]
    ctx.bf16 = bf16


def _linear_backward(ctx, dy):
    x, w, y = ctx.saved_tensors
    dx, dw, dbias, dpos = linear_bwd_op(dy, x, w, y, ctx.has_bias, ctx.pos_len,
                                        ctx.needs_input_grad[0], ctx.bf16)
    return (dx if ctx.needs_input_grad[0] else None, dw, dbias if ctx.has_bias else None,
            dpos if ctx.pos_len else None, None, None)


linear_op.register_autograd(_linear_backward, setup_context=_linear_setup)


def linear(x, w, bias=None, pos=None, relu=False, bf16=False):
    if w.dim() == 3:  # Conv1d(kernel_size=1) weight (out, in, 1)
        w = w.squeeze(-1)
    return linear_op(x, w, bias, pos, relu, bf16)


# ------------------------------------------------------------------------------------------------
# mmemo::add_ln   y = act(LN(res + gate*x))
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::add_ln", mutates_args=())
def add_ln_op(res: Optional[Tensor], x: Tensor, gate: Optional[Tensor], gamma: Tensor,
              beta: Tensor, relu: bool) -> Tuple[Tensor, Tensor]:
    _need_cuda(x)
    return _add_ln_fwd(x.dtype == BF, res, x, gate, gamma, beta, relu)


@add_ln_op.register_fake
def _(res, x, gate, gamma, beta, relu):
    return torch.empty_like(x), x.new_empty(2, x.numel() // x.shape[-1], dtype=F32)


@torch.library.custom_op("mmemo::add_ln_bwd", mutates_args=())
def add_ln_bwd_op(dy: Tensor, res: Optional[Tensor], x: Tensor, gate: Optional[Tensor],
                  gamma: Tensor, y: Tensor, stat: Tensor, relu: bool) -> List[Tensor]:
    dres, dx, dpar = _add_ln_bwd(x.dtype == BF, dy.contiguous(), res, x, gate, gamma, y, stat, relu,
                                 res is not None)
    return [dres if dres is not None else torch.empty(0, device=x.device), dx, dpar]


def _add_ln_setup(ctx, inputs, output):
    res, x, gate, gamma, beta, relu = inputs
    y, stat = output
    ctx.save_for_backward(res, x, gate, gamma, y, stat)
    ctx.relu = relu
    ctx.set_materialize_grads(False)


def _add_ln_backward(ctx, dy, _dstat):
    res, x, gate, gamma, y, stat = ctx.saved_tensors
    d = x.shape[-1]
    dres, dx, dpar = add_ln_bwd_op(dy, res, x, gate, gamma, y, stat, ctx.relu)
    return (dres if res is not None else None, dx, dpar[0:1] if gate is not None else None,
            dpar[1:1 + d], dpar[1 + d:], None)


add_ln_op.register_autograd(_add_ln_backward, setup_context=_add_ln_setup)


def add_ln(res, x, gate, gamma, beta, relu=False):
    return add_ln_op(res, x, gate, gamma, beta, relu)[0]


# ------------------------------------------------------------------------------------------------
# mmemo::resattn  (the attention core on already-projected q/k/v; unit-testable piece of kernel a)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::resattn", mutates_args=())
def resattn_op(q: Tensor, k: Tensor, v: Tensor, mask: Optional[Tensor], s_prev: Optional[Tensor],
               c: Optional[Tensor], n_heads: int) -> Tuple[Tensor, Tensor, Tensor]:
    _need_cuda(q, k, v)
    q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
    o, s, stat = _attn_fwd(q.dtype == BF, q, k, v, mask, s_prev, c, n_heads, True)
    return o, s, stat


@torch.library.custom_op("mmemo::resattn_bwd", mutates_args=())
def resattn_bwd_op(do: Tensor, ds_next: Optional[Tensor], q: Tensor, k: Tensor, v: Tensor,
                   mask: Optional[Tensor], s: Tensor, s_prev: Optional[Tensor],
                   c: Optional[Tensor], o: Tensor, stat: Tensor, n_heads: int) -> List[Tensor]:
    q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
    dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    ds_prev, dc = _attn_bwd(q.dtype == BF, do.contiguous(), q, k, v, mask, s, s_prev, c,
                            None if ds_next is None else ds_next.contiguous(), o, stat, n_heads,
                            dq, dk, dv, True)
    return [dq, dk, dv, ds_prev if ds_prev is not None else torch.empty(0, device=q.device),
            dc if dc is not None else torch.empty(0, device=q.device)]


def _resattn_setup(ctx, inputs, output):
    q, k, v, mask, s_prev, c, H = inputs
    o, s, stat = output
    ctx.save_for_backward(q, k, v, mask, s, s_prev, c, o, stat)
    ctx.H = H
    ctx.set_materialize_grads(False)


def _resattn_backward(ctx, do, ds, _dstat):
    q, k, v, mask, s, s_prev, c, o, stat = ctx.saved_tensors
    if do is None:
        do = torch.zeros_like(o)
    dq, dk, dv, dsp, dc = resattn_bwd_op(do, ds, q, k, v, mask, s, s_prev, c, o, stat, ctx.H)
    has_prev = s_prev is not None
    return (dq, dk, dv, None, dsp if has_prev else None,
            dc if (has_prev and c is not None) else None, None)


resattn_op.register_autograd(_resattn_backward, setup_context=_resattn_setup)


# ------------------------------------------------------------------------------------------------
# mmemo::pool  — concat + mean||max pooling over a segment table (float32 output)
# segs: n_groups*n_slots tensors, group-major; group g tensors are (B, L_g, d)
# ------------------------------------------------------------------------------------------------
def _seg_table(segs: Sequence[Tensor], n_groups: int):
    n_slots = len(segs) // n_groups
    ptrs = (C.c_void_p * len(segs))(*[t.data_ptr() for t in segs])
    lens = (C.c_int64 * n_groups)(*[segs[g * n_slots].shape[1] for g in range(n_groups)])
    return ptrs, lens, n_slots


@torch.library.custom_op("mmemo::pool", mutates_args=())
def pool_op(segs: Sequence[Tensor], n_groups: int) -> Tuple[Tensor, Tensor]:
    _need_cuda(*segs)
    segs = [t.contiguous() for t in segs]
    ptrs, lens, n_slots = _seg_table(segs, n_groups)
    B, _, d = segs[0].shape
    bf16 = segs[0].dtype == BF
    out = torch.empty(B, 2 * n_slots * d, dtype=F32, device=segs[0].device)
    amax = torch.empty(B, n_slots * d, dtype=torch.int32, device=segs[0].device)
    _call(f"mmemo_pool_fwd_{_sfx(bf16)}", ptrs, lens, n_groups, n_slots, B, d, out.data_ptr(),
          amax.data_ptr(), _stream())
    return out, amax


@torch.library.custom_op("mmemo::pool_bwd", mutates_args=())
def pool_bwd_op(dout: Tensor, amax: Tensor, like: Sequence[Tensor], n_groups: int) -> List[Tensor]:
    dsegs = [torch.empty(t.shape, dtype=t.dtype, device=t.device) for t in like]
    ptrs, lens, n_slots = _seg_table(dsegs, n_groups)
    B, _, d = dsegs[0].shape
    _call(f"mmemo_pool_bwd_{_sfx(dsegs[0].dtype == BF)}", dout.contiguous().data_ptr(),
          amax.data_ptr(), ptrs, lens, n_groups, n_slots, B, d, _stream())
    return dsegs


def _pool_setup(ctx, inputs, output):
    segs, n_groups = inputs
    ctx.save_for_backward(output[1], *segs)
    ctx.n_groups = n_groups
    ctx.set_materialize_grads(False)


def _pool_backward(ctx, dout, _damax):
    amax, *segs = ctx.saved_tensors
    return pool_bwd_op(dout, amax, segs, ctx.n_groups), None


pool_op.register_autograd(_pool_backward, setup_context=_pool_setup)


def pool(segs: Sequence[Tensor], n_groups: int = 3) -> Tensor:
    return pool_op(list(segs), n_groups)[0]


def pool_multi(towers: Sequence[Sequence[Tensor]], n_groups: int = 3) -> List[Tensor]:
    """Inference pooling of several trunks (same B, d, lengths) in one call: ``pool`` of every
    tower's segment list, without argmax and without autograd."""
    segs = [[t.contiguous() for t in tw] for tw in towers]
    _need_cuda(*segs[0])
    n_slots = len(segs[0]) // n_groups
    B, _, d = segs[0][0].shape
    _, lens, _ = _seg_table(segs[0], n_groups)
    outs = [torch.empty(B, 2 * n_slots * d, dtype=F32, device=segs[0][0].device) for _ in segs]
    _call(f"mmemo_pool_fwd_multi_{_sfx(segs[0][0].dtype == BF)}", len(segs),
          _arr(C.c_void_p, [t.data_ptr() for tw in segs for t in tw]), lens, n_groups, n_slots,
          B, d, _arr(C.c_void_p, [o.data_ptr() for o in outs]), _stream())
    return outs


def ensemble_head(kind: int, members: Sequence, B: int, P: int, F: int, d: int, n_cls: int,
                  out: Tensor, member_out: Optional[Tensor] = None) -> None:
    """``out`` (float32, (B, P, C) or (B, C)) = mean over ``members`` (``_lib.EnsembleMember``)
    of their heads (include/mmemo.h mmemo_ensemble_head_fwd).  ``member_out`` (float32, (K,) +
    out.shape): also each member's own output (mmemo_ensemble_head_fwd_members)."""
    _need_cuda(out)
    arr = (_lib.EnsembleMember * len(members))(*members)
    if member_out is None:
        _call("mmemo_ensemble_head_fwd", kind, len(members), C.cast(arr, C.c_void_p), B, P, F, d,
              n_cls, LN_EPS, out.data_ptr(), _stream())
        return
    assert member_out.dtype == F32 and member_out.is_contiguous()
    assert member_out.shape == (len(members),) + tuple(out.shape)
    _call("mmemo_ensemble_head_fwd_members", kind, len(members), C.cast(arr, C.c_void_p), B, P, F,
          d, n_cls, LN_EPS, out.data_ptr(), member_out.data_ptr(), _stream())


FOLD_UQ_MAX_CLASSES = 1024


def fold_uncertainty(logits: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Fold logits ``(K, *rows, C)`` (float32 or bfloat16, contiguous, CUDA) -> (mean_prob,
    var_prob, entropy, expected_entropy, mutual_info, label): float32 ``(*rows, C)`` twice,
    float32 ``(*rows)`` three times and int64 ``(*rows)`` (include/mmemo.h
    mmemo_fold_uncertainty_*).  One launch; no autograd."""
    if not isinstance(logits, Tensor) or logits.dim() < 2:
        raise ValueError("fold_uncertainty: logits must be a tensor of shape (K, ..., C)")
    if logits.dtype not in (F32, BF):
        raise TypeError(f"fold_uncertainty: logits must be float32 or bfloat16, got {logits.dtype}")
    _need_cuda(logits)
    if not logits.is_contiguous():
        raise ValueError("fold_uncertainty: logits must be contiguous")
    K, rows, n_cls = logits.shape[0], tuple(logits.shape[1:-1]), logits.shape[-1]
    if K < 1 or n_cls < 1:
        raise ValueError(f"fold_uncertainty: need K >= 1 folds and C >= 1 classes, got shape "
                         f"{tuple(logits.shape)}")
    if n_cls > FOLD_UQ_MAX_CLASSES:
        raise ValueError(f"fold_uncertainty: C = {n_cls} classes, at most {FOLD_UQ_MAX_CLASSES}")
    N = math.prod(rows)
    dev = logits.device
    mean_p = torch.empty(*rows, n_cls, dtype=F32, device=dev)
    var_p = torch.empty(*rows, n_cls, dtype=F32, device=dev)
    ent, exp_ent, mi = (torch.empty(rows, dtype=F32, device=dev) for _ in range(3))
    label = torch.empty(rows, dtype=torch.int64, device=dev)
    _call(f"mmemo_fold_uncertainty_{_sfx(logits.dtype == BF)}", logits.data_ptr(), K, N, n_cls,
          mean_p.data_ptr(), var_p.data_ptr(), ent.data_ptr(), exp_ent.data_ptr(), mi.data_ptr(),
          label.data_ptr(), _stream())
    return mean_p, var_p, ent, exp_ent, mi, label


# ------------------------------------------------------------------------------------------------
# heads and losses (float32)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::state_transfer", mutates_args=())
def state_transfer_op(feats: Tensor, trans: Tensor) -> Tensor:
    _need_cuda(feats)
    feats, trans = feats.float().contiguous(), trans.contiguous()
    B, P, C2 = feats.shape
    out = torch.empty(B, P, C2 // 2, dtype=F32, device=feats.device)
    _call("mmemo_state_transfer_fwd", feats.data_ptr(), trans.data_ptr(), out.data_ptr(), B, P,
          C2 // 2, _stream())
    return out


@torch.library.custom_op("mmemo::state_transfer_bwd", mutates_args=())
def state_transfer_bwd_op(dout: Tensor, feats: Tensor, trans: Tensor, out: Tensor) -> List[Tensor]:
    feats, trans = feats.float().contiguous(), trans.contiguous()
    B, P, C2 = feats.shape
    dfeats = torch.empty_like(feats)
    dtrans = torch.zeros_like(trans)
    _call("mmemo_state_transfer_bwd", dout.contiguous().data_ptr(), feats.data_ptr(),
          trans.data_ptr(), out.data_ptr(), dfeats.data_ptr(), dtrans.data_ptr(), B, P, C2 // 2,
          _stream())
    return [dfeats, dtrans]


def _st_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1], output)


def _st_backward(ctx, dout):
    feats, trans, out = ctx.saved_tensors
    dfeats, dtrans = state_transfer_bwd_op(dout, feats, trans, out)
    return dfeats.to(feats.dtype), dtrans


state_transfer_op.register_autograd(_st_backward, setup_context=_st_setup)


@torch.library.custom_op("mmemo::bilinear_head", mutates_args=())
def bilinear_head_op(this_feat: Tensor, last_feat: Tensor, trans: Tensor, gamma: Tensor,
                     beta: Tensor, w: Tensor, bias: Tensor) -> Tuple[Tensor, Tensor]:
    _need_cuda(this_feat)
    th, la = this_feat.float().contiguous(), last_feat.float().contiguous()
    B, Cn = th.shape
    out = torch.empty(B, Cn, dtype=F32, device=th.device)
    z = torch.empty(B, Cn, dtype=F32, device=th.device)
    _call("mmemo_bilinear_head_fwd", th.data_ptr(), la.data_ptr(), trans.contiguous().data_ptr(),
          gamma.data_ptr(), beta.data_ptr(), w.contiguous().data_ptr(), bias.data_ptr(),
          out.data_ptr(), z.data_ptr(), B, Cn, LN_EPS, _stream())
    return out, z


@torch.library.custom_op("mmemo::bilinear_head_bwd", mutates_args=())
def bilinear_head_bwd_op(dout: Tensor, this_feat: Tensor, last_feat: Tensor, trans: Tensor,
                         gamma: Tensor, beta: Tensor, w: Tensor, z: Tensor) -> List[Tensor]:
    th, la = this_feat.float().contiguous(), last_feat.float().contiguous()
    B, Cn = th.shape
    dev = th.device
    dth, dla = torch.empty_like(th), torch.empty_like(la)
    dT = torch.zeros(Cn, Cn, Cn, dtype=F32, device=dev)
    dg, db = torch.zeros(Cn, dtype=F32, device=dev), torch.zeros(Cn, dtype=F32, device=dev)
    dw = torch.zeros(Cn, 2 * Cn, dtype=F32, device=dev)
    dbias = torch.zeros(Cn, dtype=F32, device=dev)
    _call("mmemo_bilinear_head_bwd", dout.contiguous().data_ptr(), th.data_ptr(), la.data_ptr(),
          trans.contiguous().data_ptr(), gamma.data_ptr(), beta.data_ptr(),
          w.contiguous().data_ptr(), z.data_ptr(), dth.data_ptr(), dla.data_ptr(), dT.data_ptr(),
          dg.data_ptr(), db.data_ptr(), dw.data_ptr(), dbias.data_ptr(), B, Cn, LN_EPS, _stream())
    return [dth, dla, dT, dg, db, dw, dbias]


def _bh_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:6], output[1])
    ctx.set_materialize_grads(False)


def _bh_backward(ctx, dout, _dz):
    th, la, trans, gamma, beta, w, z = ctx.saved_tensors
    dth, dla, dT, dg, db, dw, dbias = bilinear_head_bwd_op(dout, th, la, trans, gamma, beta, w, z)
    return dth.to(th.dtype), dla.to(la.dtype), dT, dg, db, dw, dbias


bilinear_head_op.register_autograd(_bh_backward, setup_context=_bh_setup)


def bilinear_head(this_feat, last_feat, trans, gamma, beta, w, bias):
    return bilinear_head_op(this_feat, last_feat, trans, gamma, beta, w, bias)[0]


@torch.library.custom_op("mmemo::circle_loss", mutates_args=())
def circle_loss_op(logits: Tensor, labels: Tensor) -> Tensor:
    _need_cuda(logits)
    C_ = logits.shape[-1]
    lg = logits.float().contiguous()
    lb = labels.to(F32).contiguous()
    loss = torch.empty(logits.shape[:-1], dtype=F32, device=logits.device)
    _call("mmemo_circle_loss_fwd", lg.data_ptr(), lb.data_ptr(), loss.data_ptr(),
          lg.numel() // C_, C_, _stream())
    return loss


@torch.library.custom_op("mmemo::circle_loss_bwd", mutates_args=())
def circle_loss_bwd_op(dloss: Tensor, logits: Tensor, labels: Tensor) -> Tensor:
    C_ = logits.shape[-1]
    lg = logits.float().contiguous()
    lb = labels.to(F32).contiguous()
    dl = torch.empty_like(lg)
    _call("mmemo_circle_loss_bwd", dloss.to(F32).contiguous().data_ptr(), lg.data_ptr(),
          lb.data_ptr(), dl.data_ptr(), lg.numel() // C_, C_, _stream())
    return dl


def _cl_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _cl_backward(ctx, dloss):
    logits, labels = ctx.saved_tensors
    return circle_loss_bwd_op(dloss, logits, labels).to(logits.dtype), None


circle_loss_op.register_autograd(_cl_backward, setup_context=_cl_setup)


@torch.library.custom_op("mmemo::rdrop_kl", mutates_args=())
def rdrop_kl_op(logits: Tensor) -> Tensor:
    _need_cuda(logits)
    lg = logits.float().contiguous()
    out = torch.empty((), dtype=F32, device=logits.device)
    _call("mmemo_rdrop_kl_fwd", lg.data_ptr(), out.data_ptr(), lg.shape[0], lg.shape[1], _stream())
    return out


@torch.library.custom_op("mmemo::rdrop_kl_bwd", mutates_args=())
def rdrop_kl_bwd_op(dout: Tensor, logits: Tensor) -> Tensor:
    lg = logits.float().contiguous()
    dl = torch.empty_like(lg)
    _call("mmemo_rdrop_kl_bwd", dout.to(F32).contiguous().data_ptr(), lg.data_ptr(), dl.data_ptr(),
          lg.shape[0], lg.shape[1], _stream())
    return dl


def _rk_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])


def _rk_backward(ctx, dout):
    (logits,) = ctx.saved_tensors
    return rdrop_kl_bwd_op(dout, logits).to(logits.dtype)


rdrop_kl_op.register_autograd(_rk_backward, setup_context=_rk_setup)


# ------------------------------------------------------------------------------------------------
# mean(x^2) (the encoder benchmark's synthetic loss) — one launch per direction
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::sq_mean", mutates_args=())
def sq_mean_op(x: Tensor) -> Tensor:
    _need_cuda(x)
    x = x.contiguous()
    out = torch.zeros((), dtype=F32, device=x.device)
    _call(f"mmemo_sqmean_fwd_{_sfx(x.dtype == BF)}", x.data_ptr(), x.numel(), out.data_ptr(),
          _stream())
    return out


@torch.library.custom_op("mmemo::sq_mean_bwd", mutates_args=())
def sq_mean_bwd_op(dloss: Tensor, x: Tensor) -> Tensor:
    x = x.contiguous()
    dx = torch.empty_like(x)
    _call(f"mmemo_sqmean_bwd_{_sfx(x.dtype == BF)}", x.data_ptr(),
          dloss.to(F32).contiguous().data_ptr(), x.numel(), dx.data_ptr(), _stream())
    return dx


def _sq_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])


def _sq_backward(ctx, dloss):
    (x,) = ctx.saved_tensors
    return sq_mean_bwd_op(dloss, x)


sq_mean_op.register_autograd(_sq_backward, setup_context=_sq_setup)


def cast_bf16(x: Tensor) -> Tensor:
    """float32 -> bf16 copy of a tensor that needs no gradient (raw inputs), libmmemo's vector
    cast instead of ATen's generic copy kernel."""
    x = x.contiguous()
    y = torch.empty(x.shape, dtype=BF, device=x.device)
    _call("mmemo_cast_f32_to_bf16", x.data_ptr(), y.data_ptr(), x.numel(), _stream())
    return y


# ------------------------------------------------------------------------------------------------
# dropout (counter-based; forward and backward are the same kernel with the same seed)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::dropout", mutates_args=())
def dropout_op(x: Tensor, p: float, seed: int) -> Tensor:
    _need_cuda(x)
    x = x.contiguous()
    y = torch.empty_like(x)
    _call(f"mmemo_dropout_{_sfx(x.dtype == BF)}", x.data_ptr(), y.data_ptr(), x.numel(), p,
          seed & 0xFFFFFFFFFFFFFFFF, _stream())
    return y


def _do_setup(ctx, inputs, output):
    ctx.p, ctx.seed = inputs[1], inputs[2]


def _do_backward(ctx, dy):
    return dropout_op(dy, ctx.p, ctx.seed), None, None


dropout_op.register_autograd(_do_backward, setup_context=_do_setup)

_dropout_counter = [0]
_dropout_step = {}     # device -> int64 scalar mixed into the grouped-dropout seeds at run time


def next_dropout_seed() -> int:
    """A fresh 63-bit seed per call, derived from torch's seed (``torch.manual_seed`` controls it)."""
    _dropout_counter[0] += 1
    seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + _dropout_counter[0] * 0xD1B54A32D192ED03)
    return seed & 0x7FFFFFFFFFFFFFFF


def dropout(x: Tensor, p: float, training: bool) -> Tensor:
    if not training or p <= 0.0:
        return x
    return dropout_op(x, float(p), next_dropout_seed())


def dropout_step(dev) -> Tensor:
    """Device scalar added to every grouped-dropout seed when the kernel RUNS.  Python-side seeds
    are frozen when a training step is captured into a CUDA graph; a captured ``advance_dropout_step``
    (one increment per replay) makes every replay draw new masks."""
    dev = torch.device(dev)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    t = _dropout_step.get(dev)
    if t is None:
        t = _dropout_step[dev] = torch.zeros(1, dtype=torch.int64, device=dev)
    return t


def advance_dropout_step(dev="cuda") -> None:
    dropout_step(dev).add_(1)


def site_seeds(seed: int, G: int, site: int, n_sites: int = 2) -> List[int]:
    """One seed per (problem, dropout site) of a grouped layer."""
    return [(seed + (n_sites * g + site + 1) * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF
            for g in range(G)]


def _dropout_group(xs, ys, p: float, seeds) -> None:
    """ys[i] = dropout(xs[i]) in one call (one launch per 64 tensors); xs[i] is ys[i] = in place.
    Forward and backward use the same seeds (same masks)."""
    if p <= 0.0 or not xs:
        return
    bf16 = xs[0].dtype == BF
    step = dropout_step(xs[0].device)
    assert all(t.is_contiguous() for t in xs) and all(t.is_contiguous() for t in ys)
    _call(f"mmemo_dropout_multi_{_sfx(bf16)}", len(xs),
          _arr(C.c_void_p, [t.data_ptr() for t in xs]), _arr(C.c_void_p, [t.data_ptr() for t in ys]),
          _arr(C.c_int64, [t.numel() for t in xs]), _arr(C.c_uint64, list(seeds)), float(p),
          step.data_ptr(), _stream())
