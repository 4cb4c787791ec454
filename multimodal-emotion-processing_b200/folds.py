"""Grouped training of the k cross-validation folds (SURVEY.md §8f-4): one forward and one backward
for all folds' models instead of one per fold.

``forward(models, inputs)`` returns ``[models[k](*inputs[k]) for k]`` with autograd to each
model's own parameters, for k models of ONE of ``realformer.State_Transfer``,
``cmu_mosei.Concat_Trans``, ``ren_mme.Base_model``, ``rencecps.Concat_Linear`` or
``robot_demo.Multi_class`` (equal
state_dict shapes and ``n_heads`` / ``n_layers``, all in train or all in eval mode; ``ValueError``
otherwise).  The folds' batch sizes may differ.  One call runs, for all folds together:

- the modality projections as one grouped GEMM (bf16 mode; ``group_ops.proj_group_op``, or with
  the projections' own training dropout ``group_ops.proj_drop_group_op``, the mask drawn in the
  GEMM epilogue; ``Multi_class``'s three visual projections write the column thirds of one stream)
  and, for ``Base_model``, the towers' shared LayerNorm as one grouped LayerNorm (``ln_group_op``);
- every tower of every fold through one ``fusion_trunk_multi``;
- one grouped pooling (``mmemo_pool_fwd_multi_arg_*`` / ``mmemo_pool_bwd_multi_*``);
- the float32 head linears as grouped SIMT GEMMs (``mmemo_linear_*_grouped_f32``), with the
  grouped LayerNorm + ReLU and grouped dropout of ``State_Transfer``'s feature head between them;
- the bilinear or state-transfer head of every fold in one launch (``csrc/folds.cu``).

``circle_losses`` and ``rdrop_kl`` are the losses of every fold in one launch each, forward and
backward.  A ``trainer.fit_folds`` step for Ren-MME is then::

    ls = folds.forward(ms, [b[:12] for b in bs])
    return [c + r for c, r in zip(folds.circle_losses(ls, [b[12] for b in bs]), folds.rdrop_kl(ls))]

and for robot_demo's 4 folds (robot_demo.py:497-524; a batch is the 8 inputs then the labels)::

    return folds.circle_losses(folds.forward(ms, [b[:8] for b in bs]), [b[8] for b in bs])

Dropout.  The grouped trunk and head draw their masks from one seed per grouped call and a
per-problem index (``ops.site_seeds``), so a fold trained in the group draws different masks from
the ones it would draw alone.  Both are valid i.i.d. keep-(1-p) masks; with every dropout p = 0
the results equal the per-fold forward and backward: the grouped pooling, head linears, heads and
losses produce the bits of the per-model kernels (the float32 SIMT GEMM splits K per problem and
sums the partial tiles in a fixed order), so the activation gradients the trunk rounds to bf16 are
the same; parameter gradients summed with float atomics (head parameters, LayerNorm, scalar gates)
agree to float rounding.

Out of scope: fp32 grouping of the trunk's GEMMs and attention (the float32 parity mode runs them
per problem), and ``dp.GradReducer``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch
from torch import Tensor

from . import ops
from .blocks import as_mask, fusion_trunk_multi, is_bf16
from .cmu_mosei import Concat_Trans
from .ensemble import _check_members
from .group_ops import dropout_group_op, ln_bwd_group, ln_fwd_group, project, project_cat
from .ops import BF, F32, LN_EPS, _arr, _p
from .realformer import State_Transfer
from .ren_mme import Base_model
from .rencecps import Concat_Linear
from .robot_demo import Multi_class

# the families folds.forward groups (ensemble.Ensemble takes the first four; robot_demo.Ensemble
# serves Multi_class)
_FAMILIES = (State_Transfer, Concat_Trans, Base_model, Concat_Linear, Multi_class)


def _call(name, *args):          # late-bound: tests stub ops._call / ops._stream
    return ops._call(name, *args)


def _stream():
    return ops._stream()


def _vp(ts):
    return _arr(C.c_void_p, [_p(t) for t in ts])


def _i64(vals):
    return _arr(C.c_int64, [int(v) for v in vals])


def _sfx(t: Tensor) -> str:
    return "bf16" if t.dtype == BF else "f32"


def _views(flat: Tensor, ts: Sequence[Tensor]) -> List[Tensor]:
    """Consecutive views of ``flat`` shaped like ``ts`` (the parameter gradients of a grouped
    backward live in ONE zero-filled buffer: one fill; the ops return the buffer and the autograd
    glue takes the views, since a custom op's outputs may not alias each other)."""
    out, o = [], 0
    for t in ts:
        out.append(flat[o:o + t.numel()].view(t.shape))
        o += t.numel()
    return out


def _zeros_for(ts: Sequence[Tensor]) -> Tensor:
    return torch.zeros(sum(t.numel() for t in ts), dtype=F32, device=ts[0].device)


def _grads(grads, like):
    return [g if g is not None else torch.zeros_like(t) for g, t in zip(grads, like)]


# ------------------------------------------------------------------------------------------------
# grouped pooling of many towers (per-tower batch sizes), with argmax and backward
# ------------------------------------------------------------------------------------------------
N_POOL_GROUPS = 3


def _pool_layout(segs: Sequence[Tensor], n_towers: int):
    per = len(segs) // n_towers
    n_slots = per // N_POOL_GROUPS
    lens = _i64([segs[g * n_slots].shape[1] for g in range(N_POOL_GROUPS)])
    Bs = [segs[t * per].shape[0] for t in range(n_towers)]
    return per, n_slots, lens, Bs


@torch.library.custom_op("mmemo::pool_group", mutates_args=())
def pool_group_op(segs: Sequence[Tensor], n_towers: int) -> List[Tensor]:
    """``ops.pool`` of ``n_towers`` towers (``segs``: tower-major, each tower's segment list as
    ``ops.pool`` takes it); returns [pooled_0 .. pooled_{T-1}, argmax_0 .. argmax_{T-1}]."""
    ops._need_cuda(*segs)
    segs = [t.contiguous() for t in segs]
    per, n_slots, lens, Bs = _pool_layout(segs, n_towers)
    d = segs[0].shape[2]
    dev = segs[0].device
    outs = [torch.empty(b, 2 * n_slots * d, dtype=F32, device=dev) for b in Bs]
    amax = [torch.empty(b, n_slots * d, dtype=torch.int32, device=dev) for b in Bs]
    _call(f"mmemo_pool_fwd_multi_arg_{_sfx(segs[0])}", n_towers, _vp(segs), lens, N_POOL_GROUPS,
          n_slots, _i64(Bs), d, _vp(outs), _vp(amax), _stream())
    return outs + amax


@pool_group_op.register_fake
def _(segs, n_towers):
    per, n_slots, _, Bs = _pool_layout(segs, n_towers)
    d = segs[0].shape[2]
    return ([segs[0].new_empty(b, 2 * n_slots * d, dtype=F32) for b in Bs] +
            [segs[0].new_empty(b, n_slots * d, dtype=torch.int32) for b in Bs])


@torch.library.custom_op("mmemo::pool_group_bwd", mutates_args=())
def pool_group_bwd_op(douts: Sequence[Tensor], amax: Sequence[Tensor], like: Sequence[Tensor],
                      n_towers: int) -> List[Tensor]:
    dsegs = [torch.empty(t.shape, dtype=t.dtype, device=t.device) for t in like]
    per, n_slots, lens, Bs = _pool_layout(dsegs, n_towers)
    douts = [g.contiguous() for g in douts]
    _call(f"mmemo_pool_bwd_multi_{_sfx(dsegs[0])}", n_towers, _vp(douts), _vp(amax), _vp(dsegs),
          lens, N_POOL_GROUPS, n_slots, _i64(Bs), dsegs[0].shape[2], _stream())
    return dsegs


def _pool_group_setup(ctx, inputs, output):
    segs, n_towers = inputs
    ctx.n_towers = n_towers
    ctx.save_for_backward(*output[n_towers:], *segs)


def _pool_group_backward(ctx, grads):
    T = ctx.n_towers
    saved = ctx.saved_tensors
    amax, segs = saved[:T], saved[T:]
    douts = [g if g is not None else torch.zeros(a.shape[0], 2 * a.shape[1], dtype=F32,
                                                 device=a.device)
             for g, a in zip(grads[:T], amax)]
    return list(pool_group_bwd_op(douts, list(amax), list(segs), T)), None


pool_group_op.register_autograd(_pool_group_backward, setup_context=_pool_group_setup)


def pool_group(tower_segs: Sequence[Sequence[Tensor]]) -> List[Tensor]:
    """Pooled float32 features of every tower (``fusion_trunk_multi(..., pool=False)`` output)."""
    return pool_group_op([t for tw in tower_segs for t in tw], len(tower_segs))[:len(tower_segs)]


# ------------------------------------------------------------------------------------------------
# grouped float32 linears (the head linears: ops.linear(..., bf16=False) of every fold)
# ------------------------------------------------------------------------------------------------
def _ld(x: Tensor) -> int:
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype == F32
    return x.stride(0)


@torch.library.custom_op("mmemo::linear_group", mutates_args=())
def linear_group_op(xs: Sequence[Tensor], ws: Sequence[Tensor],
                    biases: Sequence[Tensor]) -> List[Tensor]:
    """y_g = x_g w_g^T (+ b_g) in float32; x_g (M_g, K) with unit inner stride (row slices of a
    wider tensor are read in place); bias entries with numel() == 0 mean none."""
    ops._need_cuda(*xs)
    ys = [torch.empty(x.shape[0], w.shape[0], dtype=F32, device=x.device) for x, w in zip(xs, ws)]
    _call("mmemo_linear_fwd_grouped_f32", len(xs), _vp(xs), _i64(_ld(x) for x in xs),
          _vp([w.detach() for w in ws]), _i64(w.stride(0) for w in ws),
          _vp([b if b.numel() else None for b in biases]), _vp(ys), _i64(y.stride(0) for y in ys),
          _i64(x.shape[0] for x in xs), _i64(w.shape[0] for w in ws),
          _i64(w.shape[1] for w in ws), _stream())
    return ys


@linear_group_op.register_fake
def _(xs, ws, biases):
    return [x.new_empty(x.shape[0], w.shape[0], dtype=F32) for x, w in zip(xs, ws)]


@torch.library.custom_op("mmemo::linear_group_bwd", mutates_args=())
def linear_group_bwd_op(dys: Sequence[Tensor], xs: Sequence[Tensor], ws: Sequence[Tensor],
                        has_bias: Sequence[bool], need_dx: Sequence[bool]) -> List[Tensor]:
    """Returns [dx_g or empty] + [dw_g] + [dbias_g or empty]."""
    dev = dys[0].device
    G = len(dys)
    dys = [d.contiguous() for d in dys]
    dws = [torch.empty(w.shape, dtype=F32, device=dev) for w in ws]
    dbs = [torch.empty(w.shape[0], dtype=F32, device=dev) if hb else torch.empty(0, device=dev)
           for w, hb in zip(ws, has_bias)]
    _call("mmemo_linear_bwd_w_grouped_f32", G, _vp(dys), _i64(d.stride(0) for d in dys), _vp(xs),
          _i64(_ld(x) for x in xs), _vp(dws), _i64(w.stride(0) for w in dws),
          _vp([b if hb else None for b, hb in zip(dbs, has_bias)]), _i64(x.shape[0] for x in xs),
          _i64(w.shape[0] for w in ws), _i64(w.shape[1] for w in ws), _stream())
    dxs = [torch.empty(x.shape, dtype=F32, device=dev) if nd else torch.empty(0, device=dev)
           for x, nd in zip(xs, need_dx)]
    ix = [g for g in range(G) if need_dx[g]]
    if ix:
        _call("mmemo_linear_bwd_x_grouped_f32", len(ix), _vp([dys[g] for g in ix]),
              _i64(dys[g].stride(0) for g in ix), _vp([ws[g].detach() for g in ix]),
              _i64(ws[g].stride(0) for g in ix), _vp([dxs[g] for g in ix]),
              _i64(dxs[g].stride(0) for g in ix), _i64(xs[g].shape[0] for g in ix),
              _i64(ws[g].shape[0] for g in ix), _i64(ws[g].shape[1] for g in ix), _stream())
    return dxs + dws + dbs


def _linear_group_setup(ctx, inputs, output):
    xs, ws, biases = inputs
    ctx.G = len(xs)
    ctx.has_bias = [b.numel() > 0 for b in biases]
    ctx.save_for_backward(*xs, *ws)


def _linear_group_backward(ctx, grads):
    G = ctx.G
    t = ctx.saved_tensors
    xs, ws = t[:G], t[G:]
    need_dx = list(ctx.needs_input_grad[0])
    dys = [g if g is not None else torch.zeros(x.shape[0], w.shape[0], device=x.device)
           for g, x, w in zip(grads, xs, ws)]
    res = linear_group_bwd_op(dys, list(xs), list(ws), ctx.has_bias, need_dx)
    dxs, dws, dbs = res[:G], res[G:2 * G], res[2 * G:]
    return ([dxs[g] if need_dx[g] else None for g in range(G)], list(dws),
            [dbs[g] if ctx.has_bias[g] else None for g in range(G)])


linear_group_op.register_autograd(_linear_group_backward, setup_context=_linear_group_setup)


def linear_group(xs, ws, biases=None) -> List[Tensor]:
    dev = xs[0].device
    biases = biases if biases is not None else [None] * len(xs)
    return list(linear_group_op(list(xs), list(ws),
                                [b if b is not None else torch.empty(0, device=dev)
                                 for b in biases]))


# ------------------------------------------------------------------------------------------------
# grouped LayerNorm (+ ReLU) with autograd, over ln_fwd_group / ln_bwd_group
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::ln_group", mutates_args=())
def ln_group_op(xs: Sequence[Tensor], gammas: Sequence[Tensor], betas: Sequence[Tensor],
                relu: bool) -> List[Tensor]:
    """y_g = act(LN(x_g; gamma_g, beta_g)) of every problem in one grouped call; returns
    [y_0 .. y_{G-1}, stat_0 .. stat_{G-1}]."""
    ops._need_cuda(*xs)
    xs = [x.contiguous() for x in xs]
    n = len(xs)
    ys, stats = ln_fwd_group(xs[0].dtype == BF, [None] * n, xs, [None] * n, list(gammas),
                             list(betas), relu)
    return ys + stats


@ln_group_op.register_fake
def _(xs, gammas, betas, relu):
    return ([torch.empty_like(x) for x in xs] +
            [x.new_empty(2, x.numel() // x.shape[-1], dtype=F32) for x in xs])


@torch.library.custom_op("mmemo::ln_group_bwd", mutates_args=())
def ln_group_bwd_op(dys: Sequence[Tensor], xs: Sequence[Tensor], gammas: Sequence[Tensor],
                    stats: Sequence[Tensor]) -> List[Tensor]:
    """Returns [dx_g] + [dpar]: dpar (G, 1 + 2d) = (unused | dgamma_g | dbeta_g) per row (no ReLU:
    the caller masks dy)."""
    n = len(xs)
    d = xs[0].shape[-1]
    xs = [x.contiguous() for x in xs]
    dpar = torch.zeros(n, 1 + 2 * d, dtype=F32, device=xs[0].device)
    _, dxs = ln_bwd_group(xs[0].dtype == BF, [dy.contiguous() for dy in dys], [None] * n, xs,
                          [None] * n, list(gammas), list(stats), False, list(dpar.unbind(0)))
    return dxs + [dpar]


def _ln_group_setup(ctx, inputs, output):
    xs, gammas, betas, relu = inputs
    n = len(xs)
    ctx.n, ctx.relu = n, relu
    ctx.save_for_backward(*xs, *gammas, *output)


def _ln_group_backward(ctx, grads):
    n = ctx.n
    t = ctx.saved_tensors
    xs, gammas, ys, stats = t[:n], t[n:2 * n], t[2 * n:3 * n], t[3 * n:]
    dys = _grads(grads[:n], ys)
    if ctx.relu:          # fused ReLU: mask the incoming gradient once (as ops.linear_bwd_op)
        dys = [torch.where(y > 0, dy, torch.zeros((), dtype=dy.dtype, device=dy.device))
               for y, dy in zip(ys, dys)]
    res = ln_group_bwd_op(dys, list(xs), list(gammas), list(stats))
    d = xs[0].shape[-1]
    dpar = res[n]
    return (list(res[:n]), [dpar[g, 1:1 + d] for g in range(n)],
            [dpar[g, 1 + d:] for g in range(n)], None)


ln_group_op.register_autograd(_ln_group_backward, setup_context=_ln_group_setup)


def ln_group(xs, gammas, betas, relu: bool = False) -> List[Tensor]:
    return list(ln_group_op(list(xs), list(gammas), list(betas), relu)[:len(xs)])


# ------------------------------------------------------------------------------------------------
# grouped heads
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::bilinear_group", mutates_args=())
def bilinear_group_op(ths: Sequence[Tensor], las: Sequence[Tensor], transes: Sequence[Tensor],
                      gammas: Sequence[Tensor], betas: Sequence[Tensor], ws: Sequence[Tensor],
                      biases: Sequence[Tensor]) -> List[Tensor]:
    """``ops.bilinear_head`` of every member in one launch; returns [out_g] + [z_g]."""
    ops._need_cuda(*ths)
    n, Cn = len(ths), ths[0].shape[1]
    dev = ths[0].device
    ths, las = [t.contiguous() for t in ths], [t.contiguous() for t in las]
    outs = [torch.empty(t.shape[0], Cn, dtype=F32, device=dev) for t in ths]
    zs = [torch.empty(t.shape[0], Cn, dtype=F32, device=dev) for t in ths]
    _call("mmemo_bilinear_head_fwd_multi", n, _vp(ths), _vp(las), _vp(transes), _vp(gammas),
          _vp(betas), _vp(ws), _vp(biases), _vp(outs), _vp(zs), _i64(t.shape[0] for t in ths), Cn,
          LN_EPS, _stream())
    return outs + zs


@bilinear_group_op.register_fake
def _(ths, las, transes, gammas, betas, ws, biases):
    return [torch.empty_like(t) for t in ths] * 2


@torch.library.custom_op("mmemo::bilinear_group_bwd", mutates_args=())
def bilinear_group_bwd_op(douts: Sequence[Tensor], ths: Sequence[Tensor], las: Sequence[Tensor],
                          transes: Sequence[Tensor], gammas: Sequence[Tensor],
                          betas: Sequence[Tensor], ws: Sequence[Tensor],
                          zs: Sequence[Tensor]) -> List[Tensor]:
    """Returns [dthis_g] + [dlast_g] + [flat]: flat holds dtrans, dgamma, dbeta, dw, dbias of
    every member (``_bilinear_pars``)."""
    n, Cn = len(ths), ths[0].shape[1]
    dth = [torch.empty_like(t) for t in ths]
    dla = [torch.empty_like(t) for t in las]
    like = _bilinear_pars(transes, gammas, ws)
    flat = _zeros_for(like)
    par = _views(flat, like)
    dT, dg, db, dw, dbias = (par[i::5] for i in range(5))
    _call("mmemo_bilinear_head_bwd_multi", n, _vp([d.contiguous() for d in douts]), _vp(ths),
          _vp(las), _vp(transes), _vp(gammas), _vp(betas), _vp(ws), _vp(zs), _vp(dth), _vp(dla),
          _vp(dT), _vp(dg), _vp(db), _vp(dw), _vp(dbias), _i64(t.shape[0] for t in ths), Cn,
          LN_EPS, _stream())
    return dth + dla + [flat]


def _bilinear_pars(transes, gammas, ws):
    return [p for g in range(len(transes)) for p in
            (transes[g], gammas[g], gammas[g], ws[g], gammas[g])]


def _bilinear_group_setup(ctx, inputs, output):
    ths, las, transes, gammas, betas, ws, biases = inputs
    n = len(ths)
    ctx.n = n
    ctx.save_for_backward(*[t.contiguous() for t in ths], *[t.contiguous() for t in las],
                          *transes, *gammas, *betas, *ws, *output[n:])


def _bilinear_group_backward(ctx, grads):
    n = ctx.n
    t = ctx.saved_tensors
    ths, las, transes, gammas, betas, ws, zs = (list(t[i * n:(i + 1) * n]) for i in range(7))
    res = bilinear_group_bwd_op(_grads(grads[:n], zs), ths, las, transes, gammas, betas, ws, zs)
    par = _views(res[2 * n], _bilinear_pars(transes, gammas, ws))
    return (list(res[:n]), list(res[n:2 * n])) + tuple(par[i::5] for i in range(5))


bilinear_group_op.register_autograd(_bilinear_group_backward, setup_context=_bilinear_group_setup)


@torch.library.custom_op("mmemo::state_transfer_group", mutates_args=())
def state_transfer_group_op(feats: Sequence[Tensor], transes: Sequence[Tensor]) -> List[Tensor]:
    """``ops.state_transfer_op`` of every member (feats_g (B_g, P, 2C) float32) in one launch."""
    ops._need_cuda(*feats)
    feats = [f.contiguous() for f in feats]
    _, P, C2 = feats[0].shape
    outs = [torch.empty(f.shape[0], P, C2 // 2, dtype=F32, device=f.device) for f in feats]
    _call("mmemo_state_transfer_fwd_multi", len(feats), _vp(feats), _vp(transes), _vp(outs),
          _i64(f.shape[0] for f in feats), P, C2 // 2, _stream())
    return outs


@state_transfer_group_op.register_fake
def _(feats, transes):
    return [f.new_empty(f.shape[0], f.shape[1], f.shape[2] // 2) for f in feats]


@torch.library.custom_op("mmemo::state_transfer_group_bwd", mutates_args=())
def state_transfer_group_bwd_op(douts: Sequence[Tensor], feats: Sequence[Tensor],
                                transes: Sequence[Tensor], outs: Sequence[Tensor]) -> List[Tensor]:
    n = len(feats)
    _, P, C2 = feats[0].shape
    dfeats = [torch.empty_like(f) for f in feats]
    flat = _zeros_for(transes)
    dtrans = _views(flat, transes)
    _call("mmemo_state_transfer_bwd_multi", n, _vp([d.contiguous() for d in douts]), _vp(feats),
          _vp(transes), _vp(outs), _vp(dfeats), _vp(dtrans), _i64(f.shape[0] for f in feats), P,
          C2 // 2, _stream())
    return dfeats + [flat]


def _st_group_setup(ctx, inputs, output):
    feats, transes = inputs
    ctx.n = len(feats)
    ctx.save_for_backward(*[f.contiguous() for f in feats], *transes, *output)


def _st_group_backward(ctx, grads):
    n = ctx.n
    t = ctx.saved_tensors
    feats, transes, outs = list(t[:n]), list(t[n:2 * n]), list(t[2 * n:])
    res = state_transfer_group_bwd_op(_grads(grads, outs), feats, transes, outs)
    return list(res[:n]), _views(res[n], transes)


state_transfer_group_op.register_autograd(_st_group_backward, setup_context=_st_group_setup)


# ------------------------------------------------------------------------------------------------
# grouped losses
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("mmemo::circle_group", mutates_args=())
def circle_group_op(logits: Sequence[Tensor], labels: Sequence[Tensor],
                    weights: Sequence[Tensor]) -> List[Tensor]:
    """One float32 scalar per member: (circle_loss(logits_g, labels_g) [* weights_g]).mean();
    weights entries with numel() == 0 mean none."""
    ops._need_cuda(*logits)
    Cn = logits[0].shape[-1]
    lg = [t.float().contiguous() for t in logits]
    lb = [t.to(F32).contiguous() for t in labels]
    wt = [w.to(F32).contiguous() if w.numel() else None for w in weights]
    out = [torch.empty((), dtype=F32, device=t.device) for t in lg]
    _call("mmemo_circle_loss_fwd_multi", len(lg), _vp(lg), _vp(lb), _vp(wt),
          _i64(t.numel() // Cn for t in lg), Cn, _vp(out), _stream())
    return out


@circle_group_op.register_fake
def _(logits, labels, weights):
    return [t.new_empty((), dtype=F32) for t in logits]


@torch.library.custom_op("mmemo::circle_group_bwd", mutates_args=())
def circle_group_bwd_op(dloss: Sequence[Tensor], logits: Sequence[Tensor], labels: Sequence[Tensor],
                        weights: Sequence[Tensor]) -> List[Tensor]:
    Cn = logits[0].shape[-1]
    lg = [t.float().contiguous() for t in logits]
    lb = [t.to(F32).contiguous() for t in labels]
    wt = [w.to(F32).contiguous() if w.numel() else None for w in weights]
    dl = [torch.empty_like(t) for t in lg]
    _call("mmemo_circle_loss_bwd_multi", len(lg), _vp([d.to(F32).contiguous() for d in dloss]),
          _vp(lg), _vp(lb), _vp(wt), _vp(dl), _i64(t.numel() // Cn for t in lg), Cn, _stream())
    return dl


def _circle_group_setup(ctx, inputs, output):
    logits, labels, weights = inputs
    ctx.n = len(logits)
    ctx.save_for_backward(*logits, *labels, *weights)


def _circle_group_backward(ctx, grads):
    n = ctx.n
    t = ctx.saved_tensors
    logits, labels, weights = list(t[:n]), list(t[n:2 * n]), list(t[2 * n:])
    dl = circle_group_bwd_op([g if g is not None else torch.zeros((), device=logits[0].device)
                              for g in grads], logits, labels, weights)
    return [d.to(l.dtype) for d, l in zip(dl, logits)], [None] * n, [None] * n


circle_group_op.register_autograd(_circle_group_backward, setup_context=_circle_group_setup)


@torch.library.custom_op("mmemo::rdrop_group", mutates_args=())
def rdrop_group_op(logits: Sequence[Tensor]) -> List[Tensor]:
    """``ops.rdrop_kl_op`` of every member (logits_g (B_g, C), B_g even) in one launch."""
    ops._need_cuda(*logits)
    lg = [t.float().contiguous() for t in logits]
    out = [torch.empty((), dtype=F32, device=t.device) for t in lg]
    _call("mmemo_rdrop_kl_fwd_multi", len(lg), _vp(lg), _i64(t.shape[0] for t in lg),
          lg[0].shape[1], _vp(out), _stream())
    return out


@rdrop_group_op.register_fake
def _(logits):
    return [t.new_empty((), dtype=F32) for t in logits]


@torch.library.custom_op("mmemo::rdrop_group_bwd", mutates_args=())
def rdrop_group_bwd_op(douts: Sequence[Tensor], logits: Sequence[Tensor]) -> List[Tensor]:
    lg = [t.float().contiguous() for t in logits]
    dl = [torch.empty_like(t) for t in lg]
    _call("mmemo_rdrop_kl_bwd_multi", len(lg), _vp([d.to(F32).contiguous() for d in douts]),
          _vp(lg), _vp(dl), _i64(t.shape[0] for t in lg), lg[0].shape[1], _stream())
    return dl


def _rdrop_group_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[0])


def _rdrop_group_backward(ctx, grads):
    logits = list(ctx.saved_tensors)
    dl = rdrop_group_bwd_op([g if g is not None else torch.zeros((), device=logits[0].device)
                             for g in grads], logits)
    return [d.to(l.dtype) for d, l in zip(dl, logits)]


rdrop_group_op.register_autograd(_rdrop_group_backward, setup_context=_rdrop_group_setup)


# ------------------------------------------------------------------------------------------------
# public interface
# ------------------------------------------------------------------------------------------------
def circle_losses(logits: Sequence[Tensor], labels: Sequence[Tensor],
                  weights: Optional[Sequence[Tensor]] = None) -> List[Tensor]:
    """One scalar per fold: ``multi_circle_loss(logits[k], labels[k]).mean()`` (cmu-mosei,
    rencecps and Ren-MME's ``multi_loss``), or with ``weights[k]`` (one weight per row)
    ``(multi_circle_loss(logits[k], labels[k]) * weights[k]).mean()`` (others/realformer.py:312
    with the window mask).  One launch forward and one backward for all folds."""
    if len(labels) != len(logits) or (weights is not None and len(weights) != len(logits)):
        raise ValueError("logits, labels and weights must have one entry per fold")
    dev = logits[0].device
    ws = [torch.empty(0, device=dev)] * len(logits) if weights is None else list(weights)
    return list(circle_group_op(list(logits), list(labels), ws))


def rdrop_kl(logits: Sequence[Tensor]) -> List[Tensor]:
    """``ren_mme.rdrop_kl(logits[k])`` of every fold, one launch forward and one backward."""
    return list(rdrop_group_op(list(logits)))


def forward(models: Sequence[torch.nn.Module], inputs: Sequence[Sequence]) -> List[Tensor]:
    """``[models[k](*inputs[k]) for k]`` as one grouped forward (and backward) for all folds; see
    the module docstring."""
    models, inputs = list(models), [tuple(a) for a in inputs]
    if len(models) != len(inputs):
        raise ValueError(f"{len(models)} models but {len(inputs)} input tuples")
    _check_members(models, _FAMILIES)
    if len({m.training for m in models}) > 1:
        raise ValueError("all models must be in the same train / eval mode")
    for args in inputs:
        ops._need_cuda(*[a for a in args if isinstance(a, Tensor)])
    m0 = models[0]
    if isinstance(m0, Multi_class):
        return _multi_class(models, inputs)
    if isinstance(m0, State_Transfer):
        return _state_transfer(models, inputs)
    if isinstance(m0, Concat_Linear):
        return _concat_linear(models, inputs)
    return _bilinear(models, inputs)


def _unify(u, x3, poss=(None, None, None)):
    return [(x, c.weight, p) for x, c, p in zip(x3, (u.linguistic, u.visual, u.acoustic), poss)]


def _project(probs, drop_p=0.0):
    """``drop_p`` > 0: the projections' own dropout (between the GEMM and the position add) in
    the grouped GEMM's epilogue, one seed per call."""
    return project([x for x, _, _ in probs], [w for _, w, _ in probs], None,
                   [p for _, _, p in probs], bf16=is_bf16(), drop_p=drop_p,
                   seed=ops.next_dropout_seed() if drop_p > 0 else 0)


def _heads(models, pooled_last, pooled_this, w_last, w_this, norms):
    lin = linear_group([x for pair in zip(pooled_last, pooled_this) for x in pair],
                       [w for pair in zip(w_last, w_this) for w in pair])
    return list(bilinear_group_op(lin[1::2], lin[0::2], [m.trans for m in models],
                                  [n.weight for n in norms], [n.bias for n in norms],
                                  [m.out.weight for m in models], [m.out.bias for m in models])
                [:len(models)])


def _bilinear(models, inputs):
    """cmu-mosei/run.py:321-339 / Ren-MME/run.py:273-292 for every fold: two towers each."""
    towers = []                     # (tower module, (l, v, a), masks) in fold-major order
    for m, args in zip(models, inputs):
        if isinstance(m, Concat_Trans):
            l, v, a, lm, vm, am = args
            for i, t in enumerate((m.intensity, m.stimulation)):
                towers.append((t, (l[:, i], v[:, i], a[:, i]),
                               {"l": as_mask(lm[:, i]), "v": as_mask(vm[:, i]),
                                "a": as_mask(am[:, i])}))
        else:
            for t, (x, y, z) in zip((m.intensity, m.stimulation), ((0, 4, 8), (2, 6, 10))):
                towers.append((t, (args[x], args[y], args[z]),
                               {"l": as_mask(args[x + 1]), "v": as_mask(args[y + 1]),
                                "a": as_mask(args[z + 1])}))
    ys = _project([p for t, x3, _ in towers for p in _unify(t.unify_dimension, x3)])
    if isinstance(models[0], Base_model):
        # Ren-MME/run.py:158-166: each tower's LayerNorm over its three projections, all towers of
        # all folds in one grouped call
        lns = [t.unify_dimension.norm1 for t, _, _ in towers for _ in range(3)]
        ys = ln_group(ys, [u.weight for u in lns], [u.bias for u in lns])
    trunk = [(t.multimodal_blocks, {"l": ys[3 * i], "v": ys[3 * i + 1], "a": ys[3 * i + 2]}, mk)
             for i, (t, _, mk) in enumerate(towers)]
    pooled = pool_group(fusion_trunk_multi(trunk, towers[0][0].n_layers, keep_all=True,
                                           pool=False))
    norms = [m.norm1 if isinstance(m, Concat_Trans) else m.norm3 for m in models]
    return _heads(models, pooled[0::2], pooled[1::2],
                  [m.intensity.classifier.weight for m in models],
                  [m.stimulation.classifier.weight for m in models], norms)


def _concat_linear(models, inputs):
    """rencecps/run.py:130-148 for every fold: feat (B, 2, F); the halves are read in place."""
    feats = [args[0] for args in inputs]
    return _heads(models, [f[:, 0] for f in feats], [f[:, 1] for f in feats],
                  [m.intensity.weight for m in models], [m.stimulation.weight for m in models],
                  [m.norm for m in models])


def _state_transfer(models, inputs):
    """others/realformer.py:266-286 for every fold: the B*P windows folded into the batch."""
    fs = [m.feature for m in models]
    shapes, masks, probs = [], [], []
    for f, args in zip(fs, inputs):
        l, v, a, lm, vm, am = args
        B, P = l.shape[0], l.shape[1]
        shapes.append((B, P))
        fold = lambda t, B=B, P=P: t.reshape(B * P, *t.shape[2:])
        l, v, a = fold(l), fold(v), fold(a)
        masks.append({"l": as_mask(fold(lm)), "v": as_mask(fold(vm)), "a": as_mask(fold(am))})
        probs += _unify(f.unify_dimension, (l, v, a), f.positions(l, v, a))
    ys = _project(probs, float(fs[0].unify_dimension.drop.p) if fs[0].training else 0.0)
    trunk = [(f.multimodal_blocks, {"l": ys[3 * i], "v": ys[3 * i + 1], "a": ys[3 * i + 2]},
              masks[i]) for i, f in enumerate(fs)]
    pooled = pool_group(fusion_trunk_multi(trunk, fs[0].n_layers, keep_all=False, pool=False))
    h = linear_group(pooled, [f.fully_connected.weight for f in fs],
                     [f.fully_connected.bias for f in fs])
    h = ln_group(h, [f.normalization.weight for f in fs], [f.normalization.bias for f in fs],
                 relu=True)
    p = float(fs[0].drop.p)
    if fs[0].training and p > 0:
        h = list(dropout_group_op(h, p, ops.next_dropout_seed()))
    o = linear_group(h, [m.classifier.weight for m in models], [m.classifier.bias for m in models])
    return list(state_transfer_group_op([x.view(B, P, -1) for x, (B, P) in zip(o, shapes)],
                                        [m.trans for m in models]))


def _multi_class(models, inputs):
    """robot_demo.py:377-441 for every fold: five biased projections per fold (the three visual
    ones write the column thirds of one (B, L, d) stream) with their dropout and position tables
    as ONE grouped projection, every fold's trunk as one tower of ``fusion_trunk_multi``, one
    grouped pooling and one grouped classifier linear."""
    xs, ws, bs, poss, spans, masks = [], [], [], [], [], []
    for m, args in zip(models, inputs):
        if len(args) != 8:
            raise ValueError(f"Multi_class takes 8 inputs per fold, got {len(args)}")
        l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask = args
        u = m.unify_dimension
        for x, c in zip((l, v_256, v_512, v_1024, a),
                        (u.linguistic, u.visual_256, u.visual_512, u.visual_1024, u.acoustic)):
            xs.append(x)
            ws.append(c.weight)
            bs.append(c.bias)
        spans += [1, 3, 1]
        poss += [e.position_embeddings.weight for e in
                 (m.linguistic_position, m.visual_position, m.acoustic_position)]
        masks.append({"l": as_mask(l_mask), "v": as_mask(v_mask), "a": as_mask(a_mask)})
    m0 = models[0]
    p = float(m0.unify_dimension.drop.p) if m0.training else 0.0
    ys = project_cat(xs, ws, bs, spans, poss, is_bf16(), p,
                     ops.next_dropout_seed() if p > 0 else 0)
    trunk = [(m.multimodal_blocks, {"l": ys[3 * i], "v": ys[3 * i + 1], "a": ys[3 * i + 2]},
              masks[i]) for i, m in enumerate(models)]
    pooled = pool_group(fusion_trunk_multi(trunk, m0.n_layers, keep_all=True, pool=False))
    return linear_group(pooled, [m.classifier.weight for m in models],
                        [m.classifier.bias for m in models])
