"""Grouped fusion-trunk layers: layer i of ALL chains as one autograd node and one launch per kernel.

The nine chains of a fusion trunk (others/realformer.py:232-257, cmu-mosei/run.py:278-313,
Ren-MME/run.py:230-265, robot_demo.py:399-434) are mutually independent (they share only their
read-only inputs l, v, a), and so are the two towers of ``Concat_Trans`` / ``Base_model`` and the
members of an inference ensemble.  The reference walks them one after the other: 9 x n_layers
blocks x ~18 launches of microsecond kernels per trunk.  Here layer i of every chain is ONE custom
op whose forward / backward issue one GROUPED launch per kernel kind (weight casts, Q|KV
projections, attention, output projection, LayerNorm, FFN, weight gradients ...) with the
per-problem pointers in a table - ~8 launches per layer forward and ~10 backward, independent of
the number of chains.  A block called on its own (``blocks.py``, K = V) is a group of one problem.

Problem g of a group: q-stream ``qs[g]`` (B, Lq_g, d), source ``kvs[g]`` (B, Lk_g, d) (K = V, like
every caller in the reference), mask ``masks[g]`` (B, Lk_g), previous scores ``s_prevs[g]`` or none,
and the block's parameters.  Lengths and batch sizes may differ between problems; d, n_heads and the
block type are shared.  Score tensors are allocated with a row stride padded to 8 elements
(``ops.score_stride``) when the mma.sync attention kernels take the group.

float32 (parity) mode runs the same code with the per-problem launchers (no grouped fp32 GEMM /
attention kernels exist; that mode is not the performance path).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch
from torch import Tensor

from . import _lib, ops
from .ops import BF, F32, LN_EPS, _act_dtype, _arr, _p, _weight


def _call(name, *args):          # late-bound: tests stub ops._call / ops._stream
    return ops._call(name, *args)


def _stream():
    return ops._stream()

N_FULL = 15      # wq wk wv wo  n1w n1b n2w n2b  f1w f1b f2w f2b  a b c
N_LITE = 5       # wo(proj) wm(minus, (d,2d)) nw nb c


def _e(dev) -> Tensor:
    return torch.empty(0, device=dev)


def _opt(t: Tensor) -> Optional[Tensor]:
    return t if t.numel() else None


# ------------------------------------------------------------------------------------------------
# grouped LayerNorm / column sums (one library call per group, which launches per 40 problems;
# per-problem launches when the vector kernels do not take a shape)
# ------------------------------------------------------------------------------------------------
def _vpa(ts):
    return _arr(C.c_void_p, [_p(t) for t in ts])


def ln_fwd_group(bf16: bool, res, xs, gates, gammas, betas, relu=False):
    """y_g = act(LN(res_g + gate_g * x_g)); returns ([y], [stat (2, M)])."""
    ys = [torch.empty_like(x) for x in xs]
    stats = [torch.empty(2, x.numel() // x.shape[-1], dtype=F32, device=x.device) for x in xs]
    d = xs[0].shape[-1]
    ok = False
    if len(xs) > 1 and all(x.is_contiguous() for x in xs) and \
            all(r is None or r.is_contiguous() for r in res):
        ok = ops._try_call(
            f"mmemo_add_ln_fwd_grouped_{'bf16' if bf16 else 'f32'}",
            len(xs), _vpa(res), _vpa(xs), _vpa(gates), _vpa(gammas), _vpa(betas), _vpa(ys),
            _vpa([s[0] for s in stats]), _vpa([s[1] for s in stats]),
            _arr(C.c_int64, [x.numel() // d for x in xs]), d, LN_EPS, int(relu), _stream())
    if not ok:
        for i, x in enumerate(xs):
            ys[i], stats[i] = ops._add_ln_fwd(bf16, res[i], x, gates[i], gammas[i], betas[i], relu)
    return ys, stats


def ln_bwd_group(bf16: bool, dys, res, xs, gates, gammas, stats, want_dres: bool, dpars,
                 dxsums=None):
    """Backward of ln_fwd_group (no ReLU).  dpars[g] = zero-initialised float32 [1 + 2d] slot
    (dgate | dgamma | dbeta); dxsums[g] (optional, zero-initialised [d]) receives colsum(dx).
    Returns ([dres] or Nones, [dx])."""
    d = xs[0].shape[-1]
    dxs = [torch.empty_like(x) for x in xs]
    dres = [torch.empty_like(x) if want_dres else None for x in xs]
    ok = False
    if len(xs) > 1 and all(t.is_contiguous() for t in list(xs) + list(dys)) and \
            all(r is None or r.is_contiguous() for r in res):
        ok = ops._try_call(
            f"mmemo_add_ln_bwd_grouped_{'bf16' if bf16 else 'f32'}",
            len(xs), _vpa(dys), _vpa(res), _vpa(xs), _vpa(gates), _vpa(gammas),
            _vpa([s[0] for s in stats]), _vpa([s[1] for s in stats]), _vpa(dres), _vpa(dxs),
            _vpa([dp if g is not None else None for dp, g in zip(dpars, gates)]),
            _vpa([dp[1:] for dp in dpars]), _vpa([dp[1 + d:] for dp in dpars]),
            _vpa(dxsums if dxsums is not None else [None] * len(xs)),
            _arr(C.c_int64, [x.numel() // d for x in xs]), d, _stream())
    if not ok:
        for i, x in enumerate(xs):
            dres[i], dxs[i], _ = ops._add_ln_bwd(
                bf16, dys[i], res[i], x, gates[i], gammas[i], None, stats[i], False, want_dres,
                dpar=dpars[i], dxsum=None if dxsums is None else dxsums[i])
    return dres, dxs


def colsum_group(bf16: bool, xs, outs):
    """outs[g] (zero-initialised float32 [N]) += column sums of xs[g] (M_g, N)."""
    N = xs[0].shape[-1]
    if bf16 and len(xs) > 1 and N % 8 == 0 and all(x.is_contiguous() for x in xs):
        if ops._try_call("mmemo_colsum_grouped_bf16", len(xs), _vpa(xs), _vpa(outs),
                         _arr(C.c_int64, [x.numel() // N for x in xs]), N, _stream()):
            return
    for x, o in zip(xs, outs):
        ops._rowsum(bf16, x.reshape(-1, N), o)


def merge_shared_grads(bf16: bool, inputs, grads):
    """``grads[i]`` is the gradient of ``inputs[i]`` (None = undefined).  Entries whose inputs are
    the SAME tensor (a modality stream is the query of three chains and the source of three) are
    summed into the first one's buffer with one grouped launch; the other entries become None, so
    autograd receives one gradient per distinct tensor instead of adding them pairwise."""
    groups = {}
    for i, (x, gx) in enumerate(zip(inputs, grads)):
        if gx is not None:
            groups.setdefault((x.data_ptr(), tuple(x.shape), tuple(x.stride()), x.dtype), []).append(i)
    multi = [ix for ix in groups.values() if len(ix) > 1]
    if not multi:
        return list(grads)
    out = list(grads)
    todo = []
    for ix in multi:
        gs = [grads[i] for i in ix]
        if len(ix) > 8 or not all(g_.is_contiguous() and g_.dtype == gs[0].dtype and
                                  g_.data_ptr() % 16 == 0 for g_ in gs):
            tot = gs[0]
            for g_ in gs[1:]:
                tot = tot + g_
            out[ix[0]] = tot
        else:
            todo.append(gs)
        for i in ix[1:]:
            out[i] = None
    for dt in dict.fromkeys(gs[0].dtype for gs in todo):
        part = [gs for gs in todo if gs[0].dtype == dt]
        _call(f"mmemo_sum_grouped_{'bf16' if dt == BF else 'f32'}", len(part),
              _vpa([gs[0] for gs in part]), _arr(C.c_int, [len(gs) for gs in part]),
              _vpa([g_ for gs in part for g_ in gs]), _arr(C.c_int64, [gs[0].numel() for gs in part]),
              _stream())
    return out


# ------------------------------------------------------------------------------------------------
# grouped attention core
# ------------------------------------------------------------------------------------------------
def _mma_group_ok(bf16: bool, qs, kvs, H: int, same_kv: bool) -> bool:
    """True when the group's attention runs as grouped mma.sync launches (forward and backward);
    the scores of such a group use the padded row stride."""
    # A group of one problem (a block called on its own) takes the per-problem entry points
    # instead: they pick the tcgen05 kernels where those are faster (resattn_tc.cu, and
    # resattn_tc2.cu for Lk = 256, which the check below does not exclude), and its scores keep
    # the reference's unpadded (B, H, Lq, Lk) layout.  Fusion trunks have at least 9 problems.
    if not bf16 or len(qs) < 2:
        return False
    lib = _lib.load()
    d = qs[0].shape[-1]
    hd = d // H
    for q, kv in zip(qs, kvs):
        Lq, Lk = q.shape[1], kv.shape[1]
        if lib.mmemo_resattn_uses_tensor_cores(Lq, Lk, hd, d):
            return False        # hd = 64, L = 128: the tcgen05 kernels are faster
        if not (lib.mmemo_resattn_uses_mma(Lq, Lk, hd, d, int(same_kv), 0) and
                lib.mmemo_resattn_uses_mma(Lq, Lk, hd, d, int(same_kv), 1)):
            return False
    return True


def attn_fwd_group(bf16, qs, ks, vs, masks, s_prevs, cs, H, want_s, grouped):
    """Returns ([o], [s or None], [stat]).  ``grouped``: one mma.sync launch, padded score stride."""
    dt = _act_dtype(bf16)
    os_, ss, stats, probs = [], [], [], []
    if not grouped:
        for g, q in enumerate(qs):
            o, s, st = ops._attn_fwd(bf16, q, ks[g], vs[g], masks[g], s_prevs[g], cs[g], H, want_s)
            os_.append(o), ss.append(s), stats.append(st)
        return os_, ss, stats
    for g, q in enumerate(qs):
        B, Lq, d = q.shape
        Lk = ks[g].shape[1]
        lds = ops.score_stride(Lk)
        o = torch.empty(B, Lq, d, dtype=dt, device=q.device)
        s = torch.empty(B, H, Lq, lds, dtype=dt, device=q.device) if want_s else None
        st = torch.empty(B, H, Lq, 2, dtype=F32, device=q.device)
        sp = s_prevs[g]
        assert sp is None or sp.shape[-1] == lds, "previous scores must use the padded stride"
        probs.append(ops._attn_problem(q, ks[g], vs[g], masks[g], sp, cs[g], s, o, st, H, lds))
        os_.append(o), ss.append(s), stats.append(st)
    if not ops._attn_group_call("mmemo_resattn_fwd_grouped_bf16", probs):
        raise RuntimeError("grouped attention forward rejected a shape it reported as supported")
    return os_, ss, stats


def attn_bwd_group(bf16, dos, qs, ks, vs, masks, ss, s_prevs, cs, ds_nexts, os_, stats, H, dqs, dks,
                   dvs, want_dsprev, dcs, grouped):
    """Fills dqs / dks / dvs; returns [ds_prev or None].  dcs[g]: zero-initialised float32 [1]."""
    dt = _act_dtype(bf16)
    out = []
    if not grouped:
        for g, q in enumerate(qs):
            dsp, _ = ops._attn_bwd(bf16, dos[g], q, ks[g], vs[g], masks[g], ss[g], s_prevs[g], cs[g],
                                   ds_nexts[g], os_[g], stats[g], H, dqs[g], dks[g], dvs[g],
                                   want_dsprev, dc_out=dcs[g])
            out.append(dsp)
        return out
    probs = []
    for g, q in enumerate(qs):
        B, Lq, d = q.shape
        Lk = ks[g].shape[1]
        lds = ops.score_stride(Lk)
        sp = s_prevs[g]
        dsp = None
        if sp is not None and want_dsprev:
            dsp = torch.empty(B, H, Lq, lds, dtype=dt, device=q.device)
        probs.append(ops._attn_problem(q, ks[g], vs[g], masks[g], sp, cs[g], None, os_[g], stats[g],
                                       H, lds, d_o=dos[g], s=ss[g], ds_next=ds_nexts[g], dq=dqs[g],
                                       dk=dks[g], dv=dvs[g], ds_prev=dsp,
                                       dc=dcs[g] if sp is not None else None))
        out.append(dsp)
    if not ops._attn_group_call("mmemo_resattn_bwd_grouped_bf16", probs):
        raise RuntimeError("grouped attention backward rejected a shape it reported as supported")
    return out


# ------------------------------------------------------------------------------------------------
# mmemo::trunk_full — layer i of G chains of FULL RealFormer blocks
#   (others/realformer.py:182-209 == robot_demo.py:347-374), one node
# outputs per problem (12): h2 s qp kvp o stat x h1 st1 f1 f2 st2
# ------------------------------------------------------------------------------------------------
FULL_OUT = 12


@torch.library.custom_op("mmemo::trunk_full", mutates_args=())
def trunk_full_op(qs: Sequence[Tensor], kvs: Sequence[Tensor], masks: Sequence[Tensor],
                  s_prevs: Sequence[Tensor], params: Sequence[Tensor], n_heads: int, bf16: bool,
                  emit_s: bool, drop_p: float, drop_seed: int) -> List[Tensor]:
    """``drop_p`` > 0: the block's two training dropouts — on the projected attention output
    (others/realformer.py:203  robot_demo.py:368) and at the end of the FFN (:167 / :333) — as one
    in-place grouped launch each, masks regenerated from ``drop_seed`` in the backward."""
    ops._need_cuda(*qs, *kvs)
    G = len(qs)
    dt, dev = _act_dtype(bf16), qs[0].device
    d = qs[0].shape[-1]
    P = [params[N_FULL * g:N_FULL * (g + 1)] for g in range(G)]
    qs = [q.contiguous() for q in qs]
    kvs = [qs[g] if kvs[g].data_ptr() == qs[g].data_ptr() and kvs[g].shape == qs[g].shape
           else kvs[g].contiguous() for g in range(G)]
    masks_ = [_opt(m) for m in masks]
    sp = [s_prevs[g] if len(s_prevs) else None for g in range(G)]
    if bf16:   # every bf16 weight shadow of the layer in one cast launch
        ops.shadow_bf16_block([grp for p in P for grp in
                               ([p[0]], [p[1], p[2]], [p[3]], [p[8]], [p[10]])])
    dff = P[0][8].shape[0]
    # Q projection and fused [K|V] projection (N = 2d) of every chain: one grouped GEMM
    qps = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    kvps = [torch.empty(*kv.shape[:2], 2 * d, dtype=dt, device=dev) for kv in kvs]
    items = []
    for g in range(G):
        items.append((qs[g], _weight(bf16, P[g][0]), None, qps[g].view(-1, d), False))
        items.append((kvs[g], _weight(bf16, P[g][1], P[g][2]), None, kvps[g].view(-1, 2 * d), False))
    ops._linear_fwd_group(bf16, items)
    ks = [t[..., :d] for t in kvps]
    vs = [t[..., d:] for t in kvps]
    grouped = _mma_group_ok(bf16, qs, kvs, n_heads, False)
    os_, ss, stats = attn_fwd_group(bf16, qps, ks, vs, masks_, sp, [p[14] for p in P], n_heads,
                                    emit_s, grouped)
    # output projection, gated residual + LN1
    xs = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_fwd_group(bf16, [(os_[g], _weight(bf16, P[g][3]), None, xs[g].view(-1, d), False)
                                 for g in range(G)])
    ops._dropout_group(xs, xs, drop_p, ops.site_seeds(drop_seed, G, 0))
    h1s, st1s = ln_fwd_group(bf16, qs, xs, [p[12] for p in P], [p[4] for p in P],
                             [p[5] for p in P])
    # FFN (bias + ReLU fused in the first GEMM's epilogue), gated residual + LN2
    f1s = [torch.empty(*q.shape[:2], dff, dtype=dt, device=dev) for q in qs]
    f2s = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_fwd_group(bf16, [(h1s[g], _weight(bf16, P[g][8]), P[g][9], f1s[g].view(-1, dff), True)
                                 for g in range(G)])
    ops._linear_fwd_group(bf16, [(f1s[g], _weight(bf16, P[g][10]), P[g][11], f2s[g].view(-1, d), False)
                                 for g in range(G)])
    ops._dropout_group(f2s, f2s, drop_p, ops.site_seeds(drop_seed, G, 1))
    h2s, st2s = ln_fwd_group(bf16, h1s, f2s, [p[13] for p in P], [p[6] for p in P],
                             [p[7] for p in P])
    out = []
    for g in range(G):
        out += [h2s[g], ss[g] if ss[g] is not None else _e(dev), qps[g], kvps[g], os_[g], stats[g],
                xs[g], h1s[g], st1s[g], f1s[g], f2s[g], st2s[g]]
    return out


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64          # floats: 256-byte aligned


def _full_zlen(d: int, dff: int) -> int:
    return _pad64(2 * (1 + 2 * d) + d + dff + 1) + 4 * d * d + 2 * dff * d


def _full_zviews(z: Tensor, d: int, dff: int):
    """Per-problem zero buffer: [dp2 (1+2d) | dp1 (1+2d) | db_f2 (d) | db_f1 (dff) | dc (1) | pad
    to 256 B] then dWq (d,d) dWkv (2d,d) dWo (d,d) dWf1 (dff,d) dWf2 (d,dff)."""
    dp2, dp1 = z[:1 + 2 * d], z[1 + 2 * d:2 * (1 + 2 * d)]
    o = 2 * (1 + 2 * d)
    db_f2, db_f1, dc = z[o:o + d], z[o + d:o + d + dff], z[o + d + dff:o + d + dff + 1]
    ws, o = [], _pad64(o + d + dff + 1)
    for sh in [(d, d), (2 * d, d), (d, d), (dff, d), (d, dff)]:
        ws.append(z[o:o + sh[0] * sh[1]].view(sh))
        o += sh[0] * sh[1]
    return dp2, dp1, db_f2, db_f1, dc, ws


def _full_pgrads(z: Tensor, d: int, dff: int) -> List[Tensor]:
    """The gradient of every parameter of a full block (order: N_FULL) as a view of its buffer."""
    dp2, dp1, db_f2, db_f1, dc, ws = _full_zviews(z, d, dff)
    return [ws[0], ws[1][:d], ws[1][d:], ws[2], dp1[1:1 + d], dp1[1 + d:], dp2[1:1 + d], dp2[1 + d:],
            ws[3], db_f1, ws[4], db_f2, dp1[0:1], dp2[0:1], dc]


def full_grad_unit(params: Sequence[Tensor]):
    """(key parameter, [(parameter, offset in floats)], total floats) of a full block's gradient
    buffer, for dp.GradReducer; the offsets are those of the views the backward hands to autograd."""
    d, dff = params[0].shape[0], params[8].shape[0]
    z = torch.empty(_full_zlen(d, dff), device="meta")
    offsets = [g.storage_offset() for g in _full_pgrads(z, d, dff)]
    return params[0], list(zip(params, offsets)), z.numel()


@torch.library.custom_op("mmemo::trunk_full_bwd", mutates_args=())
def trunk_full_bwd_op(dh2s: Sequence[Tensor], ds_nexts: Sequence[Tensor], qs: Sequence[Tensor],
                      kvs: Sequence[Tensor], masks: Sequence[Tensor], s_prevs: Sequence[Tensor],
                      saved: Sequence[Tensor], params: Sequence[Tensor], n_heads: int, bf16: bool,
                      need_dsprev: bool, drop_p: float, drop_seed: int) -> List[Tensor]:
    """Returns per problem [dq, dkv, ds_prev] (empty placeholders where undefined) followed by ONE
    float32 buffer holding every parameter gradient of the group (layout: _full_zviews)."""
    G = len(qs)
    dt, dev = _act_dtype(bf16), qs[0].device
    d = qs[0].shape[-1]
    P = [params[N_FULL * g:N_FULL * (g + 1)] for g in range(G)]
    S = [saved[(FULL_OUT - 1) * g:(FULL_OUT - 1) * (g + 1)] for g in range(G)]
    # saved per problem: s qp kvp o stat x h1 st1 f1 f2 st2
    ss = [_opt(s[0]) for s in S]
    qps, kvps, os_, stats = [s[1] for s in S], [s[2] for s in S], [s[3] for s in S], [s[4] for s in S]
    xs, h1s, st1s = [s[5] for s in S], [s[6] for s in S], [s[7] for s in S]
    f1s, f2s, st2s = [s[8] for s in S], [s[9] for s in S], [s[10] for s in S]
    dff = P[0][8].shape[0]
    qs = [q.contiguous() for q in qs]
    same = [kvs[g].data_ptr() == qs[g].data_ptr() and kvs[g].shape == qs[g].shape for g in range(G)]
    kvs = [qs[g] if same[g] else kvs[g].contiguous() for g in range(G)]
    masks_ = [_opt(m) for m in masks]
    sp = [s_prevs[g] if len(s_prevs) else None for g in range(G)]
    dsn = [_opt(t) for t in ds_nexts]
    dh2s = [t.contiguous() for t in dh2s]
    zlen = _full_zlen(d, dff)
    # data parallel: every block's buffer is a region of an all-reduce bucket, zero-filled by the
    # reducer (dp.GradReducer, ops.register_zbuf_dest) - no fill here, no gradient copies later
    zbs = ops.claim_zbufs([p[0] for p in P], zlen)
    if zbs is None:
        zall = torch.zeros(G * zlen, dtype=F32, device=dev)      # ONE fill for every "+=" output
        zbs = [zall[g * zlen:(g + 1) * zlen] for g in range(G)]
    else:
        zall = _e(dev)
    Z = [_full_zviews(zbs[g], d, dff) for g in range(G)]
    # LN2: h2 = LN(h1 + b*f2); colsum(df2) = the FFN-2 bias gradient comes out of the same pass
    if drop_p > 0:   # the FFN-2 bias sees the gradient BEFORE the dropout: mask first, then column sums
        dh1s, df2s = ln_bwd_group(bf16, dh2s, h1s, f2s, [p[13] for p in P], [p[6] for p in P], st2s,
                                  True, [z[0] for z in Z])
        ops._dropout_group(df2s, df2s, drop_p, ops.site_seeds(drop_seed, G, 1))
        colsum_group(bf16, [t.view(-1, d) for t in df2s], [z[2] for z in Z])
    else:
        dh1s, df2s = ln_bwd_group(bf16, dh2s, h1s, f2s, [p[13] for p in P], [p[6] for p in P], st2s,
                                  True, [z[0] for z in Z], [z[2] for z in Z])
    # FFN backward: df1 = (df2 W2) * (f1 > 0) fused in the epilogue; dh1 += df1 W1
    df1s = [torch.empty(f.shape, dtype=dt, device=dev) for f in f1s]
    ops._linear_bwd_x_group(bf16, [(df2s[g], _weight(bf16, P[g][10]), df1s[g].view(-1, dff), False,
                                    f1s[g].view(-1, dff)) for g in range(G)])
    ops._linear_bwd_x_group(bf16, [(df1s[g], _weight(bf16, P[g][8]), dh1s[g].view(-1, d), True)
                                   for g in range(G)])
    colsum_group(bf16, [t.view(-1, dff) for t in df1s], [z[3] for z in Z])
    # LN1: h1 = LN(q + a*x)
    dqs, dxs = ln_bwd_group(bf16, dh1s, qs, xs, [p[12] for p in P], [p[4] for p in P], st1s, True,
                            [z[1] for z in Z])
    ops._dropout_group(dxs, dxs, drop_p, ops.site_seeds(drop_seed, G, 0))
    # output projection
    dos = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_bwd_x_group(bf16, [(dxs[g], _weight(bf16, P[g][3]), dos[g].view(-1, d), False)
                                   for g in range(G)])
    # attention core
    dqps = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    dkvps = [torch.empty(t.shape, dtype=dt, device=dev) for t in kvps]
    grouped = _mma_group_ok(bf16, qs, kvs, n_heads, False)
    dsps = attn_bwd_group(bf16, dos, qps, [t[..., :d] for t in kvps], [t[..., d:] for t in kvps],
                          masks_, ss, sp, [p[14] for p in P], dsn, os_, stats, n_heads, dqps,
                          [t[..., :d] for t in dkvps], [t[..., d:] for t in dkvps], need_dsprev,
                          [z[4] for z in Z], grouped)
    # projections: dq += dqp Wq ; dkv = dkvp [Wk;Wv]  (same tensor for q and kv: two ordered passes)
    dkvs = [None if same[g] else torch.empty(kvs[g].shape, dtype=dt, device=dev) for g in range(G)]
    first, second = [], []
    for g in range(G):
        first.append((dqps[g], _weight(bf16, P[g][0]), dqs[g].view(-1, d), True))
        kvitem = (dkvps[g], _weight(bf16, P[g][1], P[g][2]),
                  (dqs[g] if same[g] else dkvs[g]).view(-1, d), same[g])
        (second if same[g] else first).append(kvitem)
    ops._linear_bwd_x_group(bf16, first)
    if second:
        ops._linear_bwd_x_group(bf16, second)
    # the five weight gradients of every chain: one grouped launch per 48 problems
    items = []
    for g in range(G):
        w = Z[g][5]
        items += [(df2s[g].view(-1, d), f1s[g].view(-1, dff), w[4]),
                  (df1s[g].view(-1, dff), h1s[g].view(-1, d), w[3]),
                  (dxs[g].view(-1, d), os_[g].view(-1, d), w[2]),
                  (dqps[g].view(-1, d), qs[g].view(-1, d), w[0]),
                  (dkvps[g].view(-1, 2 * d), kvs[g].view(-1, d), w[1])]
    ops._linear_bwd_w_group(bf16, items, zeroed=True)
    # one gradient per distinct input tensor (shared modality streams): grouped sum, not autograd adds
    merged = merge_shared_grads(bf16, list(qs) + list(kvs), list(dqs) + list(dkvs))
    dqs, dkvs = merged[:G], merged[G:]
    out = []
    for g in range(G):
        out += [dqs[g] if dqs[g] is not None else _e(dev), dkvs[g] if dkvs[g] is not None else _e(dev),
                dsps[g] if dsps[g] is not None else _e(dev)]
    return out + [zall]


def _trunk_full_setup(ctx, inputs, output):
    qs, kvs, masks, s_prevs, params, H, bf16, emit_s, drop_p, drop_seed = inputs
    G = len(qs)
    ctx.G, ctx.cfg, ctx.has_prev = G, (H, bf16), len(s_prevs) > 0
    ctx.drop = (drop_p, drop_seed)
    ctx.n_params = len(params)
    saved = []
    for g in range(G):
        saved += list(output[FULL_OUT * g + 1:FULL_OUT * (g + 1)])
    ctx.save_for_backward(*qs, *kvs, *masks, *s_prevs, *saved, *params)
    ctx.set_materialize_grads(False)


def _trunk_full_backward(ctx, grads):
    G = ctx.G
    H, bf16 = ctx.cfg
    t = list(ctx.saved_tensors)
    qs, kvs, masks = t[:G], t[G:2 * G], t[2 * G:3 * G]
    o = 3 * G
    s_prevs = t[o:o + G] if ctx.has_prev else []
    o += G if ctx.has_prev else 0
    ns = (FULL_OUT - 1) * G
    saved, params = t[o:o + ns], t[o + ns:]
    dev = qs[0].device
    dh2s, dsn = [], []
    for g in range(G):
        gh, gs = grads[FULL_OUT * g], grads[FULL_OUT * g + 1]
        dh2s.append(gh if gh is not None else torch.zeros_like(qs[g]))
        dsn.append(gs if gs is not None else _e(dev))
    need_dsprev = ctx.has_prev and any(ctx.needs_input_grad[3])
    res = trunk_full_bwd_op(dh2s, dsn, qs, kvs, masks, s_prevs, saved, params, H, bf16, need_dsprev,
                            *ctx.drop)
    zall = res[-1]
    d = qs[0].shape[-1]
    dff = params[8].shape[0]
    zlen = _full_zlen(d, dff)
    dqs, dkvs, dsps, pgrads = [], [], [], []
    for g in range(G):
        dq, dkv, dsp = res[3 * g:3 * g + 3]
        dqs.append(dq if dq.numel() else None)
        dkvs.append(dkv if dkv.numel() else None)
        dsps.append(dsp if dsp.numel() else None)
        zb = zall[g * zlen:(g + 1) * zlen] if zall.numel() else ops.zbuf_region(params[N_FULL * g])
        pg = _full_pgrads(zb, d, dff)
        pgrads += pg[:-1] + [pg[-1] if ctx.has_prev else None]
    n_prev = G if ctx.has_prev else 0
    return (dqs, dkvs, [None] * G, dsps if need_dsprev else [None] * n_prev, pgrads, None, None,
            None, None, None)


trunk_full_op.register_autograd(_trunk_full_backward, setup_context=_trunk_full_setup)


# ------------------------------------------------------------------------------------------------
# mmemo::trunk_lite — layer i of G chains of LITE blocks (cmu-mosei/run.py:236-262,
#   Ren-MME/run.py:188-214): attention on the raw streams, proj, LN(minus([q | x]))
# outputs per problem (7): out s o stat x y st
# ------------------------------------------------------------------------------------------------
LITE_OUT = 7


@torch.library.custom_op("mmemo::trunk_lite", mutates_args=())
def trunk_lite_op(qs: Sequence[Tensor], kvs: Sequence[Tensor], masks: Sequence[Tensor],
                  s_prevs: Sequence[Tensor], params: Sequence[Tensor], n_heads: int, bf16: bool,
                  emit_s: bool, drop_p: float, drop_seed: int) -> List[Tensor]:
    """``drop_p`` > 0: the lite block's two training dropouts — ``drop(proj(att))`` and
    ``drop(norm(minus(..)))`` (Ren-MME/run.py:208,212  cmu-mosei/run.py:256,260) — one in-place
    grouped launch each."""
    ops._need_cuda(*qs, *kvs)
    G = len(qs)
    dt, dev = _act_dtype(bf16), qs[0].device
    d = qs[0].shape[-1]
    P = [params[N_LITE * g:N_LITE * (g + 1)] for g in range(G)]
    qs = [q.contiguous() for q in qs]
    kvs = [qs[g] if kvs[g].data_ptr() == qs[g].data_ptr() and kvs[g].shape == qs[g].shape
           else kvs[g].contiguous() for g in range(G)]
    masks_ = [_opt(m) for m in masks]
    sp = [s_prevs[g] if len(s_prevs) else None for g in range(G)]
    if bf16:
        ops.shadow_bf16_block([[w] for p in P for w in (p[0], p[1])])
    grouped = _mma_group_ok(bf16, qs, kvs, n_heads, True)
    os_, ss, stats = attn_fwd_group(bf16, qs, kvs, kvs, masks_, sp, [p[4] for p in P], n_heads,
                                    emit_s, grouped)
    xs = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_fwd_group(bf16, [(os_[g], _weight(bf16, P[g][0]), None, xs[g].view(-1, d), False)
                                 for g in range(G)])
    ops._dropout_group(xs, xs, drop_p, ops.site_seeds(drop_seed, G, 0))
    # y = [q | x] Wm^T as two accumulating grouped GEMMs over the halves of Wm (no concat copy)
    ys = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    wms = [_weight(bf16, P[g][1]) for g in range(G)]
    ops._linear_fwd_group(bf16, [(qs[g], wms[g][:, :d], None, ys[g].view(-1, d), False, False)
                                 for g in range(G)])
    ops._linear_fwd_group(bf16, [(xs[g], wms[g][:, d:], None, ys[g].view(-1, d), False, True)
                                 for g in range(G)])
    outs, sts = ln_fwd_group(bf16, [None] * G, ys, [None] * G, [p[2] for p in P], [p[3] for p in P])
    ops._dropout_group(outs, outs, drop_p, ops.site_seeds(drop_seed, G, 1))
    out = []
    for g in range(G):
        out += [outs[g], ss[g] if ss[g] is not None else _e(dev), os_[g], stats[g], xs[g], ys[g],
                sts[g]]
    return out


def _lite_zlen(d: int) -> int:
    return _pad64(2 + 2 * d) + 3 * d * d


def _lite_zviews(z: Tensor, d: int):
    """[dpn (1+2d) | dc (1) | pad to 256 B] then dWo (d,d), dWm (d,2d)."""
    o = _pad64(2 + 2 * d)
    dpn, dc = z[:1 + 2 * d], z[1 + 2 * d:2 + 2 * d]
    dwo = z[o:o + d * d].view(d, d)
    dwm = z[o + d * d:o + 3 * d * d].view(d, 2 * d)
    return dpn, dc, dwo, dwm


def _lite_pgrads(z: Tensor, d: int) -> List[Tensor]:
    """The gradient of every parameter of a lite block (order: N_LITE) as a view of its buffer."""
    dpn, dc, dwo, dwm = _lite_zviews(z, d)
    return [dwo, dwm, dpn[1:1 + d], dpn[1 + d:], dc]


def lite_grad_unit(params: Sequence[Tensor]):
    """Like full_grad_unit for a lite block."""
    d = params[0].shape[0]
    z = torch.empty(_lite_zlen(d), device="meta")
    offsets = [g.storage_offset() for g in _lite_pgrads(z, d)]
    return params[0], list(zip(params, offsets)), z.numel()


@torch.library.custom_op("mmemo::trunk_lite_bwd", mutates_args=())
def trunk_lite_bwd_op(douts: Sequence[Tensor], ds_nexts: Sequence[Tensor], qs: Sequence[Tensor],
                      kvs: Sequence[Tensor], masks: Sequence[Tensor], s_prevs: Sequence[Tensor],
                      saved: Sequence[Tensor], params: Sequence[Tensor], n_heads: int, bf16: bool,
                      need_dsprev: bool, drop_p: float, drop_seed: int) -> List[Tensor]:
    G = len(qs)
    dt, dev = _act_dtype(bf16), qs[0].device
    d = qs[0].shape[-1]
    P = [params[N_LITE * g:N_LITE * (g + 1)] for g in range(G)]
    S = [saved[(LITE_OUT - 1) * g:(LITE_OUT - 1) * (g + 1)] for g in range(G)]
    # saved per problem: s o stat x y st
    ss = [_opt(s[0]) for s in S]
    os_, stats, xs, ys, sts = ([s[i] for s in S] for i in range(1, 6))
    qs = [q.contiguous() for q in qs]
    same = [kvs[g].data_ptr() == qs[g].data_ptr() and kvs[g].shape == qs[g].shape for g in range(G)]
    kvs = [qs[g] if same[g] else kvs[g].contiguous() for g in range(G)]
    masks_ = [_opt(m) for m in masks]
    sp = [s_prevs[g] if len(s_prevs) else None for g in range(G)]
    dsn = [_opt(t) for t in ds_nexts]
    douts = [t.contiguous() for t in douts]
    if drop_p > 0:   # gradient through the output dropout (out of place: douts belong to autograd)
        masked = [torch.empty_like(t) for t in douts]
        ops._dropout_group(douts, masked, drop_p, ops.site_seeds(drop_seed, G, 1))
        douts = masked
    zlen = _lite_zlen(d)
    zbs = ops.claim_zbufs([p[0] for p in P], zlen)       # (see trunk_full_bwd_op)
    if zbs is None:
        zall = torch.zeros(G * zlen, dtype=F32, device=dev)
        zbs = [zall[g * zlen:(g + 1) * zlen] for g in range(G)]
    else:
        zall = _e(dev)
    Z = [_lite_zviews(zbs[g], d) for g in range(G)]
    _, dys = ln_bwd_group(bf16, douts, [None] * G, ys, [None] * G, [p[2] for p in P], sts, False,
                          [z[0] for z in Z])
    wms = [_weight(bf16, P[g][1]) for g in range(G)]
    # minus: dx = dy Wm[:, d:]; proj: do = dx Wo
    dxs = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_bwd_x_group(bf16, [(dys[g], wms[g][:, d:], dxs[g].view(-1, d), False)
                                   for g in range(G)])
    ops._dropout_group(dxs, dxs, drop_p, ops.site_seeds(drop_seed, G, 0))
    dos = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    ops._linear_bwd_x_group(bf16, [(dxs[g], _weight(bf16, P[g][0]), dos[g].view(-1, d), False)
                                   for g in range(G)])
    # attention core (Q = q, K = V = kv): dk and dv both flow into kv -> the kernel sums them when
    # it is handed the same buffer for both
    grouped = _mma_group_ok(bf16, qs, kvs, n_heads, True)
    dqs = [torch.empty(q.shape, dtype=dt, device=dev) for q in qs]
    dks = [torch.empty(kv.shape, dtype=dt, device=dev) for kv in kvs]
    dvs = dks if grouped else [torch.empty(kv.shape, dtype=dt, device=dev) for kv in kvs]
    dsps = attn_bwd_group(bf16, dos, qs, kvs, kvs, masks_, ss, sp, [p[4] for p in P], dsn, os_,
                          stats, n_heads, dqs, dks, dvs, need_dsprev, [z[1] for z in Z], grouped)
    if not grouped:
        dks = [dk + dv for dk, dv in zip(dks, dvs)]
    # minus, q half: dq += dy Wm[:, :d]  (accumulates onto the attention's dq)
    ops._linear_bwd_x_group(bf16, [(dys[g], wms[g][:, :d], dqs[g].view(-1, d), True)
                                   for g in range(G)])
    dkv_out = []
    for g in range(G):
        if same[g]:        # q and kv are one tensor: a single gradient
            dqs[g] = dqs[g] + dks[g]
            dkv_out.append(_e(dev))
        else:
            dkv_out.append(dks[g])
    # weight gradients: dWo = dx^T o; dWm = dy^T [q | x] as two GEMMs into the halves of dWm
    items = []
    for g in range(G):
        _, _, dwo, dwm = Z[g]
        items += [(dxs[g].view(-1, d), os_[g].view(-1, d), dwo),
                  (dys[g].view(-1, d), qs[g].view(-1, d), dwm[:, :d]),
                  (dys[g].view(-1, d), xs[g].view(-1, d), dwm[:, d:])]
    ops._linear_bwd_w_group(bf16, items, zeroed=True)
    merged = merge_shared_grads(bf16, list(qs) + list(kvs),
                                list(dqs) + [t if t.numel() else None for t in dkv_out])
    dqs, dkvs = merged[:G], merged[G:]
    out = []
    for g in range(G):
        out += [dqs[g] if dqs[g] is not None else _e(dev), dkvs[g] if dkvs[g] is not None else _e(dev),
                dsps[g] if dsps[g] is not None else _e(dev)]
    return out + [zall]


def _trunk_lite_setup(ctx, inputs, output):
    qs, kvs, masks, s_prevs, params, H, bf16, emit_s, drop_p, drop_seed = inputs
    G = len(qs)
    ctx.G, ctx.cfg, ctx.has_prev = G, (H, bf16), len(s_prevs) > 0
    ctx.drop = (drop_p, drop_seed)
    saved = []
    for g in range(G):
        saved += list(output[LITE_OUT * g + 1:LITE_OUT * (g + 1)])
    ctx.save_for_backward(*qs, *kvs, *masks, *s_prevs, *saved, *params)
    ctx.set_materialize_grads(False)


def _trunk_lite_backward(ctx, grads):
    G = ctx.G
    H, bf16 = ctx.cfg
    t = list(ctx.saved_tensors)
    qs, kvs, masks = t[:G], t[G:2 * G], t[2 * G:3 * G]
    o = 3 * G
    s_prevs = t[o:o + G] if ctx.has_prev else []
    o += G if ctx.has_prev else 0
    ns = (LITE_OUT - 1) * G
    saved, params = t[o:o + ns], t[o + ns:]
    dev = qs[0].device
    douts, dsn = [], []
    for g in range(G):
        gh, gs = grads[LITE_OUT * g], grads[LITE_OUT * g + 1]
        douts.append(gh if gh is not None else torch.zeros_like(qs[g]))
        dsn.append(gs if gs is not None else _e(dev))
    need_dsprev = ctx.has_prev and any(ctx.needs_input_grad[3])
    res = trunk_lite_bwd_op(douts, dsn, qs, kvs, masks, s_prevs, saved, params, H, bf16, need_dsprev,
                            *ctx.drop)
    zall = res[-1]
    d = qs[0].shape[-1]
    zlen = _lite_zlen(d)
    dqs, dkvs, dsps, pgrads = [], [], [], []
    for g in range(G):
        dq, dkv, dsp = res[3 * g:3 * g + 3]
        dqs.append(dq if dq.numel() else None)
        dkvs.append(dkv if dkv.numel() else None)
        dsps.append(dsp if dsp.numel() else None)
        zb = zall[g * zlen:(g + 1) * zlen] if zall.numel() else ops.zbuf_region(params[N_LITE * g])
        pg = _lite_pgrads(zb, d)
        pgrads += pg[:-1] + [pg[-1] if ctx.has_prev else None]
    n_prev = G if ctx.has_prev else 0
    return (dqs, dkvs, [None] * G, dsps if need_dsprev else [None] * n_prev, pgrads, None, None,
            None, None, None)


trunk_lite_op.register_autograd(_trunk_lite_backward, setup_context=_trunk_lite_setup)


# ------------------------------------------------------------------------------------------------
# mmemo::proj_group — the modality projections ("unify dimension") of one or several towers:
#   y_g = x_g W_g^T (+ bias_g) (+ position table)  with x_g the RAW float32 features
#   (others/realformer.py:133-143,225-227; cmu-mosei/run.py:207-214; Ren-MME/run.py:158-166;
#   robot_demo.py:293-311).  bf16 mode only.
# The features arrive as float32 with widths the tensor-core GEMM's TMA cannot address (300, 35,
# 74, 205: rows are not 16-byte multiples), so the per-problem launchers ran them on the CUDA-core
# GEMM — the largest mandatory HBM read of Ren-MME (278 MB / step) at ~4 % of the HBM roofline.
# Here ONE launch casts all inputs (and weights) to bf16 with the row length padded to 8, ONE
# grouped tcgen05 launch does all projections (bias / position table fused in its epilogue), and the
# bf16 copy - half the bytes - is what backward re-reads for the weight gradients.
# ------------------------------------------------------------------------------------------------
def _pad8(k: int) -> int:
    return (k + 7) // 8 * 8


def _cast_pad(pairs) -> None:
    """pairs: [(float32 2-D source, bf16 (M, Kp) destination)], one launch per 16 tensors."""
    for i in range(0, len(pairs), 16):
        part = pairs[i:i + 16]
        _call("mmemo_cast_pad_f32_to_bf16_multi", len(part),
              _arr(C.c_void_p, [s.data_ptr() for s, _ in part]),
              _arr(C.c_int64, [s.stride(0) for s, _ in part]),
              _arr(C.c_void_p, [d.data_ptr() for _, d in part]),
              _arr(C.c_int64, [d.stride(0) for _, d in part]),
              _arr(C.c_int64, [s.shape[0] for s, _ in part]),
              _arr(C.c_int64, [s.shape[1] for s, _ in part]), _stream())


def _w2d(w: Tensor) -> Tensor:
    w = w.detach()
    return w.reshape(w.shape[0], -1)          # Conv1d(k=1) weight (N, K, 1) == Linear weight (N, K)


def _padded_shadow(w: Tensor, todo: list) -> Tensor:
    """bf16 (N, Kp) zero-padded shadow of a float32 weight; cached like ops.shadow_bf16 (keyed on
    the parameter's version counter).  Cache misses are appended to ``todo`` for one cast launch."""
    w2 = _w2d(w)
    key = (w.data_ptr(), w._version, tuple(w2.shape))
    hit = ops._shadow_pad.get(key)
    if hit is not None:
        return hit
    for k in [k for k in ops._shadow_pad if k[0] == w.data_ptr()]:
        del ops._shadow_pad[k]
    out = torch.empty(w2.shape[0], _pad8(w2.shape[1]), dtype=BF, device=w.device)
    todo.append((w2 if w2.is_contiguous() else w2.contiguous(), out))
    ops._shadow_pad[key] = out
    return out


@torch.library.custom_op("mmemo::proj_group", mutates_args=())
def proj_group_op(xs: Sequence[Tensor], ws: Sequence[Tensor], biases: Sequence[Tensor],
                  poss: Sequence[Tensor]) -> List[Tensor]:
    """Returns [y_0 .. y_{G-1}, xb_0 .. xb_{G-1}] (xb = the padded bf16 copy of x, saved for the
    weight gradient).  biases / poss entries with numel() == 0 mean "none"."""
    ops._need_cuda(*xs)
    G = len(xs)
    todo, xbs, wps, ys, items = [], [], [], [], []
    for g in range(G):
        x = xs[g]
        K = x.shape[-1]
        x2 = x.reshape(-1, K)
        x2 = x2 if x2.stride(1) == 1 else x2.contiguous()
        xb = torch.empty(x2.shape[0], _pad8(K), dtype=BF, device=x.device)
        todo.append((x2, xb))
        xbs.append(xb)
    for g in range(G):
        wps.append(_padded_shadow(ws[g], todo))
    _cast_pad(todo)
    for g in range(G):
        N = wps[g].shape[0]
        pos = _opt(poss[g])
        if pos is not None:
            assert xs[g].dim() == 3 and pos.shape[0] == xs[g].shape[1], \
                "position table length != seq length"
        y = torch.empty(*xs[g].shape[:-1], N, dtype=BF, device=xs[g].device)
        ys.append(y)
        items.append((xbs[g], wps[g], _opt(biases[g]), y.view(-1, N), False, False, pos))
    ops._linear_fwd_group(True, items)
    return ys + xbs


def _proj_zlayout(Ns, Kps, has_bias, pos_lens):
    """Offsets (floats, 256-byte aligned) of [dW_g (N, Kp) | dbias_g (N) | dpos_g (L, N)] per
    problem inside the one zero-filled gradient buffer, and its total length."""
    offs, tot = [], 0
    for g in range(len(Ns)):
        for n in (Ns[g] * Kps[g], Ns[g] if has_bias[g] else 0, pos_lens[g] * Ns[g]):
            offs.append(tot)
            tot += (n + 63) // 64 * 64
    return offs, tot


@torch.library.custom_op("mmemo::proj_group_bwd", mutates_args=())
def proj_group_bwd_op(dys: Sequence[Tensor], xbs: Sequence[Tensor], ws: Sequence[Tensor],
                      has_bias: Sequence[bool], pos_lens: Sequence[int],
                      need_dx: Sequence[bool]) -> List[Tensor]:
    """Returns [z] + [dx_g (float32 (M, K)) or empty]: z = ONE zero-initialised float32 buffer with
    every parameter gradient of the group (layout: _proj_zlayout; dW_g padded to (N, Kp))."""
    G = len(dys)
    dev = dys[0].device
    Ns = [_w2d(w).shape[0] for w in ws]
    Ks = [_w2d(w).shape[1] for w in ws]
    Kps = [_pad8(k) for k in Ks]
    dys = [dy.contiguous().view(-1, n) for dy, n in zip(dys, Ns)]
    offs, tot = _proj_zlayout(Ns, Kps, has_bias, pos_lens)
    z = torch.zeros(tot, dtype=F32, device=dev)
    dwp = [z[offs[3 * g]:offs[3 * g] + Ns[g] * Kps[g]].view(Ns[g], Kps[g]) for g in range(G)]
    ops._linear_bwd_w_group(True, [(dys[g], xbs[g], dwp[g]) for g in range(G)], zeroed=True)
    by_n = {}
    for g in range(G):
        if has_bias[g]:
            by_n.setdefault(Ns[g], []).append(g)
        if pos_lens[g]:
            dp = z[offs[3 * g + 2]:offs[3 * g + 2] + pos_lens[g] * Ns[g]].view(pos_lens[g], Ns[g])
            ops._rowsum(True, dys[g], dp, period=pos_lens[g])
    for n, gs in by_n.items():
        colsum_group(True, [dys[g] for g in gs],
                     [z[offs[3 * g + 1]:offs[3 * g + 1] + n] for g in gs])
    dxs = []
    for g in range(G):
        if need_dx[g]:
            todo: list = []
            wp = _padded_shadow(ws[g], todo)
            _cast_pad(todo)
            dxb = torch.empty(dys[g].shape[0], Kps[g], dtype=BF, device=dev)
            ops._linear_bwd_x(True, dys[g], wp, dxb)
            dxs.append(dxb[:, :Ks[g]].float())
        else:
            dxs.append(_e(dev))
    return [z] + dxs


def _proj_setup(ctx, inputs, output):
    xs, ws, biases, poss = inputs
    G = len(xs)
    ctx.G = G
    ctx.has_bias = [b.numel() > 0 for b in biases]
    ctx.pos_lens = [p.shape[0] if p.numel() else 0 for p in poss]
    ctx.x_shapes = [tuple(x.shape) for x in xs]
    ctx.save_for_backward(*output[G:], *ws)
    ctx.set_materialize_grads(False)


def _proj_backward(ctx, grads):
    G = ctx.G
    t = list(ctx.saved_tensors)
    xbs, ws = t[:G], t[G:]
    need_dx = list(ctx.needs_input_grad[0])
    Ns = [_w2d(w).shape[0] for w in ws]
    Ks = [_w2d(w).shape[1] for w in ws]
    Kps = [_pad8(k) for k in Ks]
    dys = []
    for g in range(G):
        if grads[g] is None:
            dys.append(torch.zeros(*ctx.x_shapes[g][:-1], Ns[g], dtype=BF, device=xbs[g].device))
        else:
            dys.append(grads[g])
    res = proj_group_bwd_op(dys, xbs, ws, ctx.has_bias, ctx.pos_lens, need_dx)
    z, dxs = res[0], res[1:]
    offs, _ = _proj_zlayout(Ns, Kps, ctx.has_bias, ctx.pos_lens)
    dws, dbs, dps = [], [], []
    for g in range(G):
        dw = z[offs[3 * g]:offs[3 * g] + Ns[g] * Kps[g]].view(Ns[g], Kps[g])
        if Kps[g] != Ks[g]:
            dw = dw[:, :Ks[g]].contiguous()
        dws.append(dw.view(ws[g].shape))
        dbs.append(z[offs[3 * g + 1]:offs[3 * g + 1] + Ns[g]] if ctx.has_bias[g] else None)
        L = ctx.pos_lens[g]
        dps.append(z[offs[3 * g + 2]:offs[3 * g + 2] + L * Ns[g]].view(L, Ns[g]) if L else None)
    return ([dxs[g].view(ctx.x_shapes[g]) if need_dx[g] else None for g in range(G)], dws, dbs, dps)


proj_group_op.register_autograd(_proj_backward, setup_context=_proj_setup)


@torch.no_grad()
def project_into(xs, ws, biases, outs, poss=None) -> None:
    """Inference-only (no autograd) form of the grouped projection, bf16 mode with float32 inputs:
    problem g writes ``x_g w_g^T + b_g (+ pos_g)`` into ``outs[g]``, a (rows, N_g) bf16 2-D view
    that may be a COLUMN SLICE of a wider buffer — the reference's ``cat`` of several projections
    (robot_demo.py:304-311) without the concat kernel — and ``pos_g`` may likewise be a column
    slice of the (L, d) table added after that concat (robot_demo.py:415-417).  An input tensor
    that several problems share (the members of an ensemble read the same features) is cast once.
    One cast launch per 16 tensors and ONE tensor-core launch for all problems (up to 48)."""
    ops._need_cuda(*xs)
    G = len(xs)
    poss = poss if poss is not None else [None] * G
    todo, xbs, wps, cast = [], [], [], {}
    for x in xs:
        xb = cast.get(id(x))
        if xb is None:
            K = x.shape[-1]
            x2 = x.reshape(-1, K)
            x2 = x2 if x2.stride(1) == 1 else x2.contiguous()
            xb = torch.empty(x2.shape[0], _pad8(K), dtype=BF, device=x.device)
            todo.append((x2, xb))
            cast[id(x)] = xb
        xbs.append(xb)
    for w in ws:
        wps.append(_padded_shadow(w, todo))
    _cast_pad(todo)
    items = []
    for g in range(G):
        pos = poss[g]
        if pos is not None:
            assert xs[g].dim() == 3 and pos.shape[0] == xs[g].shape[1] and pos.stride(1) == 1, \
                "position table length != seq length"
        assert outs[g].dim() == 2 and outs[g].shape == (xbs[g].shape[0], wps[g].shape[0])
        items.append((xbs[g], wps[g], biases[g], outs[g], False, False, pos))
    ops._linear_fwd_group(True, items)


def project(xs, ws, biases=None, poss=None, bf16: bool = False) -> List[Tensor]:
    """Modality projections of one or several towers.  bf16 mode with float32 inputs: the grouped
    cast + tensor-core path above; otherwise the per-problem ``ops.linear`` (float32 parity mode,
    or inputs that are already bf16)."""
    G = len(xs)
    biases = biases if biases is not None else [None] * G
    poss = poss if poss is not None else [None] * G
    if bf16 and all(x.dtype == F32 for x in xs):
        dev = xs[0].device
        ys = proj_group_op(list(xs), list(ws), [b if b is not None else _e(dev) for b in biases],
                           [p if p is not None else _e(dev) for p in poss])
        return list(ys[:G])
    return [ops.linear(x, w, b, p, bf16=bf16) for x, w, b, p in zip(xs, ws, biases, poss)]
