"""Shared host-side building blocks of the drop-in modules (precision switch, the two
``Attention_Block`` flavours, the 9-chain fusion trunk).  All compute goes through ``ops``.
"""
from __future__ import annotations

import contextlib
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn as nn

from . import group_ops, ops

_STATE = {"bf16": False}


def set_precision(mode: str) -> None:
    """'fp32' (parity mode, default) or 'bf16' (bf16 activations/GEMM operands, fp32 accumulate,
    fp32 master parameters and gradients)."""
    if mode not in ("fp32", "bf16"):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    _STATE["bf16"] = mode == "bf16"


def get_precision() -> str:
    return "bf16" if _STATE["bf16"] else "fp32"


@contextlib.contextmanager
def precision(mode: str):
    old = get_precision()
    set_precision(mode)
    try:
        yield
    finally:
        set_precision(old)


def is_bf16() -> bool:
    return _STATE["bf16"]


def as_act(x: torch.Tensor) -> torch.Tensor:
    """Cast an activation to the compute dtype of the current precision mode."""
    want = torch.bfloat16 if _STATE["bf16"] else torch.float32
    if x.dtype == want:
        return x
    if want == torch.bfloat16 and x.dtype == torch.float32 and x.is_cuda and not x.requires_grad:
        return ops.cast_bf16(x)          # raw inputs: libmmemo's vector cast
    return x.to(want)


def as_mask(m: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if m is None:
        return None
    m = m if m.dtype == torch.float32 else m.float()
    return m if m.is_contiguous() else m.contiguous()


def _split_check(dim: int, n_heads: int) -> None:
    # reference: split_last asserts through view(); an indivisible dim raises there as well
    if dim % n_heads != 0:
        raise RuntimeError(f"dim {dim} is not divisible by n_heads {n_heads}")


def _group_of_one(blk: nn.Module, op, q, kv, mask, scores, emit_scores: bool):
    """``blk`` on K = V as a trunk group of one problem (``group_ops``): one autograd node for the
    whole block, training dropout included; returns ``(out, scores or None)``."""
    same = q is kv
    q = as_act(q)
    kv = q if same else as_act(kv)
    m = as_mask(mask)
    drop_p = float(blk.drop.p) if blk.training else 0.0
    out = op([q], [kv], [m if m is not None else torch.empty(0, device=q.device)],
             [scores] if scores is not None else [], blk._params(), blk.n_heads, is_bf16(),
             emit_scores, drop_p, ops.next_dropout_seed() if drop_p > 0 else 0)
    return out[0], (out[1] if out[1].numel() else None)


class FullAttentionBlock(nn.Module):
    """RealFormer block with QKV projections, ReZero-gated post-LN and FFN.
    Reference: others/realformer.py:154-209 (ffn multiplier from the global ``FFN``) and
    robot_demo.py:324-374 (ffn is a ctor argument).  state_dict keys are the reference's."""

    def __init__(self, dim: int, n_heads: int, ffn: int, drop: float = 0.0):
        super().__init__()
        _split_check(dim, n_heads)
        self.w_qkv = nn.ModuleList([nn.Linear(dim, dim, bias=False) for _ in range(3)])
        self.n_heads = n_heads
        self.drop = nn.Dropout(drop)
        self.proj = nn.Linear(dim, dim, bias=False)
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim)
        self.ffn = nn.Sequential(nn.Linear(dim, ffn * dim), nn.ReLU(), nn.Linear(ffn * dim, dim),
                                 nn.Dropout(drop))
        self.a = nn.Parameter(torch.FloatTensor([0]), requires_grad=True)
        self.b = nn.Parameter(torch.FloatTensor([0]), requires_grad=True)
        self.c = nn.Parameter(torch.FloatTensor([0]), requires_grad=True)

    def _params(self) -> List[torch.Tensor]:
        return [self.w_qkv[0].weight, self.w_qkv[1].weight, self.w_qkv[2].weight, self.proj.weight,
                self.norm1.weight, self.norm1.bias, self.norm2.weight, self.norm2.bias,
                self.ffn[0].weight, self.ffn[0].bias, self.ffn[2].weight, self.ffn[2].bias,
                self.a, self.b, self.c]

    def mmemo_grad_unit(self):
        """dp.GradReducer protocol: the parameters whose gradients the fused backward accumulates
        into ONE zero-filled buffer, with their offsets (the reducer carves that buffer out of an
        all-reduce bucket, so nothing is copied)."""
        return group_ops.full_grad_unit(self._params())

    def multi_head_attention(self, q, k, v, mask, scores=None):
        """Projected attention + output projection; returns (drop(proj(att v)), scores)."""
        bf = is_bf16()
        q, k, v = as_act(q), as_act(k), as_act(v)
        qp = ops.linear(q, self.w_qkv[0].weight, bf16=bf)
        kp = ops.linear(k, self.w_qkv[1].weight, bf16=bf)
        vp = ops.linear(v, self.w_qkv[2].weight, bf16=bf)
        o, s, _ = ops.resattn_op(qp, kp, vp, as_mask(mask), scores, self.c, self.n_heads)
        x = ops.linear(o, self.proj.weight, bf16=bf)
        return ops.dropout(x, self.drop.p, self.training), s

    def forward(self, q, k, v, mask, scores=None, emit_scores: bool = True):
        """``emit_scores=False`` (not a reference argument; used by the fusion trunk for the last
        layer of a chain, whose scores feed nothing) skips writing the score tensor and returns
        ``(q, None)``; the default returns the scores like the reference."""
        if k is v:
            return _group_of_one(self, group_ops.trunk_full_op, q, k, mask, scores, emit_scores)
        bf = is_bf16()
        x, s = self.multi_head_attention(q, k, v, mask, scores)
        q = as_act(q)
        h1 = ops.add_ln(q, x, self.a, self.norm1.weight, self.norm1.bias)
        f = ops.linear(h1, self.ffn[0].weight, self.ffn[0].bias, relu=True, bf16=bf)
        f = ops.linear(f, self.ffn[2].weight, self.ffn[2].bias, bf16=bf)
        f = ops.dropout(f, self.drop.p, self.training)
        h2 = ops.add_ln(h1, f, self.b, self.norm2.weight, self.norm2.bias)
        return h2, s


class LiteAttentionBlock(nn.Module):
    """Residual-attention block without QKV projections: ``LN(minus([q | proj(att)]))``.
    Reference: cmu-mosei/run.py:217-262 (LayerNorm named ``norm1``) and Ren-MME/run.py:169-214
    (``norm2``)."""

    def __init__(self, dim: int, n_heads: int, ffn: int, drop: float = 0.0, norm_name: str = "norm1"):
        super().__init__()
        _split_check(dim, n_heads)
        self.n_heads = n_heads
        self.drop = nn.Dropout(drop)
        self.proj = nn.Linear(dim, dim, bias=False)
        self.minus = nn.Linear(dim * 2, dim, bias=False)
        setattr(self, norm_name, nn.LayerNorm(dim))
        self._norm_name = norm_name
        self.c = nn.Parameter(torch.FloatTensor([0]), requires_grad=True)

    @property
    def _norm(self) -> nn.LayerNorm:
        return getattr(self, self._norm_name)

    def _params(self) -> List[torch.Tensor]:
        n = self._norm
        return [self.proj.weight, self.minus.weight, n.weight, n.bias, self.c]

    def mmemo_grad_unit(self):
        """dp.GradReducer protocol (see FullAttentionBlock.mmemo_grad_unit)."""
        return group_ops.lite_grad_unit(self._params())

    def multi_head_attention(self, q, k, v, mask, scores=None):
        bf = is_bf16()
        q, k, v = as_act(q), as_act(k), as_act(v)
        o, s, _ = ops.resattn_op(q, k, v, as_mask(mask), scores, self.c, self.n_heads)
        x = ops.linear(o, self.proj.weight, bf16=bf)
        return ops.dropout(x, self.drop.p, self.training), s

    def forward(self, q, k, v, mask, scores=None, emit_scores: bool = True):
        if k is v:
            return _group_of_one(self, group_ops.trunk_lite_op, q, k, mask, scores, emit_scores)
        bf = is_bf16()
        n = self._norm
        x, s = self.multi_head_attention(q, k, v, mask, scores)
        y = ops.linear(torch.cat([as_act(q), x], dim=-1), self.minus.weight, bf16=bf)
        y = ops.add_ln(None, y, None, n.weight, n.bias)
        return ops.dropout(y, self.drop.p, self.training), s


# (query modality, source modality) in the reference's fixed order:
# others/realformer.py:232-257, cmu-mosei/run.py:278-313 — ll lv la vv vl va aa al av
CHAINS = [("l", "l"), ("l", "v"), ("l", "a"), ("v", "v"), ("v", "l"), ("v", "a"),
          ("a", "a"), ("a", "l"), ("a", "v")]


def fusion_trunk(blocks: Sequence[nn.Module], n_layers: int, feats: Dict[str, torch.Tensor],
                 masks: Dict[str, torch.Tensor], keep_all: bool) -> torch.Tensor:
    """Run the nine chains and pool.  Block ``n_layers*chain + i`` is layer i of a chain; scores
    restart at None per chain; the q-stream evolves while k = v = the un-evolved source modality.
    Returns the float32 pooled features (B, 6*d*(n_layers if keep_all else 1))."""
    return fusion_trunk_multi([(blocks, feats, masks)], n_layers, keep_all)[0]


def fusion_trunk_multi(towers, n_layers: int, keep_all: bool, pool: bool = True) -> List:
    """Several independent trunks of the same architecture at once — the two towers of
    ``Concat_Trans`` / ``Base_model`` (cmu-mosei/run.py:330-331, Ren-MME/run.py:283-284), the
    members of an ensemble (robot_demo.py:610-614).  ``towers`` = [(blocks, feats, masks), ...];
    returns one pooled tensor per tower, or with ``pool=False`` each tower's list of pooling
    segments (the input of ``ops.pool`` / ``ops.pool_multi``).  Layer i of every chain of every
    tower is one grouped op (``group_ops``); training dropout (Ren-MME and robot_demo train with
    p = 0.1) runs inside it as one grouped launch per dropout site."""
    blk0 = towers[0][0][0]
    drop_p = float(blk0.drop.p) if blk0.training else 0.0
    bf = is_bf16()
    full = isinstance(blk0, FullAttentionBlock)
    op = group_ops.trunk_full_op if full else group_ops.trunk_lite_op
    n_out = group_ops.FULL_OUT if full else group_ops.LITE_OUT
    qs, kvs, ms = [], [], []
    for _, feats, masks in towers:
        act = {k: as_act(v) for k, v in feats.items()}      # one cast per modality
        for qm, sm in CHAINS:
            qs.append(act[qm])
            kvs.append(act[sm])
            ms.append(masks[sm] if masks[sm] is not None else torch.empty(0, device=act[qm].device))
    G = len(qs)
    s_prev: List[torch.Tensor] = []
    per_chain: List[List[torch.Tensor]] = [[] for _ in range(G)]
    for i in range(n_layers):
        params = [p for blocks, _, _ in towers for ci in range(len(CHAINS))
                  for p in blocks[n_layers * ci + i]._params()]
        emit = i + 1 < n_layers                 # the last layer's scores feed nothing
        res = op(qs, kvs, ms, s_prev, params, blk0.n_heads, bf, emit, drop_p,
                 ops.next_dropout_seed() if drop_p > 0 else 0)
        qs = [res[n_out * g] for g in range(G)]
        s_prev = [res[n_out * g + 1] for g in range(G)] if emit else []
        for g in range(G):
            if keep_all or i + 1 == n_layers:
                per_chain[g].append(qs[g])
    segs = []
    for t in range(len(towers)):
        outs: Dict[str, List[torch.Tensor]] = {"l": [], "v": [], "a": []}
        for ci, (qm, _) in enumerate(CHAINS):
            outs[qm] += per_chain[t * len(CHAINS) + ci]
        # feature concat per modality, position concat in the order (l, a, v), mean||max pooling
        segs.append(outs["l"] + outs["a"] + outs["v"])
    return [ops.pool(s, 3) for s in segs] if pool else segs
