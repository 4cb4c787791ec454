"""Drop-in modules for the reference script ``others/realformer.py`` (CMU-MOSEI, 6 emotions,
full RealFormer blocks, 6-window state-transfer head).  Same class names, constructor and forward
signatures and ``state_dict`` keys as the reference; compute runs in libmmemo (sm_100a).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .blocks import FullAttentionBlock, as_act, as_mask, fusion_trunk, is_bf16

# module-level constants the reference classes read at construction time
# (others/realformer.py:23-38); kept as overridable defaults
FFN = 2
DROP = 0.0


class Unify_Dimension_Conv1d(nn.Module):
    """others/realformer.py:133-143: three bias-free Conv1d(k=1) == per-position linears."""

    def __init__(self, l_dim, v_dim, a_dim, dim):
        super().__init__()
        self.linguistic = nn.Conv1d(l_dim, dim, kernel_size=1, bias=False)
        self.visual = nn.Conv1d(v_dim, dim, kernel_size=1, bias=False)
        self.acoustic = nn.Conv1d(a_dim, dim, kernel_size=1, bias=False)
        self.drop = nn.Dropout(DROP)

    def forward(self, l, v, a, pos=(None, None, None)):
        from .group_ops import project
        convs = (self.linguistic, self.visual, self.acoustic)
        p = float(self.drop.p) if self.training else 0.0
        # all three projections (+ fused position tables) as one group (group_ops.project); the
        # reference order drop(conv(x)) THEN + position is kept in the GEMM epilogue
        return tuple(project([l, v, a], [c.weight for c in convs], None, list(pos), bf16=is_bf16(),
                             drop_p=p, seed=ops.next_dropout_seed() if p > 0 else 0))


class Position_Embedding(nn.Module):
    """others/realformer.py:145-152: returns E[arange(max_len)] broadcast over the batch (the
    caller adds it).  In the fused model path the table is added inside the projection GEMM."""

    def __init__(self, max_len, dim):
        super().__init__()
        self.position_embeddings = nn.Embedding(max_len, dim)
        self.len = max_len

    def forward(self, x):
        w = self.position_embeddings.weight
        return as_act(w)[None].expand(x.size(0), self.len, w.shape[1])


class Attention_Block(FullAttentionBlock):
    """others/realformer.py:154-209.  ``Attention_Block(dim, n_heads)``; FFN multiplier and dropout
    come from the module globals ``FFN`` / ``DROP`` like in the reference."""

    def __init__(self, dim, n_heads):
        super().__init__(dim, n_heads, FFN, DROP)


class Multi_class(nn.Module):
    """others/realformer.py:211-264."""

    def __init__(self, l_dim, v_dim, a_dim, dim, l_len, v_len, a_len, n_heads, n_layers, ffn):
        super().__init__()
        self.unify_dimension = Unify_Dimension_Conv1d(l_dim, v_dim, a_dim, dim)
        self.linguistic_position = Position_Embedding(l_len, dim)
        self.visual_position = Position_Embedding(v_len, dim)
        self.acoustic_position = Position_Embedding(a_len, dim)
        self.n_layers = n_layers
        self.multimodal_blocks = nn.ModuleList([Attention_Block(dim, n_heads)
                                                for _ in range(9 * n_layers)])
        self.fully_connected = nn.Linear(dim * 6, dim)
        self.normalization = nn.LayerNorm(dim)
        self.drop = nn.Dropout(DROP)

    def positions(self, l, v, a):
        """The three position tables, after checking the sequence lengths against them."""
        for x, pe in ((l, self.linguistic_position), (v, self.visual_position),
                      (a, self.acoustic_position)):
            if x.shape[1] != pe.len:  # the reference's `l + position(l)` broadcast would fail too
                raise RuntimeError(f"sequence length {x.shape[1]} != position table {pe.len}")
        return (self.linguistic_position.position_embeddings.weight,
                self.visual_position.position_embeddings.weight,
                self.acoustic_position.position_embeddings.weight)

    def _tower(self, l, v, a, l_mask, v_mask, a_mask):
        """(blocks, projected + position-added features, masks) - the input of
        ``fusion_trunk_multi`` (others/realformer.py:225-231)."""
        l, v, a = self.unify_dimension(l, v, a, self.positions(l, v, a))   # position add fused
        return (self.multimodal_blocks, {"l": l, "v": v, "a": a},
                {"l": as_mask(l_mask), "v": as_mask(v_mask), "a": as_mask(a_mask)})

    def forward(self, l, v, a, l_mask, v_mask, a_mask):
        blocks, feats, masks = self._tower(l, v, a, l_mask, v_mask, a_mask)
        x = fusion_trunk(blocks, self.n_layers, feats, masks, keep_all=False)
        x = ops.linear(x, self.fully_connected.weight, self.fully_connected.bias)   # float32 head
        x = ops.add_ln(None, x, None, self.normalization.weight, self.normalization.bias, relu=True)
        return ops.dropout(x, self.drop.p, self.training)


class State_Transfer(nn.Module):
    """others/realformer.py:266-286.  Inputs carry a window dim: l (B,P,L,D), masks (B,P,L).  The P
    windows are independent until the (B,P,6) recurrence, so they are folded into the batch."""

    def __init__(self, l_dim, v_dim, a_dim, dim, l_len, v_len, a_len, n_heads, n_layers, ffn):
        super().__init__()
        self.feature = Multi_class(l_dim=l_dim, v_dim=v_dim, a_dim=a_dim, dim=dim, l_len=l_len,
                                   v_len=v_len, a_len=a_len, n_heads=n_heads, n_layers=n_layers,
                                   ffn=ffn)
        self.classifier = nn.Linear(dim, 6 * 2)
        self.trans = nn.Parameter(torch.rand(6, 6), requires_grad=True)

    def forward(self, l, v, a, l_mask, v_mask, a_mask):
        B, P = l.shape[0], l.shape[1]
        fold = lambda t: t.reshape(B * P, *t.shape[2:])
        f = self.feature(fold(l), fold(v), fold(a), fold(l_mask), fold(v_mask), fold(a_mask))
        f = ops.linear(f, self.classifier.weight, self.classifier.bias)
        return ops.state_transfer_op(f.view(B, P, -1), self.trans)


def multi_circle_loss(y_pred, y_true):
    """others/realformer.py:289-298: per-row multi-label circle loss."""
    return ops.circle_loss_op(y_pred, y_true)
