"""Drop-in modules for the reference script ``robot_demo.py`` (dim 192, five biased input
projections, full RealFormer blocks, plain linear classifier; ensemble inference)."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .blocks import FullAttentionBlock, as_act, as_mask, fusion_trunk_multi, is_bf16
from .ensemble import GraphedEnsemble

DROP = 0.1  # robot_demo.py:41


class Unify_Dimension_Conv1d(nn.Module):
    """robot_demo.py:293-311: five biased Conv1d(k=1); v = cat(v256, v512, v1024 projections)."""

    def __init__(self, dim, l_dim=768, dim_1024=1024, dim_512=512, dim_256=256, a_dim=40):
        super().__init__()
        self.linguistic = nn.Conv1d(l_dim, dim, kernel_size=1)
        self.visual_1024 = nn.Conv1d(dim_1024, dim // 3, kernel_size=1)
        self.visual_512 = nn.Conv1d(dim_512, dim // 3, kernel_size=1)
        self.visual_256 = nn.Conv1d(dim_256, dim // 3, kernel_size=1)
        self.acoustic = nn.Conv1d(a_dim, dim, kernel_size=1)
        self.drop = nn.Dropout(DROP)

    def forward(self, l, v_256, v_512, v_1024, a):
        bf = is_bf16()
        convs = (self.linguistic, self.visual_256, self.visual_512, self.visual_1024, self.acoustic)
        xs = (l, v_256, v_512, v_1024, a)
        if not (self.training and self.drop.p > 0):
            from .group_ops import project
            yl, y256, y512, y1024, ya = project(list(xs), [c.weight for c in convs],
                                                [c.bias for c in convs], bf16=bf)
        else:
            yl, y256, y512, y1024, ya = (
                ops.dropout(ops.linear(x, c.weight, c.bias, bf16=bf), self.drop.p, True)
                for x, c in zip(xs, convs))
        return yl, torch.cat((y256, y512, y1024), 2), ya


class Position_Embedding(nn.Module):
    """robot_demo.py:314-321."""

    def __init__(self, max_len, dim):
        super().__init__()
        self.position_embeddings = nn.Embedding(max_len, dim)
        self.len = max_len

    def forward(self, x):
        w = self.position_embeddings.weight
        return as_act(w)[None].expand(x.size(0), self.len, w.shape[1])


class Attention_Block(FullAttentionBlock):
    """robot_demo.py:324-374."""

    def __init__(self, dim, n_heads, ffn):
        super().__init__(dim, n_heads, ffn, DROP)


class Multi_class(nn.Module):
    """robot_demo.py:377-441 (``fully_connected`` / ``normalization`` exist but are unused)."""

    def __init__(self, dim, l_len, v_len, a_len, n_heads, n_layers, ffn):
        super().__init__()
        self.unify_dimension = Unify_Dimension_Conv1d(dim)
        self.linguistic_position = Position_Embedding(l_len, dim)
        self.visual_position = Position_Embedding(v_len, dim)
        self.acoustic_position = Position_Embedding(a_len, dim)
        self.n_layers = n_layers
        self.multimodal_blocks = nn.ModuleList([Attention_Block(dim, n_heads, ffn)
                                                for _ in range(9 * n_layers)])
        self.fully_connected = nn.Linear(dim * 6, dim)
        self.normalization = nn.LayerNorm(dim)
        self.drop = nn.Dropout(DROP)
        self.classifier = nn.Linear(dim * 6 * n_layers, 7)

    def _tower(self, l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask):
        """(blocks, projected + position-embedded features, masks) for ``fusion_trunk_multi``."""
        l, v, a = self.unify_dimension(l, v_256, v_512, v_1024, a)
        l = l + self.linguistic_position(l)
        v = v + self.visual_position(v)
        a = a + self.acoustic_position(a)
        return (self.multimodal_blocks, {"l": l, "v": v, "a": a},
                {"l": as_mask(l_mask), "v": as_mask(v_mask), "a": as_mask(a_mask)})

    def forward(self, l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask):
        x = fusion_trunk_multi([self._tower(l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask)],
                               self.n_layers, keep_all=True)[0]
        return ops.linear(x, self.classifier.weight, self.classifier.bias)


def multi_circle_loss(y_pred, y_true):
    """robot_demo.py:444-453."""
    return ops.circle_loss_op(y_pred, y_true)


def sigmoids(pred, offset):
    """robot_demo.py:594-595 helper of demo_output: sigmoid with per-class logit offsets."""
    return torch.sigmoid(pred - offset)


class Ensemble(GraphedEnsemble):
    """Ensemble-of-models inference of ``demo_output`` / ``f1_calculation`` (robot_demo.py:526-581,
    597-622; SURVEY.md §8f-2): ``pred = (model_1(x) + ... + model_n(x)) / n`` under ``eval()`` and
    ``no_grad()``.

    The reference runs the members one after the other and moves every prediction to the host.  At
    batch 1 each member is ~350 launches of microsecond kernels, so the request is launch-bound.
    Here the members run on their own CUDA streams (forked from and joined into the caller's
    stream) and the whole request — input staging, all members, the average — is captured once per
    input shape into a CUDA graph and replayed (``ensemble.GraphedEnsemble``: call ``refresh()``
    after loading new weights in bf16 mode).
    """

    NAMES = ("l", "v_256", "v_512", "v_1024", "a", "l_mask", "v_mask", "a_mask")
    # logit offsets of the six printed emotions (robot_demo.py:609)
    OFFSETS = {"happy": 0.1, "sad": 0.1, "angry": -0.1, "disgust": 0.0, "surprise": 0.1, "fear": 0.0}

    def __init__(self, models, use_graph: bool = True):
        super().__init__(models, use_graph)
        self._streams = None

    def _forward(self, args):
        """All members at once.  Members that are this module's ``Multi_class`` with one
        architecture run as ONE group: layer i of every chain of every member (4 x 9 = 36
        problems) is one launch per kernel kind (``fusion_trunk_multi``; weights stay per member -
        the problem tables carry each member's own pointers, nothing is copied or stacked).  Other
        member types run concurrently on side streams, joined before the average."""
        ms = self.models
        if all(isinstance(m, Multi_class) for m in ms) and \
                len({(m.n_layers, len(m.multimodal_blocks)) for m in ms}) == 1:
            towers = self._towers_joint(args) if is_bf16() and args[0].dtype == torch.float32 \
                else [m._tower(*args) for m in ms]
            pooled = fusion_trunk_multi(towers, ms[0].n_layers, keep_all=True)
            preds = [ops.linear(x, m.classifier.weight, m.classifier.bias)
                     for m, x in zip(ms, pooled)]
        else:
            cur = torch.cuda.current_stream()
            if self._streams is None or len(self._streams) != len(ms):
                self._streams = [torch.cuda.Stream() for _ in ms]
            preds = []
            for m, s in zip(ms, self._streams):
                s.wait_stream(cur)
                with torch.cuda.stream(s):
                    preds.append(m(*args))
            for s in self._streams:
                cur.wait_stream(s)
        pred = preds[0]
        for p in preds[1:]:            # same summation order as robot_demo.py:614
            pred = pred + p
        return pred / len(preds)

    def _towers_joint(self, args):
        """``Multi_class._tower`` of every member from ONE grouped projection launch (bf16 mode):
        the 5 input projections of all members are problems of one tensor-core launch whose
        epilogue adds bias and position table; the three visual projections write the column
        thirds of one (B, L, d) buffer and add the matching thirds of the visual table, so the
        reference's ``cat`` + three ``x + position`` kernels per member disappear."""
        from .group_ops import project_into
        l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask = args
        masks = {"l": as_mask(l_mask), "v": as_mask(v_mask), "a": as_mask(a_mask)}
        xs, ws, bs, outs, poss, towers = [], [], [], [], [], []
        for m in self.models:
            u = m.unify_dimension
            d = u.linguistic.weight.shape[0]
            t = d // 3
            pl, pv, pa = (e.position_embeddings.weight.detach() for e in
                          (m.linguistic_position, m.visual_position, m.acoustic_position))
            yl = torch.empty(*l.shape[:2], d, dtype=torch.bfloat16, device=l.device)
            yv = torch.empty(*v_256.shape[:2], 3 * t, dtype=torch.bfloat16, device=l.device)
            ya = torch.empty(*a.shape[:2], d, dtype=torch.bfloat16, device=l.device)
            yv2 = yv.view(-1, 3 * t)
            for x, conv, out, pos in (
                    (l, u.linguistic, yl.view(-1, d), pl),
                    (v_256, u.visual_256, yv2[:, 0:t], pv[:, 0:t]),
                    (v_512, u.visual_512, yv2[:, t:2 * t], pv[:, t:2 * t]),
                    (v_1024, u.visual_1024, yv2[:, 2 * t:3 * t], pv[:, 2 * t:3 * t]),
                    (a, u.acoustic, ya.view(-1, d), pa)):
                xs.append(x); ws.append(conv.weight); bs.append(conv.bias.detach())
                outs.append(out); poss.append(pos)
            towers.append((m.multimodal_blocks, {"l": yl, "v": yv, "a": ya}, masks))
        project_into(xs, ws, bs, outs, poss)
        return towers

    @torch.no_grad()
    def __call__(self, l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask):
        return self._run((l, v_256, v_512, v_1024, a, l_mask, v_mask, a_mask))

    def emotions(self, pred: torch.Tensor) -> dict:
        """The scores ``demo_output`` prints for sample 0: sigmoid(logit - offset), rounded to 2
        places (robot_demo.py:594-595, 615-622)."""
        p = pred[0].detach().float().cpu()
        return {k: round(float(torch.sigmoid(p[i] - off)), 2)
                for i, (k, off) in enumerate(self.OFFSETS.items())}
