"""Ensemble inference of the k cross-validation fold models of one family (SURVEY.md §8f-2):
``pred = (model_1(x) + ... + model_k(x)) / k`` under ``eval()`` and ``no_grad()``
(others/realformer.py:418-420, Ren-MME/run.py:560, robot_demo.py:610-615; the reference scripts sum
the logits, which is k times this mean).

``Ensemble`` serves ``realformer.State_Transfer``, ``cmu_mosei.Concat_Trans``,
``ren_mme.Base_model`` and ``rencecps.Concat_Linear`` members.  One request is, for all members
together: one cast of every distinct raw input and one grouped projection GEMM (bf16 mode), one
grouped LayerNorm (``Base_model``), one ``fusion_trunk_multi`` over every tower of every member, one
grouped pooling launch and one ensemble-head launch that computes each member's classifier linears
and head and writes only the member mean.  ``GraphedEnsemble`` captures a request per input shape
into a CUDA graph and replays it; ``robot_demo.Ensemble`` uses it as well.

Uncertainty.  ``Ensemble(...)(*batch, return_uncertainty=True)`` returns ``(logits, unc)``:
``logits`` is bitwise the output of the same call without the flag, and ``unc`` an ``Uncertainty``
computed from the k members' own logits (the head launch also writes them, then one
``fold_uncertainty`` launch reduces them).  With ``p_i = softmax(logits of member i)`` over the C
classes, natural logarithms (entropies in nats) and one value per utterance (per window for
``State_Transfer``):

- ``mean_prob``        ``(..., C)``  ``(1/k) sum_i p_i``; each row sums to 1.
- ``variance``         ``(..., C)``  ``(1/(k-1)) sum_i (p_i - mean_prob)^2`` per class: how much the
                                      folds disagree (unbiased; 0 when k = 1).
- ``entropy``          ``(...)``     ``-sum_c mean_prob log mean_prob``, the predictive entropy,
                                      in [0, log C].
- ``expected_entropy`` ``(...)``     ``(1/k) sum_i -sum_c p_i log p_i``: the uncertainty each fold
                                      reports on its own (noise in the input itself).
- ``mutual_info``      ``(...)``     ``entropy - expected_entropy``, the part due to the folds
                                      disagreeing; >= 0 (clamped at 0 against rounding; 0 when
                                      k = 1).
- ``label``            ``(...)``     int64, ``argmax mean_prob`` (the first on ties).  This is the
                                      argmax of the mean probability, which can differ from the
                                      argmax of the mean logits.

``fold_uncertainty(fold_logits)`` is the same reduction for any ``(k, ..., C)`` float32 / bfloat16
CUDA tensor (one sm_100a kernel, ``csrc/uncertainty.cu``); ``fold_uncertainty_reference`` computes
it with PyTorch operations on any device, in float64, and is what the tests compare against.
"""
from __future__ import annotations

from typing import NamedTuple

import torch

from . import _lib, ops
from .blocks import as_mask, fusion_trunk_multi, get_precision, is_bf16
from .cmu_mosei import Concat_Trans
from .group_ops import ln_fwd_group, project_into
from .realformer import State_Transfer
from .ren_mme import Base_model
from .rencecps import Concat_Linear


class GraphedEnsemble:
    """Members in ``eval()`` mode and a request replayed from a CUDA graph captured per input shape
    (and precision mode).  Subclasses define ``_forward(args) -> Tensor``.  Weights are read at
    replay time from the members' parameters (float32 mode); in bf16 mode the graph uses the bf16
    weight shadows that existed at capture time, so call ``refresh()`` after loading new weights.
    ``use_graph=False`` runs ``_forward`` directly."""

    def __init__(self, models, use_graph: bool = True):
        self.models = list(models)
        if not self.models:
            raise ValueError("Ensemble needs at least one model")
        for m in self.models:
            m.eval()
        self.use_graph = use_graph
        self._graphs = {}      # input-shape key -> (graph, static inputs, static output)

    def refresh(self) -> None:
        """Drop the captured graphs (after load_state_dict / precision changes)."""
        self._graphs.clear()

    def _forward(self, args):
        raise NotImplementedError

    @torch.no_grad()
    def _run(self, args, *flags):
        """``_forward(args, *flags)``, a Tensor or a tuple of Tensors; ``flags`` are part of the
        graph key."""
        ops._need_cuda(*args)
        if not self.use_graph:
            return self._forward(args, *flags)
        key = flags + (get_precision(),) + tuple((tuple(t.shape), t.dtype) for t in args)
        entry = self._graphs.get(key)
        if entry is None:
            static_in = [torch.empty_like(t) for t in args]
            for s, t in zip(static_in, args):
                s.copy_(t)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):          # warm-up off the capture: allocator, shadows
                for _ in range(2):
                    self._forward(static_in, *flags)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = self._forward(static_in, *flags)
            entry = (graph, static_in, static_out)
            self._graphs[key] = entry
        graph, static_in, static_out = entry
        torch._foreach_copy_(static_in, list(args))
        graph.replay()
        if isinstance(static_out, tuple):
            return tuple(t.clone() for t in static_out)
        return static_out.clone()


class Uncertainty(NamedTuple):
    """How sure a k-fold ensemble is, per row of its output (definitions: module docstring)."""
    mean_prob: torch.Tensor         # (..., C) float32
    variance: torch.Tensor          # (..., C) float32
    entropy: torch.Tensor           # (...) float32, nats
    expected_entropy: torch.Tensor  # (...) float32, nats
    mutual_info: torch.Tensor       # (...) float32, nats
    label: torch.Tensor             # (...) int64


def fold_uncertainty(fold_logits: torch.Tensor) -> Uncertainty:
    """``Uncertainty`` of fold logits ``(k, ..., C)`` (float32 or bfloat16, contiguous, CUDA) in one
    kernel launch on the current stream.  CPU tensors raise; use ``fold_uncertainty_reference``."""
    return Uncertainty(*ops.fold_uncertainty(fold_logits))


def fold_uncertainty_reference(fold_logits: torch.Tensor,
                               dtype: torch.dtype = torch.float64) -> Uncertainty:
    """The reduction of ``fold_uncertainty`` with PyTorch operations, on any device: computed in
    ``dtype`` (float64 by default; float32 gives an eager baseline at the kernel's precision) from
    the max-subtracted logits, returned as float32 (label int64)."""
    if fold_logits.dim() < 2 or fold_logits.shape[0] < 1 or fold_logits.shape[-1] < 1:
        raise ValueError("fold logits must have shape (K, ..., C) with K >= 1 and C >= 1, got "
                         f"{tuple(fold_logits.shape)}")
    x = fold_logits.to(dtype)
    k = x.shape[0]
    z = x - x.amax(-1, keepdim=True)
    e = z.exp()
    s = e.sum(-1, keepdim=True)
    p = e / s
    fold_h = s.squeeze(-1).log() - torch.where(p > 0, p * z, torch.zeros_like(p)).sum(-1)
    mean = p.mean(0)
    var = (p - mean).square().sum(0) / (k - 1) if k > 1 else torch.zeros_like(mean)
    h = -torch.special.xlogy(mean, mean).sum(-1)
    eh = fold_h.mean(0)
    mi = (h - eh).clamp_min(0) if k > 1 else torch.zeros_like(h)
    return Uncertainty(mean.float(), var.float(), h.float(), eh.float(), mi.float(),
                       mean.argmax(-1))


_FAMILIES = (State_Transfer, Concat_Trans, Base_model, Concat_Linear)


def _arch(m):
    """(n_heads, n_layers) of a member's trunk; (None, None) for Concat_Linear."""
    if isinstance(m, State_Transfer):
        f = m.feature
        return f.multimodal_blocks[0].n_heads, f.n_layers
    if isinstance(m, (Concat_Trans, Base_model)):
        return m.intensity.multimodal_blocks[0].n_heads, m.intensity.n_layers
    if hasattr(m, "multimodal_blocks"):   # robot_demo.Multi_class (it imports this module)
        return m.multimodal_blocks[0].n_heads, m.n_layers
    return None, None


def _check_members(models, families=_FAMILIES) -> None:
    """One class of ``families``, equal state_dict shapes and equal n_heads / n_layers."""
    if not models:
        raise ValueError("Ensemble needs at least one model")
    cls = type(models[0])
    if cls not in families:
        raise ValueError(f"Ensemble members must be one of {[c.__name__ for c in families]}, "
                         f"got {cls.__name__}")
    shapes0 = {k: tuple(v.shape) for k, v in models[0].state_dict().items()}
    for i, m in enumerate(models[1:], 1):
        if type(m) is not cls:
            raise ValueError(f"member {i} is a {type(m).__name__}, member 0 a {cls.__name__}")
        shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        if set(shapes) != set(shapes0):
            raise ValueError(f"member {i} has state_dict keys {sorted(set(shapes) ^ set(shapes0))} "
                             "that member 0 lacks or has")
        for k, s in shapes.items():
            if s != shapes0[k]:
                raise ValueError(f"member {i}: {k} has shape {s}, member 0 {shapes0[k]}")
        for what, a, b in zip(("n_heads", "n_layers"), _arch(m), _arch(models[0])):
            if a != b:
                raise ValueError(f"member {i} has {what} {a}, member 0 {b}")


def _p(t: torch.Tensor) -> int:
    t = t.detach()
    assert t.dtype == torch.float32 and t.is_contiguous()
    return t.data_ptr()


class Ensemble(GraphedEnsemble):
    """``Ensemble([model_1, ..., model_k])(*batch_args)``: the mean of the members' logits, float32,
    shaped like one member's output.  Members: k fold models of ONE of ``State_Transfer``,
    ``Concat_Trans``, ``Base_model`` or ``Concat_Linear`` with equal state_dict shapes and equal
    ``n_heads`` / ``n_layers`` (``ValueError`` otherwise); the call takes the members' own forward
    arguments, on CUDA.  ``return_uncertainty=True`` returns ``(logits, Uncertainty)`` instead
    (module docstring); ``logits`` is unchanged."""

    def __init__(self, models, use_graph: bool = True):
        models = list(models)
        _check_members(models)
        super().__init__(models, use_graph)

    @torch.no_grad()
    def __call__(self, *args, return_uncertainty: bool = False):
        if not return_uncertainty:
            return self._run(args)
        logits, *unc = self._run(args, True)
        return logits, Uncertainty(*unc)

    def _forward(self, args, uncertainty: bool = False):
        """The mean logits, or with ``uncertainty`` the tuple (mean logits, *Uncertainty)."""
        m0 = self.models[0]
        if isinstance(m0, State_Transfer):
            return self._state_transfer(args, uncertainty)
        if isinstance(m0, Concat_Linear):
            return self._concat_linear(args[0], uncertainty)
        return self._bilinear(args, uncertainty)

    def _head(self, kind, mem, B, P, F, d, n_cls, shape, device, uncertainty):
        """One ensemble-head launch into a new (shape) float32 output; with ``uncertainty`` it also
        writes every member's output and one fold_uncertainty launch reduces them."""
        out = torch.empty(shape, dtype=torch.float32, device=device)
        if not uncertainty:
            ops.ensemble_head(kind, mem, B, P, F, d, n_cls, out)
            return out
        folds = torch.empty((len(mem),) + tuple(shape), dtype=torch.float32, device=device)
        ops.ensemble_head(kind, mem, B, P, F, d, n_cls, out, folds)
        return (out,) + ops.fold_uncertainty(folds)

    # -- shared pieces ------------------------------------------------------------------------
    @staticmethod
    def _project(problems):
        """problems: [(x, w, pos or None)] -> x w^T (+ pos) in the activation dtype.  bf16 mode with
        float32 inputs: every distinct input cast once and ONE grouped GEMM (``project_into``)."""
        bf = is_bf16()
        if bf and all(x.dtype == torch.float32 for x, _, _ in problems):
            outs, flat = [], []
            for x, w, _ in problems:
                y = torch.empty(*x.shape[:-1], w.shape[0], dtype=torch.bfloat16, device=x.device)
                outs.append(y)
                flat.append(y.view(-1, w.shape[0]))
            project_into([x for x, _, _ in problems], [w for _, w, _ in problems],
                         [None] * len(problems), flat, [p for _, _, p in problems])
            return outs
        return [ops.linear(x, w, None, p, bf16=bf) for x, w, p in problems]

    @staticmethod
    def _unify(u, x3, poss=(None, None, None)):
        return [(x, c.weight, p) for x, c, p in
                zip(x3, (u.linguistic, u.visual, u.acoustic), poss)]

    # -- families -----------------------------------------------------------------------------
    def _state_transfer(self, args, uncertainty):
        """others/realformer.py:266-286 for every member: the B*P windows folded into the batch."""
        l, v, a, l_mask, v_mask, a_mask = args
        B, P = l.shape[0], l.shape[1]
        fold = lambda t: t.reshape(B * P, *t.shape[2:])
        l, v, a = fold(l), fold(v), fold(a)
        masks = {"l": as_mask(fold(l_mask)), "v": as_mask(fold(v_mask)), "a": as_mask(fold(a_mask))}
        fs = [m.feature for m in self.models]
        probs = [p for f in fs for p in self._unify(f.unify_dimension, (l, v, a), f.positions(l, v, a))]
        ys = self._project(probs)
        towers = [(f.multimodal_blocks, {"l": ys[3 * i], "v": ys[3 * i + 1], "a": ys[3 * i + 2]},
                   masks) for i, f in enumerate(fs)]
        pooled = ops.pool_multi(fusion_trunk_multi(towers, fs[0].n_layers, keep_all=False,
                                                   pool=False))
        mem = []
        for m, f, x in zip(self.models, fs, pooled):
            mem.append(_lib.EnsembleMember(
                x0=_p(x), ld0=x.shape[1], x1=None, ld1=0, w0=_p(f.fully_connected.weight), w1=None,
                b0=_p(f.fully_connected.bias), ln_gamma=_p(f.normalization.weight),
                ln_beta=_p(f.normalization.bias), w_out=_p(m.classifier.weight),
                b_out=_p(m.classifier.bias), trans=_p(m.trans)))
        d, n_cls = f.fully_connected.weight.shape[0], m.trans.shape[0]
        return self._head(_lib.HEAD_STATE_TRANSFER, mem, B, P, pooled[0].shape[1], d, n_cls,
                          (B, P, n_cls), l.device, uncertainty)

    def _bilinear(self, args, uncertainty):
        """cmu-mosei/run.py:321-339 / Ren-MME/run.py:273-292 for every member: two towers each."""
        if isinstance(self.models[0], Concat_Trans):
            l, v, a, l_mask, v_mask, a_mask = args
            feats = [tuple(t[:, i] for t in (l, v, a)) for i in (0, 1)]
            mk = [tuple(as_mask(t[:, i]) for t in (l_mask, v_mask, a_mask)) for i in (0, 1)]
        else:
            feats = [(args[0], args[4], args[8]), (args[2], args[6], args[10])]
            mk = [tuple(as_mask(args[j]) for j in (1, 5, 9)), tuple(as_mask(args[j]) for j in (3, 7, 11))]
        masks = [{"l": m3[0], "v": m3[1], "a": m3[2]} for m3 in mk]
        towers_of = [(m.intensity, m.stimulation) for m in self.models]
        probs = [p for ts in towers_of for i, t in enumerate(ts)
                 for p in self._unify(t.unify_dimension, feats[i])]
        ys = self._project(probs)
        if isinstance(self.models[0], Base_model):
            # Ren-MME/run.py:158-166: the tower's LayerNorm over its three projections, all towers
            # of all members in one grouped call
            lns = [t.unify_dimension.norm1 for ts in towers_of for t in ts for _ in range(3)]
            n = len(ys)
            ys, _ = ln_fwd_group(ys[0].dtype == torch.bfloat16, [None] * n, ys, [None] * n,
                                 [u.weight for u in lns], [u.bias for u in lns])
        towers, k = [], 0
        for ts in towers_of:
            for i, t in enumerate(ts):
                towers.append((t.multimodal_blocks, {"l": ys[k], "v": ys[k + 1], "a": ys[k + 2]},
                               masks[i]))
                k += 3
        pooled = ops.pool_multi(fusion_trunk_multi(towers, towers_of[0][0].n_layers, keep_all=True,
                                                   pool=False))
        mem = []
        for i, m in enumerate(self.models):
            last, this = pooled[2 * i], pooled[2 * i + 1]
            norm = m.norm1 if isinstance(m, Concat_Trans) else m.norm3
            mem.append(self._bilinear_member(last, this, m.intensity.classifier.weight,
                                             m.stimulation.classifier.weight, norm, m.out, m.trans))
        return self._bilinear_head(mem, pooled[0].shape[0], pooled[0].shape[1], pooled[0].device,
                                   uncertainty)

    def _concat_linear(self, feat, uncertainty):
        """rencecps/run.py:130-148 for every member: feat (B, 2, F); the two halves are read through
        row strides."""
        feat = feat if feat.dtype == torch.float32 else feat.float()
        feat = feat if feat.is_contiguous() else feat.contiguous()
        B, _, F = feat.shape
        mem = [self._bilinear_member(feat[:, 0], feat[:, 1], m.intensity.weight,
                                     m.stimulation.weight, m.norm, m.out, m.trans)
               for m in self.models]
        return self._bilinear_head(mem, B, F, feat.device, uncertainty)

    @staticmethod
    def _bilinear_member(last, this, w_last, w_this, norm, out, trans):
        return _lib.EnsembleMember(
            x0=last.data_ptr(), ld0=last.stride(0), x1=this.data_ptr(), ld1=this.stride(0),
            w0=_p(w_last), w1=_p(w_this), b0=None, ln_gamma=_p(norm.weight), ln_beta=_p(norm.bias),
            w_out=_p(out.weight), b_out=_p(out.bias), trans=_p(trans))

    def _bilinear_head(self, mem, B, F, device, uncertainty):
        n_cls = self.models[0].trans.shape[0]
        return self._head(_lib.HEAD_BILINEAR, mem, B, 1, F, 0, n_cls, (B, n_cls), device,
                          uncertainty)
