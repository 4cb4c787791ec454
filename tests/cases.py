"""Small parity cases shared by the CPU (oracle-vs-reference / oracle-vs-golden) tests, the golden
generator and the GPU parity tests.  One entry per reference model family (SURVEY.md §8b).

Each case knows how to
  * build the REFERENCE model (``ref_model(ns)``; ns = oracle.refload.load(...)),
  * build OUR drop-in module (``our_model(pkg)``; pkg = mmemo_b200),
  * make a seeded batch, call either model on it, and compute the family's training loss,
  * run the oracle on a state_dict.
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass, field
from typing import Callable, Dict, List

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import mmemo_oracle as O  # noqa: E402
import mmemo_b200.synth as synth  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


@dataclass
class Case:
    name: str
    family: str                      # key of oracle.refload.FILES
    overrides: Dict[str, float]      # reference module-level constants to override
    ref_model: Callable              # ns -> nn.Module
    our_model: Callable              # pkg -> nn.Module
    batch: Callable                  # () -> dict of CPU tensors
    call: Callable                   # (model, batch) -> logits
    oracle: Callable                 # (state_dict, batch) -> logits
    loss: Callable                   # (logits, batch, lossfns) -> scalar
    grad_inputs: List[str] = field(default_factory=list)


def _circle_mean(logits, batch, L):
    return L.multi_circle_loss(logits, batch["label"]).mean()


def _window_loss(logits, batch, L):
    return (L.multi_circle_loss(logits, batch["label"]) * batch["wmask"]).mean()


def _renmme_loss(logits, batch, L):
    return L.multi_loss(logits, batch["label"]) + L.rdrop_kl(logits)


def _sq_mean(out, batch, L):
    # projection on a fixed random cotangent (mean(out^2) of a LayerNorm output is ~constant)
    return (out.float() * batch["dy"]).mean()


# ------------------------------------------------------------------------------------------
RF = dict(l_dim=20, v_dim=7, a_dim=10, dim=16, l_len=6, v_len=5, a_len=7, n_heads=2, n_layers=2,
          ffn=2)
MOSEI = dict(dim=24, l_len=6, v_len=9, a_len=12, n_heads=2, n_layers=2, ffn=1)
MOSEI_D = (20, 7, 10)
REN = dict(dim=32, l_len=5, v_len=7, a_len=11, n_heads=4, n_layers=1, ffn=1)
REN_D = (24, 20, 13)
ROBOT = dict(dim=24, l_len=5, v_len=8, a_len=8, n_heads=2, n_layers=2, ffn=2)
CHAIN = dict(dim=32, n_heads=4, n_layers=3, B=2, L=16)


def _rf_call(m, b):
    return m(b["l"], b["v"], b["a"], b["l_mask"], b["v_mask"], b["a_mask"])


def _robot_call(m, b):
    return m(b["l"], b["v_256"], b["v_512"], b["v_1024"], b["a"], b["l_mask"], b["v_mask"],
             b["a_mask"])


class _RefChain(torch.nn.Module):
    """BASELINE config 2 chain built from a given Attention_Block class (reference or ours)."""

    def __init__(self, block_cls, dim, n_heads, n_layers):
        super().__init__()
        self.blocks = torch.nn.ModuleList([block_cls(dim, n_heads) for _ in range(n_layers)])

    def forward(self, x, mask):
        q, s = x, None
        for blk in self.blocks:
            q, s = blk(q, x, x, mask, s)
        return q


def _chain_oracle(sd, b):
    pres = [f"blocks.{i}." for i in range(CHAIN["n_layers"])]
    return O.encoder_chain(sd, pres, b["x"], b["mask"], CHAIN["n_heads"])[0]


CASES: Dict[str, Case] = {}


def _add(c: Case):
    CASES[c.name] = c


_add(Case(
    name="realformer_state_transfer", family="realformer", overrides=dict(DROP=0.0, FFN=2),
    ref_model=lambda ns: ns.State_Transfer(**RF),
    our_model=lambda pkg: pkg.realformer.State_Transfer(**RF),
    batch=lambda: synth.realformer_batch(seed=11, B=3, P=3, L=(6, 5, 7), D=(20, 7, 10)),
    call=_rf_call,
    oracle=lambda sd, b: O.realformer_state_transfer(sd, b["l"], b["v"], b["a"], b["l_mask"],
                                                     b["v_mask"], b["a_mask"], 2, 2),
    loss=_window_loss, grad_inputs=["l", "v", "a"]))

_add(Case(
    name="mosei_concat_trans", family="mosei",
    overrides=dict(DROP=0.0, L_DIM=MOSEI_D[0], V_DIM=MOSEI_D[1], A_DIM=MOSEI_D[2]),
    ref_model=lambda ns: ns.Concat_Trans(**MOSEI),
    our_model=lambda pkg: pkg.cmu_mosei.Concat_Trans(**MOSEI, l_dim=MOSEI_D[0], v_dim=MOSEI_D[1],
                                                     a_dim=MOSEI_D[2]),
    batch=lambda: synth.mosei_batch(seed=12, B=4, L=(6, 9, 12), D=MOSEI_D),
    call=_rf_call,
    oracle=lambda sd, b: O.mosei_concat_trans(sd, b["l"], b["v"], b["a"], b["l_mask"], b["v_mask"],
                                              b["a_mask"], 2, 2),
    loss=_circle_mean, grad_inputs=["l", "v", "a"]))

_add(Case(
    name="renmme_base_model", family="renmme",
    overrides=dict(DROP=0.0, L_DIM=REN_D[0], V_DIM=REN_D[1], A_DIM=REN_D[2]),
    ref_model=lambda ns: ns.Base_model(**REN),
    our_model=lambda pkg: pkg.ren_mme.Base_model(**REN, l_dim=REN_D[0], v_dim=REN_D[1],
                                                 a_dim=REN_D[2]),
    batch=lambda: synth.renmme_batch(seed=13, B=6, L=(5, 7, 11), D=REN_D),
    call=lambda m, b: m(*b["inputs"]),
    oracle=lambda sd, b: O.renmme_base_model(sd, *b["inputs"], n_heads=4, n_layers=1),
    loss=_renmme_loss))

_add(Case(
    name="rencecps_concat_linear", family="rencecps", overrides=dict(DROP=0.0),
    ref_model=lambda ns: ns.Concat_Linear(48),
    our_model=lambda pkg: pkg.rencecps.Concat_Linear(48),
    batch=lambda: synth.rencecps_batch(seed=14, B=5, dim=48),
    call=lambda m, b: m(b["feat"]),
    oracle=lambda sd, b: O.rencecps_concat_linear(sd, b["feat"]),
    loss=_circle_mean, grad_inputs=["feat"]))

_add(Case(
    name="robot_multi_class", family="robot", overrides=dict(DROP=0.0),
    ref_model=lambda ns: ns.Multi_class(**ROBOT),
    our_model=lambda pkg: pkg.robot_demo.Multi_class(**ROBOT),
    batch=lambda: synth.robot_batch(seed=15, B=2, L=(5, 8, 8)),
    call=_robot_call,
    oracle=lambda sd, b: O.robot_multi_class(sd, b["l"], b["v_256"], b["v_512"], b["v_1024"],
                                             b["a"], b["l_mask"], b["v_mask"], b["a_mask"], 2, 2),
    loss=_circle_mean, grad_inputs=["l", "a"]))

_add(Case(
    name="encoder_chain", family="realformer", overrides=dict(DROP=0.0, FFN=2),
    ref_model=lambda ns: _RefChain(ns.Attention_Block, CHAIN["dim"], CHAIN["n_heads"],
                                   CHAIN["n_layers"]),
    our_model=lambda pkg: _RefChain(pkg.realformer.Attention_Block, CHAIN["dim"], CHAIN["n_heads"],
                                    CHAIN["n_layers"]),
    batch=lambda: synth.encoder_batch(seed=16, B=CHAIN["B"], L=CHAIN["L"], d=CHAIN["dim"]),
    call=lambda m, b: m(b["x"], b["mask"]),
    oracle=_chain_oracle,
    loss=_sq_mean, grad_inputs=["x"]))


# ------------------------------------------------------------------------------------------
def seeded_state(model: torch.nn.Module, seed: int = 1) -> Dict[str, torch.Tensor]:
    """state_dict of ``model`` with the zero-initialised gates re-drawn from U(-0.5, 0.5)."""
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return synth.randomize_gates(sd, seed)


def run_with_grads(fn, state: Dict[str, torch.Tensor], batch, loss_fn, lossfns, grad_inputs):
    """Generic fwd+bwd: ``fn(state, batch) -> logits``; returns logits, loss, param grads (only
    those that receive one) and grads of the requested float inputs."""
    st = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in state.items()}
    b = dict(batch)
    for k in grad_inputs:
        b[k] = batch[k].clone().requires_grad_(True)
    logits = fn(st, b)
    loss = loss_fn(logits, b, lossfns)
    loss.backward()
    grads = {k: v.grad.detach() for k, v in st.items() if v.grad is not None}
    igrads = {k: b[k].grad.detach() for k in grad_inputs}
    return logits.detach(), loss.detach(), grads, igrads


def run_module_with_grads(model, case: Case, batch, lossfns):
    b = dict(batch)
    for k in case.grad_inputs:
        b[k] = batch[k].clone().requires_grad_(True)
    model.zero_grad(set_to_none=True)
    logits = case.call(model, b)
    loss = case.loss(logits, b, lossfns)
    loss.backward()
    grads = {k: p.grad.detach() for k, p in model.named_parameters() if p.grad is not None}
    igrads = {k: b[k].grad.detach() for k in case.grad_inputs}
    return logits.detach(), loss.detach(), grads, igrads


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """max |a-b| / max |b| (the 'relative' of BASELINE.json's tolerances: relative to the
    tensor's scale, robust to exact zeros)."""
    a, b = a.double().cpu(), b.double().cpu()
    den = b.abs().max().item()
    num = (a - b).abs().max().item()
    return num / den if den > 0 else num


def golden_path(name: str) -> str:
    return os.path.join(GOLDEN_DIR, name + ".pt")


# ------------------------------------------------------------------------------------------
def trunk_per_block(towers, n_layers: int, keep_all: bool, pool: bool = True):
    """``blocks.fusion_trunk_multi`` walked chain by chain through each block's own ``forward``
    (a trunk group of one problem per call): the reference the grouped trunk is compared with."""
    from mmemo_b200 import blocks, ops
    segs = []
    for blks, feats, masks in towers:
        outs = {"l": [], "v": [], "a": []}
        for ci, (qm, sm) in enumerate(blocks.CHAINS):
            q, s, src = feats[qm], None, feats[sm]
            for i in range(n_layers):
                q, s = blks[n_layers * ci + i](q, src, src, masks[sm], s,
                                               emit_scores=i + 1 < n_layers)
                if keep_all or i + 1 == n_layers:
                    outs[qm].append(q)
        segs.append(outs["l"] + outs["a"] + outs["v"])
    return [ops.pool(t, 3) for t in segs] if pool else segs


def use_per_block_trunk(monkeypatch) -> None:
    """Make every model family run its fusion trunks through ``trunk_per_block``."""
    import mmemo_b200
    for mod in (mmemo_b200.cmu_mosei, mmemo_b200.ren_mme, mmemo_b200.robot_demo):
        monkeypatch.setattr(mod, "fusion_trunk_multi", trunk_per_block)
    monkeypatch.setattr(mmemo_b200.realformer, "fusion_trunk",
                        lambda blks, n_layers, feats, masks, keep_all:
                        trunk_per_block([(blks, feats, masks)], n_layers, keep_all)[0])
