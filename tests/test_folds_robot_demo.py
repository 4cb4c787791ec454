"""CPU tests of ``folds.forward`` for ``robot_demo.Multi_class`` with the library calls stubbed (as
in test_folds_forward.py): argument checks, and the library calls of one grouped training step
(forward, circle losses, backward) for k = 1, 2, 5 folds with the reference's dropout."""
from collections import Counter

import pytest
import torch

import mmemo_b200
from mmemo_b200 import folds, ops, synth
from mmemo_b200.robot_demo import Multi_class

KW = dict(dim=24, l_len=5, v_len=8, a_len=8, n_heads=2, n_layers=2, ffn=2)
NAMES = ("l", "v_256", "v_512", "v_1024", "a", "l_mask", "v_mask", "a_mask")


class _FakeLib:
    def mmemo_resattn_uses_tensor_cores(self, *a):
        return 0

    def mmemo_resattn_uses_mma(self, *a):
        return 1


@pytest.fixture()
def stub(monkeypatch):
    """Records the names of every library call (and torch.cat calls as "torch.cat")."""
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append(name))
    monkeypatch.setattr(ops, "_try_call", lambda name, *a: calls.append(name) or True)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(ops._lib, "load", lambda: _FakeLib())
    cat = torch.cat
    monkeypatch.setattr(torch, "cat", lambda *a, **k: calls.append("torch.cat") or cat(*a, **k))
    ops.clear_shadow_cache()
    yield calls
    ops.clear_shadow_cache()


def _batch(B):
    b = synth.robot_batch(seed=5, B=B, L=(5, 8, 8))
    return [b[k] for k in NAMES], b["label"]


def _grouped_step(ms, batches):
    ls = folds.forward(ms, [b[0] for b in batches])
    losses = folds.circle_losses(ls, [b[1] for b in batches])
    total = losses[0]
    for x in losses[1:]:
        total = total + x
    total.backward()
    return ls


def _own_step(m, args, label):
    ops.circle_loss_op(m(*args), label).mean().backward()


def _calls(stub, fn):
    fn()                    # the first step also casts the bf16 weight shadows
    stub.clear()
    fn()
    return Counter(stub)


def test_argument_errors(stub):
    args = _batch(3)[0]
    with pytest.raises(ValueError, match="Multi_class"):
        folds.forward([Multi_class(**KW), mmemo_b200.rencecps.Concat_Linear(48)], [args, args])
    other = Multi_class(**KW)
    other.n_layers = 1          # same parameters, walked as a 1-layer trunk of 18 chains
    with pytest.raises(ValueError, match="n_layers"):
        folds.forward([Multi_class(**KW), other], [args, args])
    with pytest.raises(ValueError, match="input tuples"):
        folds.forward([Multi_class(**KW), Multi_class(**KW)], [args])
    with pytest.raises(ValueError, match="8 inputs"):
        folds.forward([Multi_class(**KW)], [args[:5]])


def test_ensemble_still_rejects_multi_class():
    with pytest.raises(ValueError, match="Multi_class"):
        mmemo_b200.ensemble.Ensemble([Multi_class(**KW)])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_step_calls_do_not_grow_with_folds(stub, mode):
    """Pooling, classifier linear and loss calls per step are the same for k = 1, 2, 5 folds (one
    on a smaller batch); at k = 1 the grouped step makes no more calls than the model's own."""
    with mmemo_b200.precision(mode):
        per_k = {}
        for k in (1, 2, 5):
            ms = [Multi_class(**KW).train() for _ in range(k)]
            bs = [_batch(3 if i == k - 1 and k > 1 else 4) for i in range(k)]
            per_k[k] = _calls(stub, lambda: _grouped_step(ms, bs))
        m = Multi_class(**KW).train()
        own = _calls(stub, lambda: _own_step(m, *_batch(4)))
    assert sum(per_k[1].values()) <= sum(own.values()), (per_k[1], own)
    fixed = {n for n in per_k[1] if n.startswith(("mmemo_pool_", "mmemo_linear_fwd_grouped_f32",
                                                  "mmemo_linear_bwd_w_grouped_f32",
                                                  "mmemo_linear_bwd_x_grouped_f32",
                                                  "mmemo_circle"))}
    assert {"mmemo_pool_fwd_multi_arg_" + ("bf16" if mode == "bf16" else "f32"),
            "mmemo_linear_fwd_grouped_f32", "mmemo_circle_loss_fwd_multi"} <= fixed
    for k in (2, 5):
        for n in fixed:
            assert per_k[k][n] == per_k[1][n], (k, n, per_k[k])


@pytest.mark.parametrize("k", [1, 2, 5])
def test_grouped_projection_is_one_gemm_and_one_reduction(stub, k):
    """bf16 with dropout: the 5k projections are one epilogue-dropout GEMM forward and one
    reduction + one weight-gradient GEMM backward, with no separate dropout, position-add or
    concat kernels."""
    with mmemo_b200.precision("bf16"):
        ms = [Multi_class(**KW).train() for _ in range(k)]
        assert ms[0].unify_dimension.drop.p > 0
        bs = [_batch(3 if i == k - 1 and k > 1 else 4) for i in range(k)]
        c = _calls(stub, lambda: _grouped_step(ms, bs))
    assert c["mmemo_linear_fwd_grouped_dropout_bf16"] == 1
    assert c["mmemo_proj_dropout_bwd_bf16"] == 1
    # 5k input casts (the weight shadows are cached), 16 tensors per launch
    assert c["mmemo_cast_pad_f32_to_bf16_multi"] == -(-5 * k // 16)
    assert "torch.cat" not in c
    assert not {"mmemo_dropout_f32", "mmemo_dropout_bf16", "mmemo_rowsum_bf16"} & set(c)


def test_module_training_projection_is_grouped(stub):
    """robot_demo's own Unify_Dimension_Conv1d in training mode: one fused projection launch
    instead of five linears and five dropouts."""
    with mmemo_b200.precision("bf16"):
        m = Multi_class(**KW).train()
        c = _calls(stub, lambda: _own_step(m, *_batch(4)))
    assert c["mmemo_linear_fwd_grouped_dropout_bf16"] == 1
    assert c["mmemo_proj_dropout_bwd_bf16"] == 1
    assert not {"mmemo_dropout_f32", "mmemo_dropout_bf16"} & set(c)


def test_unused_parameters_get_no_gradient(stub):
    ms = [Multi_class(**KW).train() for _ in range(2)]
    _grouped_step(ms, [_batch(4), _batch(3)])
    for m in ms:
        for mod in (m.fully_connected, m.normalization):
            assert all(p.grad is None for p in mod.parameters())
        assert m.unify_dimension.visual_512.weight.grad is not None
        assert m.visual_position.position_embeddings.weight.grad.shape == (8, 24)
