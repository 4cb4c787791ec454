"""CPU tests of ``mmemo_b200.folds`` with the library calls stubbed (as in test_ensemble.py):
argument checks, and the library calls of one grouped training step (forward, losses, backward)
for k = 1, 2, 5 folds against one model's own step."""
from collections import Counter

import pytest
import torch

import mmemo_b200
from mmemo_b200 import folds, ops, synth


class _FakeLib:
    def mmemo_resattn_uses_tensor_cores(self, *a):
        return 0

    def mmemo_resattn_uses_mma(self, *a):
        return 1


@pytest.fixture()
def stub(monkeypatch):
    """Records the names of every library call."""
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append(name))
    monkeypatch.setattr(ops, "_try_call", lambda name, *a: calls.append(name) or True)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(ops._lib, "load", lambda: _FakeLib())
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.0)
    ops.clear_shadow_cache()
    yield calls
    ops.clear_shadow_cache()


# (constructor, batch(B) -> (forward args, labels, weights or None), uses R-Drop)
def _st():
    kw = dict(l_dim=20, v_dim=7, a_dim=10, dim=16, l_len=6, v_len=5, a_len=7, n_heads=2, n_layers=2,
              ffn=2)

    def batch(B):
        b = synth.realformer_batch(seed=1, B=B, P=4, L=(6, 5, 7), D=(20, 7, 10))
        return ([b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], b["label"],
                b["wmask"].float())
    return lambda: mmemo_b200.realformer.State_Transfer(**kw), batch, False


def _ct():
    kw = dict(dim=24, l_len=6, v_len=9, a_len=12, n_heads=2, n_layers=1, ffn=1, l_dim=20, v_dim=7,
              a_dim=10)

    def batch(B):
        b = synth.mosei_batch(seed=2, B=B, L=(6, 9, 12), D=(20, 7, 10))
        return [b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], b["label"], None
    return lambda: mmemo_b200.cmu_mosei.Concat_Trans(**kw), batch, False


def _bm():
    kw = dict(dim=32, l_len=5, v_len=7, a_len=11, n_heads=4, n_layers=1, ffn=1, l_dim=24, v_dim=20,
              a_dim=13)

    def batch(B):
        b = synth.renmme_batch(seed=3, B=B, L=(5, 7, 11), D=(24, 20, 13))
        return list(b["inputs"]), b["label"], None
    return lambda: mmemo_b200.ren_mme.Base_model(**kw), batch, True


def _cl():
    def batch(B):
        b = synth.rencecps_batch(seed=4, B=B, dim=48)
        return [b["feat"]], b["label"], None
    return lambda: mmemo_b200.rencecps.Concat_Linear(48), batch, False


FAMILIES = {"State_Transfer": _st, "Concat_Trans": _ct, "Base_model": _bm, "Concat_Linear": _cl}


def _own_step(m, args, label, weight, rdrop):
    lg = m(*args)
    loss = ops.circle_loss_op(lg, label)
    loss = (loss * weight).mean() if weight is not None else loss.mean()
    if rdrop:
        loss = loss + ops.rdrop_kl_op(lg)
    loss.backward()


def _grouped_step(ms, batches, rdrop):
    ls = folds.forward(ms, [b[0] for b in batches])
    ws = None if batches[0][2] is None else [b[2] for b in batches]
    losses = folds.circle_losses(ls, [b[1] for b in batches], ws)
    if rdrop:
        losses = [c + r for c, r in zip(losses, folds.rdrop_kl(ls))]
    total = losses[0]
    for x in losses[1:]:
        total = total + x
    total.backward()
    return ls


def _calls(stub, fn):
    fn()                    # the first step also casts the bf16 weight shadows
    stub.clear()
    fn()
    return Counter(stub)


def test_argument_errors(stub):
    ctor, batch, _ = _ct()
    args = batch(4)[0]
    with pytest.raises(ValueError, match="input tuples"):
        folds.forward([ctor(), ctor()], [args])
    with pytest.raises(ValueError, match="Concat_Linear"):
        folds.forward([ctor(), mmemo_b200.rencecps.Concat_Linear(48)], [args, args])
    with pytest.raises(ValueError, match="shape"):
        folds.forward([mmemo_b200.rencecps.Concat_Linear(48), mmemo_b200.rencecps.Concat_Linear(32)],
                      [args, args])
    with pytest.raises(ValueError, match="train"):
        folds.forward([ctor().train(), ctor().eval()], [args, args])
    with pytest.raises(ValueError, match="one entry per fold"):
        folds.circle_losses([torch.zeros(2, 7)], [])


def test_cpu_inputs_raise():
    ctor, batch, _ = _cl()
    with pytest.raises(RuntimeError, match="CUDA"):
        folds.forward([ctor()], [batch(4)[0]])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_step_calls_do_not_grow_with_folds(stub, family, mode):
    """One grouped training step (forward, losses, backward) makes the same library calls for
    k = 1, 2 and 5 folds (one fold with a smaller batch), with the exception the grouped GEMMs and
    LayerNorms of the trunk chunk their tables (48 / 40 problems) and the float32 parity mode runs
    the trunk's GEMMs and attention per problem.  At k = 1 it makes no more calls than one model's
    own step."""
    ctor, batch, rdrop = FAMILIES[family]()
    with mmemo_b200.precision(mode):
        per_k = {}
        for k in (1, 2, 5):
            ms = [ctor().train() for _ in range(k)]
            bs = [batch(4 if i == k - 1 and k > 1 else 6) for i in range(k)]
            per_k[k] = _calls(stub, lambda: _grouped_step(ms, bs, rdrop))
        m = ctor().train()
        own = _calls(stub, lambda: _own_step(m, *batch(6), rdrop))
    assert sum(per_k[1].values()) <= sum(own.values()), (per_k[1], own)
    heads = {n for n in per_k[1] if n.startswith(("mmemo_pool_", "mmemo_linear_fwd_grouped_f32",
                                                    "mmemo_linear_bwd_x_grouped_f32",
                                                    "mmemo_linear_bwd_w_grouped_f32",
                                                    "mmemo_state_transfer", "mmemo_bilinear",
                                                    "mmemo_circle", "mmemo_rdrop"))}
    assert heads
    for k in (2, 5):
        for n in heads:
            assert per_k[k][n] == per_k[1][n], (k, n, per_k[k])
    if mode == "bf16" and family != "State_Transfer":
        grow = {n: per_k[5][n] - per_k[1][n] for n in per_k[5] if per_k[5][n] != per_k[1][n]}
        assert set(grow) <= {"mmemo_linear_fwd_grouped_bf16", "mmemo_linear_bwd_w_grouped_bf16",
                             "mmemo_linear_bwd_x_grouped_bf16", "mmemo_add_ln_fwd_grouped_bf16",
                             "mmemo_add_ln_bwd_grouped_bf16", "mmemo_cast_pad_f32_to_bf16_multi",
                             "mmemo_colsum_grouped_bf16", "mmemo_resattn_fwd_grouped_bf16",
                             "mmemo_resattn_bwd_grouped_bf16", "mmemo_cast_f32_to_bf16_multi",
                             "mmemo_dropout_multi_bf16", "mmemo_sum_grouped_bf16"}, grow


@pytest.mark.parametrize("family", list(FAMILIES))
def test_one_pooling_head_and_loss_call_per_direction(stub, family):
    ctor, batch, rdrop = FAMILIES[family]()
    with mmemo_b200.precision("bf16"):
        ms = [ctor().train() for _ in range(3)]
        bs = [batch(6), batch(6), batch(4)]
        c = _calls(stub, lambda: _grouped_step(ms, bs, rdrop))
    pool = 0 if family == "Concat_Linear" else 1
    assert c["mmemo_pool_fwd_multi_arg_bf16"] == pool and c["mmemo_pool_bwd_multi_bf16"] == pool
    head = "state_transfer" if family == "State_Transfer" else "bilinear_head"
    assert c[f"mmemo_{head}_fwd_multi"] == 1 and c[f"mmemo_{head}_bwd_multi"] == 1
    assert c["mmemo_circle_loss_fwd_multi"] == 1 and c["mmemo_circle_loss_bwd_multi"] == 1
    assert c["mmemo_rdrop_kl_fwd_multi"] == c["mmemo_rdrop_kl_bwd_multi"] == int(rdrop)
    n_lin = 2 if family == "State_Transfer" else 1
    for n in ("fwd", "bwd_x", "bwd_w"):
        want = 0 if (n == "bwd_x" and family == "Concat_Linear") else n_lin
        assert c[f"mmemo_linear_{n}_grouped_f32"] == want, c
    assert not any(n in c for n in ("mmemo_circle_loss_fwd", "mmemo_bilinear_head_fwd",
                                    "mmemo_state_transfer_fwd", "mmemo_pool_fwd_bf16",
                                    "mmemo_linear_fwd_f32"))


def test_outputs_have_each_folds_shape(stub):
    ctor, batch, _ = _st()
    ms = [ctor().train() for _ in range(3)]
    bs = [batch(3), batch(3), batch(2)]
    ls = folds.forward(ms, [b[0] for b in bs])
    assert [tuple(x.shape) for x in ls] == [(3, 4, 6), (3, 4, 6), (2, 4, 6)]
    losses = folds.circle_losses(ls, [b[1] for b in bs], [b[2] for b in bs])
    assert len(losses) == 3 and all(x.shape == () for x in losses)
