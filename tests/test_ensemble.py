"""CPU tests of ``mmemo_b200.ensemble.Ensemble`` with the library calls stubbed (as in
test_host_plumbing.py): constructor checks, output shapes, and the calls one request makes."""
from collections import Counter

import pytest
import torch

import mmemo_b200
from mmemo_b200 import ops, synth
from mmemo_b200.ensemble import Ensemble

GEMM = "mmemo_linear_fwd_grouped_bf16"


class _FakeLib:
    def mmemo_resattn_uses_tensor_cores(self, *a):
        return 0

    def mmemo_resattn_uses_mma(self, *a):
        return 1


@pytest.fixture()
def stub(monkeypatch):
    """Records (name, args) of every library call."""
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(ops, "_try_call", lambda name, *a: calls.append((name, a)) or True)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(ops._lib, "load", lambda: _FakeLib())
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.0)
    ops.clear_shadow_cache()
    yield calls
    ops.clear_shadow_cache()


# small shapes of the four families: (constructor, batch -> forward args, output shape)
def _st():
    kw = dict(l_dim=20, v_dim=7, a_dim=10, dim=16, l_len=6, v_len=5, a_len=7, n_heads=2, n_layers=2,
              ffn=2)
    b = synth.realformer_batch(seed=1, B=3, P=4, L=(6, 5, 7), D=(20, 7, 10))
    return (lambda: mmemo_b200.realformer.State_Transfer(**kw),
            [b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], (3, 4, 6))


def _ct():
    kw = dict(dim=24, l_len=6, v_len=9, a_len=12, n_heads=2, n_layers=1, ffn=1, l_dim=20, v_dim=7,
              a_dim=10)
    b = synth.mosei_batch(seed=2, B=4, L=(6, 9, 12), D=(20, 7, 10))
    return (lambda: mmemo_b200.cmu_mosei.Concat_Trans(**kw),
            [b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], (4, 7))


def _bm():
    kw = dict(dim=32, l_len=5, v_len=7, a_len=11, n_heads=4, n_layers=1, ffn=1, l_dim=24, v_dim=20,
              a_dim=13)
    b = synth.renmme_batch(seed=3, B=6, L=(5, 7, 11), D=(24, 20, 13))
    return lambda: mmemo_b200.ren_mme.Base_model(**kw), list(b["inputs"]), (6, 9)


def _cl():
    b = synth.rencecps_batch(seed=4, B=5, dim=48)
    return lambda: mmemo_b200.rencecps.Concat_Linear(48), [b["feat"]], (5, 9)


FAMILIES = {"State_Transfer": _st, "Concat_Trans": _ct, "Base_model": _bm, "Concat_Linear": _cl}
# bf16 library calls of ONE member's eval() forward at these families' BASELINE shapes
ONE_MEMBER = {"State_Transfer": 21, "Concat_Trans": 14, "Base_model": 20, "Concat_Linear": 1}


def _request(calls, ens, args):
    """Calls of one steady-state request (the first one also casts the weight shadows)."""
    ens(*args)
    calls.clear()
    out = ens(*args)
    return out, list(calls)


def test_constructor_errors(stub):
    ctor, _, _ = _ct()
    with pytest.raises(ValueError, match="at least one"):
        Ensemble([])
    with pytest.raises(ValueError, match="Linear"):
        Ensemble([torch.nn.Linear(2, 2)])
    with pytest.raises(ValueError, match="Concat_Linear"):
        Ensemble([ctor(), mmemo_b200.rencecps.Concat_Linear(48)])
    with pytest.raises(ValueError, match="shape"):
        Ensemble([mmemo_b200.rencecps.Concat_Linear(48), mmemo_b200.rencecps.Concat_Linear(32)])
    kw = dict(dim=24, l_len=6, v_len=9, a_len=12, n_layers=1, ffn=1, l_dim=20, v_dim=7, a_dim=10)
    with pytest.raises(ValueError, match="n_heads"):
        Ensemble([mmemo_b200.cmu_mosei.Concat_Trans(n_heads=2, **kw),
                  mmemo_b200.cmu_mosei.Concat_Trans(n_heads=4, **kw)])
    m = ctor().train()
    ens = Ensemble([m])
    assert not m.training and ens.models == [m]


def test_cpu_inputs_raise():
    ctor, args, _ = _cl()
    with pytest.raises(RuntimeError, match="CUDA"):
        Ensemble([ctor()])(*args)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_output_shape_and_one_pool_and_head_call(stub, family, mode):
    ctor, args, shape = FAMILIES[family]()
    ens = Ensemble([ctor() for _ in range(3)], use_graph=False)
    with mmemo_b200.precision(mode):
        out, calls = _request(stub, ens, args)
    assert out.shape == shape and out.dtype == torch.float32
    names = Counter(n for n, _ in calls)
    assert names["mmemo_ensemble_head_fwd"] == 1
    pools = sum(v for k, v in names.items() if k.startswith("mmemo_pool"))
    assert pools == (0 if family == "Concat_Linear" else 1)
    assert pools == names[f"mmemo_pool_fwd_multi_{'bf16' if mode == 'bf16' else 'f32'}"]
    if family == "Base_model":       # the towers' shared LayerNorm: one grouped call, 6 per member
        ln = [a[0] for n, a in calls if n.startswith("mmemo_add_ln_fwd_grouped")]
        assert ln.count(18) == 1 and not any(n.startswith("mmemo_add_ln_fwd_f") or
                                             n == "mmemo_add_ln_fwd_bf16" for n, _ in calls)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_bf16_calls_do_not_grow_with_members(stub, family):
    """bf16: a 4-member request makes no more library calls than ONE member's forward does today.
    Only the grouped GEMM grows with the members, and only by its 48-problem chunks: its problems
    scale with K and every logical GEMM group still ends in at most one partial chunk."""
    ctor, args, _ = FAMILIES[family]()
    per_k, gemm = {}, {}
    with mmemo_b200.precision("bf16"):
        for K in (1, 2, 4, 5):
            ens = Ensemble([ctor() for _ in range(K)], use_graph=False)
            calls = _request(stub, ens, args)[1]
            per_k[K] = Counter(n for n, _ in calls)
            gemm[K] = [a[0] for n, a in calls if n == GEMM]
    assert sum(per_k[4].values()) <= ONE_MEMBER[family], per_k[4]
    base = {k: v for k, v in per_k[1].items() if k != GEMM}
    for K, c in per_k.items():
        assert {k: v for k, v in c.items() if k != GEMM} == base, (K, c)
        assert all(n <= 48 for n in gemm[K]) and sum(gemm[K]) == K * sum(gemm[1]), (K, gemm[K])
        assert sum(n < 48 for n in gemm[K]) <= len(gemm[1]), (K, gemm[K])


@pytest.mark.parametrize("family", ["State_Transfer", "Concat_Trans", "Base_model"])
def test_each_raw_input_is_cast_once(stub, family):
    """bf16: every distinct raw input appears once among the cast problems of a request, whatever
    the number of members; the casts read the caller's tensors (or, for the halves of a
    (B, 2, L, D) input, one copy each)."""
    ctor, args, _ = FAMILIES[family]()
    n_inputs = 3 if family == "State_Transfer" else 6
    with mmemo_b200.precision("bf16"):
        for K in (1, 4):
            ens = Ensemble([ctor() for _ in range(K)], use_graph=False)
            _, calls = _request(stub, ens, args)
            srcs = [p for n, a in calls if n == "mmemo_cast_pad_f32_to_bf16_multi"
                    for p in list(a[1])[:a[0]]]
            assert len(srcs) == n_inputs and len(set(srcs)) == n_inputs, (K, srcs)


def test_realformer_tower_matches_the_other_families(stub):
    m = mmemo_b200.realformer.Multi_class(20, 7, 10, 16, 6, 5, 7, 2, 2, 2)
    l, v, a = torch.randn(2, 6, 20), torch.randn(2, 5, 7), torch.randn(2, 7, 10)
    blocks, feats, masks = m._tower(l, v, a, torch.ones(2, 6), torch.ones(2, 5), torch.ones(2, 7))
    assert blocks is m.multimodal_blocks
    assert {k: tuple(t.shape) for k, t in feats.items()} == {"l": (2, 6, 16), "v": (2, 5, 16),
                                                            "a": (2, 7, 16)}
    assert set(masks) == {"l", "v", "a"}
    with pytest.raises(RuntimeError):
        m._tower(torch.randn(2, 9, 20), v, a, torch.ones(2, 9), torch.ones(2, 5), torch.ones(2, 7))
