"""Fold-ensemble uncertainty (mmemo_b200.ensemble: Uncertainty, fold_uncertainty,
fold_uncertainty_reference, Ensemble(..., return_uncertainty=True)).

CPU: the PyTorch reference against a per-row NumPy / SciPy computation, its invariants, argument
errors, and the library calls of a request (library stubbed as in test_ensemble.py).
GPU: the fold_uncertainty kernel against the reference over k, C, B and both input dtypes; the
head's per-member outputs; each of the four families end to end with the flag on and off."""
import math
from collections import Counter

import numpy as np
import pytest
import scipy.special
import scipy.stats
import torch

import mmemo_b200
from mmemo_b200 import ops, synth
from mmemo_b200.ensemble import (Ensemble, Uncertainty, fold_uncertainty,
                                 fold_uncertainty_reference)

DEV = "cuda"


def _logits(K, B, C, seed, dtype=torch.float32, device="cpu"):
    """Random fold logits with rows of very different scales: O(1), O(100) and O(1e4) offsets, so
    that the max subtraction matters and some probabilities underflow to exactly 0."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(K, B, C, generator=g, dtype=torch.float64) * 3
    if B:
        scale = torch.tensor([1.0, 40.0, 1.0, 0.01])[torch.arange(B) % 4].view(1, B, 1)
        shift = torch.tensor([0.0, 0.0, 1e4, -300.0])[torch.arange(B) % 4].view(1, B, 1)
        x = x * scale + shift
    return x.to(dtype).to(device)


def _naive(x: np.ndarray):
    """Row by row with scipy: softmax, scipy.stats.entropy (natural log)."""
    K, B, C = x.shape
    out = {k: [] for k in Uncertainty._fields}
    for b in range(B):
        p = np.stack([scipy.special.softmax(x[k, b]) for k in range(K)])
        mean = p.mean(0)
        h = scipy.stats.entropy(mean)
        eh = np.mean([scipy.stats.entropy(p[k]) for k in range(K)])
        out["mean_prob"].append(mean)
        out["variance"].append(p.var(0, ddof=1) if K > 1 else np.zeros(C))
        out["entropy"].append(h)
        out["expected_entropy"].append(eh)
        out["mutual_info"].append(max(h - eh, 0.0) if K > 1 else 0.0)
        out["label"].append(int(np.argmax(mean)))
    shapes = {"mean_prob": (B, C), "variance": (B, C)}
    return {k: np.asarray(v, dtype=np.float64).reshape(shapes.get(k, (B,))) for k, v in out.items()}


def _check_invariants(u: Uncertainty, C: int, atol: float):
    if u.entropy.numel() == 0:
        return
    assert (u.mutual_info >= -atol).all()
    assert (u.entropy <= math.log(C) + atol).all() and (u.entropy >= -atol).all()
    assert (u.expected_entropy <= u.entropy + atol).all()
    ones = torch.ones(u.entropy.shape, dtype=torch.float64, device=u.entropy.device)
    assert torch.allclose(u.mean_prob.double().sum(-1), ones, atol=10 * atol)
    assert (u.variance >= 0).all()


# ------------------------------------------------------------------------------------------------
# CPU: the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 5, 10])
@pytest.mark.parametrize("C", [1, 3, 7, 33])
@pytest.mark.parametrize("B", [0, 1, 17])
def test_reference_matches_scipy(K, B, C):
    x = _logits(K, B, C, seed=100 * K + 10 * C + B)
    ref = fold_uncertainty_reference(x)
    want = _naive(x.double().numpy())
    for name in ("mean_prob", "variance", "entropy", "expected_entropy", "mutual_info"):
        got = getattr(ref, name)
        assert got.dtype == torch.float32 and got.shape == want[name].shape, name
        np.testing.assert_allclose(got.numpy(), want[name], rtol=1e-6, atol=1e-7, err_msg=name)
    assert ref.label.dtype == torch.int64
    np.testing.assert_array_equal(ref.label.numpy(), want["label"])
    _check_invariants(ref, C, 1e-6)
    if K == 1:
        assert not ref.variance.any() and not ref.mutual_info.any()
    if C == 1:
        assert (ref.mean_prob == 1).all() and not ref.entropy.any() and not ref.label.any()


def test_reference_keeps_leading_row_dims_and_accepts_bf16():
    x = _logits(3, 8, 5, seed=1).view(3, 2, 4, 5)
    ref = fold_uncertainty_reference(x)
    assert ref.mean_prob.shape == (2, 4, 5) and ref.entropy.shape == (2, 4) == ref.label.shape
    flat = fold_uncertainty_reference(x.view(3, 8, 5))
    assert torch.equal(ref.entropy.view(8), flat.entropy)
    xb = x.bfloat16()
    assert torch.equal(fold_uncertainty_reference(xb).mean_prob, fold_uncertainty_reference(xb.float()).mean_prob)


def test_identical_folds_have_no_disagreement():
    x = _logits(1, 16, 7, seed=2).expand(6, 16, 7).contiguous()
    ref = fold_uncertainty_reference(x)
    assert ref.variance.abs().max() < 1e-12 and ref.mutual_info.abs().max() < 1e-6
    assert torch.allclose(ref.entropy, ref.expected_entropy, atol=1e-6)


def test_reference_rejects_bad_shapes():
    for shape in ((5,), (0, 3, 4), (2, 3, 0)):
        with pytest.raises(ValueError, match="K >= 1"):
            fold_uncertainty_reference(torch.zeros(shape))


def test_kernel_op_validates_arguments(monkeypatch):
    with pytest.raises(RuntimeError, match="CUDA"):
        fold_uncertainty(torch.zeros(2, 3, 4))
    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    with pytest.raises(ValueError, match=r"\(K, \.\.\., C\)"):
        fold_uncertainty(torch.zeros(4))
    with pytest.raises(TypeError, match="float32 or bfloat16"):
        fold_uncertainty(torch.zeros(2, 3, 4, dtype=torch.float16))
    with pytest.raises(ValueError, match="contiguous"):
        fold_uncertainty(torch.zeros(2, 4, 3).transpose(1, 2))
    with pytest.raises(ValueError, match="C >= 1"):
        fold_uncertainty(torch.zeros(2, 3, 0))
    with pytest.raises(ValueError, match="at most 1024"):
        fold_uncertainty(torch.zeros(2, 3, 1025))


# ------------------------------------------------------------------------------------------------
# CPU: the calls of a request (library stubbed)
# ------------------------------------------------------------------------------------------------
class _FakeLib:
    def mmemo_resattn_uses_tensor_cores(self, *a):
        return 0

    def mmemo_resattn_uses_mma(self, *a):
        return 1


@pytest.fixture()
def stub(monkeypatch):
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


def _small(family, B):
    """Small members of a family, their forward arguments, and the output shape."""
    if family == "State_Transfer":
        kw = dict(l_dim=20, v_dim=7, a_dim=10, dim=16, l_len=6, v_len=5, a_len=7, n_heads=2,
                  n_layers=2, ffn=2)
        b = synth.realformer_batch(seed=1, B=B, P=4, L=(6, 5, 7), D=(20, 7, 10))
        return (lambda: mmemo_b200.realformer.State_Transfer(**kw),
                [b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], (B, 4, 6))
    if family == "Concat_Trans":
        kw = dict(dim=24, l_len=6, v_len=9, a_len=12, n_heads=2, n_layers=1, ffn=1, l_dim=20,
                  v_dim=7, a_dim=10)
        b = synth.mosei_batch(seed=2, B=B, L=(6, 9, 12), D=(20, 7, 10))
        return (lambda: mmemo_b200.cmu_mosei.Concat_Trans(**kw),
                [b[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")], (B, 7))
    if family == "Base_model":
        kw = dict(dim=32, l_len=5, v_len=7, a_len=11, n_heads=4, n_layers=1, ffn=1, l_dim=24,
                  v_dim=20, a_dim=13)
        b = synth.renmme_batch(seed=3, B=B, L=(5, 7, 11), D=(24, 20, 13))
        return lambda: mmemo_b200.ren_mme.Base_model(**kw), list(b["inputs"]), (B, 9)
    b = synth.rencecps_batch(seed=4, B=B, dim=48)
    return lambda: mmemo_b200.rencecps.Concat_Linear(48), [b["feat"]], (B, 9)


FAMILIES = ("State_Transfer", "Concat_Trans", "Base_model", "Concat_Linear")


@pytest.mark.parametrize("family", FAMILIES)
def test_flag_adds_one_reduction_launch_and_changes_nothing_else(stub, family):
    """Flag off: the request's calls are exactly those of today.  Flag on: the same calls, the
    head entry point that also writes the members' outputs, and one fold_uncertainty launch on
    (K,) + the output's shape."""
    ctor, args, shape = _small(family, 6)
    ens = Ensemble([ctor() for _ in range(3)], use_graph=False)
    with mmemo_b200.precision("bf16"):
        ens(*args)
        stub.clear()
        out = ens(*args)
        off = list(stub)
        stub.clear()
        out2, unc = ens(*args, return_uncertainty=True)
        on = list(stub)
    assert out.shape == out2.shape == shape
    names_off, names_on = Counter(n for n, _ in off), Counter(n for n, _ in on)
    assert names_off["mmemo_ensemble_head_fwd"] == 1 and "mmemo_fold_uncertainty_f32" not in names_off
    expect = names_off - Counter({"mmemo_ensemble_head_fwd": 1})
    expect.update({"mmemo_ensemble_head_fwd_members": 1, "mmemo_fold_uncertainty_f32": 1})
    assert names_on == expect
    head = [a for n, a in on if n == "mmemo_ensemble_head_fwd_members"][0]
    uq = [a for n, a in on if n == "mmemo_fold_uncertainty_f32"][0]
    n_rows = math.prod(shape[:-1])
    assert uq[1:4] == (3, n_rows, shape[-1])
    assert head[-2] == uq[0]                      # the head's member buffer is what is reduced
    assert isinstance(unc, Uncertainty)
    assert unc.mean_prob.shape == unc.variance.shape == shape
    assert unc.entropy.shape == unc.expected_entropy.shape == unc.mutual_info.shape == shape[:-1]
    assert unc.label.shape == shape[:-1] and unc.label.dtype == torch.int64


# ------------------------------------------------------------------------------------------------
# GPU: the kernel
# ------------------------------------------------------------------------------------------------
def _assert_close_to_reference(u: Uncertainty, ref: Uncertainty, atol_p, atol_h):
    for name in ("mean_prob", "variance"):
        torch.testing.assert_close(getattr(u, name).cpu(), getattr(ref, name).cpu(), rtol=1e-5,
                                   atol=atol_p, msg=name)
    for name in ("entropy", "expected_entropy", "mutual_info"):
        torch.testing.assert_close(getattr(u, name).cpu(), getattr(ref, name).cpu(), rtol=1e-5,
                                   atol=atol_h, msg=name)
    # labels: equal except where the reference's top two mean probabilities (nearly) tie
    lab, rlab = u.label.cpu(), ref.label.cpu()
    diff = lab != rlab
    if diff.any():
        mp = ref.mean_prob.cpu()
        gap = mp.gather(-1, rlab.unsqueeze(-1)) - mp.gather(-1, lab.unsqueeze(-1))
        assert (gap.squeeze(-1)[diff] <= atol_p).all(), gap.squeeze(-1)[diff]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("K", [1, 2, 5, 10])
@pytest.mark.parametrize("C", [3, 7, 33, 128])
@pytest.mark.parametrize("B", [0, 1, 1000])
def test_kernel_matches_reference(dtype, K, C, B):
    x = _logits(K, B, C, seed=7 * K + C + B, dtype=dtype, device=DEV)
    u = fold_uncertainty(x)
    assert u.mean_prob.shape == (B, C) and u.entropy.shape == (B,) and u.label.dtype == torch.int64
    ref = fold_uncertainty_reference(x.cpu())      # bf16 -> float is exact on both sides
    _assert_close_to_reference(u, ref, atol_p=1e-6, atol_h=1e-5)
    _check_invariants(u, C, 1e-5)
    if K == 1:
        assert not u.variance.any() and not u.mutual_info.any()
    u2 = fold_uncertainty(x)
    assert all(torch.equal(a, b) for a, b in zip(u, u2))


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 64, 200, 1024])
def test_kernel_other_class_counts_and_row_dims(C):
    """C = 1, the chunk boundaries and the largest C; leading row dimensions kept."""
    x = _logits(4, 24, C, seed=C, device=DEV).view(4, 2, 12, C)
    u = fold_uncertainty(x)
    assert u.mean_prob.shape == (2, 12, C) and u.label.shape == (2, 12)
    _assert_close_to_reference(u, fold_uncertainty_reference(x.cpu()), atol_p=1e-6, atol_h=1e-5)
    if C == 1:
        assert (u.mean_prob == 1).all() and not u.entropy.any() and not u.label.any()


@pytest.mark.gpu
def test_kernel_rejects_bad_arguments():
    from mmemo_b200 import _lib
    lib, st = _lib.load(), torch.cuda.current_stream().cuda_stream
    x = torch.zeros(2, 4, 5, device=DEV)
    o = torch.empty(64, device=DEV)
    lb = torch.empty(4, dtype=torch.int64, device=DEV)
    p = [o.data_ptr()] * 5 + [lb.data_ptr()]
    assert lib.mmemo_fold_uncertainty_f32(x.data_ptr(), 2, 4, 1025, *p, st) == -2
    assert lib.mmemo_fold_uncertainty_f32(x.data_ptr(), 0, 4, 5, *p, st) == -1
    assert lib.mmemo_fold_uncertainty_f32(None, 2, 4, 5, *p, st) == -1
    assert lib.mmemo_fold_uncertainty_f32(None, 2, 0, 5, *p, st) == 0       # no rows: no launch
    assert lib.mmemo_ensemble_head_fwd_members(0, 1, None, 1, 1, 8, 0, 3, 1e-5, o.data_ptr(), None,
                                               st) == -1


@pytest.mark.gpu
@pytest.mark.parametrize("kind,B,P,F,d,Cn", [(1, 7, 3, 70, 96, 6), (0, 37, 1, 300, 0, 7)])
def test_head_member_outputs(kind, B, P, F, d, Cn):
    """K = 10 members (two launch tables): y is bitwise the plain entry point's, and member k's
    output is bitwise the plain entry point's output for member k alone (a mean over one member
    is that member's output: the division by 1 is exact)."""
    import ctypes as C
    from mmemo_b200 import _lib
    from tests.test_gpu_ensemble import _head_call, _head_problem
    K = 10
    mem, keep, ref = _head_problem(kind, K, B, P, F, d, Cn, seed=3)
    shape = (B, P, Cn) if kind == _lib.HEAD_STATE_TRANSFER else (B, Cn)
    y0, y1 = torch.empty(shape, device=DEV), torch.empty(shape, device=DEV)
    ym = torch.full((K,) + shape, float("nan"), device=DEV)
    assert _head_call(kind, mem, B, P, F, d, Cn, y0) == 0
    arr = (_lib.EnsembleMember * K)(*mem)
    assert _lib.load().mmemo_ensemble_head_fwd_members(
        kind, K, C.cast(arr, C.c_void_p), B, P, F, d, Cn, ops.LN_EPS, y1.data_ptr(), ym.data_ptr(),
        torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(y0, y1)
    for k in range(K):
        own = torch.empty(shape, device=DEV)
        assert _head_call(kind, [mem[k]], B, P, F, d, Cn, own) == 0
        assert torch.equal(ym[k], own), k
    torch.testing.assert_close(ym.mean(0), ref, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------------
# GPU: end to end
# ------------------------------------------------------------------------------------------------
def _gpu_members(family, K, B):
    ctor, args, shape = _small(family, B)
    models = []
    for k in range(K):
        torch.manual_seed(k)
        m = ctor()
        m.load_state_dict(synth.randomize_gates(
            {n: v.detach().clone() for n, v in m.state_dict().items()}, seed=60 + k))
        models.append(m.to(DEV).eval())
    return models, [t.to(DEV) for t in args], shape


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_end_to_end_flag_on_and_off(family, monkeypatch):
    """K = 4 members, fp32: with the flag on the logits are bitwise those of the flag-off call
    (graphed and ungraphed), and the uncertainty matches the reference applied to the members'
    own forwards (which agree with the grouped request to ~1e-5 of the logits' scale); the
    graphed ensemble keeps one graph per flag.  bf16: flag on and off agree, and the uncertainty
    follows the members' own bf16 forwards within bf16's tolerance."""
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.0)
    mmemo_b200.set_precision("fp32")
    ops.clear_shadow_cache()
    models, args, shape = _gpu_members(family, 4, 32)
    with torch.no_grad():
        ref = fold_uncertainty_reference(torch.stack([m(*args).float() for m in models]))
    graphed, direct = Ensemble(models), Ensemble(models, use_graph=False)
    for ens in (graphed, direct):
        off = ens(*args)
        on, unc = ens(*args, return_uncertainty=True)
        assert torch.equal(on, off)
        assert unc.mean_prob.shape == shape and unc.entropy.shape == shape[:-1]
        _assert_close_to_reference(unc, ref, atol_p=5e-5, atol_h=2e-4)
        _check_invariants(unc, shape[-1], 1e-5)
        assert torch.equal(ens(*args), off)
    assert len(graphed._graphs) == 2
    try:
        with mmemo_b200.precision("bf16"), torch.no_grad():
            ref_bf = fold_uncertainty_reference(torch.stack([m(*args).float() for m in models]))
            off = graphed(*args)
            on, unc = graphed(*args, return_uncertainty=True)
        torch.testing.assert_close(on, off, rtol=1e-6, atol=1e-6)
        _check_invariants(unc, shape[-1], 1e-5)
        torch.testing.assert_close(unc.mean_prob, ref_bf.mean_prob.to(DEV), rtol=0, atol=5e-2)
        torch.testing.assert_close(unc.entropy, ref_bf.entropy.to(DEV), rtol=0, atol=1e-1)
    finally:
        mmemo_b200.set_precision("fp32")
