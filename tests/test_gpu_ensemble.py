"""Ensemble inference of k fold models on the GPU (mmemo_b200.ensemble.Ensemble): the grouped
request against the CPU oracle's mean of the members at BASELINE shapes, the graphed request against
the members called one by one, and the two kernels of csrc/ensemble.cu against the per-member ops."""
import ctypes as C

import pytest
import torch

import mmemo_b200
from mmemo_b200 import _lib, ops, synth
from mmemo_b200.ensemble import Ensemble
from oracle import mmemo_oracle as O
from tests.cases import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL32, TOLBF = 1e-4, 2e-2
ARGS6 = ("l", "v", "a", "l_mask", "v_mask", "a_mask")


@pytest.fixture(autouse=True)
def _defaults(monkeypatch):
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.0)
    mmemo_b200.set_precision("fp32")
    ops.clear_shadow_cache()
    yield
    mmemo_b200.set_precision("fp32")


# family -> (constructor, batch(seed, small) -> (device args, CPU args), oracle(sd, CPU args))
def _st(seed, small):
    b = synth.realformer_batch(seed=seed, B=8 if small else 32, P=6)
    return [b[k] for k in ARGS6]


def _ct(seed, small):
    b = synth.mosei_batch(seed=seed, B=8 if small else 32)
    return [b[k] for k in ARGS6]


def _bm(seed, small):
    return list(synth.renmme_batch(seed=seed, B=32 if small else 256)["inputs"])


def _cl(seed, small):
    return [synth.rencecps_batch(seed=seed, B=16 if small else 128)["feat"]]


FAMILIES = {
    "State_Transfer": (lambda: mmemo_b200.realformer.State_Transfer(300, 35, 74, 96, 50, 50, 50, 6, 2, 2),
                       _st, lambda sd, a: O.realformer_state_transfer(sd, *a, 6, 2)),
    "Concat_Trans": (lambda: mmemo_b200.cmu_mosei.Concat_Trans(96, 20, 100, 200, 6, 1, 1),
                     _ct, lambda sd, a: O.mosei_concat_trans(sd, *a, 6, 1)),
    "Base_model": (lambda: mmemo_b200.ren_mme.Base_model(), _bm,
                   lambda sd, a: O.renmme_base_model(sd, *a)),
    "Concat_Linear": (lambda: mmemo_b200.rencecps.Concat_Linear(2304), _cl,
                      lambda sd, a: O.rencecps_concat_linear(sd, *a)),
}


def _members(family, K, seed0=0):
    ctor = FAMILIES[family][0]
    models, sds = [], []
    for k in range(K):
        torch.manual_seed(seed0 + k)
        m = ctor()
        sd = synth.randomize_gates({n: v.detach().clone() for n, v in m.state_dict().items()},
                                   seed=50 + seed0 + k)
        m.load_state_dict(sd)
        models.append(m.to(DEV).eval())
        sds.append(sd)
    return models, sds


def _sequential_mean(models, args):
    with torch.no_grad():
        pred = models[0](*args)
        for m in models[1:]:
            pred = pred + m(*args)
    return pred / len(models)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_five_members_match_oracle_mean_at_baseline_shapes(family):
    """K = 5 fold models (differently seeded weights and gates) at the BASELINE inference shapes:
    the grouped ensemble against the oracle's mean of the members, fp32 <= 1e-4 and bf16 <= 2e-2.
    (cfg 4: ten towers, 90 attention problems per launch: above one launch table.)"""
    models, sds = _members(family, 5)
    args = FAMILIES[family][1](1234, False)
    with torch.no_grad():
        ref = sum(FAMILIES[family][2](sd, args) for sd in sds) / 5
    dev_args = [t.to(DEV) for t in args]
    for prec, tol in (("fp32", TOL32), ("bf16", TOLBF)):
        with mmemo_b200.precision(prec):
            out = Ensemble(models)(*dev_args)
        assert out.dtype == torch.float32 and out.shape == ref.shape
        err = rel_err(out, ref)
        print(f"{family} {prec}: rel err {err:.2e}")
        assert err <= tol, (prec, err)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_graphed_equals_ungraphed_equals_members_one_by_one(family):
    """fp32: the graphed request (one graph for three input seeds, a second for a smaller batch),
    the ungraphed request and the members called one by one agree to 1e-5.  bf16: after
    load_state_dict + refresh() the output follows the new weights."""
    models, _ = _members(family, 4)
    make = FAMILIES[family][1]
    ens, direct = Ensemble(models), Ensemble(models, use_graph=False)
    for seed in (1, 2, 3):
        args = [t.to(DEV) for t in make(seed, False)]
        ref = _sequential_mean(models, args)
        out = ens(*args)
        assert rel_err(out, ref) <= 1e-5 and rel_err(direct(*args), ref) <= 1e-5, seed
    assert len(ens._graphs) == 1
    args = [t.to(DEV) for t in make(4, True)]
    assert rel_err(ens(*args), _sequential_mean(models, args)) <= 1e-5
    assert len(ens._graphs) == 2
    with mmemo_b200.precision("bf16"):
        old = ens(*args)
        _, new_sds = _members(family, 4, seed0=20)
        for m, sd in zip(models, new_sds):
            m.load_state_dict(sd)
        ens.refresh()
        out = ens(*args)
        ref = _sequential_mean(models, args)
    assert rel_err(out, ref) <= TOLBF
    assert rel_err(old, ref) > 10 * TOLBF


# ------------------------------------------------------------------------------------------------
# the kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pool_multi_is_bitwise_equal_to_pool_per_tower(dtype):
    """20 towers of 3 groups x 6 slots (14 towers per launch: two launches) against
    mmemo_pool_fwd_* per tower."""
    g = torch.Generator(device=DEV).manual_seed(0)
    B, d, lens = 5, 96, (20, 37, 9)
    towers = [[torch.randn(B, L, d, generator=g, device=DEV).to(dtype) for L in lens for _ in range(6)]
              for _ in range(20)]
    got = ops.pool_multi(towers, 3)
    for tw, out in zip(towers, got):
        assert torch.equal(out, ops.pool(tw, 3))


def _head_problem(kind, K, B, P, F, d, Cn, seed=0):
    """K members' parameters and inputs, and the per-member ops' mean (the reference)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, device=DEV) * 0.3
    mem, keep, ref = [], [], None
    for _ in range(K):
        if kind == _lib.HEAD_BILINEAR:
            feat = r(B, 2, F)
            wl, wt, T, gm, bt, wo, bo = r(Cn, F), r(Cn, F), r(Cn, Cn, Cn), r(Cn) + 1, r(Cn), r(Cn, 2 * Cn), r(Cn)
            out = ops.bilinear_head(ops.linear(feat[:, 1], wt), ops.linear(feat[:, 0], wl), T, gm, bt, wo, bo)
            last, this = feat[:, 0], feat[:, 1]
            mem.append(_lib.EnsembleMember(last.data_ptr(), last.stride(0), this.data_ptr(),
                                           this.stride(0), wl.data_ptr(), wt.data_ptr(), None,
                                           gm.data_ptr(), bt.data_ptr(), wo.data_ptr(), bo.data_ptr(),
                                           T.data_ptr()))
            keep += [feat, wl, wt, T, gm, bt, wo, bo]
        else:
            x = r(B * P, F)
            wf, bf, gm, bt, wc, bc, T = r(d, F), r(d), r(d) + 1, r(d), r(2 * Cn, d), r(2 * Cn), r(Cn, Cn)
            h = ops.add_ln(None, ops.linear(x, wf, bf), None, gm, bt, relu=True)
            out = ops.state_transfer_op(ops.linear(h, wc, bc).view(B, P, 2 * Cn), T)
            mem.append(_lib.EnsembleMember(x.data_ptr(), F, None, 0, wf.data_ptr(), None,
                                           bf.data_ptr(), gm.data_ptr(), bt.data_ptr(),
                                           wc.data_ptr(), bc.data_ptr(), T.data_ptr()))
            keep += [x, wf, bf, gm, bt, wc, bc, T]
        ref = out if ref is None else ref + out
    return mem, keep, ref / K


def _head_call(kind, mem, B, P, F, d, Cn, out):
    arr = (_lib.EnsembleMember * len(mem))(*mem)
    rc = _lib.load().mmemo_ensemble_head_fwd(kind, len(mem), C.cast(arr, C.c_void_p), B, P, F, d,
                                              Cn, ops.LN_EPS, out.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("kind,B,P,F,d,Cn", [
    (_lib.HEAD_STATE_TRANSFER, 32, 6, 576, 96, 6),
    (_lib.HEAD_STATE_TRANSFER, 5, 3, 70, 1024, 16),
    (_lib.HEAD_BILINEAR, 256, 1, 768, 0, 9),
    (_lib.HEAD_BILINEAR, 37, 1, 2304, 0, 7)])
def test_ensemble_head_matches_per_member_ops(kind, B, P, F, d, Cn):
    """K = 10 members (two launch tables of 8) against ops.linear + ops.bilinear_head /
    add_ln + ops.state_transfer_op per member and their mean, <= 1e-5; two runs bitwise equal."""
    mem, keep, ref = _head_problem(kind, 10, B, P, F, d, Cn)
    shape = (B, P, Cn) if kind == _lib.HEAD_STATE_TRANSFER else (B, Cn)
    y1, y2 = torch.empty(shape, device=DEV), torch.empty(shape, device=DEV)
    assert _head_call(kind, mem, B, P, F, d, Cn, y1) == 0
    assert _head_call(kind, mem, B, P, F, d, Cn, y2) == 0
    assert torch.equal(y1, y2)
    assert rel_err(y1, ref) <= 1e-5, rel_err(y1, ref)


def test_ensemble_head_rejects_bad_arguments():
    mem, keep, _ = _head_problem(_lib.HEAD_BILINEAR, 2, 4, 1, 32, 0, 5)
    y = torch.empty(4, 17, device=DEV)
    assert _head_call(_lib.HEAD_BILINEAR, mem, 4, 1, 32, 0, 17, y) == -2       # C = 17
    mem_st, keep_st, _ = _head_problem(_lib.HEAD_STATE_TRANSFER, 1, 2, 2, 32, 8, 4)
    assert _head_call(_lib.HEAD_STATE_TRANSFER, mem_st, 2, 2, 32, 1025, 4, y) == -2   # d = 1025
    mem[1].trans = None
    assert _head_call(_lib.HEAD_BILINEAR, mem, 4, 1, 32, 0, 5, y) == -1        # null pointer
