"""k-fold training on the GPU: the multi-optimizer step (optim.step_group over
mmemo_adam_step_multi_f32 / mmemo_grad_sqnorm_multi_f32) against each fold stepped alone, and
grouped launches with more problems than one launch table holds (a 5-member bf16 ensemble: 45
attention / LayerNorm problems per call)."""
import pytest
import torch

import mmemo_b200
from mmemo_b200 import ops, synth
from mmemo_b200 import optim as mo
from oracle import mmemo_oracle as O
from tests.cases import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL32, TOLBF = 1e-4, 2e-2
ARGS = ("l", "v", "a", "l_mask", "v_mask", "a_mask")


def _folds(lrs):
    """Three Concat_Trans(96, 50, 50, 50, 6, 2, 1) folds with differently seeded weights and gates
    and their fused AdamW (clip 1.0), lr per fold."""
    models, opts = [], []
    for k, lr in enumerate(lrs):
        torch.manual_seed(k)
        m = mmemo_b200.cmu_mosei.Concat_Trans(96, 50, 50, 50, 6, 2, 1)
        m.load_state_dict(synth.randomize_gates(
            {n: v.detach().clone() for n, v in m.state_dict().items()}, seed=7 + k))
        m = m.to(DEV).train()
        models.append(m)
        opts.append(mo.AdamW(m.parameters(), lr=lr, max_grad_norm=1.0))
    return models, opts


def _loss(m, b):
    return ops.circle_loss_op(m(*[b[k] for k in ARGS]), b["label"]).mean()


@pytest.mark.parametrize("lrs", [(1e-4, 1e-4, 1e-4), (1e-4, 3e-4, 3e-5)])
def test_step_group_trains_like_each_fold_alone(lrs):
    """20 AdamW steps (clip 1.0), fp32, of three folds (fold 2 with a smaller batch): the grouped
    step (sum of the fold losses, one backward, ``step_group``) against each fold run alone
    (its own loss, backward and ``optimizer.step()``) on the same batches.  Every step, the losses
    and every parameter gradient must agree to 1e-4; the alone folds are then stepped with the
    grouped gradients, so the final parameters (1e-4) compare the two optimizer paths only.  (The
    fp32 LayerNorm parameter gradients are summed with float atomics, layernorm.cu: two runs differ
    in the last bits, and Adam's m / sqrt(v) turns such a difference in a near-zero gradient element
    into a step of size lr, so parameters trained on separately computed gradients are not
    comparable at 1e-4 after 20 steps.)  The scalar gates a, b, c are left out of the gradient
    bound, as in test_gpu_models.py: each gradient is ONE float32 sum over every score or row
    element of the layer, accumulated with atomicAdd in arbitrary order, and its terms cancel."""
    batches = [[{k: v.to(DEV) for k, v in synth.mosei_batch(seed=100 * k + s, B=8 if k < 2 else 5,
                                                         L=(50, 50, 50)).items()}
                for s in range(20)] for k in range(3)]
    alone_models, alone_opts = _folds(lrs)
    models, opts = _folds(lrs)
    worst_loss, worst_grad = 0.0, (0.0, "")
    for s in range(20):
        for o in alone_opts + opts:
            o.zero_grad()
        alone = []
        for m, bs in zip(alone_models, batches):
            loss = _loss(m, bs[s])
            loss.backward()
            alone.append(loss.item())
        ls = [_loss(m, bs[s]) for m, bs in zip(models, batches)]
        sum(ls).backward()
        for k in range(3):
            worst_loss = max(worst_loss, abs(ls[k].item() - alone[k]) / abs(alone[k]))
            for (n, p), q in zip(models[k].named_parameters(), alone_models[k].parameters()):
                assert (p.grad is None) == (q.grad is None), n     # first-layer c: no gradient
                if p.grad is not None:
                    if p.numel() > 1:      # (as test_gpu_models: see the docstring on the gates)
                        worst_grad = max(worst_grad, (rel_err(p.grad, q.grad), f"step {s} fold {k} {n}"))
                    q.grad.copy_(p.grad)
        mo.step_group(opts)
        for o in alone_opts:
            o.step()
    worst_param = (0.0, "")
    for k in range(3):
        for (n, p), q in zip(models[k].named_parameters(), alone_models[k].parameters()):
            worst_param = max(worst_param, (rel_err(p.detach(), q.detach()), f"fold {k} {n}"))
        st, st_alone = opts[k].state_dict(), alone_opts[k].state_dict()
        assert st["param_groups"] == st_alone["param_groups"]
        assert all(int(v["step"]) == 20 for v in st["state"].values())
    print(f"max relative difference: loss {worst_loss:.2e}, gradient {worst_grad}, "
          f"parameter {worst_param}")
    assert worst_loss <= TOL32
    assert worst_grad[0] <= TOL32, worst_grad
    assert worst_param[0] <= TOL32, worst_param


def test_five_member_bf16_ensemble_matches_oracle_mean():
    """robot_demo.py:610-615 with 5 members (45 chains: above the 40 problems one grouped attention
    or LayerNorm launch holds) against the ORACLE's mean of the members' logits."""
    kw = dict(dim=192, l_len=25, v_len=100, a_len=100, n_heads=6, n_layers=2, ffn=2)
    models, sds = [], []
    for i in range(5):
        torch.manual_seed(i)
        m = mmemo_b200.robot_demo.Multi_class(**kw)
        sd = synth.randomize_gates({k: v.detach().clone() for k, v in m.state_dict().items()},
                                   seed=10 + i)
        m.load_state_dict(sd)
        sds.append(sd)
        models.append(m.to(DEV).eval())
    names = mmemo_b200.robot_demo.Ensemble.NAMES
    b = synth.robot_batch(seed=53, B=32)
    with torch.no_grad():
        ref = sum(O.robot_multi_class(sd, *[b[k] for k in names], 6, 2) for sd in sds) / 5
    for prec, tol in (("bf16", TOLBF), ("fp32", TOL32)):
        with mmemo_b200.precision(prec):      # (a fresh ensemble: graphs are captured per mode)
            out = mmemo_b200.robot_demo.Ensemble(models)(*[b[k].to(DEV) for k in names])
        assert rel_err(out.float(), ref) < tol, prec


def test_step_group_mixed_optimizers_match_their_own_steps():
    """Adam with L2 decay, AdamW clipped by its own norm and AdamW unclipped, three steps with
    frozen parameters joining at step 2: ``step_group`` (two calls: the two classes) equals each
    optimizer's ``step()``."""
    shapes = [(96, 96), (7,), (300_003,), (13, 5), (1,)]

    def build():
        sets = []
        for k in range(3):
            g = torch.Generator().manual_seed(k)
            sets.append([torch.nn.Parameter(torch.randn(s, generator=g).to(DEV)) for s in shapes])
        return sets, [mo.Adam(sets[0], lr=1e-3, weight_decay=0.1),
                      mo.AdamW(sets[1], lr=2e-3, max_grad_norm=0.5),
                      mo.AdamW(sets[2], lr=1e-2, weight_decay=0.0)]

    def grads(sets, step):
        for k, ps in enumerate(sets):
            g = torch.Generator().manual_seed(1000 * step + k)
            for i, p in enumerate(ps):
                p.grad = None if step == 0 and i == 3 else (torch.randn(p.shape, generator=g) * 3).to(DEV)

    sets_a, opts_a = build()
    sets_g, opts_g = build()
    for step in range(3):
        grads(sets_a, step)
        grads(sets_g, step)
        for o in opts_a:
            o.step()
        mo.step_group(opts_g)
    for ps_a, ps_g, oa, og in zip(sets_a, sets_g, opts_a, opts_g):
        for pa, pg in zip(ps_a, ps_g):
            assert rel_err(pg.detach(), pa.detach()) < 1e-6
            assert float(og.state[pg]["step"]) == float(oa.state[pa]["step"])
            assert rel_err(og.state[pg]["exp_avg_sq"], oa.state[pa]["exp_avg_sq"]) < 1e-6


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_trunk_of_five_base_models_in_one_group_matches_each_model(prec):
    """Training path above the launch-table size: the ten towers of five ``Base_model``s (90
    chains) through ONE ``fusion_trunk_multi`` call, forward and backward, against each model's two
    towers as their own group (18 chains).  Pooled outputs and every parameter gradient agree to
    1e-4 (scalar gates left out of the gradient bound, as in test_gpu_models.py: each is one float
    sum accumulated with atomicAdd in arbitrary order)."""
    from mmemo_b200.blocks import fusion_trunk_multi
    kw = dict(dim=64, l_len=12, v_len=20, a_len=28, n_heads=4, n_layers=2, ffn=2, l_dim=24, v_dim=16,
              a_dim=8)
    models, batches = [], []
    for k in range(5):
        torch.manual_seed(k)
        m = mmemo_b200.ren_mme.Base_model(**kw)
        m.load_state_dict(synth.randomize_gates(
            {n: v.detach().clone() for n, v in m.state_dict().items()}, seed=30 + k))
        models.append(m.to(DEV).eval())          # eval: no dropout, so both runs see the same math
        b = synth.renmme_batch(seed=40 + k, B=6 if k else 4, L=(12, 20, 28), D=(24, 16, 8))
        batches.append([t.to(DEV) for t in b["inputs"]])

    def towers(m, a):
        return [m.intensity._tower(a[0], a[4], a[8], a[1], a[5], a[9]),
                m.stimulation._tower(a[2], a[6], a[10], a[3], a[7], a[11])]

    def loss_of(pooled):
        g = torch.Generator(device=DEV).manual_seed(5)
        return sum((p.float() * torch.randn(p.shape, generator=g, device=DEV)).sum() for p in pooled)

    n_layers = models[0].intensity.n_layers
    with mmemo_b200.precision(prec):
        alone_out, alone_grads = [], []
        for m, a in zip(models, batches):
            m.zero_grad()
            out = fusion_trunk_multi(towers(m, a), n_layers, keep_all=True)
            loss_of(out).backward()
            alone_out.append([o.detach().float() for o in out])
            alone_grads.append({n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})
        for m in models:
            m.zero_grad()
        out = fusion_trunk_multi([t for m, a in zip(models, batches) for t in towers(m, a)], n_layers,
                                 keep_all=True)
        sum(loss_of(out[2 * k:2 * k + 2]) for k in range(5)).backward()
    for k, m in enumerate(models):
        for i in range(2):
            assert rel_err(out[2 * k + i].detach().float(), alone_out[k][i]) <= TOL32, (k, i)
        grads = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
        assert set(grads) == set(alone_grads[k])
        worst = max((rel_err(grads[n], v), n) for n, v in alone_grads[k].items() if v.numel() > 1)
        assert worst[0] <= TOL32, (k, worst)
