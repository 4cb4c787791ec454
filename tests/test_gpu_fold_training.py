"""Grouped k-fold training on the GPU (mmemo_b200.folds): one grouped forward + losses + backward
against each fold's own forward + loss + backward (dropout off), the new multi kernels against their
per-model entry points, fit_folds with a grouped step against the per-fold step, and the dropout
contract of the grouped step."""
import copy

import pytest
import torch

import mmemo_b200
from mmemo_b200 import folds, ops, optim, synth, trainer
from oracle import mmemo_oracle as O
from tests.cases import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4
ARGS6 = ("l", "v", "a", "l_mask", "v_mask", "a_mask")


@pytest.fixture(autouse=True)
def _defaults(monkeypatch):
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.0)
    mmemo_b200.set_precision("fp32")
    ops.clear_shadow_cache()
    yield
    mmemo_b200.set_precision("fp32")


# family -> {size: (constructor, batch(seed, B) -> (args, labels, row weights or None), B, B short)}
def _st_batch(small):
    def batch(seed, B):
        kw = dict(L=(6, 5, 7), D=(20, 7, 10), P=4) if small else dict(P=6)
        b = synth.realformer_batch(seed=seed, B=B, empty_windows=True, **kw)
        return [b[k] for k in ARGS6], b["label"], b["wmask"].float()
    return batch


def _ct_batch(small):
    def batch(seed, B):
        kw = dict(L=(6, 9, 12), D=(20, 7, 10)) if small else {}
        b = synth.mosei_batch(seed=seed, B=B, **kw)
        return [b[k] for k in ARGS6], b["label"], None
    return batch


def _bm_batch(small):
    def batch(seed, B):
        kw = dict(L=(5, 7, 11), D=(24, 20, 13)) if small else {}
        b = synth.renmme_batch(seed=seed, B=B, **kw)
        return list(b["inputs"]), b["label"], None
    return batch


def _cl_batch(small):
    def batch(seed, B):
        b = synth.rencecps_batch(seed=seed, B=B, dim=48 if small else 2304)
        return [b["feat"]], b["label"], None
    return batch


R = mmemo_b200.realformer
FAMILIES = {
    "State_Transfer": {
        "small": (lambda: R.State_Transfer(20, 7, 10, 16, 6, 5, 7, 2, 2, 2), _st_batch(True), 5, 3),
        "baseline": (lambda: R.State_Transfer(300, 35, 74, 96, 50, 50, 50, 6, 2, 2),
                     _st_batch(False), 32, 20)},
    "Concat_Trans": {
        "small": (lambda: mmemo_b200.cmu_mosei.Concat_Trans(24, 6, 9, 12, 2, 1, 1, l_dim=20, v_dim=7,
                                                            a_dim=10), _ct_batch(True), 6, 4),
        "baseline": (lambda: mmemo_b200.cmu_mosei.Concat_Trans(96, 20, 100, 200, 6, 1, 1),
                     _ct_batch(False), 32, 20)},
    "Base_model": {
        "small": (lambda: mmemo_b200.ren_mme.Base_model(32, 5, 7, 11, 4, 1, 1, l_dim=24, v_dim=20,
                                                        a_dim=13), _bm_batch(True), 8, 4),
        "baseline": (lambda: mmemo_b200.ren_mme.Base_model(), _bm_batch(False), 256, 128)},
    "Concat_Linear": {
        "small": (lambda: mmemo_b200.rencecps.Concat_Linear(48), _cl_batch(True), 6, 3)},
}
CASES = [(f, s) for f, d in FAMILIES.items() for s in d]
RDROP = {"Base_model"}


def _models(ctor, k):
    ms = []
    for i in range(k):
        torch.manual_seed(100 + i)
        m = ctor()
        m.load_state_dict(synth.randomize_gates({n: t.detach().clone()
                                                 for n, t in m.state_dict().items()}, seed=7 + i))
        ms.append(m.to(DEV).train())
    return ms


def _dev(batch):
    args, lab, w = batch
    return ([a.to(DEV) for a in args], lab.to(DEV), None if w is None else w.to(DEV))


def _own_loss(m, args, lab, w, rdrop):
    lg = m(*args)
    loss = ops.circle_loss_op(lg, lab)
    loss = (loss * w).mean() if w is not None else loss.mean()
    return lg, loss + ops.rdrop_kl_op(lg) if rdrop else loss


def _grouped_losses(ms, bs, rdrop):
    ls = folds.forward(ms, [b[0] for b in bs])
    ws = None if bs[0][2] is None else [b[2] for b in bs]
    losses = folds.circle_losses(ls, [b[1] for b in bs], ws)
    if rdrop:
        losses = [c + r for c, r in zip(losses, folds.rdrop_kl(ls))]
    return ls, losses


def _grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("family,size", CASES)
def test_grouped_step_matches_each_fold(family, size, mode):
    """k = 3 differently seeded folds, the last with a smaller batch, dropout off, train mode:
    logits, per-fold losses and every parameter gradient (scalar gates aside) of one grouped step
    against each fold's own forward + loss + backward, to 1e-4 in both precisions.  (In bf16 the
    activation gradients are rounded to bf16, so this needs the grouped head, pooling and loss
    kernels to produce the bits of the per-model ones: a float32 difference of one ulp upstream can
    flip a bf16 rounding, which the parameter gradients then carry at ~1e-3.)"""
    ctor, batch, B, B_short = FAMILIES[family][size]
    rdrop = family in RDROP
    ms = _models(ctor, 3)
    ref_ms = [copy.deepcopy(m) for m in ms]
    bs = [_dev(batch(11 + i, B if i < 2 else B_short)) for i in range(3)]
    with mmemo_b200.precision(mode):
        ref = []
        for m, b in zip(ref_ms, bs):
            lg, loss = _own_loss(m, *b, rdrop)
            loss.backward()
            ref.append((lg.detach(), loss.detach(), _grads(m)))
        ls, losses = _grouped_losses(ms, bs, rdrop)
        sum(losses[1:], losses[0]).backward()
    for m, lg, loss, (rlg, rloss, rg) in zip(ms, ls, losses, ref):
        assert lg.shape == rlg.shape
        assert rel_err(lg.detach(), rlg) <= TOL, (family, rel_err(lg.detach(), rlg))
        assert abs(loss.item() - rloss.item()) <= TOL * max(1.0, abs(rloss.item()))
        g = _grads(m)
        assert set(g) == set(rg)
        for n, t in rg.items():
            if t.numel() == 1:                  # scalar gates: float-atomic sums (test_gpu_models)
                continue
            assert rel_err(g[n], t) <= TOL, (family, mode, n, rel_err(g[n], t))


def test_grouped_forward_matches_the_oracle():
    ctor, batch, B, B_short = FAMILIES["Concat_Trans"]["small"]
    ms = _models(ctor, 3)
    cpu = [batch(21 + i, B if i < 2 else B_short) for i in range(3)]
    ls = folds.forward(ms, [[a.to(DEV) for a in b[0]] for b in cpu])
    for m, lg, b in zip(ms, ls, cpu):
        sd = {n: t.detach().cpu() for n, t in m.state_dict().items()}
        ref = O.mosei_concat_trans(sd, *b[0], 2, 1)
        assert rel_err(lg.detach().cpu(), ref) <= TOL


# ---------------------------------------------------------------------------------------------
# each multi kernel against its per-model entry point, with more members than one launch holds
# ---------------------------------------------------------------------------------------------
def test_pool_multi_matches_pool_per_tower():
    torch.manual_seed(0)
    n, d, Ls = 20, 16, (5, 7, 9)                       # 16 towers per launch
    towers = []
    for t in range(n):
        B = 3 + t % 4
        towers.append([torch.randn(B, Ls[g], d, device=DEV) for g in range(3) for _ in range(3)])
    segs = [s for tw in towers for s in tw]
    out = folds.pool_group_op(segs, n)
    douts = [torch.randn_like(o) for o in out[:n]]
    dsegs = folds.pool_group_bwd_op(douts, list(out[n:]), segs, n)
    for t, tw in enumerate(towers):
        ref, amax = ops.pool_op(tw, 3)
        assert torch.equal(out[t], ref) and torch.equal(out[n + t], amax)
        rd = ops.pool_bwd_op(douts[t], amax, tw, 3)
        for a, b in zip(dsegs[9 * t:9 * t + 9], rd):
            assert torch.equal(a, b)


def test_linear_group_matches_linear():
    """y, dx and dw bit for bit (K = 576 splits: the partial tiles are summed in a fixed order, and
    each problem of the group splits as it would alone); dbias (a GEMM against a ones vector here,
    a column sum in ops.linear) to float rounding."""
    torch.manual_seed(1)
    n = 50                                             # 48 problems per launch
    xs = [torch.randn(4 + i % 5, 576, device=DEV) for i in range(n)]
    ws = [torch.randn(7 + i % 3, 576, device=DEV) for i in range(n)]
    bs = [torch.randn(w.shape[0], device=DEV) if i % 2 else None for i, w in enumerate(ws)]
    ys = folds.linear_group(xs, ws, bs)
    dys = [torch.randn_like(y) for y in ys]
    res = folds.linear_group_bwd_op(dys, xs, ws, [b is not None for b in bs], [True] * n)
    for i in range(n):
        x = xs[i].clone().requires_grad_(True)
        w = ws[i].clone().requires_grad_(True)
        b = None if bs[i] is None else bs[i].clone().requires_grad_(True)
        y = ops.linear(x, w, b)
        y.backward(dys[i])
        assert torch.equal(ys[i], y.detach())
        assert torch.equal(res[i], x.grad) and torch.equal(res[n + i], w.grad)
        if b is not None:
            assert rel_err(res[2 * n + i], b.grad) <= 1e-6


def test_bilinear_and_state_transfer_multi_match_per_model():
    torch.manual_seed(2)
    n, Cn = 40, 9                                      # 32 members per launch
    th = [torch.randn(3 + i % 6, Cn, device=DEV) for i in range(n)]
    la = [torch.randn_like(t) for t in th]
    par = [(torch.rand(Cn, Cn, Cn, device=DEV), torch.randn(Cn, device=DEV),
            torch.randn(Cn, device=DEV), torch.randn(Cn, 2 * Cn, device=DEV),
            torch.randn(Cn, device=DEV)) for _ in range(n)]
    res = folds.bilinear_group_op(th, la, *[list(p) for p in zip(*par)])
    douts = [torch.randn_like(t) for t in th]
    bwd = folds.bilinear_group_bwd_op(douts, th, la, *[list(p) for p in zip(*par)][:4],
                                      list(res[n:]))
    pv = folds._views(bwd[2 * n], folds._bilinear_pars([p[0] for p in par], [p[1] for p in par],
                                                       [p[3] for p in par]))
    for i in range(n):
        ref, z = ops.bilinear_head_op(th[i], la[i], *par[i])
        assert torch.equal(res[i], ref) and torch.equal(res[n + i], z)
        rb = ops.bilinear_head_bwd_op(douts[i], th[i], la[i], *par[i][:4], z)
        assert rel_err(bwd[i], rb[0]) <= 1e-6 and rel_err(bwd[n + i], rb[1]) <= 1e-6
        for a, b in zip(pv[5 * i:5 * i + 5], rb[2:]):
            assert rel_err(a, b) <= 1e-6
    P, Cs = 6, 6
    feats = [torch.randn(2 + i % 5, P, 2 * Cs, device=DEV) for i in range(n)]
    trans = [torch.rand(Cs, Cs, device=DEV) for _ in range(n)]
    outs = folds.state_transfer_group_op(feats, trans)
    douts = [torch.randn_like(o) for o in outs]
    bwd = folds.state_transfer_group_bwd_op(douts, feats, trans, list(outs))
    dtr = folds._views(bwd[n], trans)
    for i in range(n):
        ref = ops.state_transfer_op(feats[i], trans[i])
        assert torch.equal(outs[i], ref)
        df, dt = ops.state_transfer_bwd_op(douts[i], feats[i], trans[i], ref)
        assert torch.equal(bwd[i], df) and rel_err(dtr[i], dt) <= 1e-6


def test_loss_multi_match_per_model():
    torch.manual_seed(3)
    n, Cn = 40, 9
    lg = [torch.randn(2 * (2 + i % 7), Cn, device=DEV) for i in range(n)]
    lb = [(torch.rand_like(t) < 0.3).float() for t in lg]
    wt = [(torch.rand(t.shape[0], device=DEV) < 0.7).float() for t in lg]
    for weights in (None, wt):
        xs = [t.clone().requires_grad_(True) for t in lg]
        losses = folds.circle_losses(xs, lb, weights)
        sum(losses[1:], losses[0]).backward()
        for i in range(n):
            x = lg[i].clone().requires_grad_(True)
            per_row = ops.circle_loss_op(x, lb[i])
            ref = (per_row * weights[i]).mean() if weights is not None else per_row.mean()
            ref.backward()
            assert rel_err(losses[i].detach(), ref.detach()) <= 1e-6
            assert torch.equal(xs[i].grad, x.grad)
    xs = [t.clone().requires_grad_(True) for t in lg]
    kls = folds.rdrop_kl(xs)
    sum(kls[1:], kls[0]).backward()
    for i in range(n):
        x = lg[i].clone().requires_grad_(True)
        ref = ops.rdrop_kl_op(x)
        ref.backward()
        assert torch.equal(kls[i].detach(), ref.detach()) and torch.equal(xs[i].grad, x.grad)


# ---------------------------------------------------------------------------------------------
# fit_folds with a grouped step
# ---------------------------------------------------------------------------------------------
def test_fit_folds_with_grouped_step_matches_per_fold_step():
    """20 AdamW steps (two epochs of 10 / 10 / 7 batches: the third fold leaves the group after its
    7th batch in each epoch) with folds.forward against the per-fold step, fp32, dropout off."""
    ctor, batch, B, _ = FAMILIES["Concat_Trans"]["small"]
    n_batches = (10, 10, 7)
    data = [[_dev(batch(1000 * f + j, B)) for j in range(n_batches[f])] for f in range(3)]
    valid = [[_dev(batch(5000 + f, B))] for f in range(3)]

    def run(grouped):
        ms = _models(ctor, 3)
        opts = [optim.AdamW(m.parameters(), lr=1e-3) for m in ms]
        losses = []

        def step(ms_, bs):
            if grouped:
                out = folds.circle_losses(folds.forward(ms_, [b[0] for b in bs]),
                                          [b[1] for b in bs])
            else:
                out = [ops.circle_loss_op(m(*b[0]), b[1]).mean() for m, b in zip(ms_, bs)]
            losses.append([x.item() for x in out])
            return out
        hist = trainer.fit_folds(ms, opts, [lambda f=f: data[f] for f in range(3)],
                                 [lambda f=f: valid[f] for f in range(3)], step, epochs=2,
                                 names=["a", "b", "c"], clip=None, log=lambda s: None)
        return hist, losses
    (h0, l0), (h1, l1) = run(False), run(True)
    assert len(l0) == len(l1) == 2 * (10 + 1)
    for a, b in zip(l0, l1):
        assert len(a) == len(b)
        assert all(abs(x - y) <= TOL * max(1.0, abs(x)) for x, y in zip(a, b)), (a, b)
    for a, b in zip(h0, h1):
        for key in ("train", "valid"):
            assert all(abs(x - y) <= TOL * max(1.0, abs(x)) for x, y in zip(a[key], b[key]))


# ---------------------------------------------------------------------------------------------
# dropout contract (Base_model, p = 0.1, R-Drop pairs)
# ---------------------------------------------------------------------------------------------
def test_grouped_dropout_contract(monkeypatch):
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.1)
    ctor, batch, B, _ = FAMILIES["Base_model"]["small"]
    torch.manual_seed(0)
    m0 = ctor()
    ms = [copy.deepcopy(m0).to(DEV).train() for _ in range(2)] + _models(ctor, 1)
    bs = [_dev(batch(31, B)), _dev(batch(31, B)), _dev(batch(32, B))]

    def run():
        with torch.no_grad():
            ls = folds.forward(ms, [b[0] for b in bs])
            return ls, folds.circle_losses(ls, [b[1] for b in bs]), folds.rdrop_kl(ls)
    counter = ops._dropout_counter[0]
    a = run()
    ops._dropout_counter[0] = counter
    b = run()
    c = run()
    for x, y, z in zip(a[0], b[0], c[0]):
        assert rel_err(x, y) <= 1e-6 and rel_err(x, z) > 1e-3
    assert all(abs(x.item() - y.item()) <= 1e-6 * max(1.0, abs(x.item()))
               for x, y in zip(a[1], b[1]))
    assert all(k.item() > 0 for k in a[2])
    assert rel_err(a[0][0], a[0][1]) > 1e-3            # identical folds draw different masks
    opts = [optim.AdamW(m.parameters(), lr=1e-3) for m in ms]
    first = last = None
    for step in range(50):
        for o in opts:
            o.zero_grad()
        ls = folds.forward(ms, [b[0] for b in bs])
        losses = [x + r for x, r in zip(folds.circle_losses(ls, [b[1] for b in bs]),
                                        folds.rdrop_kl(ls))]
        sum(losses[1:], losses[0]).backward()
        optim.step_group(opts)
        vals = [x.item() for x in losses]
        first = first or vals
        last = vals
    assert all(y < x for x, y in zip(first, last)), (first, last)
