"""Grouped k-fold training of ``robot_demo.Multi_class`` (robot_demo.py:497-524 trains 4 folds) and
the projection dropout fused into the grouped projection GEMM (robot_demo.py:302-311, DROP = 0.1):

  * the epilogue draws exactly the masks ``ops._dropout_group`` draws for the contiguous (M, N_g)
    projections with the same seeds, forward and backward;
  * one grouped step equals each fold's own step with dropout off;
  * the dropout contract of the grouped path (seeded, per-fold masks, off in eval())."""
import copy

import pytest
import torch

import mmemo_b200
from mmemo_b200 import folds, group_ops, ops, optim, synth, trainer
from mmemo_b200.robot_demo import Multi_class
from oracle import mmemo_oracle as O
from tests.cases import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4
NAMES = ("l", "v_256", "v_512", "v_1024", "a", "l_mask", "v_mask", "a_mask")
SMALL = (dict(dim=24, l_len=5, v_len=8, a_len=8, n_heads=2, n_layers=2, ffn=2), (5, 8, 8), 6, 4)
NATIVE = (dict(dim=192, l_len=25, v_len=100, a_len=100, n_heads=6, n_layers=2, ffn=2),
          (25, 100, 100), 32, 20)


@pytest.fixture(autouse=True)
def _defaults(monkeypatch):
    monkeypatch.setattr(mmemo_b200.robot_demo, "DROP", 0.0)
    mmemo_b200.set_precision("fp32")
    ops.clear_shadow_cache()
    ops.dropout_step(DEV).zero_()
    yield
    mmemo_b200.set_precision("fp32")
    ops.dropout_step(DEV).zero_()


def _models(kw, k):
    ms = []
    for i in range(k):
        torch.manual_seed(100 + i)
        m = Multi_class(**kw)
        m.load_state_dict(synth.randomize_gates({n: t.detach().clone()
                                                 for n, t in m.state_dict().items()}, seed=7 + i))
        ms.append(m.to(DEV).train())
    return ms


def _batch(seed, B, L, dev=DEV):
    b = synth.robot_batch(seed=seed, B=B, L=L)
    return [b[k].to(dev) for k in NAMES], b["label"].to(dev)


def _grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


# ---------------------------------------------------------------------------------------------
# the grouped projection with dropout: forward epilogue and backward reduction
# ---------------------------------------------------------------------------------------------
def _problems(seed=0, B=4, L=(5, 9, 7), K=(20, 7, 12, 33, 10), d=48):
    """Two folds' worth of robot-like problems: spans [1, 3, 1] per fold (the three visual
    projections are column thirds of one output and share one (L, d) table)."""
    g = torch.Generator().manual_seed(seed)
    xs, ws, bs, poss, spans = [], [], [], [], []
    for _ in range(2):
        lens = (L[0], L[1], L[1], L[1], L[2])
        Ns = (d, d // 3, d // 3, d // 3, d)
        for Lq, k, n in zip(lens, K, Ns):
            xs.append(torch.randn(B, Lq, k, generator=g).to(DEV))
            ws.append((torch.randn(n, k, generator=g) / k ** 0.5).to(DEV).requires_grad_())
            bs.append((0.1 * torch.randn(n, generator=g)).to(DEV).requires_grad_())
        spans += [1, 3, 1]
        poss += [(0.1 * torch.randn(Lq, d, generator=g)).to(DEV).requires_grad_()
                 for Lq in (L[0], L[1], L[2])]
    return xs, ws, bs, poss, spans


def _masks(xs, ws, p, seed):
    """mask / (1 - p) of every problem's contiguous (M, N_g) projection, from the grouped dropout
    kernel itself (test_gpu_dropout.py)."""
    ones = [torch.ones(*x.shape[:-1], w.shape[0], device=DEV) for x, w in zip(xs, ws)]
    outs = [torch.empty_like(o) for o in ones]
    ops._dropout_group(ones, outs, p, ops.site_seeds(seed, len(xs), 0, 1))
    return outs


def _reference(xs, ws, bs, poss, spans, masks, bf16):
    """Eager cat_g((x_g W_g^T + b_g) * m_g) + pos_s, with the bf16 operand rounding in bf16 mode."""
    r = (lambda t: t.to(torch.bfloat16).float()) if bf16 else (lambda t: t)
    ys = [r(x) @ r(w).t() + b for x, w, b in zip(xs, ws, bs)]
    ys = [y * m for y, m in zip(ys, masks)]
    outs, g = [], 0
    for n, pos in zip(spans, poss):
        outs.append(torch.cat(ys[g:g + n], -1) + pos)
        g += n
    return outs


def test_epilogue_dropout_matches_explicit_masks():
    xs, ws, bs, poss, spans = _problems()
    p, seed = 0.3, 1234
    with torch.no_grad():
        outs = group_ops.project_cat(xs, ws, bs, spans, poss, True, p, seed)
        ref = _reference(xs, ws, bs, poss, spans, _masks(xs, ws, p, seed), True)
        masks = _masks(xs, ws, p, seed)
    g = 0
    for s, (n, y, yr, pos) in enumerate(zip(spans, outs, ref, poss)):
        assert y.dtype == torch.bfloat16 and y.shape == yr.shape
        m = torch.cat(masks[g:g + n], -1)
        g += n
        dropped = m == 0
        assert dropped.any() and (~dropped).any()
        # a dropped element is exactly the position-table entry (rounded once to bf16)
        pos_b = pos.detach()[None].expand_as(y).to(torch.bfloat16)
        assert torch.equal(y[dropped], pos_b[dropped]), s
        assert rel_err(y.float(), yr) <= 2e-2, (s, rel_err(y.float(), yr))
    # kept fraction on a large problem
    x = torch.randn(4096, 64, device=DEV)
    w = torch.randn(256, 64, device=DEV)
    with torch.no_grad():
        y = group_ops.project_cat([x], [w], [None], [1], [None], True, p, 99)[0]
    assert abs((y != 0).float().mean().item() - (1 - p)) < 0.01
    # p = 0: bitwise the plain grouped projection
    ones = [1] * len(xs)
    with torch.no_grad():
        a = group_ops.proj_drop_group_op(xs, ws, [b.detach() for b in bs],
                                         [torch.empty(0, device=DEV)] * len(xs), ones, 0.0, 0)
        b0 = group_ops.proj_group_op(xs, ws, [b.detach() for b in bs],
                                     [torch.empty(0, device=DEV)] * len(xs))
    assert all(torch.equal(u, v) for u, v in zip(a[:len(xs)], b0[:len(xs)]))
    # the device step counter changes the masks (and only that)
    with torch.no_grad():
        y1 = group_ops.project_cat(xs, ws, bs, spans, poss, True, p, seed)
        ops.advance_dropout_step(DEV)
        y2 = group_ops.project_cat(xs, ws, bs, spans, poss, True, p, seed)
    assert torch.equal(outs[0], y1[0])
    assert not torch.equal(y1[0], y2[0])


@pytest.mark.parametrize("mode,tol", [("fp32", 2e-4), ("bf16", 2e-2)])
def test_backward_matches_explicit_masks(mode, tol):
    xs, ws, bs, poss, spans = _problems(seed=1)
    p, seed = 0.3, 77
    bf16 = mode == "bf16"
    masks = _masks(xs, ws, p, seed)
    outs = group_ops.project_cat(xs, ws, bs, spans, poss, bf16, p, seed)
    g = torch.Generator().manual_seed(5)
    dys = [torch.randn(y.shape, generator=g).to(DEV) for y in outs]
    sum((y.float() * d).sum() for y, d in zip(outs, dys)).backward()
    got = [t.grad.clone() for t in ws + bs + poss]
    for t in ws + bs + poss:
        t.grad = None
    ref = _reference(xs, ws, bs, poss, spans, masks, bf16)
    sum((y * d).sum() for y, d in zip(ref, dys)).backward()
    for i, (a, t) in enumerate(zip(got, ws + bs + poss)):
        assert rel_err(a, t.grad) <= tol, (i, rel_err(a, t.grad))
    assert poss[1].grad.shape == poss[1].shape          # one (L, d) gradient for the visual table


# ---------------------------------------------------------------------------------------------
# one grouped step against each fold's own step (dropout off)
# ---------------------------------------------------------------------------------------------
def _own_steps(ms, bs, mode):
    out = []
    with mmemo_b200.precision(mode):
        for m, (args, lab) in zip(ms, bs):
            lg = m(*args)
            loss = ops.circle_loss_op(lg, lab).mean()
            loss.backward()
            out.append((lg.detach(), loss.detach(), _grads(m)))
    return out


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("k,size", [(1, "small"), (2, "small"), (5, "small"), (2, "native")])
def test_grouped_step_matches_each_fold(k, size, mode):
    """Logits, losses and every parameter gradient of one grouped step against each fold's own
    step, to 1e-4.  In bf16 the grouped projection adds the position table before its one bf16
    rounding, where the per-fold module rounds the projection and then adds the table in bf16: a
    one-ulp difference of the trunk inputs that the bf16 trunk gradients amplify (to tens of
    percent on single block parameters at these shapes, logits within 1e-2).  So in bf16 the
    logits are compared at 2e-2 with the models' tables, and the gradients with zero tables,
    where both paths round the same values; the position-table gradients are then sums of the
    same bf16 gradients in another order (float atomics), 5e-3."""
    kw, L, B, B_short = SMALL if size == "small" else NATIVE
    bs = [_batch(11 + i, B if i < k - 1 or k == 1 else B_short, L) for i in range(k)]
    for zero_tables in ((False,) if mode == "fp32" else (False, True)):
        ms = _models(kw, k)
        if zero_tables:
            for m in ms:
                for e in (m.linguistic_position, m.visual_position, m.acoustic_position):
                    e.position_embeddings.weight.data.zero_()
        ref = _own_steps([copy.deepcopy(m) for m in ms], bs, mode)
        with mmemo_b200.precision(mode):
            ls = folds.forward(ms, [b[0] for b in bs])
            losses = folds.circle_losses(ls, [b[1] for b in bs])
            sum(losses[1:], losses[0]).backward()
        exact = mode == "fp32" or zero_tables
        lg_tol = TOL if exact else 2e-2
        for m, lg, loss, (rlg, rloss, rg) in zip(ms, ls, losses, ref):
            assert lg.shape == rlg.shape == (lg.shape[0], 7)
            assert rel_err(lg.detach(), rlg) <= lg_tol, rel_err(lg.detach(), rlg)
            assert abs(loss.item() - rloss.item()) <= lg_tol * max(1.0, abs(rloss.item()))
            got = _grads(m)
            assert set(got) == set(rg)
            for mod in (m.fully_connected, m.normalization):
                assert all(p.grad is None for p in mod.parameters())
            if not exact:
                continue
            for n, t in rg.items():
                if t.numel() == 1:
                    continue
                tol = 5e-3 if mode == "bf16" and "position" in n else TOL
                assert rel_err(got[n], t) <= tol, (n, rel_err(got[n], t))


def test_grouped_forward_matches_the_oracle():
    """Golden case weights (tests/golden/robot_multi_class.pt), every fold, fp32."""
    from tests import cases
    sd = torch.load(cases.golden_path("robot_multi_class"))["state"]
    kw = SMALL[0]
    ms = []
    for _ in range(2):
        m = Multi_class(**kw)
        m.load_state_dict(sd)
        ms.append(m.to(DEV).eval())
    cpu = [synth.robot_batch(seed=31 + i, B=3 - i, L=SMALL[1]) for i in range(2)]
    with torch.no_grad():
        ls = folds.forward(ms, [[b[k].to(DEV) for k in NAMES] for b in cpu])
    for lg, b in zip(ls, cpu):
        ref = O.robot_multi_class(sd, *[b[k] for k in NAMES], kw["n_heads"], kw["n_layers"])
        assert rel_err(lg.cpu(), ref) <= TOL


# ---------------------------------------------------------------------------------------------
# dropout contract at the reference's p = 0.1
# ---------------------------------------------------------------------------------------------
def test_grouped_dropout_contract(monkeypatch):
    monkeypatch.setattr(mmemo_b200.robot_demo, "DROP", 0.1)
    kw, L, B, _ = SMALL
    torch.manual_seed(0)
    m0 = Multi_class(**kw)
    ms = [copy.deepcopy(m0).to(DEV).train() for _ in range(2)]
    assert ms[0].unify_dimension.drop.p == 0.1
    b = _batch(41, B, L)
    with mmemo_b200.precision("bf16"):
        counter = ops._dropout_counter[0]
        a1 = [x.detach() for x in folds.forward(ms, [b[0], b[0]])]
        ops._dropout_counter[0] = counter
        a2 = [x.detach() for x in folds.forward(ms, [b[0], b[0]])]
        assert all(torch.equal(x, y) for x, y in zip(a1, a2))     # seed pinned: same outputs
        assert not torch.equal(a1[0], a1[1])                      # each fold its own masks
        for m in ms:
            m.eval()
        with torch.no_grad():
            e = folds.forward(ms, [b[0], b[0]])
            own = [m(*b[0]) for m in ms]
        assert all(rel_err(x, y) <= 2e-2 for x, y in zip(e, own))
        assert torch.equal(e[0], e[1])


def test_fp32_dropout_step_matches_explicit_masks(monkeypatch):
    """A float32 grouped step with projection dropout: the projections equal the explicit-mask
    reference (the masks ops._dropout_group draws for the step's seed), and so do their weight
    and position-table gradients."""
    kw, L, B, _ = SMALL
    ms = _models(kw, 2)
    for m in ms:
        m.unify_dimension.drop.p = 0.1
    bs = [_batch(51 + i, B, L) for i in range(2)]
    captured = {}
    real = group_ops.project_cat

    def spy(xs, ws, biases, spans, poss, bf16=False, drop_p=0.0, seed=0):
        captured.update(xs=xs, ws=ws, bs=biases, poss=poss, spans=spans, p=drop_p, seed=seed)
        return real(xs, ws, biases, spans, poss, bf16, drop_p, seed)
    monkeypatch.setattr(folds, "project_cat", spy)
    ls = folds.forward(ms, [b[0] for b in bs])
    assert captured["p"] == pytest.approx(0.1)
    c = captured
    masks = _masks(c["xs"], c["ws"], c["p"], c["seed"])
    ws2 = [w.detach().reshape(w.shape[0], -1).clone().requires_grad_() for w in c["ws"]]
    pos2 = [p.detach().clone().requires_grad_() for p in c["poss"]]
    ref = _reference(c["xs"], ws2, [b.detach() for b in c["bs"]], pos2, c["spans"], masks, False)
    outs = real(c["xs"], c["ws"], c["bs"], c["spans"], c["poss"], False, c["p"], c["seed"])
    for y, yr in zip(outs, ref):
        assert rel_err(y.detach(), yr.detach()) <= TOL
    g = torch.Generator().manual_seed(9)
    dys = [torch.randn(y.shape, generator=g).to(DEV) for y in outs]
    for m in ms:
        m.zero_grad(set_to_none=True)
    sum((y * d).sum() for y, d in zip(outs, dys)).backward()
    sum((y * d).sum() for y, d in zip(ref, dys)).backward()
    for w, w2 in zip(c["ws"], ws2):
        assert rel_err(w.grad.reshape(w2.shape), w2.grad) <= TOL
    for p_, p2 in zip(c["poss"], pos2):
        assert rel_err(p_.grad, p2.grad) <= TOL
    assert all(torch.isfinite(x).all() for x in ls)


# ---------------------------------------------------------------------------------------------
# trainer.fit_folds with the grouped step
# ---------------------------------------------------------------------------------------------
def test_fit_folds_with_grouped_step_matches_per_fold_step():
    kw, L, B, _ = SMALL
    n_batches = (6, 6, 4)
    data = [[_batch(1000 * f + j, B, L) for j in range(n_batches[f])] for f in range(3)]
    valid = [[_batch(5000 + f, B, L)] for f in range(3)]

    def run(grouped):
        ms = _models(kw, 3)
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
    assert len(l0) == len(l1)
    for a, b in zip(l0, l1):
        assert all(abs(x - y) <= TOL * max(1.0, abs(x)) for x, y in zip(a, b)), (a, b)
    for a, b in zip(h0, h1):
        for key in ("train", "valid"):
            assert all(abs(x - y) <= TOL * max(1.0, abs(x)) for x, y in zip(a[key], b[key]))
