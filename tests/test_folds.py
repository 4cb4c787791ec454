"""CPU tests of k-fold training: the launches ``optim.step_group`` issues (kernel calls stubbed,
like test_host_plumbing.py) and ``trainer.fit_folds`` against one ``trainer.fit`` per fold."""
import os

import pytest
import torch

from mmemo_b200 import ops, optim, trainer


@pytest.fixture()
def stub(monkeypatch):
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(ops, "_try_call", lambda name, *a: calls.append((name, a)) or True)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(optim, "_check", lambda ts, what: None)
    yield calls


def _fold_optimizers(n_folds, n_tensors, clip):
    opts = []
    for k in range(n_folds):
        ps = [torch.nn.Parameter(torch.zeros(3)) for _ in range(n_tensors)]
        for p in ps:
            p.grad = torch.ones(3)
        opts.append(optim.AdamW(ps, lr=1e-3 * (k + 1), max_grad_norm=clip))
    return opts


@pytest.mark.parametrize("clip", [None, 1.0])
@pytest.mark.parametrize("n_folds,n_tensors", [(1, 50), (3, 50), (5, 100), (2, 48)])
def test_step_group_makes_one_norm_and_one_update_call(stub, clip, n_folds, n_tensors):
    """Whatever K and the tensor count: the library splits the tensors into launches itself."""
    opts = _fold_optimizers(n_folds, n_tensors, clip)
    optim.step_group(opts)
    names = [c[0] for c in stub]
    assert names == (["mmemo_grad_sqnorm_multi_f32"] if clip else []) + ["mmemo_adam_step_multi_f32"]
    assert all(a[0] == n_folds * n_tensors for _, a in stub)
    # per-tensor lr / step / norm slot: the lr and slot of the fold the tensor belongs to
    lrs, steps, slots = [], [], []
    for name, a in stub:
        if name == "mmemo_adam_step_multi_f32":
            lrs += list(a[6])[:a[0]]
            steps += list(a[7])[:a[0]]
            slots += list(a[9])[:a[0]]
            assert (a[14] is not None) == (clip is not None)
    assert slots == [k for k in range(n_folds) for _ in range(n_tensors)]
    assert lrs == pytest.approx([1e-3 * (k + 1) for k in slots])
    assert steps == [1] * (n_folds * n_tensors)
    for o in opts:
        assert all(float(o.state[p]["step"]) == 1.0 for p in o.param_groups[0]["params"])


def test_step_group_rejects_other_optimizers(stub):
    p = torch.nn.Parameter(torch.zeros(2))
    with pytest.raises(TypeError):
        optim.step_group([torch.optim.Adam([p])])


def _toy(k):
    torch.manual_seed(k)
    return torch.nn.Linear(4, 2)


def _data(k, n_batches, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(3, 4, generator=g), torch.randn(3, 2, generator=g)) for _ in range(n_batches)]


def _step(m, b):
    return ((m(b[0]) - b[1]) ** 2).mean()


# validation losses that fold 1 never improves on after epoch 2 (stops early), the others do
SCRIPTS = [[1.0, 0.9, 0.8, 0.85, 0.7, 0.6, 0.65, 0.5],
           [1.0, 0.5, 0.6, 0.7, 0.8, 0.9, 0.95, 0.99],
           [2.0, 1.9, 1.95, 1.97, 1.98, 1.5, 1.4, 1.3]]
N_TRAIN = [3, 5, 2]           # batches per epoch differ between the folds


def _setup():
    models = [_toy(k) for k in range(3)]
    opts = [torch.optim.Adam(m.parameters(), lr=1e-2 * (k + 1)) for k, m in enumerate(models)]
    epoch = {k: 0 for k in range(3)}

    def train_iter(k):
        return lambda: iter(_data(k, N_TRAIN[k], seed=10 * k + epoch[k]))

    def valid_iter(k):
        def make():
            epoch[k] += 1
            return iter([SCRIPTS[k][epoch[k] - 1]] * 2)
        return make

    def valid_step(m, b):
        return torch.tensor(b + 0.0 * float(_step(m, _data(0, 1, 0)[0])))

    return models, opts, [train_iter(k) for k in range(3)], [valid_iter(k) for k in range(3)], \
        valid_step


def test_fit_folds_equals_one_fit_per_fold(tmp_path):
    log_a, log_b = tmp_path / "alone", tmp_path / "grouped"
    models, opts, tr, va, vstep = _setup()
    alone = [trainer.fit(models[k], opts[k], tr[k], va[k], _step, vstep, epochs=8,
                         name=f"fold_{k}", log_dir=str(log_a), sched_patience=1, log=lambda s: None)
             for k in range(3)]
    models_g, opts_g, tr_g, va_g, vstep_g = _setup()
    seen = []

    def train_group(ms, bs):
        seen.append(len(ms))
        return [_step(m, b) for m, b in zip(ms, bs)]

    grouped = trainer.fit_folds(models_g, opts_g, tr_g, va_g, train_group,
                                lambda ms, bs: [vstep_g(m, b) for m, b in zip(ms, bs)], epochs=8,
                                names=[f"fold_{k}" for k in range(3)], log_dir=str(log_b),
                                sched_patience=1, log=lambda s: None)
    assert len(alone[1]["valid"]) == 6 and len(alone[0]["valid"]) == 8     # fold 1 stopped early
    assert max(seen) == 3 and min(seen) == 1                  # folds leave an epoch when done
    for h_a, h_g in zip(alone, grouped):
        assert h_g["train"] == h_a["train"]
        assert h_g["valid"] == h_a["valid"]
        assert h_g["lrs"] == h_a["lrs"]
        assert os.path.basename(h_g["best"]) == os.path.basename(h_a["best"])
    assert sorted(os.listdir(log_a)) == sorted(os.listdir(log_b))
    for f in os.listdir(log_a):
        if f.endswith(".pt"):
            sa, sg = torch.load(log_a / f), torch.load(log_b / f)
            assert all(torch.equal(sa[k], sg[k]) for k in sa), f
        else:
            assert open(log_a / f).read() == open(log_b / f).read()
    for m_a, m_g in zip(models, models_g):
        assert all(torch.equal(a, b) for a, b in zip(m_a.parameters(), m_g.parameters()))


def test_fit_folds_checks_its_arguments():
    with pytest.raises(ValueError):
        trainer.fit_folds([_toy(0)], [], [], [], lambda ms, bs: [], epochs=1, names=["a"])
