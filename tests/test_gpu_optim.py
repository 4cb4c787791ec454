"""Fused clip + Adam/AdamW (csrc/optim.cu, mmemo_b200/optim.py) against the calls the reference
loops make: nn.utils.clip_grad_norm_ + torch.optim.Adam / AdamW (others/realformer.py:314-315,342;
cmu-mosei/run.py:368-369,398), run by torch on the CPU in float32 on the same seeded tensors."""
import copy

import pytest
import torch

from mmemo_b200 import optim as mo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHAPES = [(1,), (7,), (96, 96), (13, 5), (192, 96), (3, 1, 1), (300_003,), (576,)]
LATE = 3          # this parameter gets no gradient in the first step: its step count trails by one


def _params(seed, misalign):
    g = torch.Generator().manual_seed(seed)
    cpu = [torch.nn.Parameter(torch.randn(s, generator=g)) for s in SHAPES]
    gpu = []
    for i, p in enumerate(cpu):
        if misalign and i % 2 == 0:        # contiguous view at a 4-byte offset: scalar kernel path
            buf = torch.empty(p.numel() + 1, device=DEV)
            v = buf[1:].view(p.shape)
            v.copy_(p.detach())
            gpu.append(torch.nn.Parameter(v))
        else:
            gpu.append(torch.nn.Parameter(p.detach().to(DEV)))
    return cpu, gpu


def _set_grads(cpu, gpu, seed, scale, skip=None):
    g = torch.Generator().manual_seed(seed)
    for i, (pc, pg) in enumerate(zip(cpu, gpu)):
        gr = torch.randn(pc.shape, generator=g) * scale
        pc.grad = None if i == skip else gr.clone()
        pg.grad = None if i == skip else gr.to(DEV)


@pytest.mark.parametrize("kind", ["adam", "adamw"])
@pytest.mark.parametrize("mode", ["separate_clip", "fused_clip", "no_clip"])
@pytest.mark.parametrize("misalign", [False, True])
def test_adam_matches_torch(kind, mode, misalign):
    cpu, gpu = _params(5, misalign)
    kw = dict(lr=1e-3) if kind == "adam" else dict(lr=1e-3, weight_decay=0.05)
    ref = (torch.optim.Adam if kind == "adam" else torch.optim.AdamW)(cpu, **kw)
    ours = (mo.Adam if kind == "adam" else mo.AdamW)(
        gpu, max_grad_norm=1.0 if mode == "fused_clip" else None, **kw)
    for step in range(6):
        # alternate between gradients far above and far below the clip threshold
        _set_grads(cpu, gpu, 100 + step, 1.0 if step % 2 == 0 else 1e-5,
                   skip=LATE if step == 0 else None)
        if mode != "no_clip":
            n_ref = torch.nn.utils.clip_grad_norm_(cpu, 1.0)
        if mode == "separate_clip":
            n_ours = mo.clip_grad_norm_(gpu, 1.0)
            assert abs(float(n_ours) - float(n_ref)) <= 1e-5 * float(n_ref)
            for pc, pg in zip(cpu, gpu):
                if pc.grad is not None:
                    torch.testing.assert_close(pg.grad.cpu(), pc.grad, rtol=1e-5, atol=1e-9)
        ref.step()
        ours.step()
    for i, (pc, pg) in enumerate(zip(cpu, gpu)):
        torch.testing.assert_close(pg.detach().cpu(), pc.detach(), rtol=2e-5, atol=2e-7)
        torch.testing.assert_close(ours.state[pg]["exp_avg"].cpu(), ref.state[pc]["exp_avg"],
                                   rtol=2e-5, atol=2e-7)      # a few float32 ulps of |g| ~ 1
        torch.testing.assert_close(ours.state[pg]["exp_avg_sq"].cpu(), ref.state[pc]["exp_avg_sq"],
                                   rtol=2e-5, atol=1e-9)
        assert float(ours.state[pg]["step"]) == float(ref.state[pc]["step"]) == (5 if i == LATE else 6)


def test_state_dict_round_trip_with_torch_optim():
    """A checkpoint written by torch.optim.AdamW resumes in the fused optimizer and vice versa."""
    cpu, gpu = _params(9, False)
    ref = torch.optim.AdamW(cpu, lr=2e-3)
    ours = mo.AdamW(gpu, lr=2e-3)
    _set_grads(cpu, gpu, 1, 1.0)
    ref.step()
    # (deepcopy = what a torch.save / torch.load round trip does; the live dict shares its CPU
    # ``step`` tensors with ``ref``)
    sd = copy.deepcopy(ref.state_dict())
    ours.load_state_dict(sd)            # moves exp_avg / exp_avg_sq to the parameters' device
    _set_grads(cpu, gpu, 2, 1.0)
    for pc, pg in zip(cpu, gpu):
        pg.data.copy_(pc.detach())
    ref.step()
    ours.step()
    for pc, pg in zip(cpu, gpu):
        torch.testing.assert_close(pg.detach().cpu(), pc.detach(), rtol=2e-5, atol=2e-7)
    back = torch.optim.AdamW([torch.nn.Parameter(p.detach().cpu()) for p in gpu], lr=2e-3)
    back.load_state_dict(copy.deepcopy(ours.state_dict()))
    assert float(back.state[back.param_groups[0]["params"][0]]["step"]) == 2


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_training_loop_with_fused_optimizer_tracks_torch(prec):
    """cmu-mosei Concat_Trans, 20 steps of the reference loop's  backward -> clip -> AdamW  with the
    fused optimizer vs torch.optim on an identical model copy: same loss curve.  In bf16 mode the
    GEMMs read bf16 shadows of the float32 masters, keyed on the parameters' version counters: the
    fused step (which writes through raw pointers) must invalidate them, or training would keep
    running on the initial weights while the masters move on."""
    import mmemo_b200
    from mmemo_b200 import cmu_mosei, ops, synth
    from mmemo_b200.cmu_mosei import multi_circle_loss

    mmemo_b200.set_precision(prec)
    ops.clear_shadow_cache()
    torch.manual_seed(0)
    model = cmu_mosei.Concat_Trans(96, 50, 50, 50, 6, 2, 1)
    model.load_state_dict(synth.randomize_gates(model.state_dict(), seed=2))
    m1 = model.to(DEV).train()
    m2 = copy.deepcopy(m1)
    o1 = mo.AdamW(m1.parameters(), lr=1e-3, max_grad_norm=1.0)
    o2 = torch.optim.AdamW(m2.parameters(), lr=1e-3)
    batch = {k: v.to(DEV) for k, v in synth.mosei_batch(seed=3, B=8, L=(50, 50, 50)).items()}
    args = [batch[k] for k in ("l", "v", "a", "l_mask", "v_mask", "a_mask")]
    l1s, l2s = [], []
    for _ in range(20):
        for m, o, ls, fused in ((m1, o1, l1s, True), (m2, o2, l2s, False)):
            o.zero_grad()
            loss = multi_circle_loss(m(*args), batch["label"]).mean()
            loss.backward()
            if not fused:
                torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            o.step()
            ls.append(float(loss.detach()))
    mmemo_b200.set_precision("fp32")
    assert l1s[-1] < l1s[0]
    for a, b in zip(l1s, l2s):
        # (atomics reorder fp32 sums, so the two runs are not bit-identical; SURVEY's bar for a
        # loss curve is 1 %)
        assert abs(a - b) <= 5e-3 * max(1.0, abs(b)), (l1s, l2s)
    # the fused step bumped the version counters like torch.optim's in-place update does
    assert all(p._version > 0 for p in m1.parameters() if p.grad is not None)
