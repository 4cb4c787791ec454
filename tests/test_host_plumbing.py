"""CPU tests of the host logic with the kernel launches stubbed out.

The C launchers cannot run here (no GPU), so ``ops._call`` is replaced by a recorder.  Outputs
are uninitialised memory, but everything the Python side is responsible for is exercised: op
schemas, autograd wiring of every custom op, output shapes/dtypes, which parameters receive a
gradient (must equal the reference's set, e.g. first-layer ``c`` gets none — SURVEY §7), the
sequence of launcher names, and state_dict compatibility with the reference fixtures.
"""
import pytest
import torch

import mmemo_b200
from mmemo_b200 import ops
from tests import cases


class _FakeLib:
    def mmemo_resattn_uses_tensor_cores(self, *a):
        return 0

    def mmemo_resattn_uses_mma(self, *a):
        return 1


@pytest.fixture()
def stub(monkeypatch):
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append(name))
    monkeypatch.setattr(ops, "_try_call", lambda name, *a: calls.append(name) or True)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(ops._lib, "load", lambda: _FakeLib())
    mmemo_b200.robot_demo.DROP = 0.0
    mmemo_b200.ren_mme.DROP = 0.0
    ops.clear_shadow_cache()
    yield calls
    ops.clear_shadow_cache()


class _Loss:
    multi_circle_loss = staticmethod(lambda p, t: ops.circle_loss_op(p, t))
    multi_loss = staticmethod(lambda p, t: ops.circle_loss_op(p, t).mean())
    rdrop_kl = staticmethod(lambda p: ops.rdrop_kl_op(p))


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(cases.CASES))
def test_module_wiring_matches_reference_grad_set(stub, name, mode):
    c = cases.CASES[name]
    g = torch.load(cases.golden_path(name))
    model = c.our_model(mmemo_b200).train()
    assert model.load_state_dict(g["state"]).missing_keys == []
    with mmemo_b200.precision(mode):
        logits, loss, grads, igrads = cases.run_module_with_grads(model, c, g["batch"], _Loss)
    assert logits.shape == g["logits"].shape
    assert set(grads) == set(g["grads"]), sorted(set(grads) ^ set(g["grads"]))
    for k, v in grads.items():
        assert v.shape == g["grads"][k].shape and v.dtype == torch.float32, k
    for k, v in igrads.items():
        assert v.shape == g["input_grads"][k].shape
    assert any(n.startswith("mmemo_resattn_fwd") for n in stub) or name == "rencecps_concat_linear"
    assert any(n.endswith("_bf16") for n in stub) == (mode == "bf16" and name != "rencecps_concat_linear")


def test_state_dict_keys_equal_reference(stub):
    for name, c in cases.CASES.items():
        g = torch.load(cases.golden_path(name))
        model = c.our_model(mmemo_b200)
        assert list(model.state_dict().keys()) == list(g["state"].keys()), name
        for k, v in model.state_dict().items():
            assert v.shape == g["state"][k].shape, (name, k)


def test_unfused_paths_when_k_is_not_v(stub):
    blk = mmemo_b200.realformer.Attention_Block(16, 2)
    q, k, v = torch.randn(2, 5, 16, requires_grad=True), torch.randn(2, 7, 16), torch.randn(2, 7, 16)
    out, s = blk(q, k, v, torch.ones(2, 7))
    assert out.shape == (2, 5, 16) and s.shape == (2, 2, 5, 7)
    out.sum().backward()
    assert q.grad.shape == q.shape and blk.w_qkv[2].weight.grad is not None
    lite = mmemo_b200.cmu_mosei.Attention_Block(16, 2, 1)
    out, s = lite(q, k, v, torch.ones(2, 7))
    assert out.shape == (2, 5, 16)


def test_trunk_and_single_blocks_skip_unused_score_writes(stub, monkeypatch):
    """The last layer of a chain must not write its scores (nothing consumes them) - in the grouped
    trunk (one op per layer over the nine chains) and when the blocks are called one by one (one
    problem per op) - and the drop-in blocks themselves keep returning scores afterwards
    (emit_scores is a per-call argument, not module state)."""
    from mmemo_b200 import group_ops
    groups = []
    real_g = group_ops.trunk_lite_op

    def spy_g(qs, kvs, masks, s_prevs, params, H, bf16, emit_s, drop_p, drop_seed):
        groups.append((len(qs), len(s_prevs), emit_s))
        return real_g(qs, kvs, masks, s_prevs, params, H, bf16, emit_s, drop_p, drop_seed)

    monkeypatch.setattr(group_ops, "trunk_lite_op", spy_g)
    m = mmemo_b200.cmu_mosei.Multi_ATTN(16, 4, 5, 6, 2, 2, 1, l_dim=8, v_dim=6, a_dim=7)
    args = (torch.randn(2, 4, 8), torch.randn(2, 5, 6), torch.randn(2, 6, 7), torch.ones(2, 4),
            torch.ones(2, 5), torch.ones(2, 6))
    out_g = m(*args)
    assert groups == [(9, 0, True), (9, 9, False)]
    groups.clear()
    cases.use_per_block_trunk(monkeypatch)
    out_b = m(*args)
    assert groups == [(1, 0, True), (1, 1, False)] * 9 and out_b.shape == out_g.shape
    blk = m.multimodal_blocks[1]                  # a last-layer block, called directly
    x = torch.randn(2, 4, 16)
    out, s = blk(x, x, x, torch.ones(2, 4))
    assert s is not None and s.shape == (2, 2, 4, 4)


def test_standalone_blocks_are_one_problem_trunk_groups(stub):
    """A block called on K = V runs as a trunk group of one problem, on the per-problem attention
    entry points: a ResidualEncoder forward + backward issues 66 library calls in fp32 and 52 in
    bf16, and a bf16 lite block casts its two weights in one launch and computes its three weight
    gradients in one grouped launch (12 calls)."""
    from mmemo_b200 import synth
    b = synth.encoder_batch(B=2, L=16, d=32)
    for mode, n in (("fp32", 66), ("bf16", 52)):
        stub.clear()
        ops.clear_shadow_cache()
        enc = mmemo_b200.ResidualEncoder(32, 4, 3)
        with mmemo_b200.precision(mode):
            enc(b["x"], b["mask"]).float().sum().backward()
        assert len(stub) == n, (mode, stub)
        assert not any(c.startswith("mmemo_resattn") and "grouped" in c for c in stub), stub
    stub.clear()
    blk = mmemo_b200.cmu_mosei.Attention_Block(16, 2, 1)
    q, kv = torch.randn(2, 5, 16, requires_grad=True), torch.randn(2, 7, 16, requires_grad=True)
    with mmemo_b200.precision("bf16"):
        out, s = blk(q, kv, kv, torch.ones(2, 7))
        out.float().sum().backward()
    assert len(stub) == 12 and stub.count("mmemo_linear_bwd_w_grouped_bf16") == 1, stub
    assert s.shape == (2, 2, 5, 7) and q.grad.shape == q.shape and kv.grad.shape == kv.shape


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_standalone_block_dropout_stays_on_the_trunk_op(stub, monkeypatch, mode):
    """Training dropout of a block called on its own runs inside its trunk op (one op call per
    forward, one grouped dropout launch per site and direction), not on the per-op path."""
    from mmemo_b200 import blocks, group_ops
    n_ops = []
    for name in ("trunk_full_op", "trunk_lite_op"):
        monkeypatch.setattr(group_ops, name,
                            lambda *a, _op=getattr(group_ops, name): n_ops.append(1) or _op(*a))
    x = torch.randn(2, 5, 16, requires_grad=True)
    for blk in (blocks.FullAttentionBlock(16, 2, 2, drop=0.1),
                blocks.LiteAttentionBlock(16, 2, 1, drop=0.1)):
        blk.train()
        stub.clear()
        n_ops.clear()
        with mmemo_b200.precision(mode):
            out, _ = blk(x, x, x, torch.ones(2, 5))
            out.float().sum().backward()
        assert len(n_ops) == 1, type(blk)
        sfx = "bf16" if mode == "bf16" else "f32"
        assert stub.count(f"mmemo_dropout_multi_{sfx}") == 4, stub       # 2 sites x (fwd + bwd)
        assert not any(c in ("mmemo_dropout_f32", "mmemo_dropout_bf16") for c in stub), stub


def test_grouped_trunk_launch_count(stub):
    """One grouped launch per kernel kind and layer: a State_Transfer step (2 layers x 9 chains,
    fwd+bwd) stays under 60 libmmemo launches in bf16 mode (VERDICT r1: ~350 before)."""
    m = mmemo_b200.realformer.State_Transfer(l_dim=16, v_dim=8, a_dim=8, dim=16, l_len=4, v_len=4,
                                             a_len=4, n_heads=2, n_layers=2, ffn=2).train()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith((".a", ".b", ".c")):
                p.fill_(0.3)
    b = dict(l=torch.randn(2, 3, 4, 16), v=torch.randn(2, 3, 4, 8), a=torch.randn(2, 3, 4, 8))
    ones = torch.ones(2, 3, 4)
    with mmemo_b200.precision("bf16"):
        out = m(b["l"], b["v"], b["a"], ones, ones, ones)
        ops.circle_loss_op(out, torch.zeros(2, 3, 6)).mean().backward()
    assert len(stub) <= 60, (len(stub), stub)
    assert sum(n.startswith("mmemo_resattn") for n in stub) == 4      # 2 layers x (fwd + bwd)


def test_shadow_cache_tracks_parameter_version(stub):
    w = torch.nn.Parameter(torch.randn(8, 4))
    a = ops.shadow_bf16(w)
    assert ops.shadow_bf16(w) is a
    with torch.no_grad():
        w.add_(1.0)
    assert ops.shadow_bf16(w) is not a
    assert len(ops._shadow) == 1


def test_no_cpu_fallback():
    """Without the stub, a CPU tensor must raise instead of silently computing on the host."""
    with pytest.raises(RuntimeError):
        ops.linear(torch.randn(2, 3), torch.randn(4, 3))


def test_position_length_mismatch_raises(stub):
    m = mmemo_b200.realformer.Multi_class(8, 6, 7, 16, 4, 5, 6, 2, 1, 2)
    with pytest.raises(RuntimeError):
        m(torch.randn(2, 9, 8), torch.randn(2, 5, 6), torch.randn(2, 6, 7), torch.ones(2, 9),
          torch.ones(2, 5), torch.ones(2, 6))


def test_grad_reducer_on_encoder_skips_undefined_grads(stub):
    """The first-layer ``c`` receives an UNDEFINED gradient (its hook still fires): it must stay out
    of the buckets; all other parameters end up as views of the flat buckets."""
    import socket
    import torch.distributed as dist
    from mmemo_b200 import dp, synth
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    try:
        model = mmemo_b200.ResidualEncoder(32, 4, 3)
        red = dp.GradReducer(model, world_size=2, bucket_bytes=16 << 10)
        b = synth.encoder_batch(B=2, L=16, d=32)
        for _ in range(3):
            model.zero_grad(set_to_none=True)
            red.backward((model(b["x"], b["mask"]).float() ** 2).mean())
        assert model.blocks[0].c.grad is None
        assert len(red.buckets) >= 2
        flat_ptrs = {bk.flat.untyped_storage().data_ptr() for bk in red.buckets}
        for n, p in model.named_parameters():
            if n != "blocks.0.c":
                assert p.grad.untyped_storage().data_ptr() in flat_ptrs, n
    finally:
        dist.destroy_process_group()


def test_fused_adamw_makes_one_norm_and_one_update_call(monkeypatch):
    """optim.AdamW: torch.optim-compatible param_groups / state layout, one norm and one update call
    per step with per-tensor step counts, global norm over all groups, empty groups skipped
    (Ren-MME/run.py:376-379)."""
    from mmemo_b200 import optim as mo
    calls = []
    monkeypatch.setattr(ops, "_call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(mo, "_check", lambda ts, what: None)
    w1, w2 = torch.nn.Parameter(torch.ones(5, 3)), torch.nn.Parameter(torch.ones(7))
    frozen = torch.nn.Parameter(torch.ones(2))
    opt = mo.AdamW([{"params": [w1, w2, frozen], "lr": 1e-3}, {"params": [], "lr": 1e-3}],
                   max_grad_norm=1.0)
    ref = torch.optim.AdamW([torch.nn.Parameter(torch.ones(1))])
    assert set(opt.param_groups[0]) >= {"lr", "betas", "eps", "weight_decay"}
    assert opt.param_groups[0]["weight_decay"] == ref.param_groups[0]["weight_decay"] == 1e-2
    w1.grad, w2.grad = torch.ones_like(w1), torch.ones_like(w2)
    opt.step()
    names = [n for n, _ in calls]
    assert names == ["mmemo_grad_sqnorm_multi_f32", "mmemo_adam_step_multi_f32"]
    assert calls[0][1][0] == 2 and list(calls[0][1][3]) == [0, 0]     # both norms into slot 0
    a = calls[1][1]
    assert a[0] == 2 and a[13] == 1 and list(a[7]) == [1, 1]   # two tensors, decoupled, step 1
    assert a[14] == calls[0][1][4] and a[15] == 1.0             # fused clipping by that norm
    assert set(opt.state[w1]) == {"step", "exp_avg", "exp_avg_sq"} and frozen not in opt.state
    # a parameter that starts receiving gradients later gets its own bias-correction step
    calls.clear()
    frozen.grad = torch.ones_like(frozen)
    opt.step()
    names = [n for n, _ in calls]
    assert names == ["mmemo_grad_sqnorm_multi_f32", "mmemo_adam_step_multi_f32"]
    a = calls[1][1]
    assert list(a[7])[:a[0]] == [2, 2, 1]
    assert float(opt.state[w1]["step"]) == 2 and float(opt.state[frozen]["step"]) == 1
    # ReduceLROnPlateau-style lr edits are picked up
    opt.param_groups[0]["lr"] = 5e-4
    calls.clear()
    opt.step()
    a = calls[1][1]
    assert a[0] == 3 and list(a[6])[:a[0]] == pytest.approx([5e-4] * 3)     # float32 per tensor
    with pytest.raises(ValueError):
        mo.Adam([w1], amsgrad=True)
    assert mo.Adam([w1]).param_groups[0]["weight_decay"] == 0.0


def test_block_gradient_regions_are_claimed_once_and_dropped_with_their_reducer():
    """ops.claim_zbufs: the bucket regions of a GROUP of blocks are handed out all-or-nothing, once
    per backward, only while the reducer has zero-filled them; unregister_zbuf_dests drops every
    region that lives in a removed reducer's buckets and keeps those of other reducers."""
    k1, k2 = torch.nn.Parameter(torch.zeros(2, 2)), torch.nn.Parameter(torch.zeros(2, 2))
    k3, other = torch.nn.Parameter(torch.zeros(2, 2)), torch.nn.Parameter(torch.zeros(3))
    flat_a, flat_b = torch.zeros(256), torch.zeros(256)
    ops.clear_grad_dest()
    ops.register_zbuf_dest(k1, flat_a, 0, 100)
    ops.register_zbuf_dest(k2, flat_a, 128, 100)
    ops.register_zbuf_dest(k3, flat_b, 32, 100)
    try:
        ops.grad_dest_enabled, ops.grad_dest_zeroed = True, False
        ops.begin_backward()
        assert ops.claim_zbufs([k1, k2], 100) is None                  # buckets not zero-filled
        ops.grad_dest_zeroed = True
        assert ops.claim_zbufs([k1, other], 100) is None               # one block has no region
        assert ops.claim_zbufs([k1, k2], 96) is None                   # layout mismatch
        z = ops.claim_zbufs([k1, k2], 100)
        assert [t.data_ptr() for t in z] == [flat_a.data_ptr(), flat_a[128:].data_ptr()]
        assert all(t.numel() == 100 for t in z)
        assert ops.claim_zbufs([k1, k2], 100) is None                  # second use in this backward
        ops.begin_backward()
        assert ops.claim_zbufs([k2], 100) is not None
        ops.unregister_zbuf_dests([flat_a])
        ops.begin_backward()
        assert ops.claim_zbufs([k2], 100) is None
        assert ops.claim_zbufs([k3], 100)[0].data_ptr() == flat_b[32:].data_ptr()
        ops.unregister_zbuf_dests([flat_b])
        ops.begin_backward()
        assert ops.claim_zbufs([k3], 100) is None
    finally:
        ops.grad_dest_zeroed = False
        ops.clear_grad_dest()
        ops.begin_backward()


def test_ensemble_emotion_scores_follow_demo_output():
    """robot_demo.py:594-595,609,615-622: score = 1 / (1 + exp(-x + t)) with the per-emotion
    offsets happy .1, sad .1, angry -.1, disgust 0, surprise .1, fear 0, rounded to 2 places."""
    import math

    from mmemo_b200.robot_demo import Ensemble
    ens = Ensemble([torch.nn.Linear(2, 2)])
    pred = torch.tensor([[0.3, -1.2, 2.0, 0.0, -0.1, 5.0, 9.9]])
    offs = [0.1, 0.1, -0.1, 0.0, 0.1, 0.0]
    exp = [round(1 / (1 + math.exp(-float(pred[0][i]) + offs[i])), 2) for i in range(6)]
    got = ens.emotions(pred)
    assert list(got) == ["happy", "sad", "angry", "disgust", "surprise", "fear"]
    assert all(abs(g - e) <= 0.011 for g, e in zip(got.values(), exp)), (got, exp)
    with pytest.raises(ValueError):
        Ensemble([])
    with pytest.raises(RuntimeError):          # no CPU fallback
        ens(*[torch.zeros(1, 2)] * 8)


def test_bucket_length_is_sliceable_for_any_world():
    """The all-reduce kernel needs bucket_len % (4 * world) == 0; layouts of the tested worlds
    (2, 4, 8) keep the 1024-float granularity."""
    from mmemo_b200 import dp
    ps = [torch.nn.Parameter(torch.zeros(n)) for n in (5, 96 * 96, 1, 33)]
    for world in range(1, 17):
        offs, n = dp._Bucket.layout(ps, world)
        assert n % (4 * world) == 0 and n >= offs[-1] + 33 and all(o % 32 == 0 for o in offs)
        if world in (1, 2, 4, 8, 16):
            assert n == dp._Bucket.layout(ps)[1] and n % 1024 == 0


def test_training_dropout_stays_on_the_grouped_path(stub, monkeypatch):
    """Ren-MME trains with dropout 0.1 (Ren-MME/run.py:36).  The grouped trunk keeps its launch
    count: the two dropout sites of the 18 chains are ONE grouped launch each per direction, not
    36 per-tensor kernels (and not the per-op fallback path)."""
    monkeypatch.setattr(mmemo_b200.ren_mme, "DROP", 0.1)
    m = mmemo_b200.ren_mme.Base_model(16, 4, 5, 6, 2, 1, 1, l_dim=8, v_dim=6, a_dim=7).train()
    g = torch.Generator().manual_seed(0)
    inputs = []
    for L, D in ((4, 8), (5, 6), (6, 7)):
        for _ in range(2):
            inputs += [torch.randn(2, L, D, generator=g), torch.ones(2, L)]
    with mmemo_b200.precision("bf16"):
        out = m(*inputs)
        ops.circle_loss_op(out, torch.zeros(2, 9)).mean().backward()
    assert sum(n == "mmemo_dropout_multi_bf16" for n in stub) == 4     # 2 sites x (fwd + bwd)
    assert not any(n in ("mmemo_dropout_bf16", "mmemo_dropout_f32") for n in stub)
    assert sum(n.startswith("mmemo_resattn") for n in stub) == 2
    assert len(stub) <= 60, (len(stub), stub)
