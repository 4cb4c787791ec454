"""GPU parity tests of the drop-in modules.

1. every model family vs the committed golden fixtures (= outputs of the REFERENCE's own classes,
   tests/golden/make_golden.py): float32 mode <= 1e-4 relative on logits, loss, every parameter
   gradient and input gradients; bf16 mode <= 2e-2 relative on logits;
2. BASELINE.json's full-size configurations vs the CPU oracle on the same seeded inputs;
3. size-independent properties at full size (batch-permutation equivariance, DP-shard
   equivalence of gradients, window folding).
"""
import pytest
import torch

import mmemo_b200
from mmemo_b200 import ops, synth
from oracle import mmemo_oracle as O
from tests import cases
from tests.cases import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL32, TOLBF = 1e-4, 2e-2


class Loss:
    multi_circle_loss = staticmethod(lambda p, t: ops.circle_loss_op(p, t))
    multi_loss = staticmethod(lambda p, t: ops.circle_loss_op(p, t).mean())
    rdrop_kl = staticmethod(lambda p: ops.rdrop_kl_op(p))


def assert_grads_close(ours, ref32, ref64=None, tol=TOL32):
    """max-relative error per tensor <= tol.  At BASELINE's full sizes an fp32 implementation flips
    a handful of ReLU decisions (|pre-activation| ~ 1e-7 among millions) relative to any other
    summation order; each flip moves one term of a bias / weight gradient by O(1).  The fp32 oracle
    shows the same effect against the fp64 oracle, so when ``ref64`` is given a tensor passes if its
    error vs fp64 is within 5x the oracle's own fp32-vs-fp64 error (the noise floor), and the floor
    is reported next to our number."""
    bad = []
    for k, v in ref32.items():
        if ref64 is None:
            e, lim = rel_err(ours[k], v), tol
        else:
            e = rel_err(ours[k], ref64[k])
            lim = max(tol, 5.0 * rel_err(v, ref64[k]))
            if v.numel() == 1:
                # scalar gates a/b/c: the gradient is ONE sum of millions of signed terms (e.g.
                # c.grad = sum(dS * S_prev)); its relative error measures cancellation, not a
                # per-element error, so it gets 3x headroom
                lim = max(lim, 3.0 * tol)
        if not e < lim and k.endswith(("ffn.0.weight", "ffn.0.bias")):
            # rows (= hidden units) of the first FFN linear are the direct consumers of the ReLU
            # mask: one flipped decision moves a whole row by ~1/sqrt(rows).  Require >= 99% of
            # the hidden units within tolerance and every unit within 5e-2.
            r = (ref64[k] if ref64 is not None else v).double().cpu()
            o = ours[k].double().cpu()
            den = r.abs().max().item()
            per_unit = (o - r).abs().reshape(r.shape[0], -1).max(1)[0] / den
            frac_ok = (per_unit < lim).double().mean().item()
            if frac_ok >= 0.99 and per_unit.max().item() < 5e-2:
                continue
            bad.append((k, e, lim, f"units within tol: {frac_ok:.4f}"))
        elif not e < lim:
            bad.append((k, e, lim))
    assert not bad, bad


def f64(t):
    if isinstance(t, dict):
        return {k: f64(v) for k, v in t.items()}
    return t.double() if torch.is_tensor(t) and t.is_floating_point() else t


def to_dev(b):
    if isinstance(b, dict):
        return {k: to_dev(v) for k, v in b.items()}
    if isinstance(b, (list, tuple)):
        return [to_dev(v) for v in b]
    return b.to(DEV) if torch.is_tensor(b) else b


@pytest.fixture(autouse=True)
def _defaults():
    mmemo_b200.robot_demo.DROP = 0.0
    mmemo_b200.ren_mme.DROP = 0.0
    mmemo_b200.set_precision("fp32")
    ops.clear_shadow_cache()
    yield
    mmemo_b200.set_precision("fp32")


@pytest.mark.parametrize("name", list(cases.CASES))
def test_golden_fp32(name):
    c = cases.CASES[name]
    g = torch.load(cases.golden_path(name))
    model = c.our_model(mmemo_b200).to(DEV).train()
    model.load_state_dict(g["state"])
    logits, loss, grads, igrads = cases.run_module_with_grads(model, c, to_dev(g["batch"]), Loss)
    assert rel_err(logits, g["logits"]) < TOL32
    assert abs(loss.item() - g["loss"].item()) < TOL32 * max(1.0, abs(g["loss"].item()))
    assert set(grads) == set(g["grads"])
    worst = max((rel_err(grads[k], v), k) for k, v in g["grads"].items())
    assert worst[0] < TOL32, worst
    for k, v in g["input_grads"].items():
        assert rel_err(igrads[k], v) < TOL32, k


@pytest.mark.parametrize("name", list(cases.CASES))
def test_golden_bf16_logits(name):
    c = cases.CASES[name]
    g = torch.load(cases.golden_path(name))
    model = c.our_model(mmemo_b200).to(DEV).train()
    model.load_state_dict(g["state"])
    with mmemo_b200.precision("bf16"), torch.no_grad():
        logits = c.call(model, to_dev(g["batch"]))
    assert rel_err(logits.float(), g["logits"]) < TOLBF


def test_golden_eval_mode_no_grad(name="robot_multi_class"):
    """robot_demo inference path: eval() + no_grad forward (robot_demo.py:610-614)."""
    c = cases.CASES[name]
    g = torch.load(cases.golden_path(name))
    model = c.our_model(mmemo_b200).to(DEV).eval()
    model.load_state_dict(g["state"])
    with torch.no_grad():
        logits = c.call(model, to_dev(g["batch"]))
    assert rel_err(logits, g["logits"]) < TOL32


# ------------------------------------------------------------------------------------------------
# full-size configurations vs the oracle
# ------------------------------------------------------------------------------------------------
def _model_and_state(ctor, seed=0):
    torch.manual_seed(seed)
    m = ctor().train()
    sd = cases.seeded_state(m, seed=1)
    m.load_state_dict(sd)
    return m.to(DEV), sd


@pytest.mark.parametrize("empty_windows", [False, True])
def test_cfg1a_realformer_state_transfer_full_size(empty_windows):
    """BASELINE config 1 (others/realformer.py defaults): B=32, P=6, seq 50, d=96, 6 heads, 2 layers.
    With 'no_name' empty windows (all-zero masks, zero loss weight) only the forward is compared:
    on fully masked rows c.grad = sum(dS * S_prev) cancels against -1e8 and the fp32 reference
    itself is noise there (SURVEY §8a note 1(iii): fp32 ref -4.6e-3 vs fp64 -5.3e-5)."""
    kw = dict(l_dim=300, v_dim=35, a_dim=74, dim=96, l_len=50, v_len=50, a_len=50, n_heads=6,
              n_layers=2, ffn=2)
    m, sd = _model_and_state(lambda: mmemo_b200.realformer.State_Transfer(**kw))
    b = synth.realformer_batch(seed=1234, B=32, P=6, empty_windows=empty_windows)
    c = cases.CASES["realformer_state_transfer"]
    if empty_windows:
        with torch.no_grad():
            ref = O.realformer_state_transfer(sd, b["l"], b["v"], b["a"], b["l_mask"], b["v_mask"],
                                              b["a_mask"], 6, 2)
            out = cases._rf_call(m, to_dev(b))
        assert torch.isfinite(out).all()
        assert rel_err(out, ref) < TOL32
        return
    fn = lambda s, bb: O.realformer_state_transfer(s, bb["l"], bb["v"], bb["a"], bb["l_mask"],
                                                   bb["v_mask"], bb["a_mask"], 6, 2)
    ref_logits, ref_loss, ref_grads, _ = cases.run_with_grads(fn, sd, b, c.loss, O, [])
    _, _, ref_grads64, _ = cases.run_with_grads(fn, f64(sd), f64(b), c.loss, O, [])
    logits, loss, grads, _ = cases.run_module_with_grads(
        m, cases.Case(**{**c.__dict__, "grad_inputs": []}), to_dev(b), Loss)
    assert rel_err(logits, ref_logits) < TOL32
    assert abs(loss.item() - ref_loss.item()) < TOL32 * abs(ref_loss.item())
    assert_grads_close(grads, ref_grads, ref_grads64)


def test_cfg2_encoder_chain_full_size_fp32_and_bf16():
    """BASELINE config 2: 6 x Attention_Block(512, 8), B=64, L=128."""
    dim, H, nl = 512, 8, 6
    m, sd = _model_and_state(lambda: cases._RefChain(mmemo_b200.realformer.Attention_Block, dim, H,
                                                     nl))
    b = synth.encoder_batch(seed=1234, B=64, L=128, d=dim)
    pres = [f"blocks.{i}." for i in range(nl)]
    fn = lambda s, bb: O.encoder_chain(s, pres, bb["x"], bb["mask"], H)[0]
    ref_out, ref_loss, ref_grads, ref_ig = cases.run_with_grads(fn, sd, b, cases._sq_mean, O, ["x"])
    _, _, ref_grads64, ref_ig64 = cases.run_with_grads(fn, f64(sd), f64(b), cases._sq_mean, O, ["x"])
    c = cases.CASES["encoder_chain"]
    out, loss, grads, ig = cases.run_module_with_grads(m, c, to_dev(b), Loss)
    assert rel_err(out, ref_out) < TOL32
    assert_grads_close(grads, ref_grads, ref_grads64)
    assert_grads_close(ig, ref_ig, ref_ig64)
    with mmemo_b200.precision("bf16"):
        out_bf, loss_bf, grads_bf, _ = cases.run_module_with_grads(m, c, to_dev(b), Loss)
    assert out_bf.dtype == torch.bfloat16
    assert rel_err(out_bf.float(), ref_out) < TOLBF
    # bf16 gradients are not a stated criterion; keep them sane (direction + scale)
    for k in ("blocks.0.w_qkv.0.weight", "blocks.5.ffn.2.weight", "blocks.3.proj.weight",
              "blocks.5.w_qkv.0.weight", "blocks.5.w_qkv.2.weight", "blocks.2.w_qkv.1.weight",
              "blocks.0.w_qkv.2.weight", "blocks.4.ffn.0.weight"):
        a, r = grads_bf[k].flatten().double().cpu(), ref_grads[k].flatten().double()
        cos = torch.dot(a, r) / (a.norm() * r.norm())
        assert cos > 0.98, (k, cos.item())


def test_cfg1b_mosei_native_lengths_full_batch_with_gradients():
    """cmu-mosei/run.py at its native lengths 20/100/200 (9 (Lq,Lk) combinations, Lk up to 200),
    1 layer, FULL batch 32: logits, loss and every parameter gradient in float32; bf16 logits."""
    kw = dict(dim=96, l_len=20, v_len=100, a_len=200, n_heads=6, n_layers=1, ffn=1)
    m, sd = _model_and_state(lambda: mmemo_b200.cmu_mosei.Concat_Trans(**kw))
    b = synth.mosei_batch(seed=1234, B=32)
    c = cases.CASES["mosei_concat_trans"]
    nog = cases.Case(**{**c.__dict__, "grad_inputs": []})
    fn = lambda s, bb: O.mosei_concat_trans(s, bb["l"], bb["v"], bb["a"], bb["l_mask"],
                                            bb["v_mask"], bb["a_mask"], 6, 1)
    ref_logits, ref_loss, ref_grads, _ = cases.run_with_grads(fn, sd, b, c.loss, O, [])
    _, _, ref_grads64, _ = cases.run_with_grads(fn, f64(sd), f64(b), c.loss, O, [])
    logits, loss, grads, _ = cases.run_module_with_grads(m, nog, to_dev(b), Loss)
    assert rel_err(logits, ref_logits) < TOL32
    assert abs(loss.item() - ref_loss.item()) < TOL32 * abs(ref_loss.item())
    assert set(grads) == set(ref_grads)
    assert_grads_close(grads, ref_grads, ref_grads64)
    with mmemo_b200.precision("bf16"), torch.no_grad():
        out_bf = cases._rf_call(m, to_dev(b))
    assert rel_err(out_bf.float(), ref_logits) < TOLBF


def test_cfg1a_realformer_full_size_bf16_logits():
    kw = dict(l_dim=300, v_dim=35, a_dim=74, dim=96, l_len=50, v_len=50, a_len=50, n_heads=6,
              n_layers=2, ffn=2)
    m, sd = _model_and_state(lambda: mmemo_b200.realformer.State_Transfer(**kw))
    b = synth.realformer_batch(seed=1234, B=32, P=6)
    with torch.no_grad():
        ref = O.realformer_state_transfer(sd, b["l"], b["v"], b["a"], b["l_mask"], b["v_mask"],
                                          b["a_mask"], 6, 2)
        with mmemo_b200.precision("bf16"):
            out = cases._rf_call(m, to_dev(b))
    assert rel_err(out.float(), ref) < TOLBF


def test_cfg4_renmme_full_batch_256_with_rdrop_loss():
    """Ren-MME/run.py defaults at the FULL batch BASELINE names (256 = 128 R-Drop pairs): seq
    40/76/275, dims 768/640/205, d=128, 8 heads: logits, loss (multi_loss + symmetric KL) and
    every parameter gradient in float32; bf16 logits; bf16 training step runs (tiled Lk=275
    backward) and its gradients point the same way."""
    m, sd = _model_and_state(lambda: mmemo_b200.ren_mme.Base_model())
    b = synth.renmme_batch(seed=1234, B=256)
    c = cases.CASES["renmme_base_model"]
    fn = lambda s, bb: O.renmme_base_model(s, *bb["inputs"])
    ref_logits, ref_loss, ref_grads, _ = cases.run_with_grads(fn, sd, b, c.loss, O, [])
    logits, loss, grads, _ = cases.run_module_with_grads(m, c, to_dev(b), Loss)
    assert rel_err(logits, ref_logits) < TOL32
    assert abs(loss.item() - ref_loss.item()) < TOL32 * abs(ref_loss.item())
    assert set(grads) == set(ref_grads)
    worst = max((rel_err(grads[k], v), k) for k, v in ref_grads.items())
    assert worst[0] < TOL32, worst
    # R-Drop pairs carry identical inputs and dropout is off -> the same logits (to the fp32
    # summation order of the split-K classifier GEMM, whose slices are added by atomics)
    assert torch.allclose(logits[0::2], logits[1::2], rtol=0, atol=2e-6)
    with mmemo_b200.precision("bf16"):
        logits_bf, _, grads_bf, _ = cases.run_module_with_grads(m, c, to_dev(b), Loss)
    assert rel_err(logits_bf.float(), ref_logits) < TOLBF
    for k in ("intensity.multimodal_blocks.6.proj.weight", "stimulation.multimodal_blocks.8.minus.weight",
              "intensity.unify_dimension.acoustic.weight", "stimulation.classifier.weight"):
        a, r = grads_bf[k].flatten().double().cpu(), ref_grads[k].flatten().double()
        cos = torch.dot(a, r) / (a.norm() * r.norm())
        assert cos > 0.98, (k, cos.item())


def test_cfg3_composite_text_encoder_full_size():
    """BASELINE configs[2] as worded (seq 256, batch 128, RealFormer encoder): 6 x
    Attention_Block(512, 8) on 64 (previous, current) sentence pairs = 128 sequences of 256 tokens
    -> cls|max|mean pooling -> Concat_Linear(1536).  Oracle = composition of the reference
    classes' restatements (benchlib.composite_oracle)."""
    import benchlib
    wl = benchlib.Cfg3Composite(64)
    m, sd = _model_and_state(wl.model)
    b = wl.host_batch(1234)
    fn = lambda s, bb: benchlib.composite_oracle(O, s, bb["x"], bb["mask"])
    loss_fn = lambda lg, bb, L: L.multi_circle_loss(lg, bb["label"]).mean()
    ref_logits, ref_loss, ref_grads, _ = cases.run_with_grads(fn, sd, b, loss_fn, O, [])
    _, _, ref_grads64, _ = cases.run_with_grads(fn, f64(sd), f64(b), loss_fn, O, [])
    bd = to_dev(b)
    m.zero_grad(set_to_none=True)
    logits = m(bd["x"], bd["mask"])
    loss = ops.circle_loss_op(logits, bd["label"]).mean()
    loss.backward()
    grads = {k: p.grad.detach() for k, p in m.named_parameters() if p.grad is not None}
    assert rel_err(logits, ref_logits) < TOL32
    assert abs(loss.item() - ref_loss.item()) < TOL32 * abs(ref_loss.item())
    assert set(grads) == set(ref_grads)
    assert_grads_close(grads, ref_grads, ref_grads64)
    with mmemo_b200.precision("bf16"), torch.no_grad():
        out_bf = m(bd["x"], bd["mask"])
    assert rel_err(out_bf.float(), ref_logits) < TOLBF


def test_cfg5_robot_demo_native_shapes_batch1_and_32():
    kw = dict(dim=192, l_len=25, v_len=100, a_len=100, n_heads=6, n_layers=2, ffn=2)
    m, sd = _model_and_state(lambda: mmemo_b200.robot_demo.Multi_class(**kw))
    m.eval()
    for B in (1, 32):
        b = synth.robot_batch(seed=77, B=B)
        with torch.no_grad():
            ref = O.robot_multi_class(sd, b["l"], b["v_256"], b["v_512"], b["v_1024"], b["a"],
                                      b["l_mask"], b["v_mask"], b["a_mask"], 6, 2)
            out = cases._robot_call(m, to_dev(b))
        assert rel_err(out, ref) < TOL32


def test_cfg3_rencecps_full_size():
    m, sd = _model_and_state(lambda: mmemo_b200.rencecps.Concat_Linear(2304))
    b = synth.rencecps_batch(seed=5, B=128)
    c = cases.CASES["rencecps_concat_linear"]
    ref_logits, ref_loss, ref_grads, _ = cases.run_with_grads(
        lambda s, bb: O.rencecps_concat_linear(s, bb["feat"]), sd, b, c.loss, O, [])
    logits, loss, grads, _ = cases.run_module_with_grads(
        m, cases.Case(**{**c.__dict__, "grad_inputs": []}), to_dev(b), Loss)
    assert rel_err(logits, ref_logits) < TOL32
    worst = max((rel_err(grads[k], v), k) for k, v in ref_grads.items())
    assert worst[0] < TOL32, worst


# ------------------------------------------------------------------------------------------------
# size-independent properties
# ------------------------------------------------------------------------------------------------
def test_batch_permutation_equivariance_and_dp_shard_equivalence():
    """Every op is per-sample: permuting the batch permutes the logits, and the mean of per-shard
    gradients equals the full-batch gradient (SURVEY §8e: DP is exact up to fp32 summation)."""
    kw = dict(dim=96, l_len=50, v_len=50, a_len=50, n_heads=6, n_layers=2, ffn=1)
    m, _ = _model_and_state(lambda: mmemo_b200.cmu_mosei.Concat_Trans(**kw))
    b = to_dev(synth.mosei_batch(seed=3, B=16, L=(50, 50, 50)))
    c = cases.CASES["mosei_concat_trans"]
    nog = cases.Case(**{**c.__dict__, "grad_inputs": []})
    logits, _, full, _ = cases.run_module_with_grads(m, nog, b, Loss)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(0)).to(DEV)
    pb = {k: v[perm] for k, v in b.items()}
    with torch.no_grad():
        assert torch.allclose(cases._rf_call(m, pb), logits[perm], atol=1e-5)
    acc = {k: torch.zeros_like(v) for k, v in full.items()}
    for sh in range(4):
        sl = slice(4 * sh, 4 * sh + 4)
        _, _, gsh, _ = cases.run_module_with_grads(m, nog, {k: v[sl] for k, v in b.items()}, Loss)
        for k in acc:
            acc[k] += gsh[k] / 4
    # tensors: 1e-5.  The scalar gates (c, a, b) are ONE sum with cancellation over every score /
    # activation of the batch, accumulated with atomics: their fp32 summation-order noise was
    # measured at 1.1e-5 on this case, so they get 1e-4 (still far below any real sharding error,
    # which would be O(1/shards)).
    worst = max((rel_err(acc[k], full[k]), k) for k in full if full[k].numel() > 1)
    assert worst[0] < 1e-5, worst
    worst_s = max((rel_err(acc[k], full[k]), k) for k in full if full[k].numel() == 1)
    assert worst_s[0] < 1e-4, worst_s


def test_scores_returned_by_block_match_reference_semantics():
    """Attention_Block returns post-mask pre-softmax scores, chained with c*S_prev
    (others/realformer.py:191-204)."""
    blk = mmemo_b200.realformer.Attention_Block(96, 6)
    sd = cases.seeded_state(blk, seed=4)
    blk.load_state_dict(sd)
    blk = blk.to(DEV)
    gen = torch.Generator().manual_seed(8)
    q, kv = torch.randn(4, 50, 96, generator=gen), torch.randn(4, 50, 96, generator=gen)
    mask = synth.prefix_mask(gen, (4,), 50)
    with torch.no_grad():
        o1, s1 = blk(q.to(DEV), kv.to(DEV), kv.to(DEV), mask.to(DEV))
        o2, s2 = blk(o1, kv.to(DEV), kv.to(DEV), mask.to(DEV), s1)
        r1, t1 = O.block_full(sd, "", q, kv, kv, mask, 6, None)
        r2, t2 = O.block_full(sd, "", r1, kv, kv, mask, 6, t1)
    assert rel_err(o2, r2) < TOL32
    assert rel_err(s2, t2) < 1e-6   # relative to 1.5e8: masked columns must carry c*(-1e8) - 1e8
    valid = mask[:, None, None, :].expand_as(t2) > 0
    assert rel_err(s2.cpu()[valid], t2[valid]) < TOL32


@pytest.mark.parametrize("B", [1, 32])
def test_robot_demo_graphed_ensemble_equals_sequential_members(B):
    """robot_demo.py:610-614: pred = (pred_1 + pred_2 + pred_3 + pred_4) / 4 — the CUDA-graph,
    multi-stream ensemble must return exactly what the members return one by one, also when it is
    replayed on new inputs."""
    kw = dict(dim=192, l_len=25, v_len=100, a_len=100, n_heads=6, n_layers=2, ffn=2)
    models = []
    for i in range(4):
        torch.manual_seed(i)
        m = mmemo_b200.robot_demo.Multi_class(**kw)
        m.load_state_dict(synth.randomize_gates(m.state_dict(), seed=10 + i))
        models.append(m.to(DEV).eval())
    ens = mmemo_b200.robot_demo.Ensemble(models)
    for seed in (1, 2, 3):          # first call captures, later calls replay
        b = to_dev(synth.robot_batch(seed=seed, B=B))
        args = [b[k] for k in mmemo_b200.robot_demo.Ensemble.NAMES]
        with torch.no_grad():
            ref = models[0](*args)
            for m in models[1:]:
                ref = ref + m(*args)
            ref = ref / 4
        out = ens(*args)
        assert rel_err(out, ref) < 1e-5      # (split-K atomics may reorder fp32 sums)
    assert len(ens._graphs) == 1
    emo = ens.emotions(out)
    assert list(emo) == ["happy", "sad", "angry", "disgust", "surprise", "fear"]
    assert all(0.0 <= v <= 1.0 for v in emo.values())


# ------------------------------------------------------------------------------------------------
# grouped trunk (group_ops.py) vs the blocks one by one
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["realformer_state_transfer", "mosei_concat_trans",
                                  "renmme_base_model", "robot_multi_class"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_grouped_trunk_equals_one_problem_groups(name, mode, monkeypatch):
    """One grouped op per layer over all chains / towers (9 or 18 problems) must give what the
    chain-by-chain blocks give (one-problem groups, ``cases.trunk_per_block``): float32 to
    summation order (the same launchers run per problem), bf16 to bf16 noise (different kernels:
    grouped mma.sync attention, grouped tcgen05 GEMMs), for logits AND every parameter / input
    gradient - this pins the slot layout of the grouped weight-gradient buffer."""
    c = cases.CASES[name]
    g = torch.load(cases.golden_path(name))
    model = c.our_model(mmemo_b200).to(DEV).train()
    model.load_state_dict(g["state"])
    b = to_dev(g["batch"])
    with mmemo_b200.precision(mode):
        lg_g, _, gr_g, ig_g = cases.run_module_with_grads(model, c, b, Loss)
        cases.use_per_block_trunk(monkeypatch)
        lg_b, _, gr_b, ig_b = cases.run_module_with_grads(model, c, b, Loss)
    tol = 2e-5 if mode == "fp32" else 4e-2
    assert rel_err(lg_g.float(), lg_b.float()) < tol
    assert set(gr_g) == set(gr_b)
    worst = max((rel_err(gr_g[k], v), k) for k, v in gr_b.items() if v.numel() > 1)
    assert worst[0] < tol, worst
    for k, v in ig_b.items():
        assert rel_err(ig_g[k].float(), v.float()) < tol, k


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_cfg5_ensemble_matches_oracle_mean_of_members(prec):
    """robot_demo.py:610-615 at native shapes: the grouped 4-member ensemble (36 problems per
    launch) against the ORACLE's mean of the four members' logits, B = 1 and B = 32."""
    kw = dict(dim=192, l_len=25, v_len=100, a_len=100, n_heads=6, n_layers=2, ffn=2)
    models, sds = [], []
    for i in range(4):
        torch.manual_seed(i)
        m = mmemo_b200.robot_demo.Multi_class(**kw)
        sd = synth.randomize_gates({k: v.detach().clone() for k, v in m.state_dict().items()},
                                   seed=10 + i)
        m.load_state_dict(sd)
        sds.append(sd)
        models.append(m.to(DEV).eval())
    ens = mmemo_b200.robot_demo.Ensemble(models)
    names = mmemo_b200.robot_demo.Ensemble.NAMES
    with mmemo_b200.precision(prec):
        for B in (1, 32):
            b = synth.robot_batch(seed=21 + B, B=B)
            with torch.no_grad():
                ref = sum(O.robot_multi_class(sd, *[b[k] for k in names], 6, 2) for sd in sds) / 4
            out = ens(*[b[k].to(DEV) for k in names])
            assert rel_err(out.float(), ref) < (TOL32 if prec == "fp32" else TOLBF), (prec, B)
