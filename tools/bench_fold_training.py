"""Not a test: one lockstep training step of k folds on one GPU — forward, losses, backward and the
``optim.step_group`` update — with each fold's own forward / loss / backward (the current per-fold
``train_step_group``) against one ``folds.forward`` + ``folds.circle_losses`` (+ ``folds.rdrop_kl``)
for all folds, for cfg 1a / 1b / 4 / 3-faithful (``benchlib.WORKLOADS`` shapes) and cfg5t (robot_demo training:
``Multi_class(192, 25, 100, 100, 6, 2, 2)``, ``synth.robot_batch`` at B = 32 per fold), k in
{1, 2, 3, 5}, fp32 and bf16.  Dropout is off in both variants so that they compute the same losses (the reference
trains cfg 4 with p = 0.1; grouped and per-fold steps then draw different masks).

The two variants alternate (``--reps`` rounds of ``--steps`` timed steps each, after ``--warmup``
steps of both); ms per step is the median round, from CUDA events around the timed steps.  Library
calls per step from ``ops.launch_count``; the max relative difference of the per-fold losses of the
first step from identical weights.

``--dropout`` (cfg5t): both variants are the grouped step at the reference's p = 0.1
(robot_demo.py:41), one with the modality projections as per-op linears + dropouts + concat +
position adds (the projection path before the dropout epilogue existed, kept here as
``_per_op_project_cat``) and one with the fused epilogue; ``loss_max_rel_diff`` is then not a
parity figure (the two draw different masks).  Prints one JSON line per case (with the GPU's name and power
limit, read in the same run); ``--out FILE`` also writes them there."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import benchlib  # noqa: E402
import mmemo_b200  # noqa: E402
from mmemo_b200 import folds, ops, optim, synth  # noqa: E402

DEV = "cuda"
ARGS6 = ("l", "v", "a", "l_mask", "v_mask", "a_mask")
BATCH = {"cfg1a": 32, "cfg1b": 32, "cfg4": 256, "cfg3": 128, "cfg5t": 32}   # batch per fold
ROBOT = ("l", "v_256", "v_512", "v_1024", "a", "l_mask", "v_mask", "a_mask")
# cfg -> (forward args of a batch dict, row weights or None, R-Drop term)
SPEC = {
    "cfg1a": (lambda b: [b[k] for k in ARGS6], lambda b: b["wmask"].float(), False),
    "cfg1b": (lambda b: [b[k] for k in ARGS6], lambda b: None, False),
    "cfg4": (lambda b: [b[f"x{i}"] for i in range(12)], lambda b: None, True),
    "cfg3": (lambda b: [b["feat"]], lambda b: None, False),
    "cfg5t": (lambda b: [b[k] for k in ROBOT], lambda b: None, False),
}


class _Cfg5Train:
    """robot_demo.py:497-524: the 4-fold training of Multi_class at the native lengths."""

    def __init__(self, batch):
        self.batch = batch

    def model(self):
        return mmemo_b200.robot_demo.Multi_class(192, 25, 100, 100, 6, 2, 2)

    def host_batch(self, seed):
        return synth.robot_batch(seed=seed, B=self.batch)


WORKLOADS = dict(benchlib.WORKLOADS, cfg5t=_Cfg5Train)


def _per_op_project_cat(xs, ws, biases, spans, poss, bf16=False, drop_p=0.0, seed=0):
    """The per-op projection path: one linear and one dropout per problem, concat, position add."""
    ys = [ops.dropout(ops.linear(x, w, b, bf16=bf16), drop_p, True) for x, w, b in zip(xs, ws, biases)]
    outs, g = [], 0
    for n, pos in zip(spans, poss):
        y = ys[g] if n == 1 else torch.cat(ys[g:g + n], -1)
        outs.append(y if pos is None else y + pos.to(y.dtype))
        g += n
    return outs


def _with_projection(fn, step):
    def run(ms, bs):
        keep = folds.project_cat
        folds.project_cat = fn
        try:
            return step(ms, bs)
        finally:
            folds.project_cat = keep
    return run


def _no_dropout(m):
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    return m


def _per_fold(args_of, w_of, rdrop):
    def step(ms, bs):
        out = []
        for m, b in zip(ms, bs):
            lg = m(*args_of(b))
            loss = ops.circle_loss_op(lg, b["label"])
            w = w_of(b)
            loss = (loss * w).mean() if w is not None else loss.mean()
            out.append(loss + ops.rdrop_kl_op(lg) if rdrop else loss)
        return out
    return step


def _grouped(args_of, w_of, rdrop):
    def step(ms, bs):
        ls = folds.forward(ms, [args_of(b) for b in bs])
        ws = [w_of(b) for b in bs]
        losses = folds.circle_losses(ls, [b["label"] for b in bs], None if ws[0] is None else ws)
        return [c + r for c, r in zip(losses, folds.rdrop_kl(ls))] if rdrop else losses
    return step


def _train(ms, opts, bs, step):
    for o in opts:
        o.zero_grad()
    losses = step(ms, bs)
    total = losses[0]
    for x in losses[1:]:
        total = total + x
    total.backward()
    optim.step_group(opts)
    return losses


def _time(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cfgs", default="cfg1a,cfg1b,cfg4,cfg3")
    ap.add_argument("--ks", default="1,2,3,5")
    ap.add_argument("--modes", default="bf16,fp32")
    ap.add_argument("--dropout", action="store_true",
                    help="cfg5t at p = 0.1: per-op projections against the dropout epilogue")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fold_training needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = []
    for cfg in a.cfgs.split(","):
        args_of, w_of, rdrop = SPEC[cfg]
        for mode in a.modes.split(","):
            for K in (int(k) for k in a.ks.split(",")):
                wl = WORKLOADS[cfg](BATCH[cfg])
                mmemo_b200.set_precision(mode)
                ops.clear_shadow_cache()
                base = []
                for k in range(K):
                    torch.manual_seed(k)
                    m = wl.model()
                    base.append((m if a.dropout else _no_dropout(m)).to(DEV).train())
                bs = [benchlib._to(wl.host_batch(10 + k), DEV) for k in range(K)]
                variants = {}
                pairs = (("per_fold", _per_fold(args_of, w_of, rdrop)),
                         ("grouped", _grouped(args_of, w_of, rdrop)))
                if a.dropout:
                    pairs = (("per_fold", _with_projection(_per_op_project_cat, pairs[1][1])),
                             pairs[1])
                for name, step in pairs:
                    ms = [copy.deepcopy(m) for m in base]
                    opts = [optim.AdamW(m.parameters(), lr=1e-4, max_grad_norm=1.0) for m in ms]
                    first = [x.item() for x in _train(ms, opts, bs, step)]
                    variants[name] = dict(ms=ms, opts=opts, step=step, first=first, times=[])
                for _ in range(a.warmup):
                    for v in variants.values():
                        _train(v["ms"], v["opts"], bs, v["step"])
                calls = {}
                for name, v in variants.items():
                    n0 = ops.launch_count
                    _train(v["ms"], v["opts"], bs, v["step"])
                    calls[name] = ops.launch_count - n0
                for _ in range(a.reps):
                    for v in variants.values():
                        v["times"].append(_time(lambda v=v: _train(v["ms"], v["opts"], bs,
                                                                   v["step"]), a.steps))
                diff = max(abs(x - y) / max(abs(x), 1e-12) for x, y in
                           zip(variants["per_fold"]["first"], variants["grouped"]["first"]))
                row = dict(tool="bench_fold_training", gpu=gpu, cfg=cfg, mode=mode, K=K,
                           dropout=0.1 if a.dropout else 0.0,
                           steps=a.steps, warmup=a.warmup, reps=a.reps,
                           per_fold=dict(ms=statistics.median(variants["per_fold"]["times"]),
                                         ms_all=variants["per_fold"]["times"],
                                         library_calls=calls["per_fold"]),
                           grouped=dict(ms=statistics.median(variants["grouped"]["times"]),
                                        ms_all=variants["grouped"]["times"],
                                        library_calls=calls["grouped"]),
                           loss_max_rel_diff=diff)
                row["speedup"] = row["per_fold"]["ms"] / row["grouped"]["ms"]
                line = json.dumps(row)
                print(line, flush=True)
                lines.append(line)
                del variants, base
                torch.cuda.empty_cache()
    mmemo_b200.set_precision("fp32")
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
