"""Not a test: the optimizer step of k-fold training on one GPU — K separate ``optimizer.step()``
calls (the reference's folds, one after the other) against one ``optim.step_group`` over the K
fold optimizers — for the models of cfg 1a, 1b and 4 (``benchlib.WORKLOADS``), K in {1, 2, 3, 5},
fused AdamW with clipping (``max_grad_norm=1.0``) as in the reference loops.  ``step()`` is
``step_group`` of one optimizer, so the comparison is K library-call pairs against one.

Device events around 50 steps after 10 warm-up steps; library calls per step from
``ops.launch_count``; CUDA kernels per step from ``torch.profiler`` in a separate untimed pass.
The fold models' forward / backward are not part of this measurement.  Prints one JSON line
(with the GPU's name and power limit, read in the same run); ``--out FILE`` also writes it there."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import benchlib  # noqa: E402
from mmemo_b200 import ops, optim  # noqa: E402

DEV = "cuda"


def _folds(cfg: str, K: int):
    opts = []
    for k in range(K):
        torch.manual_seed(k)
        m = benchlib.WORKLOADS[cfg](1).model().to(DEV)
        g = torch.Generator(device=DEV).manual_seed(k)
        for p in m.parameters():
            p.grad = torch.randn(p.shape, generator=g, device=DEV)
        opts.append(optim.AdamW(m.parameters(), lr=1e-4 * (k + 1), max_grad_norm=1.0))
    return opts


def _time(fn, steps: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def _counts(fn):
    n0 = ops.launch_count
    fn()
    calls = ops.launch_count - n0
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = sum(e.count for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA
                  and not e.key.startswith("Memset"))
    return calls, kernels


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_folds needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    rows = []
    for cfg in ("cfg1a", "cfg1b", "cfg4"):
        for K in (1, 2, 3, 5):
            opts = _folds(cfg, K)
            n_tensors = sum(len(g["params"]) for o in opts for g in o.param_groups)

            def sequential():
                for o in opts:
                    o.step()

            def grouped():
                optim.step_group(opts)

            t_seq = _time(sequential, a.steps, a.warmup)
            t_grp = _time(grouped, a.steps, a.warmup)
            c_seq, k_seq = _counts(sequential)
            c_grp, k_grp = _counts(grouped)
            rows.append(dict(cfg=cfg, K=K, tensors=n_tensors,
                             sequential=dict(ms=t_seq, library_calls=c_seq, cuda_kernels=k_seq),
                             step_group=dict(ms=t_grp, library_calls=c_grp, cuda_kernels=k_grp),
                             speedup=t_seq / t_grp))
    line = json.dumps(dict(tool="bench_folds", what="optimizer step of K fold models (fused AdamW, "
                           "clip 1.0): K x step() vs one optim.step_group", gpu=gpu,
                           steps=a.steps, warmup=a.warmup, results=rows))
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
