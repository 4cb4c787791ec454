"""Not a test: the fold-uncertainty reduction (ensemble.fold_uncertainty, one sm_100a kernel)
against the same reduction in eager PyTorch (ensemble.fold_uncertainty_reference on the GPU, in
float32 and in its default float64), over k folds x B rows x C classes of float32 fold logits, and
what the flag costs a whole fold-ensemble request.

Part 1, per (k, B, C): microseconds per call from CUDA events around `--iters` back-to-back calls,
the three variants alternating, after warm-up.  Nothing flushes the cache between calls: a working
set (the MB column: logits read + outputs written) below the B200's 126 MB of L2 is read from L2,
as it is when the ensemble head has just written the logits; the largest shapes are not.  Also the
kernel's bytes moved per second, and the largest difference of the kernel from the float64
reference.
Part 2: ms per graphed request of ensemble.Ensemble with k members at a BASELINE inference shape,
return_uncertainty off and on (CUDA events, alternating).
Prints the GPU name and power limit first.  Writes nothing."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mmemo_b200  # noqa: E402
from mmemo_b200 import synth  # noqa: E402
from mmemo_b200.ensemble import Ensemble, fold_uncertainty, fold_uncertainty_reference  # noqa: E402

DEV = "cuda"
SHAPES = [(k, B, C) for k in (5, 10) for B in (32, 1000, 65536) for C in (7, 128)]
ARGS6 = ("l", "v", "a", "l_mask", "v_mask", "a_mask")
REQUESTS = {   # name -> (constructor, forward arguments)
    "cfg1b Concat_Trans B=32": (
        lambda: mmemo_b200.cmu_mosei.Concat_Trans(96, 20, 100, 200, 6, 1, 1),
        lambda: [synth.mosei_batch(seed=7, B=32)[k] for k in ARGS6]),
    "cfg3 Concat_Linear B=128": (
        lambda: mmemo_b200.rencecps.Concat_Linear(2304),
        lambda: [synth.rencecps_batch(seed=7, B=128)["feat"]]),
}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def time_alternating(variants, iters, warmup, reps):
    """ms per call of each variant: `reps` rounds, each timing `iters` back-to-back calls of every
    variant in turn; the mean over the rounds."""
    for _ in range(warmup):
        for fn in variants.values():
            fn()
    torch.cuda.synchronize()
    total = {k: 0.0 for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            e1.synchronize()
            total[k] += e0.elapsed_time(e1) / iters / reps
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--members", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_uncertainty.py needs a CUDA device")
    print(gpu_info(), flush=True)
    print(f"{a.reps} rounds x {a.iters} calls per variant (alternating), {a.warmup} warm-up calls",
          flush=True)
    print("| k | B | C | MB | kernel us | eager fp32 us | eager fp64 us | speed-up vs fp32 | "
          "kernel GB/s | max abs diff vs fp64 |")
    print("|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|")
    g = torch.Generator(device=DEV).manual_seed(0)
    for k, B, C in SHAPES:
        x = torch.randn(k, B, C, generator=g, device=DEV) * 4
        variants = {"kern": lambda: fold_uncertainty(x),
                    "f32": lambda: fold_uncertainty_reference(x, torch.float32),
                    "f64": lambda: fold_uncertainty_reference(x)}
        t = time_alternating(variants, a.iters, a.warmup, a.reps)
        u, ref = fold_uncertainty(x), fold_uncertainty_reference(x)
        diff = max((p.double() - q.double()).abs().max().item() for p, q in zip(u[:5], ref[:5]))
        nbytes = k * B * C * 4 + 2 * B * C * 4 + B * (3 * 4 + 8)
        us = {n: v * 1e3 for n, v in t.items()}
        print(f"| {k} | {B} | {C} | {nbytes / 1e6:.2f} | {us['kern']:.2f} | {us['f32']:.1f} | "
              f"{us['f64']:.1f} | "
              f"{us['f32'] / us['kern']:.1f}x | {nbytes / us['kern'] / 1e3:.0f} | {diff:.1e} |",
              flush=True)

    mmemo_b200.ren_mme.DROP = 0.0
    print(f"\nGraphed ensemble.Ensemble request, k = {a.members} members, fp32 and bf16:")
    print("| request | precision | flag off ms | flag on ms | added ms |")
    print("|---|---|---:|---:|---:|")
    for name, (ctor, batch) in REQUESTS.items():
        models = []
        for i in range(a.members):
            torch.manual_seed(i)
            m = ctor()
            m.load_state_dict(synth.randomize_gates(
                {n: v.detach().clone() for n, v in m.state_dict().items()}, seed=30 + i))
            models.append(m.to(DEV).eval())
        args = [t.to(DEV) for t in batch()]
        for prec in ("fp32", "bf16"):
            with mmemo_b200.precision(prec), torch.no_grad():
                ens = Ensemble(models)
                t = time_alternating({"off": lambda: ens(*args),
                                      "on": lambda: ens(*args, return_uncertainty=True)},
                                     iters=20, warmup=3, reps=a.reps)
            print(f"| {name} | {prec} | {t['off']:.3f} | {t['on']:.3f} | "
                  f"{t['on'] - t['off']:+.3f} |", flush=True)


if __name__ == "__main__":
    main()
