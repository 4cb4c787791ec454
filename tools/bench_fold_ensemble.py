"""Not a test: request latency of a K-member fold ensemble (default K = 4) of the four model
families at the BASELINE inference shapes, both precisions, three ways of serving a request:

  sequential : the members one after the other, then their mean (what the reference scripts do:
               others/realformer.py:418-420, Ren-MME/run.py:560)
  grouped    : ensemble.Ensemble(use_graph=False)
  graphed    : ensemble.Ensemble (one CUDA graph per input shape)

ms per request from CUDA events (the three variants alternate, after warm-up), libmmemo library calls
per request, and the max relative difference of grouped / graphed against sequential.  Prints the
GPU name and power limit first.  Writes nothing."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mmemo_b200  # noqa: E402
from mmemo_b200 import ops, synth  # noqa: E402
from mmemo_b200.ensemble import Ensemble  # noqa: E402

DEV = "cuda"
ARGS6 = ("l", "v", "a", "l_mask", "v_mask", "a_mask")
CONFIGS = {   # name -> (constructor, forward arguments)
    "cfg1a State_Transfer B=32x6": (
        lambda: mmemo_b200.realformer.State_Transfer(300, 35, 74, 96, 50, 50, 50, 6, 2, 2),
        lambda: [synth.realformer_batch(seed=7, B=32, P=6)[k] for k in ARGS6]),
    "cfg1b Concat_Trans B=32": (
        lambda: mmemo_b200.cmu_mosei.Concat_Trans(96, 20, 100, 200, 6, 1, 1),
        lambda: [synth.mosei_batch(seed=7, B=32)[k] for k in ARGS6]),
    "cfg4 Base_model B=256": (
        lambda: mmemo_b200.ren_mme.Base_model(),
        lambda: list(synth.renmme_batch(seed=7, B=256)["inputs"])),
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


def calls_per_request(fn):
    fn()
    torch.cuda.synchronize()
    n0 = ops.launch_count
    fn()
    return ops.launch_count - n0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=4)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_fold_ensemble.py needs a CUDA device")
    mmemo_b200.ren_mme.DROP = 0.0
    print(gpu_info(), flush=True)
    print(f"K = {a.members} members, {a.iters} timed requests per variant (alternating), "
          f"{a.warmup} warm-up", flush=True)
    print("| config | precision | sequential ms | grouped ms | graphed ms | graphed speed-up | "
          "calls seq / grouped | max rel diff grouped, graphed |")
    print("|---|---|---:|---:|---:|---:|---:|---:|")
    for name, (ctor, batch) in CONFIGS.items():
        models = []
        for k in range(a.members):
            torch.manual_seed(k)
            m = ctor()
            m.load_state_dict(synth.randomize_gates(
                {n: v.detach().clone() for n, v in m.state_dict().items()}, seed=30 + k))
            models.append(m.to(DEV).eval())
        args = [t.to(DEV) for t in batch()]
        for prec in ("fp32", "bf16"):
            with mmemo_b200.precision(prec), torch.no_grad():
                ops.clear_shadow_cache()
                grouped, graphed = Ensemble(models, use_graph=False), Ensemble(models)

                def sequential():
                    pred = models[0](*args)
                    for m in models[1:]:
                        pred = pred + m(*args)
                    return pred / len(models)

                variants = {"seq": sequential, "grp": lambda: grouped(*args),
                            "gr": lambda: graphed(*args)}
                for _ in range(a.warmup):
                    for fn in variants.values():
                        fn()
                times = {k: 0.0 for k in variants}
                for _ in range(a.iters):
                    for k, fn in variants.items():
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        fn()
                        e1.record()
                        e1.synchronize()
                        times[k] += e0.elapsed_time(e1) / a.iters
                ref = sequential().float()
                den = ref.abs().max().item()
                d_grp = (grouped(*args) - ref).abs().max().item() / den
                d_gr = (graphed(*args) - ref).abs().max().item() / den
                c_seq, c_grp = calls_per_request(sequential), calls_per_request(lambda: grouped(*args))
            print(f"| {name} | {prec} | {times['seq']:.3f} | {times['grp']:.3f} | {times['gr']:.3f} | "
                  f"{times['seq'] / times['gr']:.2f}x | {c_seq} / {c_grp} | {d_grp:.1e}, {d_gr:.1e} |",
                  flush=True)


if __name__ == "__main__":
    main()
