#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: "train samples/s (fwd+bwd)").

Workload (BASELINE configs[1]): the RealFormer residual-attention encoder of others/realformer.py
standalone — 6 x Attention_Block(d=512, 8 heads), seq 128, batch 64 PER GPU, bf16 activations /
GEMM operands with fp32 accumulation, fp32 master weights and gradients; one step = zero_grad ->
forward -> loss = mean(out^2) -> backward (optimizer excluded, like the metric).  Synthetic N(0,1)
features with prefix masks, random-init weights with the ReZero gates drawn from U(-0.5, 0.5) (at
their 0 init every attention/FFN gradient is exactly zero).

    python bench.py --gpus N --steps K --warmup W            # ours
    python bench.py ... --dump-outputs DIR                   # + what the last timed step computed
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    torchrun --nproc-per-node N bench.py --gpus N ...        # data parallel, weak scaling

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events around K
CUDA-graph replays, max over ranks); `e2e` = the same step driven from pinned HOST buffers through
the public module API with the H2D copy of the inputs and the D2H read of the loss inside the
timed region; `roofline` = the dominant kernel family timed live with CUDA events (L2 flushed
before every launch for HBM-bound families; the L2-warm time is reported next to it);
`cpu_baseline` = the oracle (CPU port of the reference algorithm) timed on this box's host cores
on a bounded sample; `gpu_eager_baseline` = the same oracle (= the reference's eager PyTorch op
sequence) run on this GPU; `configs` = the other BASELINE.json configurations (the reference's
real models: State_Transfer, Concat_Trans, Concat_Linear, Base_model at global batch 256 sharded
over the ranks = the strong-scaling curve, robot_demo ensemble p50 latency), each with its own
device-timed value, e2e, launch count, kernel table and baselines; `dp` (N > 1) = which gradient
transport ran, the exposed communication time and a check of the reduced gradients.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the benchmark leaves the tree as it found it (which may be read-only): the project modules it
# imports are compiled in memory, no __pycache__ is written next to them
sys.dont_write_bytecode = True

import torch  # noqa: E402

METRIC = "train samples/s (fwd+bwd)"
CFG = dict(dim=512, n_heads=8, n_layers=6, ffn=2, seq_len=128, batch_per_gpu=64)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"],
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


# per array: the headline step's gradients (12.6 M values, none above 2^20) are written whole and
# its 64 x 128 x 512 output is sampled, 52 MiB in all
DUMP_MAX_ELEMS = 1 << 20


def dump_outputs(out_dir: str, arrays) -> None:
    """Write every (name, tensor) of `arrays` as out_dir/<name>.npy in float32.  A tensor of more
    than DUMP_MAX_ELEMS elements is written as the same seeded sample of its flattened elements on
    every run (ascending flat indices), so that the files of two builds compare element for
    element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays:
        a = t.detach().float().cpu()
        if a.numel() > DUMP_MAX_ELEMS:
            g = torch.Generator().manual_seed(0)
            idx = torch.randperm(a.numel(), generator=g)[:DUMP_MAX_ELEMS].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi in the background during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  In-process NVML thread (a
    sample every ~2 ms; the main thread sits in cudaDeviceSynchronize with the GIL released), with
    ``nvidia-smi -lms`` as a fallback when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20,
            "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.handle, self.stop_flag = None, None, False
        self.sm, self.mask, self.mx = [], 0, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _reasons(self):
        fn = getattr(self.nvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(self.nvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
        return int(fn(self.handle))

    def _poll(self):
        while not self.stop_flag:
            try:
                self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.handle,
                                                                      self.nvml.NVML_CLOCK_SM)))
                self.mask |= self._reasons()
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                 "100", "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(k for k, b in self.BITS.items() if self.mask & b),
                    "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# per-kernel instrumentation: CUDA events around every libmmemo launch of one eager step
# ------------------------------------------------------------------------------------------------
def _algorithmic(name: str, a: tuple):
    """(flops, bytes, shape-tag) of one launcher call from its C-ABI arguments (DESIGN.md §kernels;
    formulas of SURVEY.md §8d)."""
    bf = name.endswith("_bf16")
    e = 2 if bf else 4
    if name.startswith("mmemo_resattn") and "_grouped_" in name:
        import ctypes as C
        from mmemo_b200 import _lib
        n = a[0]
        ps = C.cast(a[1], C.POINTER(_lib.AttnProblem))
        bwd = "_bwd_" in name
        fl = by = 0
        tags = {}
        for i in range(n):
            q = ps[i]
            d, S = q.H * q.hd, q.B * q.H * q.Lq * q.Lk
            kv = 1 if q.k == q.v else 2
            if not bwd:
                by += e * q.B * d * (q.Lq + kv * q.Lk) + 4 * q.B * q.Lk + e * q.B * q.Lq * d
                by += e * S * (1 if q.s_prev else 0) + e * S * (1 if q.s_out else 0)
                fl += 4 * q.B * q.Lq * q.Lk * d
                t = f"L{q.Lq}x{q.Lk}{'+prev' if q.s_prev else ''}{'+S' if q.s_out else ''}"
            else:
                by += e * q.B * d * (2 * q.Lq + kv * q.Lk) + e * q.B * d * (q.Lq + kv * q.Lk)
                by += e * q.B * q.Lq * d
                by += e * S * ((1 if q.s else 0) + (1 if q.ds_next else 0))
                by += e * S * ((1 if q.s_prev else 0) + (1 if q.ds_prev else 0))
                fl += (8 if q.s else 10) * q.B * q.Lq * q.Lk * d
                t = (f"L{q.Lq}x{q.Lk}{'+S' if q.s else '+recompute'}{'+prev' if q.s_prev else ''}"
                     f"{'+dSnext' if q.ds_next else ''}")
            tags[t] = tags.get(t, 0) + 1
        q0 = ps[0]
        return fl, by, f"G{n}:B{q0.B}H{q0.H}hd{q0.hd}:" + ",".join(f"{v}x{k}" for k, v in tags.items())
    if name.startswith("mmemo_add_ln_fwd_grouped"):
        Ms, d = list(a[9]), a[10]
        nres = sum(1 for r in a[1] if r)
        return (8 * sum(Ms) * d, e * d * (2 * sum(Ms) + (sum(Ms) * nres // max(1, len(Ms)))),
                f"G{a[0]}:{max(Ms)}x{d}")
    if name.startswith("mmemo_add_ln_bwd_grouped"):
        Ms, d = list(a[14]), a[15]
        nres = sum(1 for r in a[2] if r)
        return (16 * sum(Ms) * d, e * d * (3 * sum(Ms) + 2 * (sum(Ms) * nres // max(1, len(Ms)))),
                f"G{a[0]}:{max(Ms)}x{d}")
    if name.startswith("mmemo_colsum_grouped"):
        Ms, N = list(a[3]), a[4]
        return sum(Ms) * N, e * sum(Ms) * N, f"G{a[0]}:{max(Ms)}x{N}"
    if name.startswith("mmemo_sum_grouped"):        # (n_out, out, n_in[], in, numel[], stream)
        n = a[0]
        by = sum(e * int(m) * (int(k) + 1) for m, k in zip(list(a[4])[:n], list(a[2])[:n]))
        return 0, by, f"G{n}"
    if "_grouped_" in name:   # host arrays of per-problem M, N, K
        i0 = 8 if name.startswith("mmemo_linear_fwd") else (9 if name.startswith("mmemo_linear_bwd_x") else 7)
        Ms, Ns, Ks = list(a[i0]), list(a[i0 + 1]), list(a[i0 + 2])
        fl = sum(2 * m * n * k for m, n, k in zip(Ms, Ns, Ks))
        if name.startswith("mmemo_linear_bwd_w"):
            by = sum(e * (m * n + m * k) + 4 * n * k for m, n, k in zip(Ms, Ns, Ks))
        else:
            by = sum(e * (m * k + n * k + m * n) for m, n, k in zip(Ms, Ns, Ks))
        shapes = [f"{m}x{n}x{k}" for m, n, k in zip(Ms, Ns, Ks)]
        if len(shapes) > 6:       # large groups: count per distinct shape
            cnt = {}
            for sh in shapes:
                cnt[sh] = cnt.get(sh, 0) + 1
            return fl, by, f"G{len(shapes)}:" + ",".join(f"{v}x{k}" for k, v in cnt.items())
        return fl, by, "+".join(shapes)
    if name.startswith("mmemo_linear_fwd"):
        M, N, K = a[10], a[11], a[12]
        ex = 4 if a[1] else e
        return 2 * M * N * K, ex * M * K + e * N * K + e * M * N, f"{M}x{N}x{K}"
    if name.startswith("mmemo_linear_bwd_x"):
        M, N, K = a[8], a[9], a[10]
        return 2 * M * N * K, e * (M * N + N * K + M * K) + (e * M * K if a[6] else 0), f"{M}x{N}x{K}"
    if name.startswith("mmemo_linear_bwd_w"):
        M, N, K = a[8], a[9], a[10]
        return 2 * M * N * K, e * (M * N + M * K) + 4 * N * K, f"{M}x{N}x{K}"
    if name.startswith("mmemo_resattn_fwd"):
        B, H, Lq, Lk, hd = a[15:20]
        d, S = H * hd, B * H * Lq * Lk
        by = e * B * d * (Lq + 2 * Lk) + 4 * B * Lk + e * B * Lq * d
        by += e * S * (1 if a[9] else 0) + e * S * (1 if a[11] else 0)
        return (4 * B * Lq * Lk * d, by,
                f"B{B}H{H}L{Lq}x{Lk}hd{hd}{'+prev' if a[9] else ''}{'+S' if a[11] else ''}")
    if name.startswith("mmemo_resattn_bwd"):
        B, H, Lq, Lk, hd = a[27:32]
        d, S = H * hd, B * H * Lq * Lk
        by = e * B * d * (2 * Lq + 2 * Lk) + e * B * d * (Lq + 2 * Lk) + e * B * Lq * d
        by += e * S * (1 if a[11] else 0) + e * S * (1 if a[14] else 0)
        by += e * S * ((1 if a[12] else 0) + (1 if a[24] else 0))
        fl = (8 if a[11] else 10) * B * Lq * Lk * d
        return (fl, by, f"B{B}H{H}L{Lq}x{Lk}hd{hd}{'+S' if a[11] else '+recompute'}"
                        f"{'+prev' if a[12] else ''}{'+dSnext' if a[14] else ''}")
    if name.startswith("mmemo_add_ln_fwd"):
        M, d = a[11], a[12]
        return 8 * M * d, e * M * d * (3 if a[0] else 2), f"{M}x{d}"
    if name.startswith("mmemo_add_ln_bwd"):
        M, d = a[20], a[21]
        return 16 * M * d, e * M * d * (3 + (2 if a[2] else 0)), f"{M}x{d}"
    if name.startswith("mmemo_rowsum"):
        M, N = a[3], a[4]
        return M * N, e * M * N, f"{M}x{N}"
    if name.startswith("mmemo_cast_pad"):            # (n, src, lds, dst, ldd, M[], K[], stream)
        n = a[0]
        el = sum(int(m) * int(k) for m, k in zip(list(a[5])[:n], list(a[6])[:n]))
        return 0, 6 * el, f"G{n}:{el}"
    if name.startswith("mmemo_cast_f32_to_bf16_multi"):
        return 0, 0, f"G{a[0]}"
    if name.startswith("mmemo_cast"):
        return 0, 6 * a[2], f"{a[2]}"
    if name.startswith("mmemo_dropout_multi"):      # read + write of every tensor
        ns = [int(v) for v in list(a[3])[:a[0]]]
        return 0, 2 * e * sum(ns), f"G{a[0]}:{sum(ns)}"
    return 0, 0, ""


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the bench workload's kernels: read
# from profiles/ncu_traffic.json, which tools/ncu_traffic.py writes from the `ncu --set full`
# capture committed under profiles/ (a profiler number for a given shape, reported next to the live
# timing; it is never measured inside bench.py and never hard-coded here)
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")


def ncu_traffic():
    try:
        with open(NCU_TRAFFIC_FILE) as fh:
            d = json.load(fh)
        src = d.get("source")
        if isinstance(src, dict):
            src = src.get("cfg2")
        return d.get("families", {}), src
    except Exception:
        return {}, None


_FLUSH = {}


def flush_l2():
    """Evict the L2 (126 MB) by READING a 256 MB buffer (leaves clean lines, unlike a fill)."""
    dev = torch.cuda.current_device()
    buf = _FLUSH.get(dev)
    if buf is None:
        buf = _FLUSH[dev] = torch.zeros(64 << 20, dtype=torch.int32, device=f"cuda:{dev}")
    return buf.amax()


def instrumented_step(step_fn, reps: int = 10, cold: bool = True):
    """Per-kernel device time, measured live with CUDA events.

    One eager step is run with a hook on every libmmemo launch.  Timing a launch in place with an
    event pair would mostly measure the host (an eager step is launch-bound: the GPU idles between
    kernels), so the FIRST launch of every kernel family (entry point + shape) is re-issued while
    its argument buffers are still alive:
      * warm: `reps` times back to back from a small CUDA graph (inputs L2-resident, as for a
        consumer that runs right after its producer inside the real step);
      * cold: 5 times, each after the L2 was evicted by reading a 256 MB buffer, timed by an event
        pair around the single launch (includes ~1-2 us of launch gap) - the honest HBM number.
    Returns {family: dict(n, ms_each (warm), ms_cold, flops, bytes)}."""
    from mmemo_b200 import ops
    real = ops._call
    fam = {}

    def measure(name, args):
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                st = torch.cuda.current_stream().cuda_stream
                for _ in range(reps):
                    real(name, *(args[:-1] + (st,)))
            g.replay()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            s.record()
            g.replay()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            return s.elapsed_time(e) / (2 * reps)
        except Exception:
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(reps):
                real(name, *args)
            e.record()
            torch.cuda.synchronize()
            return s.elapsed_time(e) / reps

    def measure_cold(name, args):
        ts = []
        for _ in range(5):
            flush_l2()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            real(name, *args)
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        ts.sort()
        return ts[len(ts) // 2]

    def hooked(name, *args):
        real(name, *args)
        try:
            fl, by, tag = _algorithmic(name, args)
        except Exception:      # an entry point without a formula: timed, no roofline numbers
            fl, by, tag = 0, 0, ""
        key = name.replace("mmemo_", "") + (":" + tag if tag else "")
        r = fam.get(key)
        if r is None:
            r = fam[key] = dict(n=0, ms_each=measure(name, args), flops=0, bytes=0)
            r["ms_cold"] = measure_cold(name, args) if cold else None
        r["n"] += 1
        r["flops"] += fl
        r["bytes"] += by

    real_try = ops._try_call

    def try_via_call(name, *args):
        real(name, *args)          # raises on any error (incl. unsupported shape)
        return True

    def hooked_try(name, *args):
        if not real_try(name, *args):
            return False
        try:
            fl, by, tag = _algorithmic(name, args)
        except Exception:      # an entry point without a formula: timed, no roofline numbers
            fl, by, tag = 0, 0, ""
        key = name.replace("mmemo_", "") + (":" + tag if tag else "")
        r = fam.get(key)
        if r is None:
            r = fam[key] = dict(n=0, ms_each=measure(name, args), flops=0, bytes=0)
            r["ms_cold"] = measure_cold(name, args) if cold else None
        r["n"] += 1
        r["flops"] += fl
        r["bytes"] += by
        return True

    ops._call = hooked
    ops._try_call = hooked_try
    try:
        step_fn()
        torch.cuda.synchronize()
    finally:
        ops._call = real
        ops._try_call = real_try
    for r in fam.values():
        r["ms"] = r["ms_each"] * r["n"]
    return fam, sum(r["ms"] for r in fam.values())


def kernel_table(fam, pk, top: int = 12):
    """Rows of the per-kernel roofline table.  Bound = tensor when the arithmetic intensity is
    above the ridge, else hbm.  `frac` is computed from the COLD time for hbm-bound families and
    from the in-step-like warm time for tensor-bound ones; both fractions are listed."""
    ridge = pk["tf_sust"] * 1e12 / (pk["hbm"] * 1e9)
    ksum = sum(r["ms"] for r in fam.values())
    rows = []
    for key, r in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]):
        ai = r["flops"] / r["bytes"] if r["bytes"] else 0.0
        bound = "tensor" if ai > ridge else "hbm"
        work = (r["flops"] / 1e12) if bound == "tensor" else (r["bytes"] / 1e9)
        peak = pk["tf_sust"] if bound == "tensor" else pk["hbm"]
        warm_s = r["ms"] * 1e-3
        cold_s = (r["ms_cold"] * r["n"] * 1e-3) if r.get("ms_cold") else None
        ach_warm = work / warm_s if warm_s else 0.0
        ach_cold = work / cold_s if cold_s else None
        use_cold = bound == "hbm" and ach_cold is not None
        ach = ach_cold if use_cold else ach_warm
        row = {"kernel": key, "launches": r["n"], "us_per_launch": 1e3 * r["ms"] / r["n"],
               "us_per_launch_cold": None if r.get("ms_cold") is None else 1e3 * r["ms_cold"],
               "share": r["ms"] / ksum if ksum else 0.0, "bound": bound, "achieved": ach,
               "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
               "frac": ach / peak if peak else None,
               "frac_l2_warm": ach_warm / peak if peak else None,
               "frac_cold": None if ach_cold is None else ach_cold / peak,
               "timing": "cold (L2 flushed)" if use_cold else "L2-warm graph replay"}
        if bound == "tensor":
            row["frac_of_burst_peak"] = ach / pk["tf_burst"]
        rows.append(row)
    return rows[:top], ksum


# ------------------------------------------------------------------------------------------------
def make_oracle_step(batch, dtype=torch.float32):
    """fwd+bwd of the same workload through the CPU oracle (port of the reference algorithm)."""
    from mmemo_b200 import ResidualEncoder, synth
    from oracle import mmemo_oracle as O
    torch.manual_seed(0)
    enc = ResidualEncoder(CFG["dim"], CFG["n_heads"], CFG["n_layers"], CFG["ffn"])
    sd = synth.randomize_gates({k: v.detach().clone() for k, v in enc.state_dict().items()})
    sd = {k: v.to(dtype).requires_grad_(True) for k, v in sd.items()}
    pres = [f"blocks.{i}." for i in range(CFG["n_layers"])]
    x, mask = batch["x"].to(dtype), batch["mask"].to(dtype)

    def step():
        for v in sd.values():
            v.grad = None
        out = O.encoder_chain(sd, pres, x, mask, CFG["n_heads"])[0]
        loss = (out.float() ** 2).mean()
        loss.backward()
        return float(loss)
    return step


def time_cpu(steps: int, warmup: int, batch_size: int):
    from mmemo_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    b = synth.encoder_batch(seed=1234, B=batch_size, L=CFG["seq_len"], d=CFG["dim"])
    step = make_oracle_step(b)
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t)
    ts.sort()
    med = ts[len(ts) // 2]
    return batch_size / med, med * 1e3


def run_reference(args, rank):
    """--impl reference: the reference algorithm's CPU path (oracle port; the reference scripts are
    not importable and /root/reference does not exist on the GPU box) on all host cores, for
    exactly --steps timed steps after --warmup warm-ups (one step = fwd+bwd of one B=64 batch,
    ~0.2-0.5 s on 16-32 cores)."""
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    B = CFG["batch_per_gpu"]
    v, ms = time_cpu(steps, warm, B)
    cores = torch.get_num_threads()
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} fwd+bwd steps of one B={B} batch, fp32, "
                                   f"torch CPU {cores} threads (median)"},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def workload_config(n_gpus):
    return {"workload": "realformer_encoder_chain(6 x Attention_Block(512, 8 heads, ffn 2), "
                        "seq 128) fwd+bwd, loss=mean(out^2)",
            "global_batch": CFG["batch_per_gpu"] * n_gpus, "batch_per_gpu": CFG["batch_per_gpu"],
            "seq_len": CFG["seq_len"], "d_model": CFG["dim"], "n_heads": CFG["n_heads"],
            "n_layers": CFG["n_layers"], "parallelism": f"dp{n_gpus}",
            "l2": "no explicit flush: one step streams ~1 GB of activations/scores/weights "
                  "through the 126 MB L2",
            "gates": "a,b,c ~ U(-0.5,0.5)"}


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations (the reference's real models)
# ------------------------------------------------------------------------------------------------
def _median(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2]


def oracle_baselines(wl, want_cpu: bool, want_gpu: bool, dev):
    """(cpu_baseline, gpu_eager_baseline) of a training workload: the oracle = the reference's
    eager PyTorch op sequence, on the host cores and on this GPU (fp32 with TF32 off = the
    reference as written; bf16 = the same modules cast with .bfloat16())."""
    import benchlib
    from oracle import mmemo_oracle as O
    cpu = gpu = None
    n = wl.batch * wl.samples_per_item
    if want_cpu:
        torch.set_num_threads(os.cpu_count() or 1)
        step = benchlib.oracle_train_step(O, wl, "cpu")
        ts = benchlib.time_wall(step, 2, 1)
        med = _median(ts)
        cpu = {"value": n / med, "unit": "samples/s", "cores": torch.get_num_threads(),
               "kind": "port", "sample": f"2 fwd+bwd steps of one B={wl.batch} batch after 1 warm-up, "
                                         f"fp32 oracle, {med * 1e3:.0f} ms/step"}
    if want_gpu:
        gpu = {"what": "reference op sequence (oracle) as eager PyTorch on this GPU, fwd+bwd, "
                       "device-resident inputs; TF32 off", "unit": "samples/s"}
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        for tag, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
            try:
                step = benchlib.oracle_train_step(O, wl, dev, dt)

                def run():
                    step()
                    torch.cuda.synchronize()
                ts = benchlib.time_wall(run, 5, 2)
                gpu[tag] = n / _median(ts)
                gpu[tag + "_ms_per_step"] = _median(ts) * 1e3
            except Exception as ex:  # e.g. out of memory for the eager score tensors
                gpu[tag] = None
                gpu[tag + "_error"] = f"{type(ex).__name__}: {str(ex)[:120]}"
            torch.cuda.empty_cache()
    return cpu, gpu


def measure_train_config(key, batch, dev, rank, world, K, W, barrier, allreduce_max, pk,
                         reducer_factory=None, shard=None, baselines=True, scaling=None,
                         instrument=True):
    """Device-timed value, e2e, launch count, per-kernel table and baselines of one training
    workload.  With `shard` = (rank, world) the batch is the GLOBAL batch and every rank runs its
    contiguous 1/world slice (strong scaling)."""
    import benchlib
    wl = benchlib.WORKLOADS[key](batch)
    local = wl
    if shard is not None:
        from mmemo_b200 import dp as mdp

        class _Sharded(type(wl)):
            def host_batch(self_inner, seed):
                return mdp.shard_batch(wl.host_batch(seed), shard[0], shard[1], align=2)
        local = _Sharded(batch)
    gs = benchlib.GraphedStep(local, dev, seed=1234, reducer_factory=reducer_factory)
    ms = allreduce_max(benchlib.time_events(gs.run, K, W, barrier))
    n_global = batch * wl.samples_per_item * (1 if shard is not None else world)
    value = n_global * K / (ms * 1e-3)
    # e2e: pinned host inputs -> H2D (copy stream, double-buffered: overlaps the previous step) ->
    # step -> loss D2H read on the host one step later; all inside the timed region
    gs.run_e2e_pipelined(3)
    barrier()
    t0 = time.perf_counter()
    last = gs.run_e2e_pipelined(K)
    torch.cuda.synchronize()
    e2e_ms = allreduce_max((time.perf_counter() - t0) * 1e3)
    out = {"name": wl.name, "baseline_config": wl.cfg, "workload": wl.description,
           "metric": wl.metric, "unit": "samples/s", "value": value, "ms_per_step": ms / K,
           "global_batch": n_global,
           "batch_per_gpu": batch * wl.samples_per_item // (shard[1] if shard is not None else 1),
           "scaling": scaling, "n_gpus": world, "steps": K, "warmup": W,
           "launches_per_step": gs.launches, "cuda_graph": gs.graph is not None, "loss": last,
           "e2e": {"value": n_global * K / (e2e_ms * 1e-3), "unit": "samples/s",
                   "ms_per_step": e2e_ms / K, "h2d_bytes_per_step": gs.h2d_bytes(),
                   "d2h_bytes_per_step": 4,
                   "how": "pinned host batch -> cudaMemcpyAsync on a copy stream (double-buffered, "
                          "overlaps the previous step) -> graph replay -> loss D2H, read on the host "
                          "one step later; wall clock over all steps"}}
    if rank == 0 and instrument:
        red = gs.reducer
        if red is not None:
            red.enabled = False
        fam, _ = instrumented_step(gs._step, reps=5)
        if red is not None:
            red.enabled = True
        rows, ksum = kernel_table(fam, pk, top=8)
        out["kernels"] = rows
        out["kernel_time_sum_ms"] = ksum
        out["kernel_families"] = len(fam)
    del gs
    torch.cuda.empty_cache()
    if rank == 0 and baselines:
        cpu, gpu = oracle_baselines(wl, world == 1, world == 1, dev)
        out["cpu_baseline"], out["gpu_eager_baseline"] = cpu, gpu
    return out


def measure_robot_ensemble(dev, n_requests: int = 200, baselines: bool = True):
    """BASELINE configs[4]: p50 request latency of the 4-model robot_demo ensemble at B=1 and
    B=32.  One request = pinned host inputs -> H2D -> Ensemble (one CUDA-graph replay) -> D2H of the
    (B,7) prediction, wall clock per request after a stream synchronise."""
    import benchlib
    import mmemo_b200
    from mmemo_b200 import ops
    res = {"name": benchlib.Cfg5.name, "baseline_config": benchlib.Cfg5.cfg,
           "workload": benchlib.Cfg5.description, "metric": benchlib.Cfg5.metric, "unit": "ms",
           "higher_is_better": False, "requests": n_requests, "batches": {}}
    for B in (1, 32):
        wl = benchlib.Cfg5(B)
        models, sds = wl.models()
        models = [m.to(dev) for m in models]
        ens = mmemo_b200.robot_demo.Ensemble(models)
        hb = wl.host_batch(77)
        host = [hb[k].pin_memory() for k in wl.NAMES]
        stat = [t.to(dev) for t in host]
        out_host = torch.zeros(B, 7, pin_memory=True)

        def request():
            for s_, h_ in zip(stat, host):
                s_.copy_(h_, non_blocking=True)
            pred = ens(*stat)
            out_host.copy_(pred, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        request()                                 # builds the request graph (warm-up + capture)
        n0 = ops.launch_count
        with torch.no_grad():
            ens._forward(stat)                    # one eager pass = what one graph replay launches
        launches = ops.launch_count - n0
        ts = sorted(benchlib.time_wall(request, n_requests, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            ens(*stat)
        e1.record()
        torch.cuda.synchronize()
        r = {"p50_ms": ts[len(ts) // 2] * 1e3, "p90_ms": ts[int(len(ts) * 0.9)] * 1e3,
             "min_ms": ts[0] * 1e3, "device_ms": e0.elapsed_time(e1) / 50,
             "samples_per_s": B / ts[len(ts) // 2], "launches_per_request": launches,
             "h2d_bytes_per_request": sum(t.numel() * 4 for t in host),
             "d2h_bytes_per_request": B * 7 * 4}
        if baselines:
            from oracle import mmemo_oracle as O
            torch.set_num_threads(os.cpu_count() or 1)
            with torch.no_grad():
                cpu_ts = benchlib.time_wall(lambda: wl.oracle_pred(O, sds, hb), 5, 1)
                r["cpu_baseline_ms"] = _median(cpu_ts) * 1e3
                r["cpu_cores"] = torch.get_num_threads()
                sdg = [{k: v.to(dev) for k, v in sd.items()} for sd in sds]
                hbg = {k: v.to(dev) for k, v in hb.items()}

                def eager():
                    p_ = wl.oracle_pred(O, sdg, hbg).cpu()
                    return p_
                r["gpu_eager_baseline_ms"] = _median(benchlib.time_wall(eager, 20, 3)) * 1e3
                ref = wl.oracle_pred(O, sds, hb)
            request()
            r["max_abs_diff_vs_oracle"] = float((out_host - ref).abs().max())
        res["batches"][f"B{B}"] = r
        del ens, models
        torch.cuda.empty_cache()
    res["value"] = res["batches"]["B1"]["p50_ms"]
    return res


def ncu_step(which: str, dev, precision: str):
    """One eager step of a workload with an NVTX range (named like bench's kernel families) around
    every libmmemo launch; the profiled region is bracketed by cudaProfilerStart/Stop."""
    import benchlib
    import mmemo_b200
    from mmemo_b200 import ops, synth
    mmemo_b200.set_precision(precision)
    if which == "cfg2":
        torch.manual_seed(0)
        model = mmemo_b200.ResidualEncoder(CFG["dim"], CFG["n_heads"], CFG["n_layers"], CFG["ffn"])
        model.load_state_dict(synth.randomize_gates(
            {k: v.detach().clone() for k, v in model.state_dict().items()}))
        model = model.to(dev).train()
        b = synth.encoder_batch(seed=1234, B=CFG["batch_per_gpu"], L=CFG["seq_len"], d=CFG["dim"])
        x, m = b["x"].to(dev), b["mask"].to(dev)

        def step():
            model.zero_grad(set_to_none=True)
            ops.sq_mean_op(model(x, m)).backward()
    else:
        bsz = {"cfg1a": 32, "cfg1b": 32, "cfg3": 128, "cfg3c": 64, "cfg4": 256}[which]
        gs = benchlib.GraphedStep(benchlib.WORKLOADS[which](bsz), dev, seed=1234, use_graph=False)
        step = gs._step
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    real, real_try = ops._call, ops._try_call

    def key_of(name, args):
        try:
            _, _, tag = _algorithmic(name, args)
        except Exception:
            tag = ""
        return name.replace("mmemo_", "") + (":" + tag if tag else "")

    def call(name, *a):
        torch.cuda.nvtx.range_push(key_of(name, a))
        try:
            real(name, *a)
        finally:
            torch.cuda.nvtx.range_pop()

    def try_call(name, *a):
        torch.cuda.nvtx.range_push(key_of(name, a))
        try:
            return real_try(name, *a)
        finally:
            torch.cuda.nvtx.range_pop()

    ops._call, ops._try_call = call, try_call
    torch.cuda.profiler.start()
    step()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    ops._call, ops._try_call = real, real_try
    print(f"ncu-step {which}: done", file=sys.stderr)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu-step", default=None, metavar="WORKLOAD",
                    help="profiling driver (no JSON line): run ONE eager step of cfg2 | cfg1a | cfg1b | "
                         "cfg3c | cfg4 between cudaProfilerStart/Stop with every libmmemo launch "
                         "inside an NVTX range named after its kernel family, for "
                         "`ncu --nvtx --print-nvtx-rename kernel --profile-from-start off`")
    ap.add_argument("--configs", default="all",
                    help="comma list of the extra BASELINE configs to measure "
                         "(cfg1a,cfg1b,cfg3,cfg3c,cfg4,cfg5), 'all' or 'none'")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (encoder output "
                         "'out', 'loss', 'grad.<parameter>') to DIR/<name>.npy as float32; arrays "
                         f"above {DUMP_MAX_ELEMS} elements as a fixed seeded sample of that many "
                         "(rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.ncu_step:
        ncu_step(args.ncu_step, dev, args.precision)
        return
    import torch.distributed as dist
    stdout_fd = None
    if world > 1:
        # stdout carries exactly ONE JSON line: native libraries (NCCL's version banner) that write
        # to file descriptor 1 during initialisation are sent to stderr until the line is printed
        sys.stdout.flush()
        stdout_fd = os.dup(1)
        os.dup2(2, 1)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line
        # the gradient all-reduce moves ~50 MB per 2 ms step: a few CTAs are plenty (measured on 2
        # GPUs: 16 CTAs, no SM reservation for the persistent kernels, is the best setting)
        os.environ.setdefault("NCCL_MAX_CTAS", "16")
        dist.init_process_group("nccl", device_id=dev)
    import mmemo_b200
    from mmemo_b200 import ops, synth
    from mmemo_b200 import dp as mdp

    W = max(3, args.warmup)
    K = args.steps
    mmemo_b200.set_precision(args.precision)
    torch.manual_seed(0)
    model = mmemo_b200.ResidualEncoder(CFG["dim"], CFG["n_heads"], CFG["n_layers"], CFG["ffn"])
    sd = synth.randomize_gates({k: v.detach().clone() for k, v in model.state_dict().items()})
    model.load_state_dict(sd)
    model = model.to(dev).train()
    B, L, d = CFG["batch_per_gpu"], CFG["seq_len"], CFG["dim"]
    batch = synth.encoder_batch(seed=1234 + rank, B=B, L=L, d=d)
    host_x, host_m = batch["x"].pin_memory(), batch["mask"].pin_memory()
    x_dev = torch.empty_like(host_x, device=dev)
    m_dev = torch.empty_like(host_m, device=dev)
    x_dev.copy_(host_x)
    m_dev.copy_(host_m)
    loss_dev = torch.zeros((), device=dev)
    host_loss = torch.zeros((), pin_memory=True)

    reducer = None
    if world > 1:   # knobs for experiments; the defaults are the product configuration
        reducer = mdp.GradReducer(
            model, world, bucket_bytes=int(float(os.environ.get("MMEMO_BUCKET_MB", "8")) * (1 << 20)),
            zero_copy=os.environ.get("MMEMO_ZERO_COPY", "1") == "1",
            sm_reserve=int(os.environ.get("MMEMO_SM_RESERVE", os.environ.get("NCCL_MAX_CTAS", "16"))),
            transport=os.environ.get("MMEMO_DP_TRANSPORT", "auto"),
            comm_blocks=int(os.environ.get("MMEMO_COMM_BLOCKS", "16")),
            symm_sm_reserve=int(os.environ.get("MMEMO_SYMM_SM_RESERVE", "16")),
            reserve_launches=int(os.environ.get("MMEMO_RESERVE_LAUNCHES", "5")))

    last_out = {}

    def step():
        model.zero_grad(set_to_none=True)
        out = model(x_dev, m_dev)
        loss = ops.sq_mean_op(out)             # mean(out^2): one libmmemo launch per direction
        if reducer is not None:
            reducer.backward(loss)
        else:
            loss.backward()
        loss_dev.copy_(loss.detach())
        if args.dump_outputs:
            last_out["out"] = out              # inside the graph: the buffer every replay rewrites

    # ---- warm-up (eager) then CUDA-graph capture of the whole step ------------------------------
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = None
    launches_per_step = 0
    if not args.no_graph:
        try:
            ops.clear_shadow_cache()          # capture the fp32->bf16 weight casts with the step
            model.zero_grad(set_to_none=True)
            n0 = ops.launch_count
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            launches_per_step = ops.launch_count - n0
        except Exception as ex:  # pragma: no cover
            if rank == 0:
                print(f"[bench] CUDA-graph capture failed ({type(ex).__name__}: {ex}); eager mode",
                      file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
    if graph is None:
        n0 = ops.launch_count
        step()
        launches_per_step = ops.launch_count - n0
    run = graph.replay if graph is not None else step
    cuda_graph = graph is not None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        run()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        run()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs,
                     [("out", last_out["out"]), ("loss", loss_dev)] +
                     [("grad." + n, p.grad) for n, p in model.named_parameters()
                      if p.grad is not None])
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / K
    value = B * world * K / (ms * 1e-3)

    # ---- end to end: pinned host inputs -> H2D -> step -> D2H loss, every step --------------------
    # Software-pipelined like a real input pipeline: the H2D copy of step i+1 runs on a copy stream
    # into a second staging buffer while step i computes; the loss of step i is read on the host one
    # step later.  Every step's inputs cross PCIe and every step's loss reaches the host inside the
    # timed region.
    copy_stream = torch.cuda.Stream()
    x_stage = [torch.empty_like(x_dev) for _ in range(2)]
    m_stage = [torch.empty_like(m_dev) for _ in range(2)]
    ev_h2d = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_loss = [torch.cuda.Event() for _ in range(2)]
    host_losses = [torch.zeros((), pin_memory=True) for _ in range(2)]

    def issue_h2d(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[s])          # compute no longer reads this stage
            x_stage[s].copy_(host_x, non_blocking=True)
            m_stage[s].copy_(host_m, non_blocking=True)
            ev_h2d[s].record(copy_stream)

    def e2e_run(n):
        last = float("nan")
        cur = torch.cuda.current_stream()
        issue_h2d(0)
        for i in range(n):
            s = i % 2
            if i + 1 < n:
                issue_h2d(i + 1)
            cur.wait_event(ev_h2d[s])
            x_dev.copy_(x_stage[s], non_blocking=True)
            m_dev.copy_(m_stage[s], non_blocking=True)
            ev_free[s].record(cur)
            run()
            host_losses[s].copy_(loss_dev, non_blocking=True)
            ev_loss[s].record(cur)
            if i >= 1:
                ev_loss[1 - s].synchronize()
                last = float(host_losses[1 - s])
        ev_loss[(n - 1) % 2].synchronize()
        return float(host_losses[(n - 1) % 2])

    e2e_run(3)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    last_loss = e2e_run(K)
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    t = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_value = B * world * K / (e2e_ms * 1e-3)

    # ---- per-kernel roofline (rank 0, eager instrumented step) ------------------------------------
    roof, kernels = None, []
    pk = peaks()
    if rank == 0:
        if reducer is not None:
            reducer.enabled = False
        fam, total_ms = instrumented_step(step)
        if reducer is not None:
            reducer.enabled = True
        kernels, ksum = kernel_table(fam, pk)
        top = kernels[0]
        traffic_tab, traffic_src = ncu_traffic()
        traffic = traffic_tab.get(top["kernel"])
        roof = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"],
                "peak": top["peak"], "unit": top["unit"], "frac": top["frac"],
                "frac_l2_warm": top["frac_l2_warm"], "frac_cold": top["frac_cold"],
                "frac_of_burst_peak": top.get("frac_of_burst_peak"),
                "traffic": traffic, "traffic_source": traffic_src if traffic else None,
                "share_of_step": top["share"], "peak_source": pk["src"],
                "how": "first launch of each kernel family re-issued inside an eager step while its "
                       "buffers are alive: 10x from a CUDA graph (L2-warm) and 5x each after an L2 "
                       "flush (cold, event pair around the launch); achieved = algorithmic "
                       "bytes|flops per launch / time per launch; hbm-bound families use the cold "
                       "time, tensor-bound ones the warm (in-step-like) time",
                "kernel_time_sum_ms": total_ms}

    # ---- data-parallel evidence (N > 1): transport, exposed communication, reduced-gradient check --
    dp_info = None
    if reducer is not None:
        # (a) step without the collectives (same bucket plumbing) -> exposed communication time
        reducer.no_comm = True
        g2 = None
        try:
            model.zero_grad(set_to_none=True)
            g2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g2):
                step()
        except Exception as ex:
            print(f"[bench] no-comm graph capture failed ({type(ex).__name__}: {ex})", file=sys.stderr)
            g2 = None
            torch.cuda.synchronize()
        run2 = g2.replay if g2 is not None else step
        for _ in range(W):
            run2()
        barrier()
        e0.record()
        for _ in range(K):
            run2()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_nocomm = float(t.item()) / K
        reducer.no_comm = False
        g2 = None
        # (b) reduced gradients of a probe (first parameter of every bucket) vs an NCCL all-reduce
        # of the ranks' local gradients
        # (a weight matrix: its gradient is a two-slice split-K sum, bit-reproducible between the
        # two backward passes compared here; LayerNorm / gate gradients are atomics-ordered)
        probes = [next((p for p in b.params if p.dim() >= 2), b.params[0]) for b in reducer.buckets]
        reducer.enabled = False
        step()
        ref = [p.grad.detach().clone() for p in probes]
        for r_ in ref:
            dist.all_reduce(r_, op=dist.ReduceOp.SUM)
            r_.div_(world)
        reducer.enabled = True
        step()
        torch.cuda.synchronize()
        err = max(float((p.grad - r_).abs().max() / r_.abs().max().clamp_min(1e-30))
                  for p, r_ in zip(probes, ref))
        dp_info = {"transport": reducer.transport, "uses_multicast": reducer.uses_multicast,
                   "kernel": "libmmemo allreduce_kernel (multimem.ld_reduce/st)"
                             if reducer.transport == "symm" else "NCCL all_reduce",
                   "buckets": len(reducer.buckets),
                   "bucket_bytes": [int(b.flat.numel()) * 4 for b in reducer.buckets],
                   "ms_per_step_without_comm": ms_nocomm,
                   "exposed_comm_us": (ms_per_step - ms_nocomm) * 1e3,
                   "grad_check": {"probe_tensors": len(probes), "max_rel_err": err,
                                  "what": "max |reduced - allreduce(local)/N| / max |ref| over the "
                                          "first weight matrix of every bucket"}}

    # ---- CPU baseline + eager-PyTorch-on-this-GPU baseline (rank 0, N=1 only) -----------------------
    cpu, gpu_eager = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cms = time_cpu(3, 1, B)
        cpu = {"value": v, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"3 fwd+bwd steps of one B={B} batch (same shapes/seeds), fp32 oracle, "
                         f"median, {cms:.0f} ms/step"}
        gpu_eager = {"what": "reference op sequence (oracle) as eager PyTorch on this GPU, fwd+bwd, "
                             "device-resident inputs, TF32 off", "unit": "samples/s"}
        for tag, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
            sd_g = {k: v_.to(dev, dt).requires_grad_(True) for k, v_ in sd.items()}
            from oracle import mmemo_oracle as O
            pres = [f"blocks.{i}." for i in range(CFG["n_layers"])]
            xg, mg = x_dev.to(dt), m_dev.to(dt)

            def eager_step():
                for v_ in sd_g.values():
                    v_.grad = None
                out = O.encoder_chain(sd_g, pres, xg, mg, CFG["n_heads"])[0]
                (out.float() ** 2).mean().backward()
                torch.cuda.synchronize()
            import benchlib
            ts = sorted(benchlib.time_wall(eager_step, 5, 2))
            gpu_eager[tag] = B / ts[len(ts) // 2]
            gpu_eager[tag + "_ms_per_step"] = ts[len(ts) // 2] * 1e3
            del sd_g
            torch.cuda.empty_cache()

    # ---- the other BASELINE configs ------------------------------------------------------------------
    graph = None
    run = None
    want = ["cfg1a", "cfg1b", "cfg3", "cfg3c", "cfg4", "cfg5"] if args.configs == "all" else \
        ([] if args.configs == "none" else args.configs.split(","))
    configs = []

    def allreduce_max(ms_):
        if world == 1:
            return ms_
        t_ = torch.tensor([ms_], device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return float(t_.item())

    base = not args.no_cpu_baseline
    for key in want:
        try:
            if key == "cfg4":
                # global batch 256 sharded over the ranks (R-Drop pairs stay together): strong scaling
                mk = None
                if world > 1:
                    mk = lambda m: mdp.GradReducer(m, world, bucket_bytes=4 << 20)   # noqa: E731
                configs.append(measure_train_config(
                    "cfg4", 256, dev, rank, world, K, W, barrier, allreduce_max, pk,
                    reducer_factory=mk, shard=(rank, world), baselines=base, scaling="strong"))
            elif world > 1:
                continue        # single-GPU legs: reported by the N=1 run only
            elif key == "cfg5":
                configs.append(measure_robot_ensemble(dev, baselines=base))
            else:
                bsz = {"cfg1a": 32, "cfg1b": 32, "cfg3": 128, "cfg3c": 64}[key]
                configs.append(measure_train_config(key, bsz, dev, rank, world, K, W, barrier,
                                                    allreduce_max, pk, baselines=base))
        except Exception as ex:   # a failed leg must not take the headline line down with it
            import traceback
            traceback.print_exc(file=sys.stderr)
            configs.append({"name": key, "error": f"{type(ex).__name__}: {str(ex)[:200]}"})
            torch.cuda.synchronize()

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision if args.precision != "fp32" else "f32",
            "data": "synthetic", "config": workload_config(world), "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "samples/s",
                    "h2d_bytes_per_step": host_x.numel() * 4 + host_m.numel() * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / K,
                    "how": "pinned host x,mask -> cudaMemcpyAsync on a copy stream (double-buffered, "
                           "overlaps the previous step) -> graph replay -> loss D2H, read on the host "
                           "one step later; all inside the timed region"},
            "gpu_launches": launches_per_step * K,
            "launches_per_step": launches_per_step,
            "cuda_graph": cuda_graph,
            "loss": last_loss,
            "roofline": roof, "cpu_baseline": cpu, "gpu_eager_baseline": gpu_eager, "dp": dp_info,
            "kernels": kernels[:12], "configs": configs,
        }
        if stdout_fd is not None:
            sys.stdout.flush()
            os.dup2(stdout_fd, 1)
        print(json.dumps(out), flush=True)
    if world > 1:
        # Tear down in a fixed order: drain the device, meet the other ranks, then leave without
        # waiting on communicator teardown (destroy_process_group() was observed to block here
        # after a captured all-reduce).
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
