#!/usr/bin/env python
"""Benchmark of the Langevin posterior-inference path (BASELINE.json metric: latent-steps/s, CIFAR-10 config).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cifar10|svhn|...]
                    [--batch B] [--mode langevin|train] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input: R calls of
sample_langevin_post_z_with_flow (train.py:307-335), each T = g_l_steps Langevin iterations on B latents per GPU
(R = `langevin_calls_per_step` = --calls-per-step, 1 by default, so that K timed steps are K calls; every call gets
fresh Philox noise and the L2 is flushed between calls).  value = N * B * T * R * K / time, inputs resident in
HBM, timed with CUDA events, max over ranks.  The primary `value` runs the fp32-equivalent arithmetic (3-pass hi|lo
forward AND data gradient); `value_bwd1pass` is the opt-in single-fp16-pass data gradient, reported next to it.
`e2e` is the same metric through the public Python API with pinned HOST buffers, host<->device copies inside the
timed region.  Prints ONE JSON line (rank 0).

Inputs, parameters and noise seeds depend on the arguments only, so `--dump-outputs DIR` (rank 0) writes the results
of the same computation on every run: what the last timed call returned, as DIR/<name>.npy (see dump_outputs), for
comparing two builds output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # BASELINE.json configs (README commands of the reference)
    "svhn": dict(dataset="svhn", nz=100, ngf=64, f_width=64, T=20, sigma=0.3, B=100, img=32),
    "cifar10": dict(dataset="cifar10", nz=128, ngf=128, f_width=64, T=40, sigma=0.3, B=100, img=32),
    "celeba_crop": dict(dataset="celeba_crop", nz=100, ngf=128, f_width=64, T=20, sigma=0.3, B=100, img=64),
    "celeba_hq256": dict(dataset="celeba_hq256", nz=100, ngf=128, f_width=128, T=20, sigma=1.0, B=8, img=256),
}
# config 4 (test mode, train.py:565-655): noise-free chains over 50 000 latents + 50 000 prior samples.  README's
# --g_l_steps 400 becomes 8 000 iterations under the reference's x20 rule (train.py:606); BASELINE.json quotes 400.
TEST_WORKLOADS = {
    "svhn_test": dict(dataset="svhn", nz=100, ngf=64, f_width=64, T=400, sigma=0.3, B=1250, img=32, noise=False,
                      total_latents=50000),
}
ALL_WORKLOADS = dict(WORKLOADS, **TEST_WORKLOADS)
ROOFLINE_LATENT_STEPS = {"svhn": 5.98e6, "cifar10": 347e3, "celeba_crop": 971e3, "celeba_hq256": 112e3}  # BASELINE.md s3
DUMP_MAX_ELEMENTS = 1 << 20   # per array: a dump of the at most 7 arrays written stays below 64 MB


def dump_outputs(directory, arrays):
    """Writes each array of `arrays` (name -> tensor) as `directory/<name>.npy`, float64 kept, anything else as
    float32.  An array of more than DUMP_MAX_ELEMENTS elements is replaced by the same seeded sample of that many of
    its flattened elements (in index order) on every run."""
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        v = t.detach().cpu().numpy()
        v = v.astype(np.float64 if v.dtype == np.float64 else np.float32)
        if v.size > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(v.size, DUMP_MAX_ELEMENTS, replace=False))
            v = v.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), v)


def exact_layer_flops(layers):
    """Per-sample FLOPs (2 x MACs whose taps land inside the output) of each ConvTranspose2d -- SURVEY.md 8a table."""
    out, hin = [], 1
    for (ci, co, k, s, p) in layers:
        hout = (hin - 1) * s - 2 * p + k
        cnt1d = sum(1 for i in range(hin) for kk in range(k) if 0 <= i * s - p + kk < hout)
        out.append(2.0 * cnt1d * cnt1d * ci * co)
        hin = hout
    return out


def flow_flops(nz, w, depth=5):
    return 2.0 * depth * 2.0 * (nz * nz + nz // 2 * w + w * w + w * nz)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(tflops=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"],
                    src="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def kernel_source_sha():
    """sha256 over the CUDA sources: ties an ncu capture under profiles/ to the kernels that were actually built."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "latent-space-normalizing-flow_b200", "csrc")
    for f in sorted(os.listdir(d)):
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def workload_config(name, w):
    """The workload keys both arms report under `config` (identical dicts => the driver's same_config check holds)."""
    return {"workload": name, "dataset": w["dataset"], "nz": w["nz"], "ngf": w["ngf"], "f_width": w["f_width"],
            "g_l_steps": w["T"], "batch_per_gpu": w["B"], "g_llhd_sigma": w["sigma"],
            "l2": "CUDA arm: L2 flushed between timed calls (256 MB written, inside the timed region); reference arm: "
                  "host CPU, not applicable"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons (B200_PROFILING.md recipe).  Started before the warm-up (nvidia-smi takes
    ~0.2 s to start); every row is time-stamped on arrival and only rows inside the timed window are summarised."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window_begin(self):
        self.t0 = time.time()

    def window_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if len(r) >= 9 and self.t0 is not None and self.t0 <= t <= self.t1 + 0.06]
        where = "timed region"
        if not rows:   # region shorter than the sampling period: take the samples closest to it
            near = sorted((abs(t - (self.t1 or 0)), r) for t, r in self.rows if len(r) >= 9)[:2]
            rows = [r for _, r in near]
            where = "nearest samples (timed region shorter than the 50 ms sampling period)"
        num = lambda v: float(v) if v.replace(".", "", 1).isdigit() else None
        sm = [num(r[1]) for r in rows if num(r[1]) is not None]
        mx = [num(r[2]) for r in rows if num(r[2]) is not None]
        pw = [num(r[3]) for r in rows if num(r[3]) is not None]
        reasons = set()
        for r in rows:
            for n, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None, "window": where}


def build_models(w, device):
    import lsnf_b200
    from lsnf_b200 import synth
    args = lsnf_b200.make_args(dataset=w["dataset"], nz=w["nz"], ngf=w["ngf"], f_width=w["f_width"],
                               g_llhd_sigma=w["sigma"], g_l_steps=w["T"], batch_size=w["B"])
    netG = lsnf_b200._netG(args).to(device).eval()
    netF = lsnf_b200._netF(args, nz=w["nz"]).to(device).eval()
    gsd = synth.generator_state(w["dataset"], w["nz"], w["ngf"], 3, seed=1)
    fsd = synth.flow_state(w["nz"], w["f_width"], 5, 1, 2, seed=1)
    netG.load_state_dict({k: torch.from_numpy(v) for k, v in gsd.items()})
    netF.load_state_dict({k: torch.from_numpy(v) for k, v in fsd.items()})
    return args, netG, netF, gsd, fsd


def oracle_rate(w, gsd, fsd, langevin_steps, repeats=1, threads=None, min_seconds=None, device="cpu", batch=None):
    """latent-steps/s of the oracle (restatement of the reference's torch path, oracle/refpath.py) -- on the host
    cores (device='cpu': the cpu_baseline / --impl reference legs) or as eager torch-CUDA on the same GPU
    (the informational `reference_cuda_eager` key).  Baseline legs only: never on the product path."""
    from oracle import refpath
    from lsnf_b200 import synth
    threads = threads or os.cpu_count() or 1
    if device == "cpu":
        torch.set_num_threads(threads)
    B = batch or w["B"]
    gp = {k: torch.from_numpy(v).to(device) for k, v in gsd.items()}
    fp = {k: torch.from_numpy(v).to(device) for k, v in fsd.items()}
    layers = refpath.generator_layers(w["dataset"], w["nz"], w["ngf"])
    x, z0, eps = synth.inputs(B, w["nz"], 3, w["img"], langevin_steps, seed=1)
    x, z0, eps = torch.from_numpy(x).to(device), torch.from_numpy(z0).to(device), torch.from_numpy(eps).to(device)
    if not w.get("noise", True):
        eps = None
    sync = (lambda: torch.cuda.synchronize()) if device != "cpu" else (lambda: None)

    def run(n):
        refpath.langevin(z0, x, gp, fp, layers, depth=5, steps=n, step_size=0.1, sigma=w["sigma"], eps=eps)
        sync()

    run(1)  # warm-up
    if min_seconds:
        # bounded sample: repeat chunks of `langevin_steps` iterations until about min_seconds of work is done
        done, t0 = 0, time.perf_counter()
        while True:
            run(langevin_steps)
            done += langevin_steps
            dt = time.perf_counter() - t0
            if dt >= min_seconds or done >= 400:
                return B * done / dt, dt, threads, done
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        run(langevin_steps)
        best = min(best, time.perf_counter() - t0)
    return B * langevin_steps / best, best, threads, langevin_steps


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


REF_SAMPLE_T = {"svhn": 20, "cifar10": 4, "celeba_crop": 4, "celeba_hq256": 2, "svhn_test": 20}
REF_SAMPLE_B = {"svhn_test": 100}   # the reference's test loader uses batches of 100 (train.py:598)


def oracle_update_seconds(w, gsd, fsd, batch, threads=None, repeats=2):
    """Seconds of ONE generator step + flow step of train.py:390-415 (autograd + torch.optim.Adam, restated by
    oracle/refpath.parameter_updates) on the host cores, best of `repeats` after a warm-up.  Baseline legs only."""
    from oracle import refpath
    from lsnf_b200 import synth
    torch.set_num_threads(threads or os.cpu_count() or 1)
    gp = {k: torch.from_numpy(v).clone().requires_grad_(True) for k, v in gsd.items()}
    fp = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in fsd.items()}
    fkeys = refpath.trainable_flow_keys(fp)
    for k in fkeys:
        fp[k] = fp[k].clone().requires_grad_(True)
    adam = lambda ps: torch.optim.Adam(ps, lr=0.0004, weight_decay=0, betas=(0.5, 0.999))   # train.py:294-295
    optG, optF = adam(list(gp.values())), adam([fp[k] for k in fkeys])
    layers = refpath.generator_layers(w["dataset"], w["nz"], w["ngf"])
    x, z, _ = synth.inputs(batch, w["nz"], 3, w["img"], 1, seed=1)
    x, z = torch.from_numpy(x), torch.from_numpy(z)
    best = float("inf")
    for i in range(repeats + 1):
        t0 = time.perf_counter()
        refpath.parameter_updates(gp, fp, z, x, layers, optG, optF, depth=5)
        if i:
            best = min(best, time.perf_counter() - t0)
    return best


def run_reference(a, w, rank, out):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the reference is pure
    Python/torch and does not travel to the GPU box) on the host cores, bounded sample per step."""
    if rank != 0:
        return
    if a.mode == "train":
        return run_reference_train(a, w, out)
    from lsnf_b200 import synth
    gsd = synth.generator_state(w["dataset"], w["nz"], w["ngf"], 3, seed=1)
    fsd = synth.flow_state(w["nz"], w["f_width"], 5, 1, 2, seed=1)
    sample_T = REF_SAMPLE_T[a.workload]
    sample_B = REF_SAMPLE_B.get(a.workload, w["B"])
    for _ in range(max(a.warmup, 1) - 1):
        oracle_rate(w, gsd, fsd, 1, batch=sample_B)
    t0 = time.perf_counter()
    total = 0.0
    for _ in range(a.steps):
        rate, dt, threads, _ = oracle_rate(w, gsd, fsd, sample_T, batch=sample_B)
        total += dt
    value = sample_B * sample_T * a.steps / total
    sample = (f"each step times {sample_T} Langevin iteration(s) of a batch of {sample_B} (a bounded sample of the "
              f"T={w['T']} call: the per-iteration cost of the loop does not depend on T) on {cpu_model()}")
    line = {"impl": "reference", "metric": "langevin_latent_steps_per_sec", "value": value, "unit": "latent-steps/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a.workload, w),
            "details": {"noise": "none needed for timing (torch CPU oracle)", "cpu": cpu_model()},
            "cpu_baseline": {"value": value, "unit": "latent-steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "latent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    out.emit(line)


def run_reference_train(a, w, out):
    """--impl reference --mode train: one whole training iteration of the reference (train.py:376-415: Langevin call,
    generator step, flow step) on the host cores -- BASELINE.json's config 1 is exactly this on the SVHN shape.  Each
    step times a bounded sample of the Langevin call (REF_SAMPLE_T iterations; the per-iteration cost does not depend
    on T) plus the two parameter updates in full; the iteration time is sample * T / REF_SAMPLE_T + updates."""
    from lsnf_b200 import synth
    gsd = synth.generator_state(w["dataset"], w["nz"], w["ngf"], 3, seed=1)
    fsd = synth.flow_state(w["nz"], w["f_width"], 5, 1, 2, seed=1)
    sample_T, B, T = REF_SAMPLE_T[a.workload], w["B"], w["T"]
    for _ in range(max(a.warmup, 1) - 1):
        oracle_rate(w, gsd, fsd, 1, batch=B)
    t0 = time.perf_counter()
    t_langevin = t_update = 0.0
    threads = os.cpu_count() or 1
    for _ in range(a.steps):
        _, dt, threads, _ = oracle_rate(w, gsd, fsd, sample_T, batch=B)
        t_langevin += dt * T / sample_T
        t_update += oracle_update_seconds(w, gsd, fsd, B, threads, repeats=1)
    iter_s = (t_langevin + t_update) / a.steps
    value = B * T / iter_s
    sample = (f"each step times {sample_T} of the {T} Langevin iterations of a batch of {B} (scaled by {T}/{sample_T}: "
              f"the per-iteration cost of the loop does not depend on T) and one full generator + flow update "
              f"(autograd + torch Adam) on {cpu_model()}")
    line = {"impl": "reference", "metric": "train_iteration_latent_steps_per_sec", "value": value,
            "unit": "latent-steps/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * iter_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "mode": "train",
            "dtype": "f32", "data": "synthetic", "config": workload_config(a.workload, w),
            "details": {"what": "Langevin + generator update + flow update (train.py:376-415) on the torch CPU oracle",
                        "ms_per_iteration": 1e3 * iter_s, "langevin_call_ms": 1e3 * t_langevin / a.steps,
                        "updates_ms": 1e3 * t_update / a.steps, "cpu": cpu_model()},
            "cpu_baseline": {"value": value, "unit": "latent-steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "latent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    out.emit(line)


class _CleanStdout:
    """Everything any library prints to stdout (NCCL's version banner, warnings) is diverted to stderr; the one JSON
    line goes to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, obj):
        sys.stdout.flush()
        os.write(self.real, (json.dumps(obj) + "\n").encode())


class Ctx:
    pass


def timed_calls(ctx, fn, n_calls):
    """n_calls invocations of fn(i) between a barrier + synchronize on both sides; CUDA-event time in ms, max over
    ranks."""
    import torch.distributed as dist
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_calls):
        fn(i)
    e1.record()
    ctx.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def main():
    sink = _CleanStdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # 70 timed calls of the default CIFAR-10 workload take about 3 s on a B200: a window long enough that clock and
    # scheduler noise stay small (`details.timed_region_s` reports it; faster workloads want more steps)
    ap.add_argument("--steps", type=int, default=70)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cifar10", choices=sorted(ALL_WORKLOADS))
    ap.add_argument("--mode", default="langevin", choices=["langevin", "train"],
                    help="train: one training iteration (Langevin + G update + F update + gradient all-reduces)")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the reference's 100)")
    ap.add_argument("--test-steps", type=int, default=None, help="svhn_test: Langevin iterations per chain (400; 8000 = "
                    "the reference's x20 rule)")
    ap.add_argument("--full-50k", action="store_true", help="svhn_test: cover all 50 000 latents (strong scaling)")
    ap.add_argument("--calls-per-step", type=int, default=None, help="Langevin calls (--mode train: training "
                    "iterations) per timed step (default 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the bwd1pass secondary measurement")
    ap.add_argument("--no-eager-ref", action="store_true", help="skip the eager torch-CUDA reference row")
    ap.add_argument("--stage-table", default=None, help="write the per-stage timing table (json) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    w = dict(ALL_WORKLOADS[a.workload])
    if a.batch:
        w["B"] = a.batch
    if a.test_steps:
        w["T"] = a.test_steps
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        run_reference(a, w, rank, sink)
        return
    if a.warmup < 3:
        a.warmup = 3
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    import torch.distributed as dist
    import lsnf_b200
    torch.cuda.set_device(local_rank)
    ctx = Ctx()
    ctx.dev = dev = torch.device("cuda", local_rank)
    ctx.world, ctx.rank = world, rank
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    ctx.barrier = barrier

    if a.mode == "train":
        from bench_train import run_train_bench
        run_train_bench(a, w, ctx, sink)
        if world > 1:
            dist.destroy_process_group()
        return

    args, netG, netF, gsd, fsd = build_models(w, dev)
    from lsnf_b200 import synth
    B, T, nz = w["B"], w["T"], w["nz"]
    noisy = bool(w.get("noise", True))
    if a.full_50k:
        per_rank = w["total_latents"] // world
        a.steps = max(1, math.ceil(per_rank / B))
    x_np, z0_np, _ = synth.inputs(B, nz, 3, w["img"], 1, seed=1 + rank)
    x, z0 = torch.from_numpy(x_np).to(dev), torch.from_numpy(z0_np).to(dev).reshape(B, nz).contiguous()
    sample_offset = rank * B
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # 2x the 126 MB L2
    out = torch.empty_like(z0)
    norms = torch.zeros(2, device=dev)

    def make_step(plan):
        def call(i):
            flush.zero_()   # L2 flush between timed calls (inside the timed region: ~0.05 ms per call)
            plan.langevin_run(z0, x, T, 0.1, w["sigma"], with_noise=noisy, eps=None, seed=1234 + i,
                              sample_offset=sample_offset, out=out, norms=norms)
        return call

    def prepare(passes):
        plan = lsnf_b200.langevin_plan(netG, netF, B, dev, passes)
        plan.ensure_generator(netG)
        plan.ensure_flow(netF, need_inverse=True)
        return plan

    plan = prepare(3)
    call = make_step(plan)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(a.warmup):
        call(i)
    barrier()
    R = a.calls_per_step or 1
    sampler.window_begin()
    ms_total = timed_calls(ctx, lambda i: call(a.warmup + i), a.steps * R)
    sampler.window_end()
    clocks = sampler.stop() if rank == 0 else None
    assert torch.isfinite(out).all(), "non-finite latents"
    if a.dump_outputs and rank == 0:   # before the secondary measurement reuses `out` and `norms`
        dump_outputs(a.dump_outputs, {"z_T": out, "gnorm_g": norms[0], "gnorm_f": norms[1]})
    value = world * B * T * a.steps * R / (ms_total * 1e-3)

    # ---- secondary: the opt-in single-fp16-pass data gradient, same workload, same timing rules ----
    value_1p = ms_1p = None
    if not a.no_secondary:
        plan1 = prepare(1)
        call1 = make_step(plan1)
        for i in range(a.warmup):
            call1(i)
        ms_1p = timed_calls(ctx, lambda i: call1(a.warmup + i), a.steps * R)
        value_1p = world * B * T * a.steps * R / (ms_1p * 1e-3)
        del plan1, call1
        lsnf_b200.clear_plans()
        plan = prepare(3)

    # ---- config 4, second half: prior sampling eps -> F^-1 -> G -> [0,1] (train.py:565-586) ----
    prior = None
    if a.workload in TEST_WORKLOADS:
        eps_s = torch.randn(B, nz, device=dev)
        for _ in range(3):
            plan.sample_prior(eps_s)
        n_s = max(a.steps, 20)
        ms_s = timed_calls(ctx, lambda i: (flush.zero_(), plan.sample_prior(eps_s)), n_s)
        prior = {"samples_per_sec": world * B * n_s / (ms_s * 1e-3), "batch_per_gpu": B, "calls": n_s,
                 "ms_per_call": ms_s / n_s, "what": "lsnf_sample_prior: flow inverse + generator forward + clamp to "
                 "[0,1], one C-ABI call, inputs resident in HBM"}

    # ---- end to end through the public API: pinned host buffers, H2D + D2H inside the timed region ----
    z0_h = torch.from_numpy(z0_np).pin_memory()
    x_h = torch.from_numpy(x_np).pin_memory()
    z_res_h = torch.empty(B, nz, 1, 1).pin_memory()
    n_res_h = torch.empty(2).pin_memory()

    def e2e_call(i):
        zd = z0_h.to(dev, non_blocking=True)
        xd = x_h.to(dev, non_blocking=True)
        zk, gn, fn = lsnf_b200.sample_langevin_post_z_with_flow(zd, xd, netG, netF, args, seed=99 + i,
                                                                sample_offset=sample_offset, steps=T,
                                                                with_noise=noisy)
        z_res_h.copy_(zk, non_blocking=True)
        n_res_h.copy_(torch.stack([gn, fn]), non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller reads the result on the host

    e2e_call(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(a.steps * R):
        e2e_call(i + 1)
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * T * a.steps * R / float(e2e_s.item())
    h2d = (z0_h.numel() * 4 + x_h.numel() * 4) * R
    d2h = (z_res_h.numel() * 4 + 8) * R

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: per-stage CUDA-event timing through lsnf_plan_run_stage ----
    pk = peaks()
    layers = synth.generator_layers(w["dataset"], nz, w["ngf"])
    exact = exact_layer_flops(layers)
    stages = plan.stages()
    reps = 10
    table = []
    for idx, info in enumerate(stages):
        for _ in range(2):
            plan.run_stage(idx)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(reps):
            plan.run_stage(idx)
        s1.record()
        torch.cuda.synchronize()
        us = s0.elapsed_time(s1) * 1e3 / reps
        alg = exact[info.layer] * B
        table.append(dict(stage=idx, kind="fwd" if info.kind == 0 else "dgrad", layer=info.layer, us=us,
                          alg_gflop=alg / 1e9, nominal_gflop=info.flops / 1e9, tflops_alg=alg / us / 1e6,
                          block_n=info.block_n, k_splits=info.k_splits, passes=info.passes))
    # the flow-prior kernel alone (it overlaps the generator stages inside the loop)
    zf = torch.from_numpy(z0_np).to(dev).reshape(B, nz).contiguous()
    for _ in range(2):
        plan.flow_forward(zf, want_grad=True)
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(reps):
        plan.flow_forward(zf, want_grad=True)
    s1.record()
    torch.cuda.synchronize()
    flow_us = s0.elapsed_time(s1) * 1e3 / reps
    gemm_us = sum(t["us"] for t in table)
    dom = max(table, key=lambda t: t["us"])
    step_us = ms_total * 1e3 / (a.steps * R) / T   # one Langevin iteration
    # DRAM traffic of the dominant launch: from the ncu --set full capture of THIS build of the kernels
    # (tools/run_final.sh writes profiles/ncu_dominant_kernel.json with the hash of the CUDA sources); a capture
    # of other sources is refused
    traffic, traffic_note = None, "no ncu capture under profiles/ for this workload"
    tpath = os.path.join(ROOT, "profiles", "ncu_dominant_kernel.json")
    if os.path.exists(tpath):
        try:
            td = json.load(open(tpath))
            if td.get("workload") != a.workload or td.get("batch_per_gpu", 100) != B:
                traffic_note = "capture under profiles/ is of another workload / batch"
            elif td.get("kernel_source_sha") != kernel_source_sha():
                traffic_note = "capture under profiles/ was taken from other kernel sources: refused"
            else:
                traffic = td.get("dram_bytes_per_launch_by_stage", {}).get(str(dom["stage"]))
                traffic_note = td.get("source")
        except Exception:
            traffic = None
    kname = "tapgemm_tc2_kernel (CTA pair, N tile 256)" if dom["block_n"] == 256 else f"tapgemm_tc_kernel<{dom['block_n']}>"
    roofline = {"bound": "tensor", "achieved": dom["tflops_alg"], "peak": pk["tflops"], "unit": "TFLOP/s",
                "frac": dom["tflops_alg"] / pk["tflops"], "traffic": traffic, "traffic_source": traffic_note,
                "kernel": f"{kname} stage {dom['stage']} ({dom['kind']} layer {dom['layer']})",
                "kernel_us": dom["us"], "alg_gflop_per_launch": dom["alg_gflop"],
                "peak_source": pk["src"] + ", burst bf16 (kernel timed alone)",
                "mma": f"tcgen05 kind::f16, fp32 TMEM accumulate; {dom['passes']} pass(es) in this stage (3 = hi*hi + "
                       "hi*lo + lo*hi of a 16-bit hi/lo split); algorithmic FLOPs count one pass",
                "share_of_iteration": dom["us"] / step_us, "all_gemm_stages_us": gemm_us, "iteration_us": step_us,
                "flow_prior_kernel_us": flow_us}
    # what the tensor pipe actually executes in that launch: every pass, zero-padded taps included
    exec_tflops = dom["nominal_gflop"] * dom["passes"] / dom["us"] * 1e3   # GFLOP per us -> TFLOP/s
    roofline["executed"] = {"mma_gflop_per_launch": dom["nominal_gflop"] * dom["passes"], "tflops": exec_tflops,
                            "frac_of_peak": exec_tflops / pk["tflops"],
                            "note": "all MMA passes and out-of-bounds (zero-filled) tap rows counted; not the roofline claim"}
    if a.stage_table:
        json.dump({"stages": table, "flow_prior_kernel_us": flow_us, "iteration_us": step_us}, open(a.stage_table, "w"), indent=1)

    cpu_b = None
    if not a.no_cpu_baseline and world == 1:   # the contract: rank 0, N=1 only (at N>1 the other ranks have left already)
        cpu_T = {"svhn": 10, "cifar10": 2, "celeba_crop": 2, "celeba_hq256": 1, "svhn_test": 10}[a.workload]
        cb = REF_SAMPLE_B.get(a.workload, B)
        rate, dt, threads, done = oracle_rate(w, gsd, fsd, cpu_T, min_seconds=12.0, batch=cb)
        cpu_b = {"value": rate, "unit": "latent-steps/s", "cores": threads, "kind": "port",
                 "sample": f"{done} Langevin iterations of a batch of {cb} of the same workload in {dt:.1f} s on "
                           f"{cpu_model()} ({threads} threads; oracle/refpath.py, torch CPU fp32)"}
    # the same oracle as eager torch-CUDA on this GPU: what a user of the reference (a GPU program, train.py:737
    # cudnn.benchmark=True) would compare against.  Informational; TF32 off so that it computes in fp32 like ours.
    eager = None
    if not a.no_eager_ref and world == 1:
        try:
            torch.backends.cudnn.benchmark = True
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            eb = REF_SAMPLE_B.get(a.workload, B)
            eT = min(T, 40)
            rate, dt, _, done = oracle_rate(w, gsd, fsd, eT, repeats=2, device=str(dev), batch=eb)
            eager = {"value": rate, "unit": "latent-steps/s", "what": f"oracle/refpath.py (restatement of train.py:307-335 "
                     f"on torch autograd) run as eager torch-CUDA on the same GPU: best of 2 calls of {done} iterations, "
                     f"batch {eb}, fp32 (TF32 off), cudnn.benchmark=True", "ms_per_iteration": dt * 1e3 / done,
                     "torch": torch.__version__}
        except Exception as e:   # informational row: never fail the bench on it
            eager = {"value": None, "error": repr(e)[:200]}

    alg_per_ls = 2 * sum(exact) + flow_flops(nz, w["f_width"])
    roof_ls = pk["tflops_sustained"] * 1e12 / alg_per_ls
    line = {
        "metric": "langevin_latent_steps_per_sec", "value": value, "unit": "latent-steps/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
        "scaling": "strong" if a.full_50k else "weak", "vs_baseline": None,
        "dtype": "fp16-hi/lo-3pass-fwd+bf16-hi/lo-3pass-bwd/f32-accumulate (fp32-equivalent)",
        "data": "synthetic",
        "config": workload_config(a.workload, w),
        "details": {"noise": "in-kernel Philox4x32-10" if noisy else "none (test-mode chain, train.py:623)",
                    "langevin_calls_per_step": R, "timed_region_s": ms_total * 1e-3,
                    "mma_passes": {"forward": 3, "data_gradient": 3},
                    "l2": f"flushed between timed calls (256 MB written, inside the timed region); per-call working set "
                          f"{plan.ws_bytes / 1e6:.0f} MB",
                    "alg_gflop_per_latent_step": alg_per_ls / 1e9,
                    "frac_of_tensor_roofline": value / world / roof_ls,
                    "ceiling_of_this_arithmetic": sum(exact) * 2 / (sum(s.flops * s.passes for s in stages) / B),
                    "roofline_denominator": f"{pk['tflops_sustained']} TFLOP/s bf16 sustained, {pk['src']}",
                    "kernel_source_sha": kernel_source_sha()},
        "value_bwd1pass": None if value_1p is None else {
            "value": value_1p, "unit": "latent-steps/s", "ms_per_step": ms_1p / a.steps,
            "frac_of_tensor_roofline": value_1p / world / roof_ls,
            "dtype": "fp16-hi/lo-3pass-fwd+fp16-1pass-bwd/f32-accumulate",
            "note": "opt-in reduced-precision data gradient (bwd_passes=1 / LSNF_BWD_PASSES=1); NOT the headline: its "
                    "arithmetic is narrower than the reference's fp32 (measured z_T margins: profiles/)"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "latent-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": a.steps * R * plan.launch_count(T),
        "roofline": roofline,
        "cpu_baseline": cpu_b,
        "reference_cuda_eager": eager,
    }
    if prior is not None:
        line["prior_sampling"] = prior
    sink.emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
