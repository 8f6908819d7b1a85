"""`bench.py --mode train`: one whole training iteration of the reference (train.py:376-415) per step, with the
parameter-gradient all-reduces INSIDE the timed region:

    z_0 ~ N(0,I);  z_k = Langevin(z_0, x)                 lsnf_langevin_run           (no collective)
    generator update:  grads -> all-reduce -> fused Adam   lsnf_generator_param_grads  (per-layer buckets on a comm stream)
    flow update:       grads -> all-reduce -> fused Adam   lsnf_flow_param_grads

B latents per GPU (weak scaling); the losses are normalised by the global batch.  Reports training-iteration
throughput as latent-steps/s (N * B * T / iteration time), the time the collectives add to an iteration (the same loop
with the all-reduces switched off, on the same ranks) and the bus bandwidth of the big all-reduce timed alone.
"""
from __future__ import annotations

import json
import time

import torch


def run_train_bench(a, w, ctx, sink):
    import torch.distributed as dist
    import bench
    import lsnf_b200
    from lsnf_b200 import synth
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    args, netG, netF, gsd, fsd = bench.build_models(w, dev)
    netG.train()
    netF.train()
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)
    B, T, nz = w["B"], w["T"], w["nz"]
    x_np, _, _ = synth.inputs(B, nz, 3, w["img"], 1, seed=1 + rank)
    x = torch.from_numpy(x_np).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def make_step(dp):
        def step(i):
            flush.zero_()
            return lsnf_b200.training_iteration(x, netG, netF, optG, optF, args, global_batch=world * B,
                                                sample_offset=rank * B, seed=1000 + i,
                                                data_parallel=None if dp else False)
        return step

    step = make_step(True)
    sampler = bench.ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    for i in range(max(a.warmup, 3)):
        step(i)
    ctx.barrier()
    R = a.calls_per_step or 1
    n_iter = a.steps * R
    last = []

    def timed_step(i):
        last[:] = step(100 + i)

    sampler.window_begin()
    ms_total = bench.timed_calls(ctx, timed_step, n_iter)
    sampler.window_end()
    clocks = sampler.stop() if rank == 0 else None
    lg, lf, gn, fn, zk = last
    assert torch.isfinite(zk).all() and torch.isfinite(lg) and torch.isfinite(lf)
    if a.dump_outputs and rank == 0:   # the parameters as the last timed iteration left them, before the runs below
        bench.dump_outputs(a.dump_outputs, {
            "loss_g": lg, "loss_f": lf, "gnorm_g": gn, "gnorm_f": fn, "z_k": zk,
            "generator_params": torch.cat([p.detach().reshape(-1) for p in netG.parameters()]),
            "flow_params": torch.cat([p.detach().reshape(-1) for p in netF.parameters()])})
    value = world * B * T * n_iter / (ms_total * 1e-3)

    # the same iterations without the collectives (every rank updates from its own shard): what the all-reduces cost
    exposed_ms = None
    busbw = None
    if world > 1:
        nodp = make_step(False)
        for i in range(3):
            nodp(i)
        ms_nodp = bench.timed_calls(ctx, lambda i: nodp(200 + i), n_iter)
        exposed_ms = (ms_total - ms_nodp) / n_iter
        # the generator's flat gradient buffer all-reduced alone
        n = sum(p.numel() for p in netG.parameters())
        buf = torch.zeros(n, dtype=torch.float32, device=dev)
        for _ in range(3):
            dist.all_reduce(buf)
        reps = 10
        ms_ar = bench.timed_calls(ctx, lambda i: dist.all_reduce(buf), reps) / reps
        busbw = {"bytes": n * 4, "ms": ms_ar, "algbw_gbs": n * 4 / ms_ar / 1e6,
                 "busbw_gbs": n * 4 / ms_ar / 1e6 * 2 * (world - 1) / world,
                 "nvlink5_peak_gbs_per_direction": 900.0}

    # end to end: the minibatch comes from pinned host memory every iteration, the two losses go back to the host
    x_h = torch.from_numpy(x_np).pin_memory()
    res_h = torch.empty(2).pin_memory()

    def e2e_step(i):
        xd = x_h.to(dev, non_blocking=True)
        lg, lf, _, _, _ = lsnf_b200.training_iteration(xd, netG, netF, optG, optF, args, global_batch=world * B,
                                                       sample_offset=rank * B, seed=5000 + i)
        res_h.copy_(torch.stack([lg, lf]), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step(0)
    ctx.barrier()
    t0 = time.perf_counter()
    for i in range(n_iter):
        e2e_step(1 + i)
    ctx.barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * T * n_iter / float(e2e_s.item())
    if rank != 0:
        return

    # split of one iteration on this rank: Langevin call alone vs the two updates
    plan = lsnf_b200.langevin_plan(netG, netF, B, dev, train=True)
    z0 = torch.randn(B, nz, device=dev)
    outz, norms = torch.empty_like(z0), torch.zeros(2, device=dev)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(5):
        plan.langevin_run(z0, x, T, 0.1, w["sigma"], with_noise=True, seed=i, out=outz, norms=norms)
    e1.record()
    torch.cuda.synchronize()
    langevin_ms = e0.elapsed_time(e1) / 5
    iter_ms = ms_total / n_iter
    n_layers = len([s for s in plan.stages() if s.kind == 0])
    line = {
        "metric": "train_iteration_latent_steps_per_sec", "value": value, "unit": "latent-steps/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_total / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "mode": "train",
        "dtype": "fp16-hi/lo-3pass-fwd+bf16-hi/lo-3pass-bwd-and-wgrad/f32-accumulate (fp32-equivalent); fp32 flow + Adam",
        "data": "synthetic", "config": bench.workload_config(a.workload, w),
        "details": {"what": "Langevin + generator update + flow update (train.py:376-415), parameter-gradient "
                            "all-reduces inside the timed region; B per GPU fixed, losses normalised by the global batch",
                    "training_iterations_per_step": R, "ms_per_iteration": iter_ms,
                    "langevin_call_ms": langevin_ms, "updates_ms": iter_ms - langevin_ms,
                    "allreduce_exposed_ms_per_iteration": exposed_ms, "allreduce_alone": busbw,
                    "grad_bytes_per_iteration": {"generator": sum(p.numel() for p in netG.parameters()) * 4,
                                                 "flow": sum(p.numel() for p in netF.parameters()) * 4},
                    "loss_g": float(lg), "loss_f": float(lf), "timed_region_s": ms_total * 1e-3,
                    "l2": "flushed between iterations (256 MB written, inside the timed region)"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "latent-steps/s", "h2d_bytes_per_step": x_h.numel() * 4 * R,
                "d2h_bytes_per_step": 8 * R},
        # Langevin call + generator update (split_z, L forward stages, gather, loss, fused seed kernel, L-1 data-gradient
        # stages, per layer 2 transposes + tap-GEMM + finalize + bias sums, 1 Adam launch) + flow update (fused kernel,
        # parameter-gradient kernel, 2 Adam launches for its 60 tensors)
        "gpu_launches": n_iter * (plan.launch_count(T) + (1 + n_layers + 1) + 1 + 1 + (n_layers - 1) + 5 * n_layers + 1
                                  + 2 + 2),
    }
    sink.emit(line)
