"""Cost of differentiating through the modules: the reference's own Langevin closure (train.py:307-335, written with
``torch.autograd.grad``) and its two parameter updates (train.py:390-415, written with ``loss.backward()``), run

    eager              the modules' differentiable torch branch (the default)
    kernel_autograd    the same code under ``lsnf_b200.kernel_autograd()``: kernels forward, their VJPs backward
    fused              the library's own entry points: ``lsnf_langevin_run`` / ``generator_update`` + ``flow_update``

at one workload (default CIFAR-10: B=100, T=40).  Prints one JSON document (ms per iteration, latent-steps/s, the
GPU's name and power limit read in the same run) and writes it to ``--out`` if given.

    python bench_autograd.py [--workload cifar10] [--calls 5] [--out profiles/r3_autograd_cifar10_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import time

import torch
import torch.nn.functional as F

LOG_2PI = math.log(2.0 * math.pi)


def reference_closure(z, x, netG, netF, steps, step_size, sigma, eps=None, with_noise=True):
    """sample_langevin_post_z_with_flow of train.py:307-335 as the reference writes it.  ``eps`` [steps,B,nz,1,1]
    injects the noise; otherwise it is drawn with ``torch.randn_like`` (train.py:326).  Returns (z_k, |grad_g|,
    |grad_f|) of the last step."""
    B = z.shape[0]
    z = z.clone().detach().requires_grad_(True)
    gn = fn = None
    for t in range(steps):
        x_hat = netG(z)                                                                   # train.py:312
        g_log_lkhd = 1.0 / (2.0 * sigma * sigma) * F.mse_loss(x_hat, x, reduction="sum")  # :313
        z_grad_g = torch.autograd.grad(g_log_lkhd, z)[0]                                  # :314
        z_f, objective, _ = netF(torch.squeeze(z), objective=torch.zeros(B, device=z.device))   # :316
        ll = (-0.5 * z_f ** 2).sum(1) + LOG_2PI + objective                               # :317-319
        f_log_lkhd = -ll.sum()                                                            # :320
        z_grad_f = torch.autograd.grad(f_log_lkhd, z)[0]                                  # :323
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)             # :324
        if eps is not None:
            z.data += step_size * eps[t]                                                  # :325-326
        elif with_noise:
            z.data += step_size * torch.randn_like(z)
        gn = z_grad_g.view(B, -1).norm(dim=1).mean()                                      # :328
        fn = z_grad_f.view(B, -1).norm(dim=1).mean()                                      # :329
    return z.detach(), gn, fn


def generator_loss(netG, z_k, x):
    """loss_g of train.py:392-393."""
    x_hat = netG(z_k.detach())
    return F.mse_loss(x_hat, x, reduction="sum") / x.shape[0]


def flow_loss(netF, z_k):
    """loss_f of train.py:405-410."""
    B = z_k.shape[0]
    z_f, objective, _ = netF(torch.squeeze(z_k.detach()).reshape(B, -1), objective=torch.zeros(B, device=z_k.device))
    ll = (-0.5 * z_f ** 2).sum(1) + LOG_2PI + objective
    return -ll.mean()


def reference_updates(netG, netF, optG, optF, z_k, x):
    """train.py:390-415 with loss.backward() (no gradient clipping: the reference's defaults)."""
    optG.zero_grad()
    loss_g = generator_loss(netG, z_k, x)
    loss_g.backward()
    optG.step()
    optF.zero_grad()
    loss_f = flow_loss(netF, z_k)
    loss_f.backward()
    optF.step()
    return loss_g.detach(), loss_f.detach()


def gpu_identity(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", f"--id={dev.index or 0}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = None
    return {"gpu": name, "power_limit": out or "unavailable"}


def timed_ms(fn, calls):
    """Host clock around `calls` calls that end in a device synchronise; ms per call."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(calls):
        fn(i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / calls


def main():
    import bench
    import lsnf_b200
    from lsnf_b200 import synth

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cifar10", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--calls", type=int, default=5, help="timed calls per arm (each a whole closure / update)")
    ap.add_argument("--eager-calls", type=int, default=2, help="timed calls of the (slow) eager closure")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_autograd.py measures the GPU path and needs a CUDA device")
    dev = torch.device("cuda:0")
    w = bench.WORKLOADS[a.workload]
    B, T, s, sigma = w["B"], w["T"], 0.1, w["sigma"]
    args, netG, netF, _, _ = bench.build_models(w, dev)
    x_np, z0_np, _ = synth.inputs(B, w["nz"], 3, w["img"], 1, seed=1)
    x = torch.from_numpy(x_np).to(dev)
    z0 = torch.from_numpy(z0_np).reshape(B, w["nz"], 1, 1).to(dev)
    res = {"workload": a.workload, "B": B, "T": T, **gpu_identity(dev), "torch": torch.__version__}

    def closure(i):
        return reference_closure(z0, x, netG, netF, T, s, sigma)

    def langevin_arm(name, fn, calls):
        fn(0)
        ms = timed_ms(fn, calls)
        res[name] = {"ms_per_call": ms, "ms_per_iteration": ms / T, "latent_steps_per_s": B * T / (ms * 1e-3),
                     "calls": calls}

    langevin_arm("closure_eager", closure, a.eager_calls)
    with lsnf_b200.kernel_autograd():
        langevin_arm("closure_kernel_autograd", closure, a.calls)
    langevin_arm("langevin_run_fused",
                 lambda i: lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=i), a.calls)

    # the parameter updates (train mode, as in a training iteration), from the latents of one Langevin call
    z_k = lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=7)[0]
    netG.train()
    netF.train()
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)

    def update_arm(name, fn, calls):
        fn(0)
        ms = timed_ms(fn, calls)
        res[name] = {"ms_per_update": ms, "calls": calls}

    update_arm("updates_eager_backward", lambda i: reference_updates(netG, netF, optG, optF, z_k, x), a.calls)
    with lsnf_b200.kernel_autograd():
        update_arm("updates_kernel_autograd_backward", lambda i: reference_updates(netG, netF, optG, optF, z_k, x),
                   a.calls)
    update_arm("updates_fused", lambda i: (lsnf_b200.generator_update(netG, optG, z_k, x, args),
                                           lsnf_b200.flow_update(netF, optF, z_k, args)), a.calls)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
