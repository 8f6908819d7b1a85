"""Cost of posterior inference from linear measurements y = A vec(G(z)) + sigma noise at one workload (B=100 at the
workload's g_l_steps), in latent-steps/s of the Langevin call, for a dense Gaussian operator A [m, n] (n = nc*H*W) with
m = n/16, n/4 and n:

    unmeasured          the fused loop on x, ``lsnf_langevin_run``
    measured_m<m>       the fused loop on y = A vec(x) + noise, ``lsnf_langevin_run_measured``
    closure_kernel_autograd_m<m>
                        the same measured chain written as the reference's closure (train.py:307-335) with
                        |A @ x_hat.view(B, -1) - y|^2, under ``lsnf_b200.kernel_autograd()``

With ``--mode train`` it times one whole training iteration (Langevin + generator update + flow update,
train.py:376-415) at the same B, in ms per iteration:

    train_iteration_unmeasured      ``training_iteration`` on x
    train_iteration_measured_m<m>   ``training_iteration(..., operator=A)`` on y
    reference_train_kernel_autograd_m<m>
                                    the reference's iteration written with |A @ x_hat.view(B, -1) - y|^2 under
                                    ``kernel_autograd()``: the closure, loss_g.backward(), loss_f.backward() and
                                    torch.optim.Adam

The arms alternate, round after round, so that drift of the box affects all of them alike.  The operator is read
from L2 after the first iteration when its packed copies fit (8 m n bytes; at CIFAR-10 and m = n, 75 MB of the 126 MB).
Prints one JSON document with the GPU's name and power limit read in the same run and writes it to ``--out`` if given.

    python bench_measured.py [--workload cifar10] [--rounds 3] [--calls 10] [--out profiles/r10_measured_cifar10_1gpu.json]
    python bench_measured.py --mode train [--workload cifar10] [--out profiles/r12_measured_train_cifar10_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import statistics

import torch

from bench_autograd import LOG_2PI, gpu_identity, timed_ms


def measured_reference_closure(z, y, A, netG, netF, steps, step_size, sigma, with_noise=True):
    """train.py:307-335 as the reference writes it, with the reconstruction term |A vec(x_hat) - y|^2.  Returns z_k."""
    B = z.shape[0]
    z = z.clone().detach().requires_grad_(True)
    for _ in range(steps):
        x_hat = netG(z)
        r = x_hat.view(B, -1) @ A.t() - y
        z_grad_g = torch.autograd.grad(1.0 / (2.0 * sigma * sigma) * torch.sum(r * r), z)[0]
        z_f, objective, _ = netF(torch.squeeze(z), objective=torch.zeros(B, device=z.device))
        ll = (-0.5 * z_f ** 2).sum(1) + LOG_2PI + objective
        z_grad_f = torch.autograd.grad(-ll.sum(), z)[0]
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)
        if with_noise:
            z.data += step_size * torch.randn_like(z)
    return z.detach()


def measured_reference_iteration(z0, y, A, netG, netF, optG, optF, steps, step_size, sigma):
    """train.py:376-415 as the reference writes it, with the measured reconstruction term in the closure and in loss_g.
    Returns (loss_g, loss_f)."""
    from bench_autograd import flow_loss
    netG.train()
    netF.train()
    B = z0.shape[0]
    z_k = measured_reference_closure(z0, y, A, netG, netF, steps, step_size, sigma)
    optG.zero_grad()
    r = netG(z_k.detach()).view(B, -1) @ A.t() - y
    loss_g = torch.sum(r * r) / B
    loss_g.backward()
    optG.step()
    optF.zero_grad()
    loss_f = flow_loss(netF, z_k)
    loss_f.backward()
    optF.step()
    return loss_g.detach(), loss_f.detach()


def main():
    import bench
    import lsnf_b200
    from lsnf_b200 import synth

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cifar10", choices=["cifar10", "svhn"])
    ap.add_argument("--rounds", type=int, default=3, help="rounds of the alternating arms; the median is reported")
    ap.add_argument("--calls", type=int, default=10, help="timed calls per fused arm and round (closure arms: a fifth)")
    ap.add_argument("--mode", default="langevin", choices=["langevin", "train"],
                    help="train: one whole training iteration per call instead of one Langevin call")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_measured.py measures the GPU path and needs a CUDA device")
    dev = torch.device("cuda:0")
    w = bench.WORKLOADS[a.workload]
    B, T, s, sigma = w["B"], w["T"], 0.1, w["sigma"]
    args, netG, netF, _, _ = bench.build_models(w, dev)
    x_np, z0_np, _ = synth.inputs(B, w["nz"], 3, w["img"], 1, seed=1)
    x = torch.from_numpy(x_np).to(dev)
    z0 = torch.from_numpy(z0_np).reshape(B, w["nz"], 1, 1).to(dev)
    n = 3 * w["img"] * w["img"]
    g = torch.Generator(device=dev).manual_seed(7)
    ops = {}
    for m in (n // 16, n // 4, n):
        A = torch.randn(m, n, device=dev, generator=g) / n ** 0.5
        ops[m] = (A, (x.view(B, -1) @ A.t() + 0.05 * torch.randn(B, m, device=dev, generator=g)).contiguous())
    res = {"workload": a.workload, "B": B, "T": T, "n": n, **gpu_identity(dev), "torch": torch.__version__,
           "rounds": a.rounds, "calls_per_round": a.calls, "operator": "Gaussian, N(0, 1/n) entries, dense fp32",
           "operator_packed_bytes": {str(m): 8 * m * n for m in ops}}

    if a.mode == "train":
        return run_train(a, res, ops, x, z0, args, netG, netF, T, s, sigma)

    def chain(m):
        if m is None:
            return lambda i: lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=i)
        A, y = ops[m]
        return lambda i: lsnf_b200.sample_langevin_post_z_with_flow(z0, y, netG, netF, args, seed=i, operator=A)

    def closure(m):
        A, y = ops[m]

        def run(i):
            with lsnf_b200.kernel_autograd():
                return measured_reference_closure(z0, y, A, netG, netF, T, s, sigma)
        return run

    arms = {"unmeasured": (chain(None), a.calls)}
    for m in ops:
        arms[f"measured_m{m}"] = (chain(m), a.calls)
    for m in ops:
        arms[f"closure_kernel_autograd_m{m}"] = (closure(m), max(2, a.calls // 5))
    ms = {k: [] for k in arms}
    for fn, _ in arms.values():
        fn(0)   # warm-up: plans, packed weights and operators, CUDA graphs of every arm
        fn(1)
    for _ in range(a.rounds):
        for k, (fn, calls) in arms.items():
            ms[k].append(timed_ms(fn, calls))
    for k in arms:
        med = statistics.median(ms[k])
        res[k] = {"ms_per_call": med, "latent_steps_per_s": B * T / (med * 1e-3),
                  "latent_steps_per_s_rounds": [B * T / (v * 1e-3) for v in ms[k]]}
    base = res["unmeasured"]["ms_per_call"]
    res["time_vs_unmeasured"] = {k: res[k]["ms_per_call"] / base for k in arms}
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


def run_train(a, res, ops, x, z0, args, netG, netF, T, s, sigma):
    import lsnf_b200
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)
    refG = torch.optim.Adam(netG.parameters(), lr=0.0004, betas=(0.5, 0.999))   # train.py:294-295
    refF = torch.optim.Adam(netF.parameters(), lr=0.0004, betas=(0.5, 0.999))
    res["mode"] = "train"

    def train(m):
        if m is None:
            return lambda i: lsnf_b200.training_iteration(x, netG, netF, optG, optF, args, seed=i, z0=z0)
        A, y = ops[m]
        return lambda i: lsnf_b200.training_iteration(y, netG, netF, optG, optF, args, seed=i, z0=z0, operator=A)

    def reference(m):
        A, y = ops[m]

        def run(i):
            with lsnf_b200.kernel_autograd():
                return measured_reference_iteration(z0, y, A, netG, netF, refG, refF, T, s, sigma)
        return run

    arms = {"train_iteration_unmeasured": (train(None), a.calls)}
    for m in ops:
        arms[f"train_iteration_measured_m{m}"] = (train(m), a.calls)
    for m in ops:
        arms[f"reference_train_kernel_autograd_m{m}"] = (reference(m), max(2, a.calls // 5))
    ms = {k: [] for k in arms}
    for fn, _ in arms.values():
        fn(0)   # warm-up: plans, packed weights and operators, CUDA graphs, optimizer state of every arm
        fn(1)
    for _ in range(a.rounds):
        for k, (fn, calls) in arms.items():
            ms[k].append(timed_ms(fn, calls))
    for k in arms:
        res[k] = {"ms_per_iteration": statistics.median(ms[k]), "ms_rounds": ms[k]}
    base = res["train_iteration_unmeasured"]["ms_per_iteration"]
    res["time_vs_unmeasured"] = {k: res[k]["ms_per_iteration"] / base for k in arms}
    res["extra_ms_vs_unmeasured"] = {k: res[k]["ms_per_iteration"] - base for k in arms}
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
