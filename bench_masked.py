"""Cost of a masked reconstruction loss (inpainting, occluded pixels, images with missing regions) at one workload
(B=100 at the workload's g_l_steps), in latent-steps/s of the Langevin call and ms per training iteration:

    unmasked            the fused loop, ``lsnf_langevin_run``
    mask_ones           the fused loop with an all-ones mask (``lsnf_langevin_run_masked``)
    mask_centre_block   the fused loop with a centre block of a quarter of the pixels hidden
    closure_kernel_autograd_masked
                        the same masked chain written as the reference's closure (train.py:307-335) with the weighted
                        loss, under ``lsnf_b200.kernel_autograd()``
    train_iteration_unmasked / train_iteration_masked
                        one ``training_iteration`` (Langevin + generator update + flow update) without / with the
                        centre-block mask

The arms alternate, round after round, so that drift of the box affects all of them alike.  Prints one JSON document
with the GPU's name and power limit read in the same run and writes it to ``--out`` if given.

    python bench_masked.py [--workload cifar10] [--rounds 3] [--calls 10] [--out profiles/r5_masked_cifar10_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import statistics

import torch

from bench_autograd import LOG_2PI, gpu_identity, timed_ms


def centre_block_mask(B, nc, img, device):
    """1 everywhere except a centred img/2 x img/2 block (a quarter of the pixels), the same for every sample."""
    m = torch.ones(B, nc, img, img, device=device)
    a, b = img // 4, img // 4 + img // 2
    m[:, :, a:b, a:b] = 0.0
    return m


def masked_reference_closure(z, x, mask, netG, netF, steps, step_size, sigma, eps=None, with_noise=True):
    """train.py:307-335 as the reference writes it, with the reconstruction term weighted per pixel:
    1/(2 sigma^2) sum m (G(z) - x)^2.  ``eps`` [steps,B,nz,1,1] injects the noise; otherwise it is drawn with
    ``torch.randn_like``.  Returns z_k."""
    B = z.shape[0]
    z = z.clone().detach().requires_grad_(True)
    for t in range(steps):
        x_hat = netG(z)
        g_log_lkhd = 1.0 / (2.0 * sigma * sigma) * torch.sum(mask * (x_hat - x) ** 2)
        z_grad_g = torch.autograd.grad(g_log_lkhd, z)[0]
        z_f, objective, _ = netF(torch.squeeze(z), objective=torch.zeros(B, device=z.device))
        ll = (-0.5 * z_f ** 2).sum(1) + LOG_2PI + objective
        z_grad_f = torch.autograd.grad(-ll.sum(), z)[0]
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)
        if eps is not None:
            z.data += step_size * eps[t]
        elif with_noise:
            z.data += step_size * torch.randn_like(z)
    return z.detach()


def main():
    import bench
    import lsnf_b200
    from lsnf_b200 import synth

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cifar10", choices=["cifar10", "svhn"])
    ap.add_argument("--rounds", type=int, default=3, help="rounds of the alternating arms; the median is reported")
    ap.add_argument("--calls", type=int, default=10, help="timed calls per arm and round")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_masked.py measures the GPU path and needs a CUDA device")
    dev = torch.device("cuda:0")
    w = bench.WORKLOADS[a.workload]
    B, T, s, sigma = w["B"], w["T"], 0.1, w["sigma"]
    args, netG, netF, _, _ = bench.build_models(w, dev)
    x_np, z0_np, _ = synth.inputs(B, w["nz"], 3, w["img"], 1, seed=1)
    x = torch.from_numpy(x_np).to(dev)
    z0 = torch.from_numpy(z0_np).reshape(B, w["nz"], 1, 1).to(dev)
    ones = torch.ones_like(x)
    block = centre_block_mask(B, 3, w["img"], dev)
    res = {"workload": a.workload, "B": B, "T": T, **gpu_identity(dev), "torch": torch.__version__,
           "rounds": a.rounds, "calls_per_round": a.calls,
           "mask_centre_block_hidden_fraction": float(1.0 - block.mean().item())}

    def chain(mask):
        return lambda i: lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=i, mask=mask)

    def closure(i):
        with lsnf_b200.kernel_autograd():
            return masked_reference_closure(z0, x, block, netG, netF, T, s, sigma)

    langevin_arms = {"unmasked": chain(None), "mask_ones": chain(ones), "mask_centre_block": chain(block),
                     "closure_kernel_autograd_masked": closure}
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)

    def train(mask):
        return lambda i: lsnf_b200.training_iteration(x, netG, netF, optG, optF, args, seed=i, z0=z0, mask=mask)

    train_arms = {"train_iteration_unmasked": train(None), "train_iteration_masked": train(block)}
    ms = {k: [] for k in list(langevin_arms) + list(train_arms)}
    for fn in list(langevin_arms.values()) + list(train_arms.values()):
        fn(0)   # warm-up: plans, packed weights, CUDA graphs of every arm
        fn(1)
    for r in range(a.rounds):
        for k, fn in list(langevin_arms.items()) + list(train_arms.items()):
            ms[k].append(timed_ms(fn, a.calls))
    for k in langevin_arms:
        med = statistics.median(ms[k])
        res[k] = {"ms_per_call": med, "latent_steps_per_s": B * T / (med * 1e-3),
                  "latent_steps_per_s_rounds": [B * T / (v * 1e-3) for v in ms[k]]}
    for k in train_arms:
        res[k] = {"ms_per_iteration": statistics.median(ms[k]), "ms_rounds": ms[k]}
    base = res["unmasked"]["latent_steps_per_s"]
    res["rate_vs_unmasked"] = {k: res[k]["latent_steps_per_s"] / base for k in langevin_arms}
    res["train_masked_vs_unmasked_time"] = res["train_iteration_masked"]["ms_per_iteration"] / \
        res["train_iteration_unmasked"]["ms_per_iteration"]
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
