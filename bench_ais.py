"""Cost of annealed importance sampling (``lsnf_ais_run``) against the Langevin loop (``lsnf_langevin_run``) on the same
plan, at one workload (B=100 at the workload's g_l_steps T: CIFAR-10 T=40, SVHN T=20):

    langevin   T Langevin iterations (Philox noise, replayed CUDA graphs)
    ais        T MALA transitions along the sigmoidal schedule with step-size adaptation: T + 1 loop iterations

Reported per arm: ms per call, latent-steps/s (B * T transitions per call) and ms per loop iteration (the AIS call runs
one iteration more than it has transitions), plus the AIS chains' mean acceptance rate.  The arms alternate, round after
round, so that drift of the box affects both alike.  Prints one JSON document with the GPU's name and power limit read
in the same run and writes it to ``--out`` if given.

    python bench_ais.py [--workload cifar10] [--rounds 5] [--calls 20] [--out profiles/r6_ais_cifar10_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import statistics

import numpy as np
import torch

from bench_autograd import gpu_identity, timed_ms


def main():
    import bench
    import lsnf_b200
    from lsnf_b200 import synth
    from lsnf_b200.ais import sigmoid_schedule

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cifar10", choices=["cifar10", "svhn"])
    ap.add_argument("--rounds", type=int, default=5, help="rounds of the alternating arms; the median is reported")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per arm and round")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ais.py measures the GPU path and needs a CUDA device")
    dev = torch.device("cuda:0")
    w = bench.WORKLOADS[a.workload]
    B, T, s, sigma = w["B"], w["T"], 0.1, w["sigma"]
    _args, netG, netF, _, _ = bench.build_models(w, dev)
    x_np, z0_np, _ = synth.inputs(B, w["nz"], 3, w["img"], 1, seed=1)
    x = torch.from_numpy(x_np).to(dev).contiguous()
    z0 = torch.from_numpy(z0_np).reshape(B, w["nz"]).to(dev).contiguous()
    plan = lsnf_b200.langevin_plan(netG, netF, B, dev, 3)
    plan.ensure_generator(netG)
    plan.ensure_flow(netF, need_inverse=True)
    betas = torch.from_numpy(sigmoid_schedule(T).astype(np.float32)).to(dev)
    rates = []

    def langevin(i):
        return plan.langevin_run(z0, x, T, s, sigma, seed=i)

    def ais(i):
        out = plan.ais_run(z0, x, betas, T, s, sigma, target_accept=0.65, seed=i)
        rates.append(out[2])
        return out

    arms = {"langevin": (langevin, T), "ais": (ais, T + 1)}
    for fn, _ in arms.values():
        fn(0)   # warm-up: eager first call, then the CUDA graphs
        fn(1)
    ms = {k: [] for k in arms}
    for r in range(a.rounds):
        for k, (fn, _) in arms.items():
            ms[k].append(timed_ms(fn, a.calls))
    res = {"workload": a.workload, "B": B, "T": T, **gpu_identity(dev), "torch": torch.__version__,
           "rounds": a.rounds, "calls_per_round": a.calls}
    for k, (_, iters) in arms.items():
        med = statistics.median(ms[k])
        res[k] = {"ms_per_call": med, "latent_steps_per_s": B * T / (med * 1e-3), "ms_per_iteration": med / iters,
                  "latent_steps_per_s_rounds": [B * T / (v * 1e-3) for v in ms[k]]}
    res["ais"]["mean_accept_rate"] = float(torch.stack(rates).mean())
    res["ais_iteration_time_vs_langevin"] = res["ais"]["ms_per_iteration"] / res["langevin"]["ms_per_iteration"]
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
