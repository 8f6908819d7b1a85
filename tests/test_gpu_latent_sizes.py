"""The generator and the Langevin loop at latent sizes outside the shipped {100, 128}.

nz sets the K extent of the first forward layer (nz = 4: 60 of its 64 K columns are zero padding; nz = 192 / 256: 3-4
K blocks), the N extent of the first layer's data gradient (nzp = nz rounded up to 128: above 128 there are two N
tiles, the second partly padding), the rows of the first layer's weight gradient (two M tiles, one ragged) and the
columns reduce_partial_kernel sums.  Every other GPU test runs nz = 100 or 128.  The generator is made kink-free with
leak = 1.0 (DESIGN.md section 2) so that every tensor is compared element-wise with the fp64 oracle."""
import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import synth
from oracle import philox, refpath
from helpers import REL_TOL, build_nets, oracle_langevin, record, rel_err, rel_l2, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = 0.3


def _gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


GEN_CASES = [(dict(dataset="svhn", nz=nz, ngf=64), B) for nz in (4, 132, 192, 256) for B in (1, 57, 130)]
GEN_CASES.append((dict(dataset="cifar10", nz=256, ngf=128), 100))   # the CTA-pair kernels at nz = 256


@pytest.mark.parametrize("c,B", GEN_CASES)
def test_generator_at_latent_size_against_fp64_oracle(c, B):
    c = dict(c, leak=1.0)
    nz = c["nz"]
    args, netG, _ = build_nets(c, DEV, seed=4)
    netG.train()
    img = synth.image_size(c["dataset"])
    x_np, z_np, _ = synth.inputs(B, nz, 3, img, 1, seed=9)
    z, x = torch.from_numpy(z_np).reshape(B, nz), torch.from_numpy(x_np)
    gy = torch.randn(B, 3, img, img, generator=torch.Generator().manual_seed(5))
    # ---- the kernels: forward, reconstruction gradient, VJP, parameter gradients on a training plan ----
    plan = netG._plan(B, torch.device(DEV))
    plan.ensure_generator(netG)
    xh = plan.generator_forward(z.to(DEV)).cpu()
    g_dgrad = plan.generator_dgrad(x.to(DEV), SIGMA).cpu()
    plan.generator_forward(z.to(DEV))
    g_vjp, _ = plan.generator_vjp(gy.to(DEV).contiguous())
    _, pairs, loss = lsnf_b200.generator_gradients(netG, z.to(DEV), x.to(DEV), B)
    named = dict(netG.named_parameters())
    got_p = {k: g.cpu() for p, g in pairs for k, q in named.items() if q is p}
    # ---- the oracle in fp64 ----
    gp = {k: v.double() for k, v in to_torch(synth.generator_state(c["dataset"], nz, c["ngf"], 3, seed=4)).items()}
    layers = refpath.generator_layers(c["dataset"], nz, c["ngf"])
    z64, x64 = z.double().reshape(B, nz, 1, 1), x.double()
    want_xh, want_dgrad = refpath.recon_grad(z64, x64, gp, layers, SIGMA, leak=1.0)
    zr = z64.clone().requires_grad_(True)
    (refpath.generator_forward(gp, zr, layers, 1.0) * gy.double()).sum().backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    want_loss = torch.nn.functional.mse_loss(refpath.generator_forward(leaves, z64, layers, 1.0), x64, reduction="sum") / B
    want_loss.backward()
    errs = {"x_hat": rel_err(xh, want_xh), "dgrad": rel_l2(g_dgrad, want_dgrad.reshape(B, nz)),
            "vjp": rel_l2(g_vjp.cpu(), zr.grad.reshape(B, nz)), "loss": abs(loss.item() - want_loss.item()) / want_loss.item()}
    errs.update({k: rel_l2(got_p[k], leaves[k].grad) for k in leaves})
    worst = max(errs, key=errs.get)
    print(f"generator {c['dataset']} ngf={c['ngf']} nz={nz} B={B}: " + ", ".join(f"{k} {e:.1e}" for k, e in errs.items()))
    record(f"r4_latent_{c['dataset']}_nz{nz}_b{B}.json", {"config": c, "B": B, "errors": errs, "worst": worst})
    # the first layer's weight and bias gradients: the two M tiles of the weight-gradient GEMM (nz > 128) and the
    # bias row sums, asserted on their own so that a failure names them
    assert errs["gen.0.weight"] < REL_TOL, errs["gen.0.weight"]
    assert errs["gen.0.bias"] < REL_TOL, errs["gen.0.bias"]
    for k, e in errs.items():
        assert e < REL_TOL, (k, e)


@pytest.mark.parametrize("nz,perm", [(192, 2), (256, 1)])
def test_langevin_chain_at_latent_size_against_oracle(nz, perm):
    # nz = 256 with the invertible 1x1 matrix does not fit the flow kernels (nz^2 alone is 256 KB); with the shuffle
    # permutation it does.  Injected noise, the reference's leak = 0.2, z_T held to the suite's 1e-4.
    B, T = 100, 10
    c = dict(dataset="svhn", nz=nz, ngf=64, f_width=64, permutation=perm, sigma=SIGMA, T=T)
    x_np, z0_np, eps_np = synth.inputs(B, nz, 3, 32, T, seed=31)
    zr, gnr, fnr = oracle_langevin(c, x_np, z0_np, eps_np, seed=2)
    args, netG, netF = build_nets(c, DEV, seed=2)
    z, gn, fn = lsnf_b200.sample_langevin_post_z_with_flow(_gpu(z0_np), _gpu(x_np), netG, netF, args, eps=_gpu(eps_np))
    e = rel_l2(z.cpu(), zr)
    print(f"svhn nz={nz} perm={perm} B={B} T={T}: z_T rel-l2 {e:.2e}, |grad_g| {gn.item():.4f} (oracle "
          f"{gnr.item():.4f}), |grad_f| {fn.item():.4f} (oracle {fnr.item():.4f})")
    record(f"r4_latent_chain_nz{nz}_perm{perm}.json", {"config": c, "B": B, "z_T_rel_l2": e})
    assert e < REL_TOL
    assert abs(gn.item() - gnr.item()) < 2e-3 * gnr.item() and abs(fn.item() - fnr.item()) < 1e-3 * fnr.item()


def test_philox_chain_graph_replay_at_latent_size_192():
    # as test_gpu_parity_real_shapes.py::test_product_configuration_philox_graph_replay_against_oracle: call 0 runs
    # eagerly, calls 1-2 replay the captured graph, bit for bit
    B, T = 100, 10
    c = dict(dataset="svhn", nz=192, ngf=64, f_width=64, sigma=SIGMA, T=T)
    x_np, z0_np, _ = synth.inputs(B, 192, 3, 32, 1, seed=23)
    seed, offset = 0x5EED00000000 + 91, 7000
    eps_np = np.stack([philox.langevin_noise(seed, offset, B, 192, t) for t in range(T)]).reshape(T, B, 192, 1, 1)
    zr, gnr, _ = oracle_langevin(c, x_np, z0_np, eps_np.astype(np.float32), seed=2)
    args, netG, netF = build_nets(c, DEV, seed=2)
    outs = []
    for call in range(3):
        z, gn, _ = lsnf_b200.sample_langevin_post_z_with_flow(_gpu(z0_np), _gpu(x_np), netG, netF, args, seed=seed,
                                                              sample_offset=offset)
        outs.append(z.cpu())
        e = rel_l2(z.cpu(), zr)
        print(f"svhn nz=192 philox call {call}: z_T rel-l2 vs oracle {e:.2e}")
        assert e < REL_TOL
        assert abs(gn.item() - gnr.item()) < 2e-3 * gnr.item()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
