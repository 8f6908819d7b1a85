"""GPU parity of the test-mode paths (SURVEY.md section 8d config 4): the fused prior-sampling pipeline
eps -> F^-1 -> G -> [0,1] (train.py:565-576), long noise-free chains replayed as chunked CUDA graphs
(train.py:602-634, g_l_steps * 20), and concurrent use of several plans / devices of one process."""
import threading

import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import synth
from oracle import philox, refpath
from helpers import REL_TOL, build_nets, oracle_langevin, rel_err, rel_l2, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("c,B", [
    (dict(dataset="svhn", nz=100, ngf=64, f_width=64), 100),          # config 4's sampling half at its true width
    (dict(dataset="cifar10", nz=128, ngf=128, f_width=64), 37),
    (dict(dataset="celeba_crop", nz=100, ngf=64, f_width=64), 5),
])
def test_prior_sampling_pipeline_against_oracle(c, B):
    args, netG, netF = build_nets(c, DEV, seed=4)
    gp = to_torch(synth.generator_state(c["dataset"], c["nz"], c["ngf"], 3, seed=4))
    fp = to_torch(synth.flow_state(c["nz"], c["f_width"], 5, 1, 2, seed=4))
    layers = refpath.generator_layers(c["dataset"], c["nz"], c["ngf"])
    eps = torch.randn(B, c["nz"], generator=torch.Generator().manual_seed(5))
    # train.py:567-573 restated on the oracle
    z_ref, _ = refpath.flow_reverse(fp, eps.clone(), torch.zeros(B), 5)
    x_ref = ((refpath.generator_forward(gp, z_ref.reshape(B, c["nz"], 1, 1), layers) + 1.0) / 2.0).clamp(min=0.0, max=1.0)
    e_dev = eps.to(DEV)
    x = lsnf_b200.sample_x(netG, netF, B, DEV, eps=e_dev)
    assert x.shape == x_ref.shape and float(x.min()) >= 0.0 and float(x.max()) <= 1.0
    assert float((x.cpu() - x_ref).abs().max()) < REL_TOL          # values live in [0, 1]: absolute = relative to range
    assert torch.equal(e_dev.cpu(), eps), "eps must not be modified (the reference's reverse pass does, model.py:436)"
    plan = lsnf_b200.langevin_plan(netG, netF, B, torch.device(DEV))
    x2, z = plan.sample_prior(e_dev, to_unit_range=False, want_z=True)
    assert rel_err(z.cpu(), z_ref) < REL_TOL
    assert float((x2.cpu() - refpath.generator_forward(gp, z_ref.reshape(B, c["nz"], 1, 1), layers)).abs().max()) < REL_TOL
    # the fused call equals the composition of the two module calls the reference makes
    with torch.no_grad():
        zf = netF(e_dev, objective=torch.zeros(B, device=DEV), reverse=True, return_obj=False)
        xk = netG(torch.reshape(zf, (B, c["nz"], 1, 1)))
    assert torch.equal(((xk + 1.0) / 2.0).clamp(min=0.0, max=1.0), x)


def _energy(c, gp, fp, layers, z, x):
    """U(z) = 1/(2 sigma^2) |G(z) - x|^2 - log p(z) per sample: what the noise-free chain descends (train.py:613-620)."""
    xh = refpath.generator_forward(gp, z.reshape(z.shape[0], -1, 1, 1), layers)
    ll, _, _ = refpath.log_prior(fp, z.reshape(z.shape[0], -1), 5)
    return 0.5 / c["sigma"] ** 2 * ((xh - x) ** 2).flatten(1).sum(1) - ll


def test_long_noise_free_chain_chunked_graph_against_oracle():
    # test mode: g_l_steps * 20 noise-free iterations (train.py:606, :623).  400 iterations = 10 replays of one
    # 40-iteration graph; the first call of the plan runs eagerly and must agree bit for bit with the replays.
    #
    # What "parity" can mean at this length: a 400-step descent through LeakyReLU kinks is NOT reproducible to 1e-4
    # by the reference itself -- its fp32 path differs from its fp64 path by 1.3e-3 on this very case, and from itself
    # by 2.2e-3 when torch's CPU thread count (= summation order) changes (measured, DESIGN.md section 2).  So:
    # the first graph chunk (40 steps) must agree to 1e-4, the end point to 2e-2, and the energy each chain has
    # descended to -- the quantity the chain optimises -- to 2e-3 relative.
    c = dict(dataset="svhn", nz=100, ngf=32, f_width=64, sigma=0.3, T=20)
    x_np, z0_np, _ = synth.inputs(6, 100, 3, 32, 1, seed=12)
    args, netG, netF = build_nets(c, DEV, seed=7)
    sampler = lsnf_b200.make_sampler(args, test_mode=True)
    z0, x = torch.from_numpy(z0_np).to(DEV), torch.from_numpy(x_np).to(DEV)
    z_eager, gn0, fn0 = sampler(z0, x, netG, netF)
    z_graph, gn1, fn1 = sampler(z0, x, netG, netF)
    assert torch.equal(z_eager, z_graph) and gn0.item() == gn1.item() and fn0.item() == fn1.item()
    trace = []
    zr, gnr, fnr = oracle_langevin(c, x_np, z0_np, None, seed=7, steps=400, trace=trace)
    z40, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, steps=40, with_noise=False)
    e40, e400 = rel_l2(z40.cpu(), trace[39]), rel_l2(z_graph.cpu(), zr)
    gp = to_torch(synth.generator_state("svhn", 100, 32, 3, seed=7))
    fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=7))
    layers = refpath.generator_layers("svhn", 100, 32)
    xc = torch.from_numpy(x_np)
    u_ours, u_ref = _energy(c, gp, fp, layers, z_graph.cpu(), xc), _energy(c, gp, fp, layers, zr, xc)
    u_start = _energy(c, gp, fp, layers, torch.from_numpy(z0_np), xc)
    du = float(((u_ours - u_ref).abs() / u_ref.abs()).max())
    print(f"noise-free chain: z_40 rel-l2 {e40:.2e}, z_400 rel-l2 {e400:.2e}, energy rel diff {du:.2e} "
          f"(start {u_start.mean():.1f} -> ours {u_ours.mean():.2f} / oracle {u_ref.mean():.2f})")
    assert e40 < REL_TOL
    assert e400 < 2e-2
    assert du < 2e-3
    assert abs(gn1.item() - gnr.item()) < 2e-2 * gnr.item() and abs(fn1.item() - fnr.item()) < 2e-2 * fnr.item()


def test_chunked_graph_keeps_the_philox_step_counter():
    # 100 noisy iterations = chunks of 40 + 40 + 20: the step index of the Philox counter must continue across the
    # chunks (read from device memory), i.e. the replay equals the eager loop, and equals the oracle fed the same noise
    c = dict(dataset="svhn", nz=100, ngf=32, f_width=64, sigma=0.3, T=100)
    B = 8
    x_np, z0_np, _ = synth.inputs(B, 100, 3, 32, 1, seed=13)
    args, netG, netF = build_nets(c, DEV, seed=7)
    z0, x = torch.from_numpy(z0_np).to(DEV), torch.from_numpy(x_np).to(DEV)
    a, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=5, sample_offset=3)   # eager
    b, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=5, sample_offset=3)   # graphs
    assert torch.equal(a, b)
    eps = np.stack([philox.langevin_noise(5, 3, B, 100, t) for t in range(100)]).reshape(100, B, 100, 1, 1)
    zr, _, _ = oracle_langevin(c, x_np, z0_np, eps.astype(np.float32), seed=7)
    # a 100-step noisy chain amplifies rounding differences more than the 20/40-step configurations do
    assert rel_l2(b.cpu(), zr) < 3 * REL_TOL


def test_two_plans_on_two_streams_from_two_threads():
    # include/lsnf.h: distinct plans may be used concurrently from distinct threads / streams
    cs = [dict(dataset="svhn", nz=100, ngf=32, f_width=64, sigma=0.3, T=10),
          dict(dataset="cifar10", nz=128, ngf=64, f_width=64, sigma=0.3, T=10)]
    nets = [build_nets(c, DEV, seed=2) for c in cs]
    inputs = [synth.inputs(9, c["nz"], 3, 32, 1, seed=3) for c in cs]
    want = []
    for (args, netG, netF), (x_np, z0_np, _) in zip(nets, inputs):
        z, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(torch.from_numpy(z0_np).to(DEV), torch.from_numpy(x_np).to(DEV),
                                                             netG, netF, args, seed=1)
        want.append(z.cpu())
    got, errs = [None, None], []

    def work(i):
        try:
            args, netG, netF = nets[i]
            x_np, z0_np, _ = inputs[i]
            st = torch.cuda.Stream(device=DEV)
            with torch.cuda.stream(st):
                for _ in range(5):
                    z, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(
                        torch.from_numpy(z0_np).to(DEV), torch.from_numpy(x_np).to(DEV), netG, netF, args, seed=1)
                st.synchronize()
            got[i] = z.cpu()
        except Exception as e:   # pragma: no cover
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process():
    # per-device kernel attributes (opt-in shared memory) and SM counts live in the plan / are prepared per device
    c = dict(dataset="cifar10", nz=128, ngf=64, f_width=64, sigma=0.3, T=3)
    x_np, z0_np, _ = synth.inputs(20, 128, 3, 32, 1, seed=3)
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        args, netG, netF = build_nets(c, dev, seed=2)
        with torch.cuda.device(dev):
            z, _, _ = lsnf_b200.sample_langevin_post_z_with_flow(torch.from_numpy(z0_np).to(dev), torch.from_numpy(x_np).to(dev),
                                                                 netG, netF, args, seed=4)
        outs.append(z.cpu())
    assert torch.equal(outs[0], outs[1])


_PDL_SCRIPT = """
import sys, numpy as np, torch
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import lsnf_b200
from lsnf_b200 import synth
from helpers import build_nets
c = dict(dataset="svhn", nz=100, ngf=64, f_width=64, sigma=0.3, T=20)
x_np, z0_np, _ = synth.inputs(100, 100, 3, 32, 1, seed=21)
args, netG, netF = build_nets(c, "cuda:0", seed=3)
z0, x = torch.from_numpy(z0_np).to("cuda:0"), torch.from_numpy(x_np).to("cuda:0")
outs = [lsnf_b200.sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=9)[0].cpu().numpy() for _ in range(2)]
np.save({out!r}, np.stack(outs))   # [eager first call, graph replay]
"""


def test_programmatic_dependent_launch_changes_no_bit(tmp_path):
    # DESIGN.md 4.7: the kernels of the loop chain by programmatic dependent launch (LSNF_PDL=0 turns it off, read once
    # per process).  It moves launches and kernel set-up earlier and nothing else, so processes with it on (the
    # default) and off must produce the same bits -- at SVHN's true width and batch, where the loop mixes 1-CTA,
    # CTA-pair / stream-K and CUDA-core kernels, eagerly and from the replayed graph.
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    got = {}
    for mode in ("0", "1"):
        out = str(tmp_path / f"z_pdl{mode}.npy")
        env = dict(os.environ, LSNF_PDL=mode)
        subprocess.run([sys.executable, "-c", _PDL_SCRIPT.format(root=root, tests=os.path.join(root, "tests"), out=out)],
                       check=True, env=env, timeout=600)
        got[mode] = np.load(out)
        assert np.isfinite(got[mode]).all()
        assert np.array_equal(got[mode][0], got[mode][1])        # eager == replay within one process
    assert np.array_equal(got["0"], got["1"])
