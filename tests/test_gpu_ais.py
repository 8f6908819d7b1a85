"""Annealed importance sampling on the fused kernels (``lsnf_ais_run``, ``lsnf_b200.ais``) against the numpy restatement
in tests/ais_oracle.py, which runs over the reference's generator and flow prior (oracle/refpath.py)."""
import math

import numpy as np
import pytest
import torch

import ais_oracle as O
from helpers import build_nets, record, to_torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _fresh_plan(netG, netF, batch):
    import lsnf_b200
    p = lsnf_b200.Plan(arch=netG.dataset, batch=batch, nz=netG.nz, ngf=netG.ngf, nc=netG.nc, f_depth=netF.f_depth,
                       f_width=netF.f_width, f_permutation=netF.f_permutation, f_coupling=netF.f_coupling,
                       leak=netG.leak, device=DEV, gemm_impl=netG.gemm_impl, bwd_passes=3)
    p.ensure_generator(netG)
    p.ensure_flow(netF, need_inverse=True)
    return p


def _oracle_energy(c, x, sigma, mask=None):
    from lsnf_b200 import synth
    from oracle import refpath
    gp = to_torch(synth.generator_state(c["dataset"], c["nz"], c["ngf"], 3, seed=1))
    fp = to_torch(synth.flow_state(c["nz"], c.get("f_width", 64), 5, 1, 2, seed=1))
    layers = refpath.generator_layers(c["dataset"], c["nz"], c["ngf"])
    return O.refpath_energy(gp, fp, layers, x, sigma, mask, leak=c.get("leak", 0.2))


def _simulated(plan, netG, n, sigma, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    z = torch.randn(n, netG.nz, device=DEV, generator=g)
    x = plan.generator_forward(z) + sigma * torch.randn(n, netG.nc, plan.img, plan.img, device=DEV, generator=g)
    return z, x.contiguous()


def _block_mask(n, img):
    m = torch.ones(n, 3, img, img, device=DEV)
    m[:, :, img // 4: 3 * img // 4, img // 4: 3 * img // 4] = 0.0
    m[1::2, 1] *= 0.5
    return m


# ---- 1. T = 1: log w = l(z_0) exactly, whatever the transition does -----------------------------------------
@pytest.mark.parametrize("dataset", ["svhn", "cifar10"])
@pytest.mark.parametrize("masked", [False, True], ids=["unmasked", "block_mask"])
def test_one_step_log_w_is_the_reconstruction_log_likelihood(dataset, masked):
    c = dict(dataset=dataset, nz=100, ngf=32)
    _args, netG, netF = build_nets(c, DEV)
    B, sigma = 8, 0.3
    plan = _fresh_plan(netG, netF, B)
    g = torch.Generator(device=DEV).manual_seed(5)
    z0 = torch.randn(B, 100, device=DEV, generator=g)
    x = (torch.rand(B, 3, plan.img, plan.img, device=DEV, generator=g) * 2 - 1).contiguous()
    m = _block_mask(B, plan.img) if masked else None
    betas = torch.tensor([0.0, 1.0], device=DEV)
    _z, lw, _r = plan.ais_run(z0, x, betas, 1, 0.1, sigma, mask=m, seed=3)
    zr = O.round_hl(z0.cpu().numpy())
    want = _oracle_energy(c, x.cpu().numpy(), sigma, None if m is None else m.cpu().numpy())(zr)[0]
    got = lw.cpu().numpy().astype(np.float64)
    err = np.abs(got - want) / np.abs(want)
    record(f"ais_one_step_{dataset}_{'masked' if masked else 'unmasked'}.json", {"max_rel_err": float(err.max())})
    assert err.max() < 1e-5, err


# ---- 2 and 6. parity with the oracle's chains under injected noise ----------------------------------------
def _parity_case(schedule, target, seed):
    c = dict(dataset="svhn", nz=100, ngf=32, leak=1.0)   # kink-free generator: gradients agree element-wise
    _args, netG, netF = build_nets(c, DEV)
    N, T, sigma, s0 = 16, 20, 0.3, 0.8   # accepts 40-65 % of the oracle's proposals: both outcomes are checked
    plan = _fresh_plan(netG, netF, N)
    zt, x = _simulated(plan, netG, N, sigma, seed)
    r = np.random.default_rng(seed)
    eps = r.normal(size=(T, N, 100)).astype(np.float32)
    u = r.uniform(size=(T, N)).astype(np.float32)
    if schedule == "ones":
        betas = np.ones(T + 1, np.float32)
        z0 = zt + 0.05 * torch.randn(N, 100, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 1))
    else:
        betas = O.sigmoid_schedule(T).astype(np.float32)
        z0 = plan.flow_inverse(torch.randn(N, 100, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed)))[0]
    z, lw, rate = plan.ais_run(z0.contiguous(), x, torch.from_numpy(betas).to(DEV), T, s0, sigma, target_accept=target,
                               eps=torch.from_numpy(eps).to(DEV), u=torch.from_numpy(u).to(DEV))
    want = O.ais(z0.cpu().numpy(), _oracle_energy(c, x.cpu().numpy().astype(np.float64), sigma), betas, step_size=s0,
                 target_accept=target, eps=eps, u=u)
    keep = want["margin"] >= 1e-3
    acc = np.rint(rate.cpu().numpy() * T).astype(np.int64)
    lw_err = np.abs(lw.cpu().numpy() - want["logw"]) / np.maximum(np.abs(want["logw"]), 1e-30)
    z_err = np.linalg.norm(z.cpu().numpy() - want["z"], axis=1) / np.linalg.norm(want["z"], axis=1)
    rec = {"excluded": int((~keep).sum()), "accept_rate": float(want["accepts"].mean() / T),
           "max_rel_err_log_w": float(lw_err[keep].max()), "max_rel_l2_z_T": float(z_err[keep].max())}
    record(f"ais_parity_{schedule}_{'adaptive' if target else 'fixed'}.json", rec)
    assert (~keep).sum() <= 1, rec
    assert 0 < want["accepts"].sum() < N * T, rec   # both outcomes occur
    np.testing.assert_array_equal(acc[keep], want["accepts"][keep])
    if schedule != "ones":
        assert lw_err[keep].max() < 1e-5, rec
    assert z_err[keep].max() < 1e-4, rec


@pytest.mark.parametrize("target", [0.0, 0.65], ids=["fixed", "adaptive"])
def test_oracle_parity_forward_ais(target):
    _parity_case("sigmoid", target, 11)


def test_constant_schedule_is_the_oracles_mala_chain():
    _parity_case("ones", 0.0, 12)


# ---- 5. graph replay and isolation --------------------------------------------------------------------------
@pytest.fixture(scope="module")
def svhn_nets():
    return build_nets(dict(dataset="svhn", nz=100, ngf=32), DEV)


def _inputs(plan, n, T, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    z0 = torch.randn(n, 100, device=DEV, generator=g)
    x = (torch.rand(n, 3, plan.img, plan.img, device=DEV, generator=g) * 2 - 1).contiguous()
    betas = torch.from_numpy(O.sigmoid_schedule(T).astype(np.float32)).to(DEV)
    return z0, x, betas


def test_graph_replay_is_bit_identical_to_the_eager_run(svhn_nets):
    _a, netG, netF = svhn_nets
    T = 100   # 101 iterations: three graph chunks of at most 40
    plan = _fresh_plan(netG, netF, 8)
    z0, x, betas = _inputs(plan, 8, T, 1)
    eager = plan.ais_run(z0, x, betas, T, 0.05, 0.3, target_accept=0.65, seed=77, sample_offset=5)   # first call
    replay = plan.ais_run(z0, x, betas, T, 0.05, 0.3, target_accept=0.65, seed=77, sample_offset=5)
    again = plan.ais_run(z0, x, betas, T, 0.05, 0.3, target_accept=0.65, seed=77, sample_offset=5)
    for a, b, c in zip(eager, replay, again):
        assert torch.equal(a, b) and torch.equal(a, c)
    assert 0 < float(eager[2].mean()) < 1


def test_philox_noise_is_keyed_like_the_oracle(svhn_nets):
    from oracle.philox import langevin_noise
    _a, netG, netF = svhn_nets
    T, n, seed, off = 3, 8, 1234, 40
    plan = _fresh_plan(netG, netF, n)
    z0, x, betas = _inputs(plan, n, T, 2)
    philox = plan.ais_run(z0, x, betas, T, 0.05, 0.3, seed=seed, sample_offset=off)
    eps = np.stack([langevin_noise(seed, off, n, 100, k) for k in range(T)])
    u = np.stack([O.philox_uniform(seed, off, n, k) for k in range(1, T + 1)])
    inj = plan.ais_run(z0, x, betas, T, 0.05, 0.3, eps=torch.from_numpy(eps).to(DEV), u=torch.from_numpy(u).to(DEV))
    for a, b in zip(philox, inj):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6)


def test_replay_sees_new_schedule_x_and_mask(svhn_nets):
    _a, netG, netF = svhn_nets
    T, n = 30, 8
    plan = _fresh_plan(netG, netF, n)
    z0, x, betas = _inputs(plan, n, T, 3)
    m = _block_mask(n, plan.img)
    plan.ais_run(z0, x, betas, T, 0.05, 0.3, mask=m, seed=9)          # eager
    plan.ais_run(z0, x, betas, T, 0.05, 0.3, mask=m, seed=9)          # captures the masked graph
    x2 = (x * 0.5).contiguous()
    b2 = torch.from_numpy(np.linspace(0, 1, T + 1).astype(np.float32) ** 2).to(DEV)
    m2 = torch.flip(m, [0]).contiguous()
    got = plan.ais_run(z0, x2, b2, T, 0.05, 0.3, mask=m2, seed=9)      # replay with new values
    ref = _fresh_plan(netG, netF, n).ais_run(z0, x2, b2, T, 0.05, 0.3, mask=m2, seed=9)   # eager on a fresh plan
    for a, b in zip(got, ref):
        assert torch.equal(a, b)


def test_all_ones_mask_is_bit_identical_to_no_mask(svhn_nets):
    _a, netG, netF = svhn_nets
    T, n = 10, 8
    plan = _fresh_plan(netG, netF, n)
    z0, x, betas = _inputs(plan, n, T, 4)
    a = plan.ais_run(z0, x, betas, T, 0.05, 0.3, seed=2)
    b = plan.ais_run(z0, x, betas, T, 0.05, 0.3, seed=2, mask=torch.ones(1, 1, 1, 1, device=DEV))
    for p, q in zip(a, b):
        assert torch.equal(p, q)


def test_langevin_after_ais_is_unchanged(svhn_nets):
    _a, netG, netF = svhn_nets
    n = 8
    plan = _fresh_plan(netG, netF, n)
    z0, x, betas = _inputs(plan, n, 50, 5)
    plan.langevin_run(z0, x, 20, 0.1, 0.3, seed=4)                   # eager
    plan.langevin_run(z0, x, 20, 0.1, 0.3, seed=4)                   # graph
    plan.ais_run(z0, x, betas, 50, 0.05, 0.3, seed=4)
    plan.ais_run(z0, x, betas, 50, 0.05, 0.3, seed=4)
    got = plan.langevin_run(z0, x, 20, 0.1, 0.3, seed=4)
    fresh = _fresh_plan(netG, netF, n)
    want = fresh.langevin_run(z0, x, 20, 0.1, 0.3, seed=4)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert plan.launch_count(20) == fresh.launch_count(20)


# ---- 3. small latent: AIS against prior importance sampling ----------------------------------------------------
def test_small_latent_ais_agrees_with_prior_importance_sampling():
    import lsnf_b200
    c = dict(dataset="svhn", nz=4, ngf=32, leak=1.0, sigma=1.0)
    args, netG, netF = build_nets(c, DEV)
    n_img, sigma = 2, 1.0
    sim = _fresh_plan(netG, netF, n_img)
    _z, x = _simulated(sim, netG, n_img, sigma, 21)
    # 512 chains: the Monte-Carlo error of the AIS estimate itself stays well below the 0.02-nat allowance
    log_px, lw, rate = lsnf_b200.ais_log_likelihood(x, netG, netF, args, chains=512, steps=1000, seed=3)
    # prior importance sampling: 2^20 draws per image through flow_inverse + generator_forward
    chunk = 1 << 15
    big = _fresh_plan(netG, netF, chunk)
    g = torch.Generator(device=DEV).manual_seed(8)
    D = 3 * 32 * 32
    C = -0.5 * D * math.log(2 * math.pi * sigma ** 2)
    res = []
    for i in range(n_img):
        ells = []
        for _ in range((1 << 20) // chunk):
            z = big.flow_inverse(torch.randn(chunk, 4, device=DEV, generator=g))[0]
            d = big.generator_forward(z) - x[i:i + 1]
            ells.append(-(d.double() ** 2).flatten(1).sum(1) / (2 * sigma ** 2))
        ell = torch.cat(ells)
        mx = ell.max()
        w = torch.exp(ell - mx)
        est = float(mx + torch.log(w.mean())) + C
        se = float(w.std() / w.mean()) / math.sqrt(w.numel())
        res.append({"is": est, "is_se": se, "ais": float(log_px[i]), "ais_log_w_std": float(lw[i].double().std()),
                    "accept": float(rate[i].mean())})
    record("ais_small_latent.json", res)
    for r in res:
        assert abs(r["ais"] - r["is"]) < 3 * r["is_se"] + 0.02, res


# ---- 4. BDMC sandwich at a true width -------------------------------------------------------------------------
def test_bdmc_sandwich_svhn():
    import lsnf_b200
    c = dict(dataset="svhn", nz=100, ngf=64)
    args, netG, netF = build_nets(c, DEV)
    out = {}
    for T in (200, 2000):
        lo, hi, _x = lsnf_b200.bdmc(netG, netF, args, 8, chains=8, steps=T, step_size=0.02, seed=17)
        out[T] = {"lower": lo.tolist(), "upper": hi.tolist(), "mean_gap": float((hi - lo).mean())}
        assert float(lo.mean()) <= float(hi.mean()) + 0.5, out
    record("ais_bdmc_svhn.json", {"config": dict(c, chains=8, images=8, sigma=0.3, step_size=0.02, target_accept=0.65),
                                  "by_steps": {str(k): v for k, v in out.items()}})
    assert out[2000]["mean_gap"] < out[200]["mean_gap"], out
