"""The oracle restatement against the fixtures written from the reference's own modules
(oracle/make_golden.py), and -- when LSNF_REFERENCE names a checkout of the reference -- against the reference live."""
import os
import sys

import numpy as np
import pytest
import torch

import lsnf_b200.synth as synth
from oracle import philox, refpath
from helpers import load_golden, rel_err, to_torch

CASES = ["svhn_small", "cifar_small", "celeba_small", "svhn_additive", "hq_flow_w128"]


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_fixture(name):
    g = load_golden(name)
    c = g["config"]
    fsd = synth.flow_state(c["nz"], c["f_width"], 5, c["coupling"], 2, seed=1)
    np.testing.assert_allclose(synth.checksum(fsd), g["f_checksum"], rtol=1e-12)
    fp = to_torch(fsd)
    B, nz = c["B"], c["nz"]
    z0 = torch.from_numpy(g["z0"])
    ll, z1, ld, gf = refpath.prior_grad(z0.reshape(B, nz), fp, 5, c["coupling"])
    assert rel_err(z1, g["flow_z1"]) < 1e-6
    assert rel_err(ld, g["flow_logdet"]) < 1e-6
    assert rel_err(ll, g["flow_ll"]) < 1e-6
    assert rel_err(gf, g["flow_grad"]) < 1e-5
    e = torch.from_numpy(g["eps"][0].reshape(B, nz))
    zi, obj = refpath.flow_reverse(fp, e, torch.zeros(B), 5, c["coupling"])
    assert rel_err(zi, g["flow_inv_z"]) < 1e-5
    assert rel_err(-obj, g["flow_inv_negobj"]) < 1e-5
    if not c["dataset"]:
        return
    gsd = synth.generator_state(c["dataset"], nz, c["ngf"], 3, seed=1)
    np.testing.assert_allclose(synth.checksum(gsd), g["g_checksum"], rtol=1e-12)
    gp = to_torch(gsd)
    layers = refpath.generator_layers(c["dataset"], nz, c["ngf"], 3)
    x = torch.from_numpy(g["x"])
    xh, gg = refpath.recon_grad(z0, x, gp, layers, c["sigma"])
    assert rel_err(xh, g["x_hat"]) < 1e-6
    assert rel_err(gg, g["grad_g"]) < 1e-5
    zT, gn, fn = refpath.langevin(z0, x, gp, fp, layers, depth=5, steps=c["T"], step_size=0.1, sigma=c["sigma"],
                                  eps=torch.from_numpy(g["eps"]), coupling=c["coupling"])
    assert rel_err(zT, g["z_T"]) < 1e-5
    assert abs(gn.item() - g["gnorm_g"]) / g["gnorm_g"] < 1e-5
    assert abs(fn.item() - g["gnorm_f"]) / g["gnorm_f"] < 1e-5
    zN, _, _ = refpath.langevin(z0, x, gp, fp, layers, depth=5, steps=c["T"], step_size=0.1, sigma=c["sigma"],
                                eps=None, coupling=c["coupling"])
    assert rel_err(zN, g["z_T_nonoise"]) < 1e-5
    # the reference's own fp32 error budget against fp64 truth stays far inside the parity tolerance
    assert rel_err(g["z_T"], g["z_T_fp64"]) < 1e-5


@pytest.mark.parametrize("name", CASES)
def test_oracle_forward_passes_match_the_reference_outputs(name):
    # test_oracle_matches_reference_live's comparison against the reference's outputs stored in the fixtures:
    # generator_forward against its netG(z), flow_forward against its netF(z) (z1, log-det)
    g = load_golden(name)
    c = g["config"]
    B, nz = c["B"], c["nz"]
    z = torch.from_numpy(g["z0"])
    z1, ld = refpath.flow_forward(to_torch(synth.flow_state(nz, c["f_width"], 5, c["coupling"], 2, seed=1)),
                                  z.reshape(B, nz), torch.zeros(B), 5, c["coupling"])
    assert rel_err(z1, g["flow_z1"]) < 1e-6 and rel_err(ld, g["flow_logdet"]) < 1e-6
    if c["dataset"]:
        gp = to_torch(synth.generator_state(c["dataset"], nz, c["ngf"], 3, seed=1))
        xh = refpath.generator_forward(gp, z, refpath.generator_layers(c["dataset"], nz, c["ngf"], 3))
        assert rel_err(xh, g["x_hat"]) < 1e-6


def test_parameter_updates_match_the_reference_training_iterations_fixture():
    # two whole training iterations of train.py:384-415 run on the reference's own modules + torch Adam
    # (oracle/make_golden.py: training_iteration_case): refpath.langevin + refpath.parameter_updates must land on the
    # same losses and the same parameters
    from oracle.make_golden import TRAIN_CASE as c, TRAIN_KEEP
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "train_update_svhn_small.npz"))
    gsd = synth.generator_state(c["dataset"], c["nz"], c["ngf"], 3, seed=1)
    fsd = synth.flow_state(c["nz"], c["f_width"], 5, c["coupling"], 2, seed=1)
    gp = {k: v.clone().requires_grad_(True) for k, v in to_torch(gsd).items()}
    fp = to_torch(fsd)
    fkeys = refpath.trainable_flow_keys(fp)
    assert len(fkeys) == 60                        # 12 trainable tensors per step that receive a gradient
    for k in fkeys:
        fp[k] = fp[k].clone().requires_grad_(True)
    adam = lambda ps: torch.optim.Adam(ps, lr=c["lr"], weight_decay=0, betas=(0.5, 0.999))
    optG, optF = adam(list(gp.values())), adam([fp[k] for k in fkeys])
    layers = refpath.generator_layers(c["dataset"], c["nz"], c["ngf"], 3)
    for it in range(c["iters"]):
        x_np, z0_np, eps_np = synth.inputs(c["B"], c["nz"], 3, 32, c["T"], seed=100 + it)
        x, z0, eps = torch.from_numpy(x_np), torch.from_numpy(z0_np), torch.from_numpy(eps_np)
        zk, _, _ = refpath.langevin(z0, x, {k: v.detach() for k, v in gp.items()}, {k: v.detach() for k, v in fp.items()},
                                    layers, depth=5, steps=c["T"], step_size=0.1, sigma=c["sigma"], eps=eps)
        lg, lf = refpath.parameter_updates(gp, fp, zk, x, layers, optG, optF, depth=5)
        assert abs(lg.item() - g["losses"][it][0]) < 1e-5 * abs(g["losses"][it][0])
        assert abs(lf.item() - g["losses"][it][1]) < 1e-5 * abs(g["losses"][it][1])
    # Adam moves every element by ~lr per step whatever the size of its gradient, so an element whose gradient is
    # within rounding of zero may land one update away on another CPU: bound the outliers, compare the bulk tightly
    lr, n_it = c["lr"], c["iters"]
    for k in TRAIN_KEEP:
        got = (gp[k] if k in gp else fp[k]).detach()
        want = torch.from_numpy(g["after:" + k])
        d = (got - want).abs()
        assert float(d.max()) <= 2.5 * lr * n_it, k
        assert float((d > 1e-6).float().mean()) < 2e-3, k
    after_g = synth.checksum({k: v.detach().numpy() for k, v in gp.items()})
    np.testing.assert_allclose(after_g, g["g_checksum_after"], rtol=1e-5)
    start = to_torch(gsd)
    assert max(float((gp[k].detach() - start[k]).abs().max()) for k in gp) > 0.5 * lr      # the parameters did move


def test_analytic_prior_gradient_matches_autograd_fp64():
    fsd = synth.flow_state(100, 64, 5, 1, 2, seed=3)
    rng = np.random.default_rng(0)
    z = rng.standard_normal((9, 100))
    ga = refpath.prior_grad_analytic(z, fsd, 5, 1)
    _, _, _, g = refpath.prior_grad(torch.from_numpy(z), to_torch(fsd, torch.float64), 5, 1)
    assert rel_err(ga, g) < 1e-10


def test_flow_inverse_roundtrip_and_fresh_logdet():
    # SURVEY.md section 4: F^-1(F(z)) == z; a fresh (unperturbed) flow has a sample-independent log-det
    fsd = synth.flow_state(100, 64, 5, 1, 2, seed=1, perturb=0.0)
    fp = to_torch(fsd, torch.float64)
    z = torch.randn(11, 100, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    y, ld = refpath.flow_forward(fp, z, torch.zeros(11, dtype=torch.float64), 5)
    zr, ld2 = refpath.flow_reverse(fp, y, ld, 5)
    assert rel_err(zr, z) < 1e-11 and float(ld2.abs().max()) < 1e-10
    sig2 = float(np.log(1.0 / (1.0 + np.exp(-2.0))))
    expect = 5 * 50 * sig2 + sum(3.0 * float(fsd[f"revnet2d_s.0.revnet2d_step_s.{i}.actnorm.logs"].astype(np.float64).sum())
                                 for i in range(5))
    assert float((ld - expect).abs().max()) < 1e-4  # |log-abs-det W| ~ 1e-6 for the fp32 QR factor


def test_state_dict_key_inventory():
    k = np.load(os.path.join(os.path.dirname(__file__), "golden", "state_dict_keys.npz"))
    assert len(k["flow_nz100_w64"]) == 85
    assert sorted(synth.flow_state(100).keys()) == sorted(str(s) for s in k["flow_nz100_w64"])
    for ds in ("svhn", "cifar10", "celeba_crop", "celeba_hq256"):
        mine = [f"{n}:{tuple(v.shape)}" for n, v in synth.generator_state(ds, 100, 8).items()]
        assert mine == [str(s) for s in k["gen_" + ds]]


REFERENCE = os.environ.get("LSNF_REFERENCE")


@pytest.mark.skipif(not (REFERENCE and os.path.exists(os.path.join(REFERENCE, "model.py"))),
                    reason="LSNF_REFERENCE does not name a checkout of the reference")
def test_oracle_matches_reference_live():
    sys.path.insert(0, REFERENCE)
    import model as ref_model
    sys.path.pop(0)
    from oracle.make_golden import ref_args
    c = dict(dataset="svhn", nz=100, ngf=16, f_width=64, coupling=1)
    fsd = synth.flow_state(100, 64, 5, 1, 2, seed=7)
    gsd = synth.generator_state("svhn", 100, 16, 3, seed=7)
    netF = ref_model._netF(ref_args(c), nz=100)
    netF.load_state_dict(to_torch(fsd))
    netG = ref_model._netG(ref_args(c))
    netG.load_state_dict(to_torch(gsd))
    z = torch.randn(4, 100, 1, 1, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        assert rel_err(refpath.generator_forward(to_torch(gsd), z, refpath.generator_layers("svhn", 100, 16)), netG(z)) < 1e-6
        a, b = refpath.flow_forward(to_torch(fsd), z.reshape(4, 100), torch.zeros(4), 5)
        ra, rb, _ = netF(z.reshape(4, 100), torch.zeros(4))
        assert rel_err(a, ra) < 1e-6 and rel_err(b, rb) < 1e-6


def test_philox_known_answers():
    # Random123 known-answer vectors for philox4x32-10
    kat = [
        ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
        ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
        ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
         [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
    ]
    for ctr, key, want in kat:
        got = philox.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))
        assert [int(v) for v in got] == want


def test_philox_noise_is_standard_normal_and_shard_invariant():
    n = philox.langevin_noise(seed=1, sample0=0, batch=4096, nz=100, step=3)
    assert abs(float(n.mean())) < 0.01 and abs(float(n.std()) - 1.0) < 0.01
    part = philox.langevin_noise(seed=1, sample0=1000, batch=10, nz=100, step=3)
    assert np.array_equal(part, n[1000:1010])
    assert not np.array_equal(n, philox.langevin_noise(seed=1, sample0=0, batch=4096, nz=100, step=4))
