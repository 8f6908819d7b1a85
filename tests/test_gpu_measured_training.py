"""Training from linear measurements y = A vec(G(z)) + sigma noise on the fused kernels
(``lsnf_generator_param_grads_measured`` through ``generator_gradients`` / ``generator_update`` /
``training_iteration`` with ``operator=``): the generator's parameter gradients and loss_g = |A vec(G(z)) - y|^2 / B
against fp64 autograd on the oracle's generator, against the masked update for the identity rows of a mask, against
the reference's loss written with ``A`` under ``kernel_autograd()``, in rescaled units, across call orders, and the
update and the whole training iteration against torch Adam on the measured oracle (tests/measured_training_oracle.py).
The worst error of every case is recorded as JSON (helpers.record)."""
import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import synth
from oracle import philox, refpath
import measured_oracle as MO
import measured_training_oracle as MTO
from helpers import REL_TOL, build_nets, record, rel_l2, to_torch
from test_gpu_param_updates import _param_keys, assert_params_close, assert_updates_agree

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SVHN = dict(dataset="svhn", nz=100, ngf=64)
CIFAR = dict(dataset="cifar10", nz=128, ngf=128)
CELEBA = dict(dataset="celeba_crop", nz=100, ngf=64)
WORST = {}


def _note(case, value):
    WORST[case] = float(value)
    record("r12_measured_training_worst_errors.json", WORST)


def _operator(kind, img, seed=0, frac=8):
    n = 3 * img * img
    if kind == "gaussian":
        return MO.gaussian_operator(n // frac, n, seed)
    return MO.avg_pool_operator(3, img)


def _problem(c, B, op, seed, frac=8, m=None):
    """(z [B,nz,1,1], y [B,m], A [m,n]) as CPU tensors: y = A vec(x) + 0.05 noise."""
    img = synth.image_size(c["dataset"])
    x_np, z_np, _ = synth.inputs(B, c["nz"], 3, img, 1, seed=seed)
    n = 3 * img * img
    A = MO.gaussian_operator(m, n, seed + 1) if m is not None else _operator(op, img, seed + 1, frac)
    y = x_np.reshape(B, -1) @ A.T
    y = (y + 0.05 * np.random.default_rng(seed + 2).standard_normal(y.shape)).astype(np.float32)
    return torch.from_numpy(z_np).reshape(B, c["nz"], 1, 1), torch.from_numpy(y), torch.from_numpy(A)


def _fused(netG, z, y, A, B, **kw):
    """(loss_g, {state_dict key: gradient}) of the fused measured update, copied out of the plan's buffer."""
    flat, pairs, loss = lsnf_b200.generator_gradients(netG, z.to(DEV), y.to(DEV), B, operator=A.to(DEV), **kw)
    names = {id(p): k for k, p in netG.named_parameters()}
    return loss.item(), {names[id(p)]: g.detach().clone().cpu() for p, g in pairs}


def _fp64(c, seed, z, y, A, leak):
    """(loss_g, {key: gradient}) by fp64 autograd on the oracle's generator (on the GPU, in fp64)."""
    gp = to_torch(synth.generator_state(c["dataset"], c["nz"], c["ngf"], 3, seed=seed), dtype=torch.float64, device=DEV)
    leaves = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    layers = refpath.generator_layers(c["dataset"], c["nz"], c["ngf"])
    loss = MTO.generator_loss(leaves, z.to(DEV), y.to(DEV), A.to(DEV), layers, leak)
    loss.backward()
    return loss.item(), {k: v.grad.cpu() for k, v in leaves.items()}


def _compare(case, got, want, tol=REL_TOL):
    (lg, gg), (lw, gw) = got, want
    le = abs(lg - lw) / abs(lw)
    errs = {k: rel_l2(gg[k].double(), gw[k].double()) for k in gw}
    _note(f"{case}_loss_rel", le)
    _note(f"{case}_worst_grad_rel_l2", max(errs.values()))
    assert le < tol, (case, le)
    for k, e in errs.items():
        assert e < tol, (case, k, e)


# ---- 1. gradients against fp64 autograd ------------------------------------------------------------------------------
@pytest.mark.parametrize("c,op,frac", [(SVHN, "gaussian", 8), (SVHN, "avgpool", 4), (CIFAR, "gaussian", 8),
                                       (CIFAR, "avgpool", 4), (CELEBA, "gaussian", 16)],
                         ids=["svhn_gaussian", "svhn_avgpool", "cifar10_gaussian", "cifar10_avgpool",
                              "celeba_crop_gaussian_n16"])
def test_measured_parameter_gradients_match_fp64_autograd(c, op, frac):
    c = dict(c, leak=1.0)           # kink-free generator: element-wise agreement is meaningful
    B = 100
    args, netG, netF = build_nets(c, DEV, seed=4)
    z, y, A = _problem(c, B, op, seed=9, frac=frac)
    _compare(f"grads_{c['dataset']}_{op}", _fused(netG, z, y, A, B), _fp64(c, 4, z, y, A, 1.0))


# ---- 2. ragged operator and batch -------------------------------------------------------------------------------------
def test_ragged_operator_and_two_tile_batch_match_fp64_autograd():
    c = dict(SVHN, leak=1.0)
    B = 129                          # two M tiles; the weight-gradient transposes at a ragged batch
    args, netG, netF = build_nets(c, DEV, seed=5)
    z, y, A = _problem(c, B, None, seed=11, m=257)
    _compare("grads_svhn_m257_B129", _fused(netG, z, y, A, B), _fp64(c, 5, z, y, A, 1.0))


# ---- 3. identity rows of a mask against the masked update -------------------------------------------------------------
def test_identity_rows_match_the_masked_generator_gradients():
    c = dict(SVHN, leak=0.2)
    B = 100
    args, netG, netF = build_nets(c, DEV, seed=6)
    x_np, z_np, _ = synth.inputs(B, 100, 3, 32, 1, seed=13)
    mask = np.ones((3, 32, 32), np.float32)
    mask[:, 6:22, 9:27] = 0.0
    mask[0, ::2] = 0.0
    A = torch.from_numpy(MO.identity_rows(mask))
    x = torch.from_numpy(x_np)
    y = x.reshape(B, -1)[:, torch.from_numpy(mask.reshape(-1) > 0)].contiguous()
    z = torch.from_numpy(z_np).reshape(B, 100, 1, 1)
    got = _fused(netG, z, y, A, B)
    flat, pairs, loss = lsnf_b200.generator_gradients(netG, z.to(DEV), x.to(DEV), B,
                                                      mask=torch.from_numpy(mask).to(DEV).expand(B, 3, 32, 32))
    names = {id(p): k for k, p in netG.named_parameters()}
    want = (loss.item(), {names[id(p)]: g.detach().clone().cpu() for p, g in pairs})
    _compare("identity_rows_vs_mask", got, want, tol=2e-5)


# ---- 4. against the reference's loss under kernel_autograd() --------------------------------------------------------
@pytest.mark.parametrize("c", [SVHN, CIFAR], ids=["svhn", "cifar10"])
def test_measured_gradients_agree_with_the_reference_loss_under_kernel_autograd(c):
    c = dict(c, leak=1.0)
    B = 100
    args, netG, netF = build_nets(c, DEV, seed=7)
    z, y, A = _problem(c, B, "gaussian", seed=15)
    got = _fused(netG, z, y, A, B)
    zd, yd, Ad = z.to(DEV), y.to(DEV), A.to(DEV)
    netG.train()                     # train.py:390-394 runs in training mode: netG(z_k) records the parameters' graph
    netG.zero_grad(set_to_none=True)
    with lsnf_b200.kernel_autograd():
        loss_g = ((netG(zd).view(B, -1) @ Ad.t() - yd) ** 2).sum() / B
        loss_g.backward()
    want = (loss_g.item(), {k: p.grad.detach().clone().cpu() for k, p in netG.named_parameters()})
    netG.zero_grad(set_to_none=True)
    _compare(f"kernel_autograd_{c['dataset']}", got, want)


# ---- 5. units -----------------------------------------------------------------------------------------------------------
def test_rescaled_operator_and_measurements_scale_loss_and_gradients_exactly():
    c = dict(SVHN, leak=1.0)
    B = 100
    args, netG, netF = build_nets(c, DEV, seed=8)
    z, y, A = _problem(c, B, "gaussian", seed=17)
    l0, g0 = _fused(netG, z, y, A, B)
    for j in (-8, -3, 5, 8):
        s = 2.0 ** j
        lj, gj = _fused(netG, z, y * s, A * s, B)
        assert lj == l0 * s * s, j
        for k in g0:
            assert torch.equal(gj[k], g0[k] * (s * s)), (j, k)
    ref = _fp64(c, 8, z, y, A, 1.0)
    worst = 0.0
    for j in (-32, -20, 20, 32):
        s = 2.0 ** j
        lj, gj = _fused(netG, z, y * s, A * s, B)
        assert np.isfinite(lj) and all(torch.isfinite(g).all() for g in gj.values()), j
        scaled = (lj / (s * s), {k: v.double() / (s * s) for k, v in gj.items()})
        _compare(f"units_2^{j}", scaled, ref)
        worst = max(worst, WORST[f"units_2^{j}_worst_grad_rel_l2"])
    _note("units_worst_grad_rel_l2", worst)


# ---- 6. determinism and state -------------------------------------------------------------------------------------------
def _train_plan(netG, netF, B, m):
    """The plan a measured ``training_iteration`` runs on."""
    p = lsnf_b200.langevin_plan(netG, netF, B, torch.device(DEV), bwd_passes=3, train=True, meas_rows=m)
    p.ensure_generator(netG)
    p.ensure_flow(netF)
    return p


def test_split_calls_repeats_and_interleaved_calls_are_bit_identical():
    c = dict(SVHN, leak=0.2, f_width=64)
    B = 100
    args, netG, netF = build_nets(c, DEV, seed=9)
    z, y, A = _problem(c, B, "gaussian", seed=19)
    x_np, _, _ = synth.inputs(B, 100, 3, 32, 1, seed=19)
    zd, yd, Ad, xd = z.reshape(B, 100).to(DEV), y.to(DEV), A.to(DEV), torch.from_numpy(x_np).to(DEV)
    plan = _train_plan(netG, netF, B, A.shape[0])
    plan.ensure_operator(Ad)
    L = len(plan.generator_grad_layout()) // 2

    def whole():
        flat, loss = plan.generator_param_grads_measured(zd, yd, B)
        return flat.clone(), loss.clone()

    def split():
        flat = torch.zeros_like(ref[0])
        flat, loss = plan.generator_param_grads_measured(zd, yd, B, flat, part=-2)
        for l in reversed(range(L)):
            plan.generator_param_grads_measured(zd, yd, B, flat, part=l, loss=loss)
        return flat.clone(), loss.clone()

    def unmeasured():
        flat, loss = plan.generator_param_grads(zd, xd, B)
        return flat.clone(), loss.clone()

    ref = whole()
    ref_u = unmeasured()
    same = lambda a, b: torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert same(whole(), ref) and same(split(), ref) and same(whole(), ref)
    # an unmeasured update and a measured Langevin call on the same plan leave the e4m3 amax words, the gradient
    # state and the workspace copy of y as the measured update expects them
    assert same(unmeasured(), ref_u)
    assert same(whole(), ref)
    plan.langevin_run_measured(zd, yd * 3.0, 5, 0.1, 0.3, seed=3)
    plan.langevin_run_measured(zd, yd * 3.0, 5, 0.1, 0.3, seed=4)    # a graph replay: y copied into the workspace
    assert same(whole(), ref) and same(unmeasured(), ref_u) and same(split(), ref)
    # layer calls need the measured prologue: right after a re-pack, and after the unmeasured prologue, they fail
    plan.invalidate()
    plan.ensure_generator(netG)
    with pytest.raises(RuntimeError, match=r"\(-3\)"):
        plan.generator_param_grads_measured(zd, yd, B, ref[0].clone(), part=0)
    plan.generator_param_grads(zd, xd, B, ref_u[0].clone(), part=-2)
    with pytest.raises(RuntimeError, match=r"\(-3\)"):
        plan.generator_param_grads_measured(zd, yd, B, ref[0].clone(), part=L - 1)
    plan.generator_param_grads_measured(zd, yd, B, ref[0].clone(), part=-2)
    with pytest.raises(RuntimeError, match=r"\(-3\)"):
        plan.generator_param_grads(zd, xd, B, ref_u[0].clone(), part=L - 1)
    assert same(whole(), ref)


# ---- 7. generator_update(operator=) against torch Adam -----------------------------------------------------------------
@pytest.mark.parametrize("leak", [1.0, 0.2])
def test_measured_generator_update_matches_torch_adam(leak):
    c = dict(SVHN, leak=leak)
    B, lr = 100, 0.0004
    args, netG, netF = build_nets(c, DEV, seed=6)
    netG.train()
    optG, _ = lsnf_b200.make_optimizers(netG, netF, args)
    gp = to_torch(synth.generator_state("svhn", 100, 64, 3, seed=6))
    start = {k: v.clone() for k, v in gp.items()}
    leaves = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    ref_opt = torch.optim.Adam(list(leaves.values()), lr=lr, betas=(0.5, 0.999))
    layers = refpath.generator_layers("svhn", 100, 64)
    A = torch.from_numpy(_operator("gaussian", 32, seed=3))
    Ad = A.to(DEV)
    for it in range(3):
        x_np, z_np, _ = synth.inputs(B, 100, 3, 32, 1, seed=50 + it)
        z = torch.from_numpy(z_np).reshape(B, 100, 1, 1)
        y = (torch.from_numpy(x_np).reshape(B, -1) @ A.t()).contiguous()
        loss = lsnf_b200.generator_update(netG, optG, z.to(DEV), y.to(DEV), args, operator=Ad)
        ref_opt.zero_grad()
        want = MTO.generator_loss(leaves, z, y, A, layers, leak)
        want.backward()
        ref_opt.step()
        assert abs(loss.item() - want.item()) < 1e-3 * want.item()
    named = dict(netG.named_parameters())
    for k in leaves:
        assert_updates_agree(named[k].detach().cpu(), leaves[k].detach(), start[k], lr, 3, k, strict=(leak == 1.0))


# ---- 8. training_iteration(operator=) against the measured oracle ------------------------------------------------------
@pytest.mark.parametrize("leak", [1.0, 0.2])
def test_measured_training_iteration_matches_the_oracle(leak):
    c = dict(SVHN, T=20, sigma=0.3, leak=leak)
    B, lr, T = 100, 0.0004, 20
    args, netG, netF = build_nets(c, DEV, seed=2)
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)
    x_np, z0_np, _ = synth.inputs(B, 100, 3, 32, 1, seed=77)
    A = torch.from_numpy(_operator("gaussian", 32, seed=5))
    y = (torch.from_numpy(x_np).reshape(B, -1) @ A.t()
         + 0.05 * torch.from_numpy(np.random.default_rng(78).standard_normal((B, A.shape[0])).astype(np.float32)))
    seed = 0xABD
    eps = np.stack([philox.langevin_noise(seed, 0, B, 100, t) for t in range(T)]).reshape(T, B, 100, 1, 1)
    lg, lf, gn, fn, zk = lsnf_b200.training_iteration(y.to(DEV), netG, netF, optG, optF, args, seed=seed,
                                                      z0=torch.from_numpy(z0_np).to(DEV), operator=A.to(DEV))
    g0 = to_torch(synth.generator_state("svhn", 100, 64, 3, seed=2))
    gp = {k: v.clone().requires_grad_(True) for k, v in g0.items()}
    fsd = synth.flow_state(100, 64, 5, 1, 2, seed=2)
    fkeys = _param_keys(fsd)
    fp = {k: torch.from_numpy(np.ascontiguousarray(v)).clone() for k, v in fsd.items()}
    fleaves = {k: fp[k].requires_grad_(True) for k in fkeys}
    layers = refpath.generator_layers("svhn", 100, 64)
    z_ref, _, _ = MO.langevin(torch.from_numpy(z0_np), y, A, {k: v.detach() for k, v in gp.items()},
                              {k: v.detach() for k, v in fp.items()}, layers, depth=5, steps=T, step_size=0.1,
                              sigma=0.3, eps=torch.from_numpy(eps.astype(np.float32)), leak=leak)
    ez = rel_l2(zk.cpu(), z_ref)
    _note(f"training_iteration_leak{leak}_zT_rel_l2", ez)
    assert ez < REL_TOL
    og = torch.optim.Adam(list(gp.values()), lr=lr, betas=(0.5, 0.999))
    of = torch.optim.Adam(list(fleaves.values()), lr=lr, betas=(0.5, 0.999))
    loss_g, loss_f = MTO.parameter_updates(gp, fp, z_ref, y, A, layers, og, of, depth=5, leak=leak)
    _note(f"training_iteration_leak{leak}_loss_g", lg.item())
    _note(f"training_iteration_leak{leak}_loss_g_oracle", loss_g.item())
    _note(f"training_iteration_leak{leak}_loss_g_rel", abs(lg.item() - loss_g.item()) / loss_g.item())
    _note(f"training_iteration_leak{leak}_loss_f_rel", abs(lf.item() - loss_f.item()) / abs(loss_f.item()))
    assert abs(lg.item() - loss_g.item()) < 1e-3 * loss_g.item()
    assert abs(lf.item() - loss_f.item()) < 1e-3 * abs(loss_f.item())
    ng, nf = dict(netG.named_parameters()), dict(netF.named_parameters())
    for k in gp:
        assert_updates_agree(ng[k].detach().cpu(), gp[k].detach(), g0[k], lr, 1, k, strict=(leak == 1.0))
    for k in fkeys:
        assert_params_close(nf[k].detach().cpu(), fp[k].detach(), lr, 1, k)


# ---- 9. error codes of the entry point on a bound plan ------------------------------------------------------------------
def test_error_codes_of_the_measured_parameter_gradients():
    c = dict(SVHN, leak=0.2)
    B, m = 8, 96
    args, netG, netF = build_nets(c, DEV, seed=1)
    n = 3 * 32 * 32
    A = torch.from_numpy(MO.gaussian_operator(m, n, 1)).to(DEV)
    z = torch.zeros(B, 100, device=DEV)
    y = torch.zeros(B, m, device=DEV)

    def plan(**kw):
        cfg = dict(train=True, meas_rows=m, bwd_passes=3)
        cfg.update(kw)
        p = lsnf_b200.Plan(arch="svhn", batch=B, nz=100, ngf=64, nc=3, f_depth=5, f_width=64, f_permutation=2,
                           f_coupling=1, leak=0.2, device=DEV, **cfg)
        p.ensure_generator(netG)
        return p

    def call(p, part=-1):
        flat = torch.zeros(max(1, int(p.lib.lsnf_generator_grad_floats(p.handle))), device=DEV)
        rc = p.lib.lsnf_generator_param_grads_measured(p.handle, z.data_ptr(), y.data_ptr(), B, flat.data_ptr(), None,
                                                       part, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return rc

    assert call(plan(meas_rows=0)) == -4                       # no operator rows
    assert call(plan(bwd_passes=1)) == -4                      # single-pass data gradient
    p = plan()
    assert call(p) == -1                                       # no operator packed
    p.ensure_operator(A)
    assert call(p, part=0) == -3                               # a layer before the prologue
    assert call(p, part=4) == -1 and call(p, part=-3) == -1    # no such part
    assert call(p) == 0
    p = plan(train=False)
    p.ensure_operator(A)
    assert call(p) == -3                                       # no training buffers
    p = plan(gemm_impl=1)
    p.ensure_operator(A)
    assert call(p) == -4                                       # the SIMT path has no weight-gradient GEMMs
