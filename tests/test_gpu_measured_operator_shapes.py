"""The measurement-operator path (y = A vec(G(z)) + sigma noise) stage by stage, at the shapes the plan accepts rather
than the two operators of tests/test_gpu_measured_inference.py: ragged operator sizes m (one row, either side of a
64-column K block and of a 128-row N tile, a last |r|^2 tile of one row, m > n), batches of one and of several 128-row
M tiles, the long split K of CelebA-HQ256, and both GEMM implementations.  Each launch of a measured iteration is read
back from the workspace and checked on the very operands it read:

* the operator's two packed copies (fp16 hi|lo of A 2^k and bf16 hi|lo of A^T 2^k), bit for bit;
* x_hat's fp16 hi|lo rows, bit for bit, and stage 2L (A x_hat 2^k) against an fp64 contraction of its operands;
* the finisher's bf16 hi|lo rows of r 2^k seed_scale, bit for bit against an fp32 restatement;
* stage 2L+1 (A^T r) against an fp64 contraction of its operands;

then the data gradient end to end against the fp64 oracle, AIS energies over |r|^2 tiles, and the path's independence
of the units of A, y and sigma: bit-identical results under a power-of-two change of units, and the fp64 oracle far
beyond the range of the 16-bit formats.  The worst error of every case is recorded as JSON (helpers.record)."""
import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import _cabi, synth
from oracle import refpath
import ais_oracle as O
import measured_oracle as MO
from helpers import REL_TOL, build_nets, per_sample_rel_l2, record, rel_l2, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = 0.3
SVHN = dict(dataset="svhn", nz=100, ngf=32, leak=1.0)       # kink-free: gradients agree sample by sample
CROP = dict(dataset="celeba_crop", nz=100, ngf=64, leak=1.0)
HQ = dict(dataset="celeba_hq256", nz=100, ngf=64, leak=1.0)
N = 3072
# (config, m, B): each edge at least once -- m = 1; 63 / 64 / 65 around a K block; 129 / 255 / 257 around an N tile and
# a 256-row |r|^2 tile; n/4 + 5; n; 2n + 1 (K of A^T r larger than that of A x_hat).  B = 1; 100; 128 (one full M
# tile); 129 and 300 (two and three M tiles, grid_x > 1 on both operator stages)
CASES = [(SVHN, 1, 1), (SVHN, 63, 100), (SVHN, 64, 128), (SVHN, 65, 129), (SVHN, 129, 300), (SVHN, 255, 1),
         (SVHN, 257, 129), (SVHN, N // 4 + 5, 100), (SVHN, N, 128), (SVHN, 2 * N + 1, 129),
         (CROP, 12288 // 8 + 3, 129), (HQ, 257, 3)]
IDS = [f"{c['dataset']}_m{m}_B{b}" for c, m, b in CASES]
SIMT_CASES = [(SVHN, 65, 129), (SVHN, N // 4 + 5, 100)]
WORST = {}


def _note(case, value):
    WORST[case] = float(value)
    record("r11_measured_operator_shapes.json", WORST)


def _ws(plan):
    return plan._ws[plan._ws_ptr - plan._ws.data_ptr():]


def _at(ws, off, shape, dtype):
    n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
    return ws[off:off + n].view(dtype).view(*shape)


def _split(v, dtype):
    hi = v.to(dtype)
    return hi, (v - hi.float()).to(dtype)


def _bits(t):
    return t.contiguous().view(torch.int16)


def _fixed_order_sum(part):
    """The split-K partials [S][B][N] summed in split order in fp32, as the finisher and the im2col seed do."""
    v = part[0].clone()
    for q in range(1, part.shape[0]):
        v = v + part[q]
    return v


def _contract(a_hi, a_lo, b_hi, b_lo, three_pass):
    """fp64 a b^T of hi|lo operands: the three products of the tensor-core passes (hi hi, hi lo, lo hi), or the whole
    (hi + lo)(hi + lo) the SIMT twin forms."""
    a_hi, a_lo, b_hi, b_lo = (t.double() for t in (a_hi, a_lo, b_hi, b_lo))
    if three_pass:
        return a_hi @ b_hi.T + a_hi @ b_lo.T + a_lo @ b_hi.T
    return (a_hi + a_lo) @ (b_hi + b_lo).T


def _errors(got, ref):
    return float((got - ref).norm() / ref.norm()), float((got - ref).abs().max() / ref.abs().max())


def _plan(netG, netF, B, m, impl=_cabi.GEMM_TCGEN05):
    p = lsnf_b200.Plan(arch=netG.dataset, batch=B, nz=netG.nz, ngf=netG.ngf, nc=netG.nc, f_depth=netF.f_depth,
                       f_width=netF.f_width, f_permutation=netF.f_permutation, f_coupling=netF.f_coupling,
                       leak=netG.leak, device=DEV, gemm_impl=impl, bwd_passes=3, meas_rows=m)
    p.ensure_generator(netG)
    p.ensure_flow(netF, need_inverse=True)
    return p


def _problem(c, m, B, seed):
    """(A, y, z, x): a Gaussian operator with N(0, 1/n) entries, y = A vec(x) + 0.05 noise."""
    img = synth.image_size(c["dataset"])
    n = 3 * img * img
    x, z, _ = synth.inputs(B, c["nz"], 3, img, 1, seed=seed)
    A = MO.gaussian_operator(m, n, seed + 1)
    y = x.reshape(B, -1) @ A.T
    y = (y + 0.05 * np.random.default_rng(seed + 2).standard_normal(y.shape)).astype(np.float32)
    return A, y, z.reshape(B, c["nz"]), x


def _oracle_grad(c, z, y, A, sigma=SIGMA):
    gp = to_torch(synth.generator_state(c["dataset"], c["nz"], c["ngf"], 3, seed=1))
    layers = refpath.generator_layers(c["dataset"], c["nz"], c["ngf"])
    z = torch.from_numpy(np.asarray(z)).reshape(len(z), -1, 1, 1)
    _, g = MO.recon_grad(z, torch.as_tensor(y), torch.as_tensor(A), gp, layers, sigma, leak=c["leak"],
                         dtype=torch.float64)
    return g.reshape(len(z), -1).numpy()


# ---- 1. the operator's packed copies, bit for bit -------------------------------------------------------------------
def _check_pack(plan, A, tag):
    """Both packed copies against the torch restatement: fp16 hi|lo of A 2^k (max|A| 2^k in [1, 2)), bf16 hi|lo of
    A^T 2^k, zeros in every padding row and column."""
    st = plan.stages()
    fwd, bwd = st[-2], st[-1]
    m, n = A.shape
    k = MO.operator_scale_exp(float(A.abs().max()))
    a = A * 2.0 ** k
    assert 1.0 <= float(a.abs().max()) < 2.0 or k in (-126, 126)
    ws = _ws(plan)
    kx, km = fwd.k_per_tap, bwd.k_per_tap
    want = torch.zeros(fwd.b_rows, 2 * kx, dtype=torch.float16, device=DEV)
    hi, lo = _split(a, torch.float16)
    want[:m, :n], want[:m, kx:kx + n] = hi, lo
    got = _at(ws, fwd.b_offset, (fwd.b_rows, 2 * kx), torch.float16)
    assert torch.equal(_bits(got), _bits(want)), (tag, "fp16 copy of A")
    want = torch.zeros(bwd.b_rows, 2 * km, dtype=torch.bfloat16, device=DEV)
    hi, lo = _split(a.T, torch.bfloat16)
    want[:n, :m], want[:n, km:km + m] = hi, lo
    got = _at(ws, bwd.b_offset, (bwd.b_rows, 2 * km), torch.bfloat16)
    assert torch.equal(_bits(got), _bits(want)), (tag, "bf16 copy of A^T")
    return k


@pytest.mark.parametrize("amax", [1.0, 2.0, float(np.nextafter(np.float32(1.0), np.float32(0.0))), 2.0 ** 40,
                                  2.0 ** -40, 2.0 ** 100, 2.0 ** -100],
                         ids=["1", "2", "1-ulp", "2^40", "2^-40", "2^100", "2^-100"])
def test_operator_packs_bit_for_bit_at_scale_edges(amax):
    _args, netG, netF = build_nets(SVHN, DEV)
    m = 65
    plan = _plan(netG, netF, 4, m)
    A = torch.from_numpy(MO.gaussian_operator(m, N, seed=7)).to(DEV)
    A = A * (0.5 / float(A.abs().max()))                 # every entry within about 0.5 ...
    A[3, 17] = -1.0                                      # ... but this one, the maximum (negative)
    A = A * float(np.float32(amax))                      # a power of two or 1 - 2^-24: max|A| = amax exactly
    assert float(A.abs().max()) == float(np.float32(amax))
    plan.ensure_operator(A)
    torch.cuda.synchronize()
    _check_pack(plan, A, amax)


# ---- 2.-4. the operator stages and the finisher on the operands they read --------------------------------------------
_RUNS = {}


def _run(c, m, B, impl=_cabi.GEMM_TCGEN05):
    """One lsnf_generator_dgrad_measured call; returns (plan, A, y, z, x_hat, grad) with the workspace it left."""
    key = (c["dataset"], m, B, impl)
    if key not in _RUNS:
        _RUNS.clear()   # one plan alive at a time: the operator copies of 2n+1 rows or HQ256 are hundreds of MB
        _args, netG, netF = build_nets(c, DEV, impl=impl)
        A, y, z, _x = _problem(c, m, B, seed=m + B)
        plan = _plan(netG, netF, B, m, impl)
        At, yt = torch.from_numpy(A).to(DEV), torch.from_numpy(y).to(DEV)
        plan.ensure_operator(At)
        x_hat = plan.generator_forward(torch.from_numpy(z).to(DEV))
        g = plan.generator_dgrad_measured(yt, SIGMA)
        torch.cuda.synchronize()
        _RUNS[key] = (plan, At, yt, z, x_hat, g)
    return _RUNS[key]


def _check_stages(c, m, B, impl, tag):
    plan, A, y, z, x_hat, _g = _run(c, m, B, impl)
    three = impl == _cabi.GEMM_TCGEN05
    st = plan.stages()
    fwd, bwd = st[-2], st[-1]
    n = A.shape[1]
    kx, km = fwd.k_per_tap, bwd.k_per_tap
    assert (fwd.n_valid, bwd.n_valid, kx, km) == (m, n, -(-n // 64) * 64, -(-m // 64) * 64)
    k = _check_pack(plan, A, tag)
    ws = _ws(plan)
    # x_hat as the fp16 hi|lo rows stage 2L reads, bit for bit
    xhl = _at(ws, fwd.a_offset, (B, 2 * kx), torch.float16)
    want = torch.zeros(B, 2 * kx, dtype=torch.float16, device=DEV)
    hi, lo = _split(x_hat.reshape(B, -1), torch.float16)
    want[:, :n], want[:, kx:kx + n] = hi, lo
    assert torch.equal(_bits(xhl), _bits(want)), "x_hat rows"
    # stage 2L: A x_hat 2^k, against fp64 over the packed operands
    a16 = _at(ws, fwd.b_offset, (fwd.b_rows, 2 * kx), torch.float16)
    part = _at(ws, fwd.out_offset, (fwd.k_splits, B, fwd.n_pad), torch.float32)
    v = _fixed_order_sum(part)
    assert not v[:, m:].any(), "padding columns of A x_hat"
    ref = _contract(xhl[:, :kx], xhl[:, kx:], a16[:m, :kx], a16[:m, kx:], three)
    e2, w2 = _errors(v[:, :m].double(), ref)
    _note(f"{tag}_stage2L_rel_l2", e2)
    _note(f"{tag}_stage2L_worst", w2)
    # the finisher: bf16 hi|lo of (sum - y 2^k) seed_scale, bit for bit; rows [m, km) stay zero
    r = (v[:, :m] - y * 2.0 ** k) * MO.sigma_seed_scale(SIGMA)
    rhl = _at(ws, bwd.a_offset, (B, 2 * km), torch.bfloat16)
    want = torch.zeros(B, 2 * km, dtype=torch.bfloat16, device=DEV)
    hi, lo = _split(r, torch.bfloat16)
    want[:, :m], want[:, km:km + m] = hi, lo
    assert torch.equal(_bits(rhl), _bits(want)), "r rows"
    # stage 2L+1: A^T r, against fp64 over the packed operands
    at16 = _at(ws, bwd.b_offset, (bwd.b_rows, 2 * km), torch.bfloat16)
    part = _at(ws, bwd.out_offset, (bwd.k_splits, B, bwd.n_pad), torch.float32)
    v = _fixed_order_sum(part)
    assert not v[:, n:].any(), "padding columns of A^T r"
    ref = _contract(rhl[:, :km], rhl[:, km:], at16[:n, :km], at16[:n, km:], three)
    e3, w3 = _errors(v[:, :n].double(), ref)
    _note(f"{tag}_stage2L+1_rel_l2", e3)
    _note(f"{tag}_stage2L+1_worst", w3)
    print(f"{tag}: k {k} splits {fwd.k_splits}/{bwd.k_splits} A x_hat {e2:.2e}/{w2:.2e} A^T r {e3:.2e}/{w3:.2e}")
    # fp32 accumulation of exactly the products the kernel forms.  Its error grows with K and with the cancellation
    # of a zero-mean operator: observed on one B200 at most 2e-6 at n = 3072, 8e-6 at 12 288 and 1.4e-5 (rel-l2) /
    # 1.2e-5 (worst) at CelebA-HQ256's K = 196 608; the SIMT twin 3e-7.  A lost fp16 lo half of one operand leaves
    # about 2^-12 = 2.4e-4, a dropped split or a wrong pitch 1e-2 and more.
    assert e2 < 5e-5 and w2 < 5e-5, (e2, w2)
    assert e3 < 5e-5 and w3 < 5e-5, (e3, w3)


@pytest.mark.parametrize("c,m,B", CASES, ids=IDS)
def test_operator_stages_match_fp64_and_the_finisher_matches_bit_for_bit(c, m, B):
    _check_stages(c, m, B, _cabi.GEMM_TCGEN05, f"{c['dataset']}_m{m}_B{B}")


# ---- 5. the data gradient end to end ---------------------------------------------------------------------------------
@pytest.mark.parametrize("c,m,B", [x for x in CASES if x[0] is not HQ], ids=[i for x, i in zip(CASES, IDS)
                                                                             if x[0] is not HQ])
def test_measured_data_gradient_matches_the_fp64_oracle(c, m, B):
    plan, A, y, z, _x_hat, g = _run(c, m, B)
    e = per_sample_rel_l2(g.cpu().numpy(), _oracle_grad(c, z, y.cpu(), A.cpu()))
    _note(f"{c['dataset']}_m{m}_B{B}_dgrad_worst_rel_l2", e.max())
    assert e.max() < REL_TOL, e.max()


@pytest.mark.parametrize("c,m,B", SIMT_CASES, ids=[f"m{m}_B{b}" for _c, m, b in SIMT_CASES])
def test_simt_twin_runs_the_operator_stages_and_agrees_with_tcgen05(c, m, B):
    tag = f"simt_m{m}_B{B}"
    _check_stages(c, m, B, _cabi.GEMM_SIMT, tag)
    g_simt = _run(c, m, B, _cabi.GEMM_SIMT)[5].cpu().numpy()
    _plan_, A, y, z, _x, g_tc = _run(c, m, B)
    e = per_sample_rel_l2(g_simt, _oracle_grad(c, z, y.cpu(), A.cpu()))
    e_tc = per_sample_rel_l2(g_tc.cpu().numpy(), g_simt)
    _note(f"{tag}_dgrad_worst_rel_l2", e.max())
    _note(f"{tag}_tc_vs_simt_worst_rel_l2", e_tc.max())
    assert e.max() < REL_TOL and e_tc.max() < REL_TOL, (e.max(), e_tc.max())


# ---- 6. AIS energy tiles and a measured chain: m = 257 (the last |r|^2 tile holds one row), B = 129 ---------------------
_T = 20


def _chain_setup():
    c = dict(SVHN, ngf=64)   # at ngf 64 the data gradient has e4m3 stages (DESIGN.md section 4.1), whose scales clamp
    m, B = 257, 129
    _args, netG, netF = build_nets(c, DEV)
    A, y, _z, _x = _problem(c, m, B, seed=5)
    x0, z0, _ = synth.inputs(B, 100, 3, 32, 1, seed=41)
    r = np.random.default_rng(9)
    eps = r.standard_normal((_T, B, 100)).astype(np.float32)
    u = r.uniform(size=(_T, B)).astype(np.float32)
    return c, netG, netF, A, y, z0.reshape(B, 100), eps, u


def _measured_outputs(netG, netF, A, y, sigma, z0, eps, u, betas):
    """(grad at z0, z_T of a T-step chain with injected eps, AIS log w with injected eps and u, T = 1 AIS log w)."""
    B, m = y.shape
    plan = _plan(netG, netF, B, m)
    plan.ensure_operator(A)
    z0t = torch.from_numpy(z0).to(DEV)
    plan.generator_forward(z0t)
    g = plan.generator_dgrad_measured(y, sigma)
    zT, _ = plan.langevin_run_measured(z0t, y, _T, 0.1, sigma, eps=torch.from_numpy(eps).to(DEV))
    _z, lw, _rate = plan.ais_run_measured(z0t, y, torch.from_numpy(betas).to(DEV), _T, 0.5, sigma,
                                          eps=torch.from_numpy(eps).to(DEV), u=torch.from_numpy(u).to(DEV))
    _z, lw1, _r = plan.ais_run_measured(z0t, y, torch.tensor([0.0, 1.0], device=DEV), 1, 0.1, sigma, seed=3)
    torch.cuda.synchronize()
    return g, zT, lw, lw1


_BASE = {}


def _base():
    if not _BASE:
        c, netG, netF, A, y, z0, eps, u = _chain_setup()
        betas = O.sigmoid_schedule(_T).astype(np.float32)
        gp = to_torch(synth.generator_state("svhn", 100, c["ngf"], 3, seed=1))
        fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=1))
        layers = refpath.generator_layers("svhn", 100, c["ngf"])
        B = len(z0)
        z_ref, _, _ = MO.langevin(torch.from_numpy(z0).reshape(B, 100, 1, 1), torch.from_numpy(y), torch.from_numpy(A),
                                  gp, fp, layers, depth=5, steps=_T, step_size=0.1, sigma=SIGMA,
                                  eps=torch.from_numpy(eps).reshape(_T, B, 100, 1, 1), leak=1.0)
        energy = MO.energy(gp, fp, layers, y, A, SIGMA, leak=1.0)
        l1 = energy(O.round_hl(z0))[0]
        _BASE.update(c=c, netG=netG, netF=netF, A=A, y=y, z0=z0, eps=eps, u=u, betas=betas, z_ref=z_ref.numpy(),
                     l1=l1, g_ref=_oracle_grad(c, z0, y, A))
        _BASE["out"] = _measured_outputs(netG, netF, torch.from_numpy(A).to(DEV), torch.from_numpy(y).to(DEV), SIGMA,
                                         z0, eps, u, betas)
    return _BASE


def test_measured_ais_and_chain_over_ragged_energy_tiles_match_the_oracle():
    b = _base()
    g, zT, _lw, lw1 = b["out"]
    e_g = per_sample_rel_l2(g.cpu().numpy(), b["g_ref"]).max()
    e_z = rel_l2(zT.cpu().numpy().reshape(b["z_ref"].shape), b["z_ref"])
    e_l = float((np.abs(lw1.cpu().numpy() - b["l1"]) / np.abs(b["l1"])).max())
    _note("ais_chain_m257_B129_dgrad_worst_rel_l2", e_g)
    _note("ais_chain_m257_B129_T20_zT_rel_l2", e_z)
    _note("ais_chain_m257_B129_T1_log_w_max_rel_err", e_l)
    assert e_g < REL_TOL and e_z < REL_TOL, (e_g, e_z)
    assert e_l < 1e-5, e_l


# ---- 7. units: A, y and sigma times 2^j --------------------------------------------------------------------------------
def _scaled(j):
    b = _base()
    c = np.float32(2.0 ** j)
    return _measured_outputs(b["netG"], b["netF"], torch.from_numpy(b["A"] * c).to(DEV),
                             torch.from_numpy(b["y"] * c).to(DEV), float(np.float32(SIGMA) * c), b["z0"], b["eps"],
                             b["u"], b["betas"])


@pytest.mark.parametrize("j", [-8, -3, 1, 5, 8])
def test_a_power_of_two_change_of_units_leaves_every_bit(j):
    """Every step of the path is exact under power-of-two scaling while values stay normal and no clamp bites."""
    want = _base()["out"]
    got = _scaled(j)
    for name, a, w in zip(("grad", "z_T", "log w", "T=1 log w"), got, want):
        assert torch.equal(a, w), (j, name, float((a - w).abs().max()))
    _note(f"units_2^{j}_max_abs_diff", 0.0)


@pytest.mark.parametrize("j", [-32, -28, -24, -20, -16, -12, 12, 16, 20, 24, 28, 32])
def test_far_changes_of_units_match_the_fp64_oracle(j):
    b = _base()
    g, zT, _lw, lw1 = _scaled(j)
    e_g = per_sample_rel_l2(g.cpu().numpy(), b["g_ref"]).max()
    e_z = rel_l2(zT.cpu().numpy().reshape(b["z_ref"].shape), b["z_ref"])
    e_l = float((np.abs(lw1.cpu().numpy() - b["l1"]) / np.abs(b["l1"])).max())
    _note(f"units_2^{j}_dgrad_worst_rel_l2", e_g)
    _note(f"units_2^{j}_zT_rel_l2", e_z)
    _note(f"units_2^{j}_T1_log_w_max_rel_err", e_l)
    assert e_g < REL_TOL and e_z < REL_TOL and e_l < 1e-5, (e_g, e_z, e_l)


@pytest.mark.parametrize("j", [16, 24, 28])
def test_large_residuals_match_the_fp64_oracle(j):
    """y far from every A vec(G(z)) (2^j noise): r, A^T r and every data-gradient tensor grow as 2^j, and the e4m3
    stages' scales follow them."""
    b = _base()
    y = (b["y"] + 2.0 ** j * np.random.default_rng(j).standard_normal(b["y"].shape)).astype(np.float32)
    B, m = y.shape
    plan = _plan(b["netG"], b["netF"], B, m)
    plan.ensure_operator(torch.from_numpy(b["A"]).to(DEV))
    z0 = torch.from_numpy(b["z0"]).to(DEV)
    plan.generator_forward(z0)
    g = plan.generator_dgrad_measured(torch.from_numpy(y).to(DEV), SIGMA)
    _z, lw1, _r = plan.ais_run_measured(z0, torch.from_numpy(y).to(DEV), torch.tensor([0.0, 1.0], device=DEV), 1, 0.1,
                                        SIGMA, seed=3)
    e_g = per_sample_rel_l2(g.cpu().numpy(), _oracle_grad(b["c"], b["z0"], y, b["A"])).max()
    gp = to_torch(synth.generator_state("svhn", 100, b["c"]["ngf"], 3, seed=1))
    fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=1))
    l1 = MO.energy(gp, fp, refpath.generator_layers("svhn", 100, b["c"]["ngf"]), y, b["A"], SIGMA,
                   leak=1.0)(O.round_hl(b["z0"]))[0]
    e_l = float((np.abs(lw1.cpu().numpy() - l1) / np.abs(l1)).max())
    _note(f"residual_2^{j}_dgrad_worst_rel_l2", e_g)
    _note(f"residual_2^{j}_T1_log_w_max_rel_err", e_l)
    assert e_g < REL_TOL and e_l < 1e-5, (e_g, e_l)


def test_heteroscedastic_rows_match_the_fp64_oracle():
    """Rows of A and y weighted by 2^u, u ~ U(-12, 12): the scaling plan.as_operator prescribes for per-row noise."""
    b = _base()
    w = (2.0 ** np.random.default_rng(21).uniform(-12, 12, size=(b["A"].shape[0], 1))).astype(np.float32)
    A, y = (b["A"] * w).astype(np.float32), (b["y"] * w.T).astype(np.float32)
    B, m = y.shape
    plan = _plan(b["netG"], b["netF"], B, m)
    plan.ensure_operator(torch.from_numpy(A).to(DEV))
    plan.generator_forward(torch.from_numpy(b["z0"]).to(DEV))
    g = plan.generator_dgrad_measured(torch.from_numpy(y).to(DEV), SIGMA)
    e = per_sample_rel_l2(g.cpu().numpy(), _oracle_grad(b["c"], b["z0"], y, A)).max()
    _note("heteroscedastic_2^U(-12,12)_dgrad_worst_rel_l2", e)
    assert e < REL_TOL, e
