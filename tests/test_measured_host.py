"""Host side of inference from linear measurements y = A vec(G(z)) + sigma noise, on the CPU: the operator and y checks
of ``plan.as_operator`` / ``plan.as_measurements`` and of the public entry points, the plan of a config with
``meas_rows`` (its first 2L stages, launches and workspace regions are those of the plan without it; the two operator
stages stay within the hardware limits and their K splits cover K exactly), the measured oracle (fp64 autograd, and
the masked oracle for identity rows), and that ``dist.langevin_sharded`` hands each rank its y shard and the whole A.
The kernels are covered by tests/test_gpu_measured_inference.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from lsnf_b200 import _cabi, ais as lais, dist as ldist, langevin as llang, synth
from lsnf_b200.plan import as_measurements, as_operator
from oracle import refpath
import masked_oracle
import measured_oracle as MO
from helpers import assert_grad_close, rel_l2, to_torch
from test_plan_tables import BASELINE_CONFIGS, SMEM_MAX, SMEM_PER_SM, launch_infos, stage_infos

B, NC, IMG = 4, 3, 32
N = NC * IMG * IMG


# ---- operator and y checks -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(N,), (8, N + 1), (8, N - 64), (2, 8, N), (0, N)])
def test_operator_of_a_wrong_shape_raises_value_error(shape):
    with pytest.raises(ValueError):
        as_operator(torch.empty(shape, device="meta"), (B, NC, IMG, IMG))


def test_operator_dtype_finiteness_and_device():
    with pytest.raises(ValueError, match="cast"):
        as_operator(torch.empty(8, N, dtype=torch.complex64, device="meta"), (B, NC, IMG, IMG))
    for bad in (float("nan"), float("inf"), -float("inf")):
        A = torch.zeros(8, N)
        A[3, 5] = bad
        with pytest.raises(ValueError, match="non-finite"):
            as_operator(A, (B, NC, IMG, IMG))
    with pytest.raises(RuntimeError, match="CUDA"):
        as_operator(torch.zeros(8, N, dtype=torch.float64), (NC, IMG, IMG))
    with pytest.raises(TypeError):
        as_operator(np.zeros((8, N), np.float32), (NC, IMG, IMG))
    a = as_operator(torch.empty(8, N, dtype=torch.float16, device="meta"), (B, NC, IMG, IMG))
    assert a.dtype == torch.float32 and a.is_contiguous() and a.shape == (8, N)


@pytest.mark.parametrize("shape", [(B, 9), (B + 1, 8), (B * 8,), (B, 8, 1)])
def test_measurements_not_batch_by_m_raise_value_error(shape):
    with pytest.raises(ValueError, match=r"\[B, m\]"):
        as_measurements(torch.empty(shape, device="meta"), torch.empty(8, N, device="meta"), B)
    y = as_measurements(torch.empty(B, 8, dtype=torch.float64, device="meta"), torch.empty(8, N, device="meta"), B)
    assert y.shape == (B, 8) and y.dtype == torch.float32


def test_mask_and_operator_together_raise_value_error():
    with pytest.raises(ValueError, match="not both"):
        llang.sample_langevin_post_z_with_flow(None, None, None, None, None, mask=object(), operator=object())
    with pytest.raises(ValueError, match="not both"):
        lais.ais_log_likelihood(None, None, None, None, chains=1, steps=1, mask=object(), operator=object())


def test_measured_log_likelihood_constant():
    c = lais.log_likelihood_constant(0.3, (B, 192), operator=torch.empty(192, N, device="meta"))
    assert c.shape == (B,) and np.allclose(c, -0.5 * 192 * np.log(2 * np.pi * 0.09))


# ---- the plan of a config with meas_rows ----------------------------------------------------------------------------
def _plan(arch, nz, ngf, batch, meas_rows, bwd_passes=0):
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=3, f_depth=5, f_width=64,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=bwd_passes,
                       meas_rows=meas_rows)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "create")
    return lib, h


@pytest.mark.parametrize("arch,nz,ngf,batch", BASELINE_CONFIGS)
def test_operator_adds_two_stages_after_an_unchanged_plan(arch, nz, ngf, batch):
    lib, h0 = _plan(arch, nz, ngf, batch, 0)
    n = 3 * synth.image_size(arch) ** 2
    s0, l0 = stage_infos(lib, h0), launch_infos(lib, h0)
    ws0 = lib.lsnf_workspace_bytes(h0)
    L2 = len(s0)
    for m in (n // 16, n // 4 + 5, n):
        lib_, h = _plan(arch, nz, ngf, batch, m)
        s, l = stage_infos(lib, h), launch_infos(lib, h)
        assert len(s) == L2 + 2
        assert [bytes(x) for x in s[:L2]] == [bytes(x) for x in s0]
        assert [bytes(x) for x in l[:L2]] == [bytes(x) for x in l0]
        # every region of the operator lies after the workspace of the plan without it
        for st in s[L2:]:
            assert min(st.a_offset, st.b_offset, st.out_offset) >= ws0
        assert lib.lsnf_workspace_bytes(h) >= ws0 + 8 * m * n
        assert lib.lsnf_langevin_launch_count(h, 20) == lib.lsnf_langevin_launch_count(h0, 20)
        _check_operator_records(s[L2:], l[L2:], m, n, batch)
        lib.lsnf_plan_destroy(h)
    lib.lsnf_plan_destroy(h0)


def _check_operator_records(stages, launches, m, n, batch):
    """The two operator stages' records: shapes, K coverage of the splits, the hardware limits."""
    for st, li, rows, k in zip(stages, launches, (m, n), (n, m)):
        kblocks = -(-k // 64)
        assert st.kind == 3 and st.epilogue == 3 and st.tap_gen_k == 1 and st.k_per_tap == 64 * kblocks
        assert st.n_valid == rows and st.n_pad % st.block_n == 0 and st.n_pad >= rows
        assert st.b_k == st.k_per_tap and st.b_rows == st.n_pad and st.passes == 3
        # the K splits cover every K block once, none empty
        per = -(-kblocks // st.k_splits)
        assert (st.k_splits - 1) * per < kblocks <= st.k_splits * per
        # the hardware limits of tests/test_plan_tables.py
        assert li.kernel == _cabi.KERNEL_SINGLE and li.block == 320 and li.smem_bytes <= SMEM_MAX
        assert li.ring_stages >= 1 and li.ring_stages * li.stage_bytes + 1280 <= li.smem_bytes
        assert li.ctas_per_sm >= 1 and li.ctas_per_sm * (li.smem_bytes + 1024) <= SMEM_PER_SM
        assert li.ctas_per_sm * li.tmem_columns <= 512
        assert (li.grid_x, li.grid_y, li.grid_z) == (-(-batch // 128), st.n_pad // st.block_n, st.k_splits)
        assert not li.tma_store and not li.stream_k and not li.cross_fp8
        # a small batch is one M tile: the splits bring the grid to about one wave or more K blocks per split
        assert li.grid_x * li.grid_y * li.grid_z >= min(148, li.grid_x * li.grid_y * kblocks // 2) * 0.5
    return stages


# the (m, B) grid of tests/test_gpu_measured_operator_shapes.py
@pytest.mark.parametrize("arch,ngf,m,batch", [
    ("svhn", 32, 1, 1), ("svhn", 32, 63, 100), ("svhn", 32, 64, 128), ("svhn", 32, 65, 129), ("svhn", 32, 129, 300),
    ("svhn", 32, 255, 1), ("svhn", 32, 257, 129), ("svhn", 32, 773, 100), ("svhn", 32, 3072, 128),
    ("svhn", 32, 6145, 129), ("celeba_crop", 64, 1539, 129), ("celeba_hq256", 64, 257, 3)])
def test_operator_stage_records_across_the_shape_grid(arch, ngf, m, batch):
    lib, h = _plan(arch, 100, ngf, batch, m)
    n = 3 * synth.image_size(arch) ** 2
    li = launch_infos(lib, h)[-2:]
    fwd, bwd = _check_operator_records(stage_infos(lib, h)[-2:], li, m, n, batch)
    lib.lsnf_plan_destroy(h)
    assert li[0].grid_x == li[1].grid_x == (1 if batch <= 128 else 2 if batch <= 256 else 3)
    if m == 1:        # A^T r has one K block: one split
        assert (bwd.k_per_tap, bwd.k_splits) == (64, 1)
    if m == 2 * n + 1:   # K of A^T r exceeds that of A x_hat: more K blocks per split there
        assert bwd.k_per_tap == 64 * -(-m // 64) > fwd.k_per_tap and bwd.k_splits >= fwd.k_splits
    if arch == "celeba_hq256":   # 3072 K blocks of A x_hat split about 50 ways over 3 N tiles
        assert fwd.k_per_tap == 196608 and fwd.n_pad == 384 and 40 <= fwd.k_splits <= 60


def test_meas_rows_is_refused_where_it_cannot_apply():
    lib = _cabi.load()
    h = C.c_void_p()
    for arch, m in (("svhn", -1), ("none", 8)):
        cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=4, nz=100, ngf=64, nc=3, f_depth=5, f_width=64,
                           f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, meas_rows=m)
        assert lib.lsnf_plan_create(C.byref(cfg), C.byref(h)) == -1
    # measured calls on an unbound plan fail cleanly
    lib_, h = _plan("svhn", 100, 64, 4, 16)
    assert lib.lsnf_pack_measurement(h, None, None) == -3
    lib.lsnf_plan_destroy(h)


# ---- the measured oracle ---------------------------------------------------------------------------------------------
def _oracle_setup(seed=3, ngf=16):
    gp = to_torch(synth.generator_state("svhn", 100, ngf, 3, seed=seed))
    fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=seed))
    layers = refpath.generator_layers("svhn", 100, ngf)
    x_np, z0_np, eps_np = synth.inputs(B, 100, 3, 32, 3, seed=seed)
    return gp, fp, layers, torch.from_numpy(x_np), torch.from_numpy(z0_np).reshape(B, 100, 1, 1), torch.from_numpy(eps_np)


def test_measured_oracle_gradient_is_fp64_autograd():
    gp, fp, layers, x, z0, eps = _oracle_setup()
    A = torch.from_numpy(MO.gaussian_operator(N // 8, N, seed=1))
    y = x.reshape(B, -1) @ A.t() + 0.05
    sigma = 0.3
    _, g32 = MO.recon_grad(z0, y, A, gp, layers, sigma)
    _, g64 = MO.recon_grad(z0, y, A, gp, layers, sigma, dtype=torch.float64)
    # fp64, written out independently of the oracle's helper
    z = z0.double().clone().requires_grad_(True)
    xh = refpath.generator_forward({k: v.double() for k, v in gp.items()}, z, layers)
    r = xh.reshape(B, -1) @ A.double().t() - y.double()
    want = torch.autograd.grad((r * r).sum() / (2.0 * sigma * sigma), z)[0]
    assert torch.allclose(g64, want, rtol=1e-12, atol=0)
    assert_grad_close(g32.reshape(B, -1).numpy(), want.reshape(B, -1).numpy(), what="measured oracle fp32 vs fp64")


def test_identity_rows_of_a_mask_are_the_masked_oracle():
    gp, fp, layers, x, z0, eps = _oracle_setup()
    mask = np.ones((NC, IMG, IMG), np.float32)
    mask[:, 8:20, 4:30] = 0.0
    mask[2, ::2] = 0.0
    A = torch.from_numpy(MO.identity_rows(mask))
    y = x.reshape(B, -1)[:, torch.from_numpy(mask.reshape(-1) > 0)]
    kw = dict(depth=5, steps=3, step_size=0.1, sigma=0.3, eps=eps.reshape(3, B, 100, 1, 1))
    zm, gm, fm = MO.langevin(z0, y, A, gp, fp, layers, **kw)
    zk, gk, fk = masked_oracle.langevin(z0, x, torch.from_numpy(mask).expand(B, NC, IMG, IMG), gp, fp, layers, **kw)
    assert rel_l2(zm, zk) < 1e-6 and gm.item() == pytest.approx(gk.item(), rel=1e-5)
    # and the 2x2 average-pooling operator is what F.avg_pool2d computes
    P = torch.from_numpy(MO.avg_pool_operator(NC, IMG))
    assert torch.allclose((x.reshape(B, -1) @ P.t()).reshape(B, NC, IMG // 2, IMG // 2),
                          torch.nn.functional.avg_pool2d(x, 2), atol=1e-6)


# ---- data parallel: each rank gets its y shard and the whole operator ------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_langevin_sharded_hands_each_rank_its_y_shard(monkeypatch, world):
    calls = []
    monkeypatch.setattr(llang, "sample_langevin_post_z_with_flow",
                        lambda z, x, netG, netF, args, **kw: calls.append((z, x, kw)) or (z, None, None))
    Bg, m = 7, 12
    z = torch.arange(Bg * 2, dtype=torch.float32).reshape(Bg, 2)
    y = torch.arange(Bg * m, dtype=torch.float32).reshape(Bg, m)
    A = torch.ones(m, N)
    for rank in range(world):
        ldist.langevin_sharded(z, y, None, None, None, seed=5, rank=rank, world=world, operator=A)
    starts = [ldist.shard_range(Bg, r, world) for r in range(world)]
    for (zz, yy, kw), (a, b) in zip(calls, starts):
        assert torch.equal(yy, y[a:b]) and torch.equal(zz, z[a:b])
        assert kw["operator"] is A and kw["sample_offset"] == a and kw["mask"] is None


# ---- the operator's scale rule (restated in tests/measured_oracle.py for the GPU tests) -------------------------------
@pytest.mark.parametrize("amax,k", [(1.0, 0), (2.0, -1), (float(np.nextafter(np.float32(1), np.float32(0))), 1),
                                    (float(np.nextafter(np.float32(2), np.float32(0))), 0), (0.5, 1), (3.0, -1),
                                    (2.0 ** 30, -30), (2.0 ** 31, -31), (2.0 ** -15, 15), (2.0 ** -31, 31),
                                    (2.0 ** 125, -125), (2.0 ** 127, -126), (3.4e38, -126), (2.0 ** -126, 126),
                                    (2.0 ** -140, 126), (0.0, 1)])
def test_operator_scale_exponent_puts_the_maximum_in_one_to_two(amax, k):
    assert MO.operator_scale_exp(amax) == k
    a = np.float32(amax)
    if a > 0 and -126 < k < 126:
        assert 1.0 <= a * np.float32(2.0 ** k) < 2.0
    # no clamp but fp32's normal range: 2^k and 2^-k are normal fp32 numbers
    assert np.isfinite(np.float32(2.0 ** k)) and np.float32(2.0 ** -k) >= np.finfo(np.float32).tiny


def test_sigma_seed_scale_restatement():
    assert [MO.sigma_seed_scale(s) for s in (0.3, 1.0, 0.6, 0.1, 2.0 ** 20)] == [8.0, 1.0, 2.0, 16.0, 1.0]
