"""Host side of masked posterior inference, on the CPU: the mask normalisation of ``plan.as_mask`` (shapes, dtypes,
errors), the masked oracle (an all-ones mask is the unmasked closure; the masked gradient is fp64 autograd of the
weighted loss), and that ``training_iteration``, ``generator_update_begin``, ``make_sampler`` and
``dist.langevin_sharded`` hand each rank its mask shard (device entry points replaced by recorders, as in
tests/test_train_dp_host_logic.py).  The kernels behind them are covered by tests/test_gpu_masked_inference.py."""
import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import dist as ldist, langevin as llang, synth, train as ltrain
from lsnf_b200.plan import as_mask
from oracle import refpath
import masked_oracle
from helpers import assert_grad_close, rel_l2, to_torch

B, NC, IMG = 4, 3, 32


# ---- mask normalisation ----------------------------------------------------------------------------------------------
# Shapes and dtypes are checked on the meta device (no data, no CUDA needed); as_mask refuses CPU tensors.
@pytest.mark.parametrize("shape", [(B, NC, IMG, IMG), (B, 1, IMG, IMG), (1, 1, IMG, IMG), (IMG, IMG), (1, NC, 1, 1),
                                   (IMG,)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.float16, torch.bool, torch.uint8, torch.int64])
def test_mask_broadcasts_to_a_contiguous_fp32_tensor_of_x_shape(shape, dtype):
    x = torch.empty(B, NC, IMG, IMG, device="meta")
    m = as_mask(torch.empty(shape, dtype=dtype, device="meta"), x)
    assert m.shape == x.shape and m.dtype == torch.float32 and m.is_contiguous() and m.device == x.device


@pytest.mark.parametrize("shape", [(B, 2, IMG, IMG), (B + 1, NC, IMG, IMG), (IMG + 1, IMG), (2, B, NC, IMG, IMG),
                                   (IMG, IMG, 1)])
def test_mask_of_a_shape_that_does_not_broadcast_raises_value_error(shape):
    x = torch.empty(B, NC, IMG, IMG, device="meta")
    with pytest.raises(ValueError):
        as_mask(torch.empty(shape, device="meta"), x)


def test_cpu_mask_raises_runtime_error_like_x():
    with pytest.raises(RuntimeError, match="CUDA"):
        as_mask(torch.ones(B, NC, IMG, IMG), torch.empty(B, NC, IMG, IMG))
    with pytest.raises(RuntimeError):
        as_mask(torch.ones(IMG, IMG, dtype=torch.bool), torch.empty(B, NC, IMG, IMG, device="meta"))
    with pytest.raises(TypeError):
        as_mask(np.ones((IMG, IMG), np.float32), torch.empty(B, NC, IMG, IMG, device="meta"))


# ---- the masked oracle -----------------------------------------------------------------------------------------------
def _oracle_setup(seed=3, ngf=16):
    gp = to_torch(synth.generator_state("svhn", 100, ngf, 3, seed=seed))
    fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=seed))
    layers = refpath.generator_layers("svhn", 100, ngf)
    x_np, z0_np, eps_np = synth.inputs(B, 100, 3, 32, 3, seed=seed)
    return gp, fp, layers, torch.from_numpy(x_np), torch.from_numpy(z0_np).reshape(B, 100, 1, 1), torch.from_numpy(eps_np)


def test_oracle_closure_with_an_all_ones_mask_is_the_unmasked_closure():
    gp, fp, layers, x, z0, eps = _oracle_setup()
    kw = dict(depth=5, steps=3, step_size=0.1, sigma=0.3, eps=eps.reshape(3, B, 100, 1, 1))
    za, ga, fa = refpath.langevin(z0, x, gp, fp, layers, **kw)
    zb, gb, fb = masked_oracle.langevin(z0, x, torch.ones_like(x), gp, fp, layers, **kw)
    assert rel_l2(zb, za) < 1e-6 and abs(gb.item() - ga.item()) < 1e-6 * ga.item() and fb.item() == pytest.approx(fa.item(), rel=1e-6)


def test_masked_oracle_gradient_is_fp64_autograd_of_the_weighted_loss():
    gp, fp, layers, x, z0, eps = _oracle_setup()
    rng = np.random.default_rng(0)
    m = torch.from_numpy(rng.random((B, NC, IMG, IMG)).astype(np.float32))
    m[0, :, 8:24, 8:24] = 0.0
    m[1] = 0.0
    sigma = 0.3
    _, g = masked_oracle.recon_grad(z0, x, m, gp, layers, sigma)
    # fp64, written out independently of the oracle's helper
    z = z0.double().clone().requires_grad_(True)
    xh = refpath.generator_forward({k: v.double() for k, v in gp.items()}, z, layers)
    loss = ((xh - x.double()) ** 2 * m.double()).sum() / (2.0 * sigma * sigma)
    want = torch.autograd.grad(loss, z)[0]
    assert_grad_close(g.reshape(B, -1).numpy(), want.reshape(B, -1).numpy(), what="masked oracle gradient vs fp64")
    assert torch.count_nonzero(g[1]).item() == 0                 # an all-zero mask removes the likelihood term
    _, g_unmasked = refpath.recon_grad(z0, x, gp, layers, sigma)
    assert rel_l2(g, g_unmasked) > 1e-2


def test_oracle_parameter_updates_weight_loss_g_by_the_mask():
    gp, fp, layers, x, z0, _ = _oracle_setup()
    m = torch.zeros_like(x)
    m[:, :, :16] = 1.0
    gl = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    fl = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in fp.items()}
    og = torch.optim.Adam(list(gl.values()), lr=1e-4)
    of = torch.optim.Adam([fl[k] for k in refpath.trainable_flow_keys(fl)], lr=1e-4)
    loss_g, _ = masked_oracle.parameter_updates(gl, fl, z0, x, m, layers, og, of, depth=5)
    xh = refpath.generator_forward(gp, z0, layers)
    assert loss_g.item() == pytest.approx(float(((xh - x)[:, :, :16] ** 2).sum()) / B, rel=1e-5)


# ---- the mask reaches every entry point, sharded per rank ------------------------------------------------------------
def test_training_iteration_passes_the_mask_to_inference_and_the_generator_update(monkeypatch):
    log = {}

    def fake_langevin(z, x, netG, netF, args, verbose=False, **kw):
        log["langevin_mask"] = kw.get("mask")
        return z.clone(), torch.tensor(1.0), torch.tensor(2.0)

    class Pending:
        def finish(self):
            return torch.tensor(3.0)

    def fake_gen_begin(netG, optG, z_k, x, args, **kw):
        log["gen_mask"] = kw.get("mask")
        return Pending()

    monkeypatch.setattr(ltrain, "sample_langevin_post_z_with_flow", fake_langevin)
    monkeypatch.setattr(ltrain, "generator_update_begin", fake_gen_begin)
    monkeypatch.setattr(ltrain, "flow_update", lambda *a, **k: torch.tensor(4.0))
    monkeypatch.setattr(llang, "langevin_plan", lambda *a, **k: None)
    args = lsnf_b200.make_args(dataset="svhn", nz=100, ngf=4, seed=5)
    netG, netF = lsnf_b200._netG(args), lsnf_b200._netF(args, nz=100)
    x = torch.zeros(6, 3, 32, 32)
    mask = torch.rand(6, 1, 32, 32)
    lsnf_b200.training_iteration(x, netG, netF, None, None, args, seed=1, mask=mask)
    assert log["langevin_mask"] is mask and log["gen_mask"] is mask
    lsnf_b200.training_iteration(x, netG, netF, None, None, args, seed=1)
    assert log["langevin_mask"] is None and log["gen_mask"] is None


class _RecordingPlan:
    """Stands in for a training plan: records the mask of every generator_param_grads call."""

    def __init__(self, netG):
        self.convs = [m for m in netG.gen if isinstance(m, torch.nn.ConvTranspose2d)]
        self.calls = []

    def ensure_generator(self, netG):
        pass

    def generator_grad_layout(self):
        sizes = [p.numel() for m in self.convs for p in (m.weight, m.bias)]
        return [(sum(sizes[:i]), s) for i, s in enumerate(sizes)]

    def generator_param_grads(self, z, x, global_batch, flat, part=-1, loss=None, *, mask=None):
        self.calls.append((part, mask))
        return flat, torch.zeros(())


def test_generator_update_normalises_the_mask_once_and_passes_it_to_the_prologue_calls(monkeypatch):
    args = lsnf_b200.make_args(dataset="svhn", nz=100, ngf=4)
    netG = lsnf_b200._netG(args)
    plan = _RecordingPlan(netG)
    plan._ggrad_flat = torch.zeros(sum(s for _, s in plan.generator_grad_layout()))
    # meta tensors: the mask logic is device-independent past the CPU check
    z, x = torch.empty(6, 100, 1, 1, device="meta"), torch.empty(6, 3, 32, 32, device="meta")
    ltrain.generator_update_begin(netG, None, z, x, args, plan=plan, mask=torch.empty(6, 1, 32, 32, device="meta"))
    (part, m), = plan.calls
    assert part == -1 and m.shape == (6, 3, 32, 32) and m.dtype == torch.float32 and m.is_contiguous()
    plan.calls.clear()
    ltrain.generator_update_begin(netG, None, z, x, args, plan=plan)
    assert plan.calls == [(-1, None)]
    with pytest.raises(ValueError):
        ltrain.generator_update_begin(netG, None, z, x, args, plan=plan, mask=torch.empty(5, 3, 32, 32, device="meta"))


def test_make_sampler_closure_keeps_the_reference_signature_and_takes_a_mask(monkeypatch):
    log = []
    monkeypatch.setattr(llang, "sample_langevin_post_z_with_flow",
                        lambda z, x, netG, netF, args, verbose=False, **kw: log.append((verbose, kw)))
    args = lsnf_b200.make_args(g_l_steps=3)
    m = object()
    llang.make_sampler(args)(1, 2, 3, 4, True, mask=m)
    llang.make_sampler(args, test_mode=True)(1, 2, 3, 4)
    assert log[0] == (True, {"mask": m})
    assert log[1] == (False, {"steps": 60, "with_noise": False, "mask": None})


@pytest.mark.parametrize("world", [2, 3])
def test_langevin_sharded_passes_each_rank_its_mask_shard(monkeypatch, world):
    seen = []
    monkeypatch.setattr(llang, "sample_langevin_post_z_with_flow",
                        lambda z, x, netG, netF, args, **kw: seen.append((z, x, kw)) or (z, 1.0, 2.0))
    n = 7
    z, x = torch.randn(n, 100, 1, 1), torch.randn(n, 3, 32, 32)
    mask = torch.rand(n, 1, 32, 32)
    shared = torch.rand(1, 1, 32, 32)
    plane = torch.rand(32, 32)
    for rank in range(world):
        a, b = ldist.shard_range(n, rank, world)
        for m, want in ((mask, mask[a:b]), (shared, shared), (plane, plane), (None, None)):
            seen.clear()
            ldist.langevin_sharded(z, x, None, None, None, seed=1, rank=rank, world=world, mask=m)
            (zs, xs, kw), = seen
            assert torch.equal(zs, z[a:b]) and torch.equal(xs, x[a:b]) and kw["sample_offset"] == a
            if want is None:
                assert kw["mask"] is None
            else:
                assert torch.equal(kw["mask"], want)
