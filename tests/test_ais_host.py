"""Host-side tests of annealed importance sampling: the AIS/MALA maths on a linear-Gaussian model with an analytic
log p(x) (tests/ais_oracle.py), the schedule, the likelihood constant, the chain aggregation and argument validation
of ``lsnf_b200.ais``."""
import math

import numpy as np
import pytest
import torch

import ais_oracle as O
from lsnf_b200 import ais


def _run_toy(model, x, chains, T, *, reverse=False, seed=0, target=0.65):
    rng = np.random.default_rng(seed)
    xr = np.repeat(x, chains, 0)
    n = xr.shape[0]
    betas = O.sigmoid_schedule(T)
    if reverse:
        betas = betas[::-1].copy()
        z0 = model.posterior_sample(xr, rng)
    else:
        z0 = rng.normal(size=(n, model.d))
    eps = rng.normal(size=(T, n, model.d))
    u = rng.uniform(size=(T, n)).astype(np.float32)
    r = O.ais(z0, model.energy(xr), betas, step_size=0.3, target_accept=target, eps=eps, u=u, round_z=False)
    lw = r["logw"].reshape(len(x), chains)
    est = O.logmeanexp(lw, 1) if not reverse else -O.logmeanexp(lw, 1)
    return est + model.C(), r


@pytest.fixture(scope="module")
def toy():
    m = O.LinearGaussian()
    _z, x = m.sample(4)
    return m, x


def test_forward_ais_converges_to_the_analytic_log_px(toy):
    m, x = toy
    est, r = _run_toy(m, x, 256, 200)
    truth = m.log_px(x)
    assert np.all(np.abs(est - truth) < 0.05), (est, truth)
    assert 0.3 < r["accepts"].mean() / 200 < 0.95


def test_forward_below_reverse_above_and_the_gap_shrinks(toy):
    m, x = toy
    truth = m.log_px(x)
    gaps = []
    for T in (5, 200):
        lo, _ = _run_toy(m, x, 64, T, seed=T)
        hi, _ = _run_toy(m, x, 64, T, reverse=True, seed=T + 1)
        # stochastic bounds: allow the Monte-Carlo error of 64 chains
        assert np.mean(lo) <= np.mean(truth) + 0.02
        assert np.mean(hi) >= np.mean(truth) - 0.02
        gaps.append(float(np.mean(hi - lo)))
    assert gaps[1] < gaps[0], gaps
    assert gaps[1] < 0.1


def test_fixed_step_is_kept_and_adaptation_moves_it(toy):
    m, x = toy
    _, r = _run_toy(m, x, 8, 20, target=0.0)
    assert np.all(r["step"] == np.float32(0.3))
    _, r = _run_toy(m, x, 8, 20, target=0.99)
    assert np.all(r["step"] < np.float32(0.3))


def test_mh_rejects_non_finite_energies():
    def energy(z):
        n = z.shape[0]
        bad = np.abs(z[:, 0]) > 0.5
        ell = np.where(bad, np.nan, -0.5 * (z * z).sum(1))
        return ell, -0.5 * (z * z).sum(1), z, z
    z0 = np.zeros((4, 2), np.float32)
    eps = np.full((1, 4, 2), 100.0)
    r = O.ais(z0, energy, [1.0, 1.0], step_size=0.1, eps=eps, u=np.full((1, 4), 1e-30, np.float32), round_z=False)
    assert np.all(r["accepts"] == 0)
    assert np.all(r["z"] == 0)


@pytest.mark.parametrize("T", [1, 2, 7, 40, 2000])
def test_sigmoid_schedule(T):
    b = ais.sigmoid_schedule(T)
    assert b.shape == (T + 1,) and b[0] == 0.0 and b[-1] == 1.0
    assert np.all(np.diff(b) > 0)
    np.testing.assert_allclose(b, b[::-1][::-1])
    np.testing.assert_allclose(b + b[::-1], 1.0, atol=1e-12)   # symmetric about the midpoint
    np.testing.assert_allclose(b, O.sigmoid_schedule(T), atol=1e-12)


def test_sigmoid_schedule_rejects_zero_steps():
    with pytest.raises(ValueError):
        ais.sigmoid_schedule(0)


def _direct_C(sigma, m):
    out = []
    for row in m.reshape(m.shape[0], -1):
        out.append(sum(-0.5 * math.log(2 * math.pi * sigma ** 2 / v) for v in row if v > 0))
    return np.array(out)


def test_constant_unmasked():
    c = ais.log_likelihood_constant(0.3, (3, 3, 4, 4))
    np.testing.assert_allclose(c, -0.5 * 48 * math.log(2 * math.pi * 0.09))


@pytest.mark.parametrize("kind", ["ones", "binary", "fractional", "broadcast"])
def test_constant_masked_against_a_direct_sum(kind):
    g = torch.Generator().manual_seed(3)
    shape = (2, 3, 4, 4)
    if kind == "ones":
        m = torch.ones(shape)
    elif kind == "binary":
        m = (torch.rand(shape, generator=g) > 0.4).float()
    elif kind == "fractional":
        m = torch.rand(shape, generator=g) * (torch.rand(shape, generator=g) > 0.3).float()
    else:
        m = (torch.rand(1, 1, 4, 4, generator=g) > 0.5).float()
    c = ais.log_likelihood_constant(0.3, shape, m)
    np.testing.assert_allclose(c, _direct_C(0.3, m.expand(shape).double().numpy()), rtol=1e-12)
    if kind == "ones":
        np.testing.assert_allclose(c, ais.log_likelihood_constant(0.3, shape), rtol=1e-12)


def test_logmeanexp_over_chains():
    a = torch.tensor([[0.0, 0.0], [1000.0, 1000.0 + math.log(3.0)], [-1e4, -1e4]], dtype=torch.float64)
    got = ais.logmeanexp(a, 1)
    np.testing.assert_allclose(got.numpy(), [0.0, 1000.0 + math.log(2.0), -1e4], rtol=1e-12)
    assert got.dtype == torch.float64 and ais.logmeanexp(a.float(), 1).dtype == torch.float64
    np.testing.assert_allclose(O.logmeanexp(a.numpy(), 1), got.numpy(), rtol=1e-12)


class _StubPlan:
    def __getattr__(self, name):
        raise AssertionError(f"plan.{name} used before the arguments were validated")


@pytest.fixture
def stub(monkeypatch):
    monkeypatch.setattr(ais, "langevin_plan", lambda *a, **k: _StubPlan())


@pytest.mark.parametrize("kw, err", [
    (dict(chains=0, steps=4), ValueError),
    (dict(chains=2, steps=0), ValueError),
    (dict(chains=2, steps=4, schedule=[0.0, 0.5, 1.0]), ValueError),
    (dict(chains=2, steps=2, schedule=[0.0, 1.5, 1.0]), ValueError),
    (dict(chains=2, steps=2, schedule=[-0.1, 0.5, 1.0]), ValueError),
    (dict(chains=2, steps=2, schedule=[0.0, float("nan"), 1.0]), ValueError),
    (dict(chains=2, steps=2, schedule=np.zeros((3, 1))), ValueError),
    (dict(chains=2, steps=2), RuntimeError),                      # x on the CPU
    (dict(chains=2, steps=2, schedule=[0.0, 0.5, 1.0]), RuntimeError),
])
def test_ais_log_likelihood_validates_its_arguments(stub, kw, err):
    x = torch.zeros(2, 3, 32, 32)
    with pytest.raises(err):
        ais.ais_log_likelihood(x, None, None, {}, **kw)


def test_bdmc_validates_its_arguments(stub):
    with pytest.raises(ValueError):
        ais.bdmc(None, None, {}, 0, chains=2, steps=2, device="cpu")
    with pytest.raises(ValueError):
        ais.bdmc(None, None, {}, 2, chains=0, steps=2, device="cpu")


def test_the_entry_point_is_bound():
    from lsnf_b200 import _cabi
    assert "lsnf_ais_run" in _cabi.EXPORTS
    assert len(_cabi.EXPORTS["lsnf_ais_run"][1]) == 17
