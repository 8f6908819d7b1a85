"""Marginal likelihood log p(x) of a trained model by annealed importance sampling (AIS) with Metropolis-adjusted
Langevin transitions, on the fused kernels (``lsnf_ais_run``, include/lsnf.h), and its bidirectional check BDMC.

The prior is a normalizing flow, so log p(z) is exact and log p(x) = log int p(x|z) p(z) dz is well defined.  Forward
AIS from exact prior samples gives a stochastic lower bound on it; reverse AIS from an exact posterior sample (available
for data simulated from the model) gives a stochastic upper bound (Grosse, Ghahramani and Adams 2015; Wu et al. 2017).
"""
from __future__ import annotations

import itertools
import math
from typing import Optional

import numpy as np
import torch

from .langevin import langevin_plan
from .model import _get

_call_counter = itertools.count()


def sigmoid_schedule(steps: int, delta: float = 4.0) -> np.ndarray:
    """The sigmoidal schedule of Grosse et al.: beta_t proportional to sigmoid(delta (2t/T - 1)), rescaled so that
    beta_0 = 0 and beta_T = 1.  Returns float64 [steps + 1], increasing."""
    if steps < 1:
        raise ValueError("steps must be at least 1")
    t = np.arange(steps + 1, dtype=np.float64)
    s = 1.0 / (1.0 + np.exp(-delta * (2.0 * t / steps - 1.0)))
    b = (s - s[0]) / (s[-1] - s[0])
    b[0], b[-1] = 0.0, 1.0
    return b


def log_likelihood_constant(sigma: float, shape, mask: Optional[torch.Tensor] = None) -> np.ndarray:
    """C = -1/2 sum_{i: m_i > 0} log(2 pi sigma^2 / m_i) per image, fp64 [B]: the normaliser of the Gaussian likelihood
    p(x|z) with per-pixel precision m_i / sigma^2 (-(D/2) log(2 pi sigma^2) without a mask).  ``shape`` is x's."""
    B = int(shape[0])
    D = int(np.prod(shape[1:]))
    l2ps = math.log(2.0 * math.pi * float(sigma) ** 2)
    if mask is None:
        return np.full(B, -0.5 * D * l2ps)
    m = mask.detach().double().expand(tuple(shape)).reshape(B, -1).cpu().numpy()
    obs = m > 0
    with np.errstate(divide="ignore"):
        lm = np.where(obs, np.log(np.where(obs, m, 1.0)), 0.0)
    return -0.5 * (obs.sum(1) * l2ps - lm.sum(1))


def logmeanexp(a: torch.Tensor, dim: int = -1) -> torch.Tensor:
    """log mean exp along ``dim`` in fp64."""
    a = a.double()
    return torch.logsumexp(a, dim=dim) - math.log(a.shape[dim])


def _check_schedule(schedule, steps: int) -> np.ndarray:
    b = np.asarray(schedule.detach().cpu() if isinstance(schedule, torch.Tensor) else schedule, dtype=np.float64)
    if b.ndim != 1 or b.shape[0] != steps + 1:
        raise ValueError(f"schedule must hold steps + 1 = {steps + 1} values (got shape {b.shape})")
    if not np.all(np.isfinite(b)) or b.min() < 0.0 or b.max() > 1.0:
        raise ValueError("schedule values must lie in [0, 1]")
    return b


def _ais_chains(x, netG, netF, args, z0, *, chains, steps, betas, step_size, target_accept, mask, seed):
    """AIS on the plan of batch B * chains: chain c of image b is row b * chains + c.  ``z0`` [B*chains, nz] or None
    (exact prior samples F^-1(eps)).  Returns (z_T, log w [B, chains], acceptance rate [B, chains], mask rows)."""
    B = x.shape[0]
    n = B * chains
    sigma = float(_get(args, "g_llhd_sigma", 0.3))
    s0 = float(_get(args, "g_l_step_size", 0.1)) if step_size is None else float(step_size)
    plan = langevin_plan(netG, netF, n, x.device, 3)
    plan.ensure_generator(netG)
    plan.ensure_flow(netF, need_inverse=True)
    xx = x.detach().float().repeat_interleave(chains, 0).contiguous()
    mm = None
    if mask is not None:
        from .plan import as_mask
        mm = as_mask(mask, x).repeat_interleave(chains, 0).contiguous()
    gen = torch.Generator(device=x.device)
    gen.manual_seed(int(seed) & (2 ** 63 - 1))
    if z0 is None:
        eps = torch.randn(n, netG.nz, device=x.device, generator=gen)
        z0 = plan.flow_inverse(eps)[0]
    bt = torch.as_tensor(betas, dtype=torch.float32).to(x.device).contiguous()
    t = 0.0 if target_accept is None else float(target_accept)
    z, lw, rate = plan.ais_run(z0.contiguous(), xx, bt, steps, s0, sigma, target_accept=t, mask=mm, seed=seed)
    return z, lw.view(B, chains), rate.view(B, chains)


def _validate(x, chains, steps, schedule):
    if int(chains) < 1:
        raise ValueError("chains must be at least 1")
    if int(steps) < 1:
        raise ValueError("steps must be at least 1")
    betas = sigmoid_schedule(int(steps)) if schedule is None else _check_schedule(schedule, int(steps))
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise RuntimeError("x must be a CUDA tensor: AIS runs on the fused kernels and has no CPU fallback")
    return betas


def ais_log_likelihood(x: torch.Tensor, netG, netF, args, *, chains: int, steps: int, schedule=None,
                       step_size: Optional[float] = None, target_accept: Optional[float] = 0.65,
                       mask: Optional[torch.Tensor] = None, seed: Optional[int] = None):
    """Forward AIS estimate of log p(x) for every image of x [B,nc,H,W]: ``chains`` chains per image from exact prior
    samples z_0 = F^-1(eps), ``steps`` MALA transitions along ``schedule`` (steps + 1 values in [0, 1], 0 -> 1; default
    the sigmoidal schedule of Grosse et al. with delta = 4).  sigma is ``args.g_llhd_sigma``; the initial step size
    ``args.g_l_step_size`` unless ``step_size`` is given; ``target_accept`` (None or <= 0: fixed) adapts it per chain.
    ``mask`` weights the likelihood per pixel as in ``sample_langevin_post_z_with_flow``.

    Returns (log_px [B] fp64, log_w [B, chains], accept_rate [B, chains]); log_px = logmeanexp over the chains of log w
    plus the likelihood's normaliser C (``log_likelihood_constant``).  E[log_px] <= log p(x): a stochastic lower bound
    that tightens as ``steps`` grows."""
    betas = _validate(x, chains, steps, schedule)
    if seed is None:
        seed = (int(_get(args, "seed", 1)) << 32) ^ (0x5A15 << 16) ^ next(_call_counter)
    sigma = float(_get(args, "g_llhd_sigma", 0.3))
    _, lw, rate = _ais_chains(x, netG, netF, args, None, chains=int(chains), steps=int(steps), betas=betas,
                              step_size=step_size, target_accept=target_accept, mask=mask, seed=seed)
    c = torch.from_numpy(log_likelihood_constant(sigma, tuple(x.shape), mask)).to(x.device)
    return logmeanexp(lw, 1) + c, lw, rate


def bdmc(netG, netF, args, n: int, *, chains: int, steps: int, schedule=None, step_size: Optional[float] = None,
         target_accept: Optional[float] = 0.65, seed: Optional[int] = None, device=None):
    """Bidirectional Monte Carlo on ``n`` images simulated from the model: z ~ p(z) (z = F^-1(eps)), x = G(z) + sigma
    noise.  Forward AIS gives a stochastic lower bound on each log p(x); reverse AIS, started from the true z (an exact
    posterior sample) along the reversed schedule, gives a stochastic upper bound.  The gap between the two bounds
    the error of either estimate on data like the model's own.  Returns (lower [n], upper [n], x [n,nc,H,W])."""
    if int(n) < 1:
        raise ValueError("n must be at least 1")
    if device is None:
        device = next(netG.parameters()).device
    device = torch.device(device)
    betas = _validate(torch.empty(0, device=device), chains, steps, schedule)
    if seed is None:
        seed = (int(_get(args, "seed", 1)) << 32) ^ (0xBD3C << 16) ^ next(_call_counter)
    sigma = float(_get(args, "g_llhd_sigma", 0.3))
    gen = torch.Generator(device=device)
    gen.manual_seed((int(seed) ^ 0x9E3779B97F4A7C15) & (2 ** 63 - 1))
    plan = langevin_plan(netG, netF, int(n), device, 3)
    plan.ensure_generator(netG)
    plan.ensure_flow(netF, need_inverse=True)
    z = plan.flow_inverse(torch.randn(int(n), netG.nz, device=device, generator=gen))[0]
    x = plan.generator_forward(z) + sigma * torch.randn(int(n), netG.nc, plan.img, plan.img, device=device,
                                                        generator=gen)
    c = torch.from_numpy(log_likelihood_constant(sigma, tuple(x.shape))).to(device)
    _, lw_f, _ = _ais_chains(x, netG, netF, args, None, chains=int(chains), steps=int(steps), betas=betas,
                             step_size=step_size, target_accept=target_accept, mask=None, seed=seed)
    z0 = z.repeat_interleave(int(chains), 0)
    _, lw_r, _ = _ais_chains(x, netG, netF, args, z0, chains=int(chains), steps=int(steps), betas=betas[::-1].copy(),
                             step_size=step_size, target_accept=target_accept, mask=None, seed=seed + 1)
    return logmeanexp(lw_f, 1) + c, -logmeanexp(lw_r, 1) + c, x
