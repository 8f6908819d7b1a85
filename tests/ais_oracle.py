"""Annealed importance sampling with Metropolis-adjusted Langevin (MALA) transitions, restated in numpy for the tests of
``lsnf_ais_run`` (include/lsnf.h).  The algorithm runs over a generic ``energy(z) -> (l, log p, -dl/dz, -dlog p/dz)``
callable, with injected proposal noise ``eps`` [T,N,nz] and uniforms ``u`` [T,N], and the library's step-size
adaptation.  Its two users: the reference's generator and flow prior from ``oracle/refpath.py`` (``refpath_energy``,
autograd gradients) and a linear-Gaussian model whose log p(x) is analytic (``LinearGaussian``).

The state is kept in fp32 as the kernels keep it; with ``round_z`` each proposal is rounded to its fp16 hi|lo value
(the point the first generator layer reads)."""
from __future__ import annotations

import math

import numpy as np
import torch

KAPPA, STEP_MIN, STEP_MAX = 0.05, 1e-5, 10.0   # csrc/lsnf_internal.cuh: AIS_KAPPA, AIS_STEP_MIN, AIS_STEP_MAX


def round_hl(v: np.ndarray) -> np.ndarray:
    """fp32 -> the value of its fp16 hi|lo split, hi + lo (split16 in csrc/lsnf_internal.cuh)."""
    v = np.asarray(v, np.float32)
    hi = v.astype(np.float16)
    lo = (v - hi.astype(np.float32)).astype(np.float16)
    return (hi.astype(np.float32) + lo.astype(np.float32)).astype(np.float32)


def ais(z0, energy, betas, *, step_size, target_accept=0.0, eps, u, round_z=True):
    """Returns dict(z [N,nz], logw [N] fp64, accepts [N], margin [N] = min_t |log u - log alpha|, step [N])."""
    betas = np.asarray(betas, np.float32)
    T = len(betas) - 1
    rnd = round_hl if round_z else (lambda a: np.asarray(a, np.float32))
    z = rnd(z0)
    ell, lp, gr, gp = energy(z)
    N = z.shape[0]
    s = np.full(N, step_size, np.float32)
    logw = np.zeros(N)
    acc = np.zeros(N, np.int64)
    margin = np.full(N, np.inf)
    zp = e2 = None
    for k in range(T + 1):
        if k >= 1:
            beta = np.float64(betas[k])
            ell1, lp1, gr1, gp1 = energy(zp)
            h = (0.5 * s.astype(np.float64) ** 2)[:, None]
            r = z.astype(np.float64) - zp + h * (gp1 + beta * gr1)
            rk = (r * r).sum(1)
            u0 = -lp - beta * ell
            u1 = -lp1 - beta * ell1
            with np.errstate(invalid="ignore", over="ignore"):
                la = u0 - u1 - rk / (2.0 * s.astype(np.float64) ** 2) + e2
            logu = np.log(np.asarray(u[k - 1], np.float32).astype(np.float64))
            ok = np.isfinite(u1) & np.isfinite(la) & (logu < la)
            margin = np.minimum(margin, np.where(np.isfinite(la), np.abs(logu - la), np.inf))
            z = np.where(ok[:, None], zp, z).astype(np.float32)
            ell, lp = np.where(ok, ell1, ell), np.where(ok, lp1, lp)
            gr, gp = np.where(ok[:, None], gr1, gr), np.where(ok[:, None], gp1, gp)
            acc += ok
            if target_accept > 0:
                with np.errstate(over="ignore"):
                    a = np.where(np.isfinite(u1) & ~np.isnan(la), np.where(la >= 0, 1.0, np.exp(np.minimum(la, 0))), 0.0)
                s = np.clip(s.astype(np.float64) * np.exp(KAPPA * (a - target_accept)), STEP_MIN,
                            STEP_MAX).astype(np.float32)
        if k == T:
            break
        logw += (np.float64(betas[k + 1]) - np.float64(betas[k])) * ell
        e = np.asarray(eps[k], np.float64)
        h = (0.5 * s.astype(np.float64) ** 2)[:, None]
        zp = rnd(z - h * (gp + np.float64(betas[k + 1]) * gr) + s[:, None].astype(np.float64) * e)
        e2 = 0.5 * (e * e).sum(1)
    return dict(z=z, logw=logw, accepts=acc, margin=margin, step=s)


def logmeanexp(a, axis=-1):
    a = np.asarray(a, np.float64)
    m = a.max(axis=axis, keepdims=True)
    return (m + np.log(np.mean(np.exp(a - m), axis=axis, keepdims=True))).squeeze(axis)


def sigmoid_schedule(T, delta=4.0):
    t = np.arange(T + 1, dtype=np.float64)
    s = 1.0 / (1.0 + np.exp(-delta * (2.0 * t / T - 1.0)))
    return (s - s[0]) / (s[-1] - s[0])


class LinearGaussian:
    """z ~ N(0, I_d), x | z ~ N(W z + c, sigma^2 / m) per dimension: log p(x) is that of N(c, W W^T + sigma^2 M^-1)."""

    def __init__(self, d=4, D=8, sigma=0.5, seed=0):
        r = np.random.default_rng(seed)
        self.W = r.normal(size=(D, d)) * 0.8
        self.c = r.normal(size=D) * 0.1
        self.sigma, self.d, self.D = sigma, d, D

    def sample(self, n, seed=1):
        r = np.random.default_rng(seed)
        z = r.normal(size=(n, self.d))
        return z, z @ self.W.T + self.c + self.sigma * r.normal(size=(n, self.D))

    def energy(self, x):
        """energy(z) for chains whose rows are observations x [N, D]."""
        W, c, s2, d = self.W, self.c, self.sigma ** 2, self.d

        def f(z):
            z = np.asarray(z, np.float64)
            res = z @ W.T + c - x
            ell = -(res * res).sum(1) / (2 * s2)
            lp = -0.5 * (z * z).sum(1) - 0.5 * d * math.log(2 * math.pi)
            return ell, lp, res @ W / s2, z
        return f

    def log_px(self, x):
        S = self.W @ self.W.T + self.sigma ** 2 * np.eye(self.D)
        r = x - self.c
        _, ld = np.linalg.slogdet(S)
        return -0.5 * (np.einsum("ni,ij,nj->n", r, np.linalg.inv(S), r) + ld + self.D * math.log(2 * math.pi))

    def posterior_sample(self, x, rng):
        P = np.eye(self.d) + self.W.T @ self.W / self.sigma ** 2
        Sig = np.linalg.inv(P)
        mu = (x - self.c) @ self.W @ Sig / self.sigma ** 2
        return mu + rng.normal(size=mu.shape) @ np.linalg.cholesky(Sig).T

    def C(self):
        return -0.5 * self.D * math.log(2 * math.pi * self.sigma ** 2)


def refpath_energy(gp, fp, layers, x, sigma, mask=None, *, depth=5, coupling=1, permutation=2, leak=0.2):
    """energy(z) of the reference's generator and flow prior (oracle/refpath.py) in fp64 for chains with observations
    x [N,nc,H,W] and per-pixel weights ``mask`` (None = 1)."""
    from oracle import refpath
    gp = {k: v.double() if v.is_floating_point() else v for k, v in gp.items()}
    fp = {k: v.double() if v.is_floating_point() else v for k, v in fp.items()}
    xt = torch.as_tensor(np.asarray(x), dtype=torch.float64)
    mt = None if mask is None else torch.as_tensor(np.asarray(mask), dtype=torch.float64)

    def f(z):
        zt = torch.tensor(np.asarray(z, np.float64), requires_grad=True)
        d = refpath.generator_forward(gp, zt.reshape(zt.shape[0], -1, 1, 1), layers, leak) - xt
        dd = d * d if mt is None else mt * d * d
        ell = -dd.flatten(1).sum(1) / (2.0 * sigma * sigma)
        gr = torch.autograd.grad(-ell.sum(), zt)[0]
        zt2 = torch.tensor(np.asarray(z, np.float64), requires_grad=True)
        lp, _z1, _ld = refpath.log_prior(fp, zt2, depth, coupling, permutation)
        gp_ = torch.autograd.grad(-lp.sum(), zt2)[0]
        return ell.detach().numpy(), lp.detach().numpy(), gr.numpy(), gp_.numpy()
    return f


def philox_uniform(seed: int, sample0: int, batch: int, step: int) -> np.ndarray:
    """float32 [batch]: the uniform of the decision made at loop iteration ``step`` (counter quad 0xFFFFFFFF, which no
    Gaussian draw uses; ``oracle/philox.py`` has the generator and the Gaussian draws)."""
    from oracle.philox import MASK, philox4x32_10
    sample = np.arange(batch, dtype=np.uint64) + np.uint64(sample0)
    ctr = np.stack([sample & MASK, sample >> np.uint64(32), np.full(batch, step, np.uint64),
                    np.full(batch, 0xFFFFFFFF, np.uint64)], axis=-1).astype(np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    bits = philox4x32_10(ctr, key)[:, 0]
    return (((bits >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)).astype(np.float32)
