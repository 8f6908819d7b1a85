"""Linear measurements y = A vec(G(z)) + sigma noise on the CPU, for the tests of measured inference: the Langevin
closure, one evaluation of its reconstruction gradient and the AIS energy of ``oracle/refpath.py`` with the
reconstruction term |A vec(G(z)) - y|^2.  The reference has no operator, so these are restatements; they reuse the
oracle's generator and flow prior unchanged.  vec is the NCHW flattening x.view(B, -1); A is [m, nc*H*W] and y [B, m].
Every function takes ``dtype`` (float32 as the reference computes, or float64)."""
from typing import Optional

import numpy as np
import torch

from oracle import refpath


def _cast(d, dtype):
    return {k: v.to(dtype) if v.is_floating_point() else v for k, v in d.items()}


def residual(x_hat: torch.Tensor, y: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    """r = A vec(x_hat) - y, [B, m]."""
    return x_hat.reshape(x_hat.shape[0], -1) @ A.t() - y


def measured_sse(x_hat: torch.Tensor, y: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    """|A vec(x_hat) - y|^2 summed over the batch."""
    r = residual(x_hat, y, A)
    return (r * r).sum()


def langevin(z0: torch.Tensor, y: torch.Tensor, A: torch.Tensor, gp, fp, layers, *, depth: int, steps: int,
             step_size: float, sigma: float, eps: Optional[torch.Tensor], leak: float = 0.2, coupling: int = 1,
             permutation: int = 2, dtype=torch.float32):
    """``refpath.langevin`` on the energy |A vec(G(z)) - y|^2 / (2 sigma^2) - log p(z).  Returns (z_T, mean_b |grad_g|,
    mean_b |grad_f|) of the last step."""
    gp, fp = _cast(gp, dtype), _cast(fp, dtype)
    y, A = y.to(dtype), A.to(dtype)
    z = z0.clone().detach().to(dtype)
    z.requires_grad_(True)
    bsz = z.shape[0]
    gn = fn = None
    for t in range(steps):
        x_hat = refpath.generator_forward(gp, z, layers, leak)
        z_grad_g = torch.autograd.grad(1.0 / (2.0 * sigma * sigma) * measured_sse(x_hat, y, A), z)[0]
        ll, _z1, _ld = refpath.log_prior(fp, z.reshape(bsz, -1), depth, coupling, permutation)
        z_grad_f = torch.autograd.grad(-ll.sum(), z)[0]
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)
        if eps is not None:
            z.data += step_size * eps[t].to(dtype)
        gn = z_grad_g.view(bsz, -1).norm(dim=1).mean()
        fn = z_grad_f.view(bsz, -1).norm(dim=1).mean()
    return z.detach(), gn, fn


def recon_grad(z: torch.Tensor, y: torch.Tensor, A: torch.Tensor, gp, layers, sigma: float, leak: float = 0.2,
               dtype=torch.float32):
    """(x_hat, d/dz [|A vec(G(z)) - y|^2 / (2 sigma^2)])."""
    gp = _cast(gp, dtype)
    z = z.clone().detach().to(dtype).requires_grad_(True)
    x_hat = refpath.generator_forward(gp, z, layers, leak)
    loss = 1.0 / (2.0 * sigma * sigma) * measured_sse(x_hat, y.to(dtype), A.to(dtype))
    return x_hat.detach(), torch.autograd.grad(loss, z)[0]


def energy(gp, fp, layers, y, A, sigma, *, depth=5, coupling=1, permutation=2, leak=0.2):
    """energy(z) -> (l, log p, -dl/dz, -dlog p/dz) in fp64 for ``tests/ais_oracle.ais``, with
    l(z) = -|A vec(G(z)) - y|^2 / (2 sigma^2)."""
    gp, fp = _cast(gp, torch.float64), _cast(fp, torch.float64)
    yt = torch.as_tensor(np.asarray(y), dtype=torch.float64)
    At = torch.as_tensor(np.asarray(A), dtype=torch.float64)

    def f(z):
        zt = torch.tensor(np.asarray(z, np.float64), requires_grad=True)
        r = residual(refpath.generator_forward(gp, zt.reshape(zt.shape[0], -1, 1, 1), layers, leak), yt, At)
        ell = -(r * r).sum(1) / (2.0 * sigma * sigma)
        gr = torch.autograd.grad(-ell.sum(), zt)[0]
        zz = zt.detach().clone().requires_grad_(True)
        lp, _z1, _ld = refpath.log_prior(fp, zz, depth, coupling, permutation)
        gpr = torch.autograd.grad(-lp.sum(), zz)[0]
        return ell.detach().numpy(), lp.detach().numpy(), gr.numpy(), gpr.numpy()
    return f


def identity_rows(mask: np.ndarray) -> np.ndarray:
    """The operator that observes the pixels where the 0/1 ``mask`` [nc,H,W] is 1: one identity row per such pixel."""
    obs = np.flatnonzero(np.asarray(mask).reshape(-1) > 0)
    A = np.zeros((len(obs), np.asarray(mask).size), np.float32)
    A[np.arange(len(obs)), obs] = 1.0
    return A


def avg_pool_operator(nc: int, img: int, f: int = 2) -> np.ndarray:
    """Super-resolution: each row averages one f x f block of one channel (m = n / f^2)."""
    h = img // f
    A = np.zeros((nc * h * h, nc * img * img), np.float32)
    for c in range(nc):
        for by in range(h):
            for bx in range(h):
                row = (c * h + by) * h + bx
                for dy in range(f):
                    for dx in range(f):
                        A[row, (c * img + by * f + dy) * img + bx * f + dx] = 1.0 / (f * f)
    return A


def gaussian_operator(m: int, n: int, seed: int) -> np.ndarray:
    """Compressed sensing: i.i.d. N(0, 1/n) entries, so that every measurement is a projection of about unit norm, as
    a pixel reading is.  (With the column-normalised N(0, 1/m) the posterior at sigma = 0.3 is n/m times sharper and the
    Langevin chain so ill-conditioned that the oracle's own fp32 and fp64 z_T differ by 9e-5 at SVHN, m = n/8, T = 20;
    with N(0, 1/n) by 3e-6.)"""
    return (np.random.default_rng(seed).standard_normal((m, n)) / np.sqrt(n)).astype(np.float32)


def operator_scale_exp(amax) -> int:
    """k of the operator's packed copies (csrc/gen_aux.cu, launch_meas_pack): max|A| 2^k in [1, 2), clamped to
    [-126, 126] so that 2^k and 2^-k are normal fp32 numbers; k = 1 for an all-zero operator."""
    a = np.float32(amax)
    e = int(np.frexp(a)[1]) if a > 0 and np.isfinite(a) else 0   # a = f 2^e, f in [0.5, 1)
    return max(-126, min(126, 1 - e))


def sigma_seed_scale(sigma) -> float:
    """csrc/lsnf_internal.cuh sigma_seed_scale: the power of two of at most 16 of 1/sigma^2 (fp32) r carries."""
    inv = np.float32(1.0) / (np.float32(sigma) * np.float32(sigma))
    s = np.float32(1.0)
    while s * 2 <= inv and s < 16:
        s = np.float32(s * 2)
    return float(s)
