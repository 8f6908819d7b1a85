"""The masked reconstruction loss on the CPU, for the tests of masked inference: the Langevin closure, one evaluation of
its reconstruction gradient and the two parameter updates of ``oracle/refpath.py`` with the reconstruction term
weighted per pixel, sum m (G(z) - x)^2.  The reference has no mask, so these are restatements; they reuse the oracle's
generator and flow prior unchanged, and with an all-ones ``mask`` they compute what the oracle's own functions compute.
``mask`` has x's shape [B,nc,H,W]."""
from typing import Optional

import torch

from oracle import refpath


def masked_sse(x_hat: torch.Tensor, x: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """sum m (x_hat - x)^2."""
    d = x_hat - x
    return (mask * d * d).sum()


def langevin(z0: torch.Tensor, x: torch.Tensor, mask: torch.Tensor, gp, fp, layers, *, depth: int, steps: int,
             step_size: float, sigma: float, eps: Optional[torch.Tensor], leak: float = 0.2, coupling: int = 1,
             permutation: int = 2, trace: Optional[list] = None):
    """``refpath.langevin`` on the energy 1/(2 sigma^2) sum m (G(z) - x)^2 - log p(z).  Returns (z_T, mean_b |grad_g|,
    mean_b |grad_f|) of the last step."""
    z = z0.clone().detach()
    z.requires_grad_(True)
    bsz = z.shape[0]
    gn = fn = None
    for t in range(steps):
        x_hat = refpath.generator_forward(gp, z, layers, leak)
        z_grad_g = torch.autograd.grad(1.0 / (2.0 * sigma * sigma) * masked_sse(x_hat, x, mask), z)[0]
        ll, _z1, _ld = refpath.log_prior(fp, z.reshape(bsz, -1), depth, coupling, permutation)
        z_grad_f = torch.autograd.grad(-ll.sum(), z)[0]
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)
        if eps is not None:
            z.data += step_size * eps[t]
        gn = z_grad_g.view(bsz, -1).norm(dim=1).mean()
        fn = z_grad_f.view(bsz, -1).norm(dim=1).mean()
        if trace is not None:
            trace.append(z.detach().clone())
    return z.detach(), gn, fn


def recon_grad(z: torch.Tensor, x: torch.Tensor, mask: torch.Tensor, gp, layers, sigma: float, leak: float = 0.2):
    """``refpath.recon_grad`` of the weighted term: (x_hat, d/dz [1/(2 sigma^2) * sum m (G(z) - x)^2])."""
    z = z.clone().detach().requires_grad_(True)
    x_hat = refpath.generator_forward(gp, z, layers, leak)
    loss = 1.0 / (2.0 * sigma * sigma) * masked_sse(x_hat, x, mask)
    return x_hat.detach(), torch.autograd.grad(loss, z)[0]


def parameter_updates(gp, fp, z_k: torch.Tensor, x: torch.Tensor, mask: torch.Tensor, layers, optG, optF, *, depth: int,
                      leak: float = 0.2, coupling: int = 1, permutation: int = 2):
    """``refpath.parameter_updates`` with loss_g = sum m (G(z_k) - x)^2 / B; the flow update is the oracle's.  ``gp`` /
    ``fp`` map state_dict keys to leaf tensors that ``optG`` / ``optF`` were built on.  Returns (loss_g, loss_f)."""
    bsz = x.shape[0]
    optG.zero_grad()
    loss_g = masked_sse(refpath.generator_forward(gp, z_k.detach(), layers, leak), x, mask) / bsz
    loss_g.backward()
    optG.step()
    optF.zero_grad()
    ll, _z1, _ld = refpath.log_prior(fp, torch.squeeze(z_k.detach()).reshape(bsz, -1), depth, coupling, permutation)
    loss_f = -ll.mean()
    loss_f.backward()
    optF.step()
    return loss_g.detach(), loss_f.detach()
