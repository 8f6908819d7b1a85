"""The two parameter updates of one training iteration from linear measurements y = A vec(G(z)) + sigma noise on the
CPU, for the tests of measured training: ``oracle/refpath.py``'s ``parameter_updates`` (train.py:390-415) with
loss_g = |A vec(G(z_k)) - y|^2 / B in place of mse_sum(G(z_k), x) / B.  The reference has no operator, so this is a
restatement, in the manner of ``masked_oracle.parameter_updates``; the inference half is ``measured_oracle.langevin``.
vec is the NCHW flattening x.view(B, -1); A is [m, nc*H*W] and y [B, m]."""
import torch

from oracle import refpath
from measured_oracle import measured_sse


def generator_loss(gp, z_k: torch.Tensor, y: torch.Tensor, A: torch.Tensor, layers, leak: float = 0.2):
    """loss_g = |A vec(G(z_k)) - y|^2 / B, in the dtype of ``gp``'s tensors (y and A are cast to it)."""
    dtype = next(iter(gp.values())).dtype
    x_hat = refpath.generator_forward(gp, z_k.detach().to(dtype), layers, leak)
    return measured_sse(x_hat, y.to(dtype), A.to(dtype)) / y.shape[0]


def parameter_updates(gp, fp, z_k: torch.Tensor, y: torch.Tensor, A: torch.Tensor, layers, optG, optF, *, depth: int,
                      leak: float = 0.2, coupling: int = 1, permutation: int = 2):
    """``refpath.parameter_updates`` with the measured generator loss; the flow update is the oracle's.  ``gp`` / ``fp``
    map state_dict keys to leaf tensors that ``optG`` / ``optF`` were built on.  Returns (loss_g, loss_f)."""
    bsz = y.shape[0]
    optG.zero_grad()
    loss_g = generator_loss(gp, z_k, y, A, layers, leak)
    loss_g.backward()
    optG.step()
    optF.zero_grad()
    ll, _z1, _ld = refpath.log_prior(fp, torch.squeeze(z_k.detach()).reshape(bsz, -1), depth, coupling, permutation)
    loss_f = -ll.mean()
    loss_f.backward()
    optF.step()
    return loss_g.detach(), loss_f.detach()
