"""``sample_langevin_post_z_with_flow`` -- the reference closure (train.py:307-335; test variant :602-634) as one
call into the CUDA library.  No autograd, no per-step Python: the whole ``g_l_steps`` loop is enqueued by
``lsnf_langevin_run`` on the caller's current stream."""
from __future__ import annotations

import itertools
from typing import Optional

import torch

from .model import _get, _netF, _netG
from .plan import default_bwd_passes, get_plan

_call_counter = itertools.count()


class AttrDict(dict):
    """Same access pattern as the reference's ``AttrDict`` (train.py:743-746)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.__dict__ = self


def make_args(**overrides) -> AttrDict:
    """Defaults of train.py:37-99 (``cli.FLAGS``); ``overrides`` use the CLI flag names."""
    from .cli import defaults
    a = AttrDict(defaults())
    unknown = set(overrides) - set(a) - {"device", "job_id", "status"}
    if unknown:
        raise TypeError(f"unknown argument(s): {sorted(unknown)}")
    a.update(overrides)
    return a


def langevin_plan(netG: _netG, netF: _netF, batch: int, device, bwd_passes: Optional[int] = None, train: bool = False):
    """The plan (workspace, packed parameters, CUDA graphs) of one (netG, netF, batch) configuration; ``train=True``
    adds the buffers of the generator parameter update so that one plan serves a whole training iteration."""
    return get_plan(arch=netG.dataset, batch=batch, nz=netG.nz, ngf=netG.ngf, nc=netG.nc, f_depth=netF.f_depth,
                    f_width=netF.f_width, f_permutation=netF.f_permutation, f_coupling=netF.f_coupling,
                    leak=netG.leak, device=device, gemm_impl=netG.gemm_impl, bwd_passes=bwd_passes, train=train)


def sample_langevin_post_z_with_flow(z, x, netG: _netG, netF: _netF, args, verbose: bool = False, *,
                                     eps: Optional[torch.Tensor] = None, steps: Optional[int] = None,
                                     with_noise: Optional[bool] = None, seed: Optional[int] = None,
                                     sample_offset: int = 0, bwd_passes: Optional[int] = None, train: bool = False,
                                     mask: Optional[torch.Tensor] = None):
    """z [B,nz,1,1], x [B,nc,H,W] -> (z_k [B,nz,1,1], mean_b|grad_g|, mean_b|grad_f|) as train.py:335 returns them.

    ``args`` supplies g_l_steps, g_l_step_size, g_l_with_noise, g_llhd_sigma (train.py:311-326).  ``eps``
    [steps,B,nz,1,1] injects the noise (parity runs); otherwise noise is drawn in-kernel from Philox keyed by
    (seed, sample_offset + b, step), so a sharded batch draws exactly the noise of the unsharded one (the latents
    then agree up to fp32 summation order: split-K / stream-K cut points depend on the tile count).  The
    diagnostics use the real batch size (the reference's ``view(args.batch_size, -1)`` breaks on a ragged batch).
    ``bwd_passes``: tensor-core passes of the reconstruction-gradient GEMMs: 3 (fp32-equivalent hi|lo split) unless
    the caller opts in to the single fp16 pass with 1 (``plan.default_bwd_passes``).
    ``mask``: per-pixel likelihood weight m for partly observed images (inpainting, occluded pixels): the energy
    becomes 1/(2 sigma^2) sum m (G(z) - x)^2 - log p(z), with 1 = observed, 0 = missing and fractions in [0, 1]
    allowed.  Any shape that broadcasts to x's, any real or bool dtype (``plan.as_mask``).  |grad_g| is then the
    norm of the masked gradient.
    """
    if not isinstance(netG, _netG) or not isinstance(netF, _netF):
        raise TypeError("netG / netF must be lsnf_b200._netG / _netF instances")
    if not (z.is_cuda and x.is_cuda):
        raise RuntimeError("sample_langevin_post_z_with_flow needs CUDA tensors: there is no CPU fallback")
    B = z.shape[0]
    if netF.nz != netG.nz:
        raise ValueError("netG and netF disagree on nz")
    T = int(_get(args, "g_l_steps", 20) if steps is None else steps)
    s = float(_get(args, "g_l_step_size", 0.1))
    sigma = float(_get(args, "g_llhd_sigma", 0.3))
    noise = bool(_get(args, "g_l_with_noise", True)) if with_noise is None else bool(with_noise)
    z2 = z.detach().reshape(B, netG.nz).contiguous().float()
    xx = x.detach().contiguous().float()
    e = None
    if eps is not None:
        e = eps.detach().reshape(T, B, netG.nz).contiguous().float()
    if seed is None:
        seed = (int(_get(args, "seed", 1)) << 32) ^ next(_call_counter)
    noisy = noise or eps is not None
    if bwd_passes is None:
        bwd_passes = default_bwd_passes(noisy_chain=noisy)
    plan = langevin_plan(netG, netF, B, z2.device, bwd_passes, train=train)
    plan.ensure_generator(netG)
    plan.ensure_flow(netF)
    out, norms = plan.langevin_run(z2, xx, T, s, sigma, with_noise=noise, eps=e, seed=seed,
                                   sample_offset=sample_offset, mask=mask)
    if verbose:
        print("Langevin posterior: z_grad_g_grad_norm={:8.3f}, z_grad_f_grad_norm={:8.3f}".format(
            norms[0].item(), norms[1].item()))
    return out.reshape(B, netG.nz, 1, 1), norms[0], norms[1]


def make_sampler(args, test_mode: bool = False):
    """Closure with the reference's exact signature ``f(z, x, netG, netF, verbose=False)``, plus the keyword-only
    ``mask`` of ``sample_langevin_post_z_with_flow``.

    ``test_mode=True`` reproduces the test variant: ``g_l_steps * 20`` iterations and no noise
    (train.py:606, :623-625)."""
    def sampler(z, x, netG, netF, verbose=False, *, mask=None):
        if test_mode:
            return sample_langevin_post_z_with_flow(z, x, netG, netF, args, verbose,
                                                    steps=int(_get(args, "g_l_steps", 20)) * 20, with_noise=False,
                                                    mask=mask)
        return sample_langevin_post_z_with_flow(z, x, netG, netF, args, verbose, mask=mask)
    return sampler


def sample_x(netG: _netG, netF: _netF, n: int, device, generator: Optional[torch.Generator] = None,
             eps: Optional[torch.Tensor] = None, to_unit_range: bool = True):
    """Prior sampling of train.py:565-576 as ONE call into the library (``lsnf_sample_prior``): eps ~ N(0,I) ->
    z = F^-1(eps) -> x = G(z) -> clamp((x + 1) / 2, 0, 1) applied in the store of the last generator kernel.
    ``eps`` [n,nz] may be supplied (parity runs); otherwise it is drawn from ``generator``."""
    if eps is None:
        eps = torch.randn(n, netG.nz, device=device, generator=generator)
    eps = eps.detach().reshape(n, netG.nz).contiguous().float()
    if netF.nz != netG.nz:
        raise ValueError("netG and netF disagree on nz")
    plan = langevin_plan(netG, netF, n, eps.device, default_bwd_passes())
    plan.ensure_generator(netG)
    plan.ensure_flow(netF, need_inverse=True)
    return plan.sample_prior(eps, to_unit_range=to_unit_range)


def reconstruction_error(batches, netG: _netG, netF: _netF, args, generator: Optional[torch.Generator] = None) -> float:
    """The reconstruction report of test mode (train.py:641-662): for every batch ``x`` [B,nc,H,W] on the GPU,
    z_0 ~ N(0,I), z_k = test-mode Langevin (``g_l_steps * 20`` noise-free iterations), x_hat = G(z_k); returns the
    mean over batches of ``mse_sum(x_hat, x) / B / nc / H / W`` (the reference divides by ``3 * img_size**2``)."""
    sampler = make_sampler(args, test_mode=True)
    total, n = 0.0, 0
    for x in batches:
        z0 = torch.randn(x.shape[0], netG.nz, 1, 1, device=x.device, generator=generator)
        z_k = sampler(z0, x, netG, netF)[0]
        x_hat = netG.generate(z_k.reshape(x.shape[0], netG.nz))
        total += float(((x_hat - x) ** 2).sum().item()) / x.shape[0] / x.shape[1] / x.shape[2] / x.shape[3]
        n += 1
    if n == 0:
        raise ValueError("no batches")
    return total / n

