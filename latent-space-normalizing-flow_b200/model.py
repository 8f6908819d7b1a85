"""Host-side mirror of the reference's module interface for the hot path: ``_netG`` (model.py:48-157) and
``_netF`` (model.py:460-498) with the same constructor arguments, ``forward`` signatures, ``state_dict`` keys and
error behaviour, so reference checkpoints load and reference call sites keep working.

Execution:
  * Inference calls (autograd not recording: ``torch.no_grad()``, or ``.eval()`` mode with no input requiring grad)
    run the hand-written CUDA kernels through the C ABI.  Non-CUDA tensors are rejected -- there is no CPU fallback.
  * When autograd IS recording (an input requires grad, or training mode with trainable parameters) the same maths
    run as ordinary differentiable torch ops, so code written against the reference modules (including its own
    autograd-based Langevin closure) keeps working.  That branch is not part of the Langevin path:
    ``sample_langevin_post_z_with_flow`` and ``train.training_iteration`` never take it.
  * Under ``lsnf_b200.kernel_autograd()`` such calls on float32 CUDA tensors instead run the kernels forward and
    their vector-Jacobian products backward (``autograd_fns``); CPU tensors and the reverse flow pass stay eager.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import autograd_fns, synth
from .plan import get_plan


def weights_init_xavier(m):
    """model.py:39-45 (applied by train.py:271-272; a no-op on the lower-case flow classes)."""
    classname = m.__class__.__name__
    if classname.find("Conv") != -1:
        nn.init.xavier_normal_(m.weight)
    elif classname.find("BatchNorm") != -1:
        m.weight.data.normal_(1, 0.02)
        m.bias.data.fill_(0)


def _get(args, name, default=None):
    if isinstance(args, dict):
        return args.get(name, default)
    return getattr(args, name, default)


def _autograd_needed(module: nn.Module, *tensors) -> bool:
    """True when the call has to record an autograd graph: grad mode is on and either an input requires grad (in any
    module mode -- the reference's own Langevin closures differentiate w.r.t. z in eval mode, train.py:565, :602-634)
    or the module is in training mode with trainable parameters (the parameter updates of train.py:390-415)."""
    if not torch.is_grad_enabled():
        return False
    if any(t.requires_grad for t in tensors if isinstance(t, torch.Tensor)):
        return True
    return module.training and any(p.requires_grad for p in module.parameters())


def _kernel_autograd(z) -> bool:
    """A differentiable call takes the kernels' autograd Functions: ``kernel_autograd`` is on and z is float32 CUDA."""
    return autograd_fns.is_enabled() and z.is_cuda and z.dtype == torch.float32


class _netG(nn.Module):
    """Generator: [ConvTranspose2d, Identity, LeakyReLU] * (L-1) + [ConvTranspose2d, Tanh]; parameters live under
    ``gen.<3i>.weight|bias`` exactly as in the reference ``nn.Sequential``."""

    def __init__(self, args):
        super().__init__()
        dataset = _get(args, "dataset")
        if dataset not in ("svhn", "cifar10", "celeba_crop", "celeba_hq256"):
            raise ValueError(dataset)                                   # model.py:154
        if _get(args, "g_batchnorm", False):
            raise NotImplementedError("g_batchnorm=True couples the samples of a batch; the per-sample Langevin "
                                      "path does not support it (SURVEY.md section 2 #12)")
        if _get(args, "g_activation", "lrelu") != "lrelu":
            raise NotImplementedError("only --g_activation lrelu is supported (SURVEY.md section 2 #11)")
        self.dataset = dataset
        self.nz, self.ngf, self.nc = int(_get(args, "nz")), int(_get(args, "ngf")), int(_get(args, "nc", 3))
        self.leak = float(_get(args, "g_activation_leak", 0.2))
        self.layers = synth.generator_layers(dataset, self.nz, self.ngf, self.nc)
        mods = []
        for i, (ci, co, k, s, p) in enumerate(self.layers):
            mods.append(nn.ConvTranspose2d(ci, co, k, s, p, bias=True))
            if i < len(self.layers) - 1:
                mods += [nn.Identity(), nn.LeakyReLU(self.leak)]
            else:
                mods.append(nn.Tanh())
        self.gen = nn.Sequential(*mods)
        self.gemm_impl = 0

    def _plan(self, batch, device, train=False, meas_rows=0):
        # a placeholder flow the generator never runs; the shuffle permutation keeps its footprint free of nz^2, so
        # that plan creation's flow shared-memory check accepts every nz
        return get_plan(arch=self.dataset, batch=batch, nz=self.nz, ngf=self.ngf, nc=self.nc, f_depth=1, f_width=4,
                        f_permutation=1, f_coupling=1, leak=self.leak, device=device, gemm_impl=self.gemm_impl,
                        train=train, meas_rows=meas_rows)

    def generate(self, z):
        """z [B,nz,1,1] or [B,nz] -> x_hat [B,nc,H,W] through the CUDA kernels (never records autograd)."""
        b = z.shape[0]
        z2 = z.detach().reshape(b, self.nz)
        if z2.dtype != torch.float32 or not z2.is_cuda:
            raise RuntimeError("_netG: the kernel path needs a float32 CUDA tensor (no CPU fallback)")
        plan = self._plan(b, z2.device)
        plan.ensure_generator(self)
        return plan.generator_forward(z2.contiguous())

    def forward(self, z):
        if _autograd_needed(self, z):
            if _kernel_autograd(z):
                return autograd_fns.generator_apply(self, z)
            return self.gen(z)
        return self.generate(z)


# ---------------------------------------------------------------------------------------------------------
# flow prior: parameter containers named as in the reference (lower-case class names on purpose, so that
# ``netF.apply(weights_init_xavier)`` stays the no-op it is upstream)
# ---------------------------------------------------------------------------------------------------------
class actnorm(nn.Module):
    def __init__(self, nz):
        super().__init__()
        self.b = nn.Parameter(torch.randn(1, nz) * 0.05)               # model.py:230
        self.register_parameter(name="bias", param=self.b)             # model.py:231 (alias)
        self.logs = nn.Parameter(torch.randn(1, nz) * 0.05)            # model.py:233


class invertible_1x1_conv(nn.Module):
    def __init__(self, nz):
        super().__init__()
        w_init = np.linalg.qr(np.random.randn(nz, nz))[0].astype("float32")   # model.py:176
        self.w = nn.Parameter(torch.tensor(w_init, dtype=torch.float))


class shuffle_features(nn.Module):
    """Fixed channel permutation (intended semantics of model.py:200-225, which is broken upstream)."""

    def __init__(self, nz):
        super().__init__()
        idx = np.random.permutation(nz)
        inv = np.empty_like(idx)
        inv[idx] = np.arange(nz)
        self.indices = nn.Parameter(torch.tensor(idx, dtype=torch.int), requires_grad=False)
        self.indices_inverse = nn.Parameter(torch.tensor(inv, dtype=torch.int), requires_grad=False)


class fc(nn.Module):
    def __init__(self, n_in, width):
        super().__init__()
        self.actnorm = actnorm(width)
        self.w = nn.Parameter(torch.randn(n_in, width) * 0.05)         # model.py:318
        self.b = nn.Parameter(torch.zeros(1, width))                   # never read (model.py:329-330)


class fc_zeros(nn.Module):
    def __init__(self, n_in, width):
        super().__init__()
        self.w = nn.Parameter(torch.zeros(n_in, width))                # model.py:340-342
        self.b = nn.Parameter(torch.zeros(1, width))
        self.logs = nn.Parameter(torch.zeros(1, width))


class f(nn.Module):
    def __init__(self, width, n_in, n_out):
        super().__init__()
        self.fc_1 = fc(n_in, width)
        self.fc_2 = fc(width, width)
        self.fc_zeros = fc_zeros(width, n_out)


class revnet2d_step(nn.Module):
    def __init__(self, hps, nz):
        super().__init__()
        self.actnorm = actnorm(nz)
        perm = int(_get(hps, "f_flow_permutation", 2))
        if perm == 1:
            self.shuffle_features = shuffle_features(nz)
            self.invertible_1x1_conv = None
        elif perm == 2:
            self.invertible_1x1_conv = invertible_1x1_conv(nz)
            self.shuffle_features = None
        else:
            raise Exception()                                           # model.py:379
        assert nz % 2 == 0                                              # model.py:383
        coupling = int(_get(hps, "f_flow_coupling", 1))
        width = int(_get(hps, "f_width", 64))
        if coupling == 0:
            self.f = f(width, nz // 2, nz // 2)
        elif coupling == 1:
            self.f = f(width, nz // 2, nz)
        else:
            raise Exception()                                           # model.py:402 / :420 (raised at call time upstream)


class revnet2d(nn.Module):
    def __init__(self, hps, nz):
        super().__init__()
        self.revnet2d_step_s = nn.ModuleList([revnet2d_step(hps, nz) for _ in range(int(_get(hps, "f_depth", 5)))])


def _an(x, m: actnorm):
    return (x + m.b) * torch.exp(m.logs * 3.0)


def _mlp(st: revnet2d_step, h):
    h = F.relu(_an(h @ st.f.fc_1.w, st.f.fc_1.actnorm))
    h = F.relu(_an(h @ st.f.fc_2.w, st.f.fc_2.actnorm))
    return (h @ st.f.fc_zeros.w + st.f.fc_zeros.b) * torch.exp(st.f.fc_zeros.logs * 3.0)


class _netF(nn.Module):
    """Flow prior; ``forward`` keeps the reference signature (model.py:473)."""

    def __init__(self, hps, nz, *args, **kwargs):
        super().__init__()
        self.hps = hps
        self.nz = int(nz)
        n_levels = int(_get(hps, "f_n_levels", 1))
        levels = []
        for i in range(n_levels):
            levels.append(revnet2d(hps, nz=self.nz))
            if i < n_levels - 1:
                raise NotImplementedError                               # model.py:470
        self.revnet2d_s = nn.ModuleList(levels)
        self.f_depth = int(_get(hps, "f_depth", 5))
        self.f_width = int(_get(hps, "f_width", 64))
        self.f_permutation = int(_get(hps, "f_flow_permutation", 2))
        self.f_coupling = int(_get(hps, "f_flow_coupling", 1))

    def _plan(self, batch, device):
        return get_plan(arch="none", batch=batch, nz=self.nz, ngf=0, nc=3, f_depth=self.f_depth, f_width=self.f_width,
                        f_permutation=self.f_permutation, f_coupling=self.f_coupling, leak=0.2, device=device)

    # ---- kernel path ----
    def _kernel_input(self, z):
        assert len(z.shape) == 2                                        # model.py:237
        if z.dtype != torch.float32 or not z.is_cuda:
            raise RuntimeError("_netF: the kernel path needs a float32 CUDA tensor (no CPU fallback)")
        return z.detach().contiguous()

    def log_prior(self, z, want_grad=False):
        """(z_out, logdet, log p(z), d(-sum log p)/dz or None) of train.py:316-323 through the fused kernel."""
        z = self._kernel_input(z)
        plan = self._plan(z.shape[0], z.device)
        plan.ensure_flow(self)
        return plan.flow_forward(z, want_grad)

    def inverse(self, eps):
        """(z, -objective) of the reverse pass (model.py:484-498) through the fused kernel; eps is not modified."""
        eps = self._kernel_input(eps)
        plan = self._plan(eps.shape[0], eps.device)
        plan.ensure_flow(self, need_inverse=True)
        return plan.flow_inverse(eps)

    # ---- differentiable torch path (parameter updates only) ----
    def _eager(self, z, objective, reverse):
        n = self.nz
        steps = self.revnet2d_s[0].revnet2d_step_s
        if not reverse:
            for st in steps:
                z = _an(z, st.actnorm)
                objective = objective + torch.sum(st.actnorm.logs * 3.0)
                if st.invertible_1x1_conv is not None:
                    w = st.invertible_1x1_conv.w
                    z = z @ w
                    objective = objective + torch.log(torch.abs(torch.det(w.double()))).float()
                else:
                    z = z.index_select(1, st.shuffle_features.indices.long())
                z1, z2 = z[:, : n // 2], z[:, n // 2:]
                h = _mlp(st, z1)
                if self.f_coupling == 0:
                    z2 = z2 + h
                else:
                    scale = torch.sigmoid(h[:, 1::2] + 2.0)
                    z2 = (z2 + h[:, 0::2]) * scale
                    objective = objective + torch.sum(torch.log(scale), dim=1)
                z = torch.cat([z1, z2], 1)
            return z, objective
        for st in reversed(list(steps)):
            z1, z2 = z[:, : n // 2], z[:, n // 2:]
            h = _mlp(st, z1)
            if self.f_coupling == 0:
                z2 = z2 - h
            else:
                scale = torch.sigmoid(h[:, 1::2] + 2.0)
                z2 = z2 / scale - h[:, 0::2]
                objective = objective - torch.sum(torch.log(scale), dim=1)
            z = torch.cat([z1, z2], 1)
            if st.invertible_1x1_conv is not None:
                w = st.invertible_1x1_conv.w
                z = z @ torch.inverse(w)
                objective = objective - torch.log(torch.abs(torch.det(w.double()))).float()
            else:
                z = z.index_select(1, st.shuffle_features.indices_inverse.long())
            z = z * torch.exp(-st.actnorm.logs * 3.0) - st.actnorm.b
            objective = objective - torch.sum(st.actnorm.logs * 3.0)
        return z, objective

    def forward(self, z, objective, init=False, reverse=False, eps=None, eps_std=None, z2_s=None, return_obj=False):
        if init:
            raise NotImplementedError("data-dependent actnorm init is never enabled upstream (train.py:316,406,614)")
        if _autograd_needed(self, z, objective):
            if not reverse and _kernel_autograd(z):
                assert len(z.shape) == 2                                # model.py:237
                z_out, logdet = autograd_fns.flow_apply(self, z)
                return z_out, objective + logdet, []                   # model.py:483
            z, objective = self._eager(z, objective, reverse)
            if not reverse:
                return z, objective, []
            return (z, -objective) if return_obj else z
        if not reverse:
            z_out, logdet, _logp, _ = self.log_prior(z)
            return z_out, objective + logdet, []                       # model.py:483
        z_out, negobj = self.inverse(z)
        if not return_obj:
            return z_out                                                # model.py:496
        return z_out, negobj - objective                                # model.py:498
