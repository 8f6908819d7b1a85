"""Autograd through the kernels: ``torch.autograd.Function``s whose backward passes are the library's vector-Jacobian
products (``lsnf_generator_vjp``, ``lsnf_flow_vjp``), so that code which differentiates ``_netG`` / ``_netF`` for any
loss -- the reference's own Langevin closure (train.py:307-335) and ``loss.backward()`` updates (train.py:390-415), a
masked reconstruction loss, extra loss terms -- runs on the CUDA kernels.  Off by default (``kernel_autograd``)."""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from .plan import flow_step_params

_enabled = False


class kernel_autograd:
    """Route differentiable ``_netG`` / ``_netF`` calls on float32 CUDA tensors through the kernels' vector-Jacobian
    products.  Usable as a call or as a context manager, like ``torch.set_grad_enabled``::

        lsnf_b200.kernel_autograd()            # on from here
        with lsnf_b200.kernel_autograd():      # on inside the block, restored after it
            ...
        lsnf_b200.kernel_autograd(False)       # off (the default)

    The setting is process-wide and read when a module's forward runs.  CPU tensors, the reverse flow pass and double
    backward stay on the eager torch branch (the last raises: the kernels' backward is not differentiable)."""

    def __init__(self, enabled: bool = True):
        global _enabled
        self.prev = _enabled
        _enabled = bool(enabled)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        global _enabled
        _enabled = self.prev
        return False


def is_enabled() -> bool:
    return _enabled


def _gradient_nodes(params):
    """The autograd nodes that accumulate into ``params`` (AccumulateGrad for leaves).  In the backward,
    ``torch._C._will_engine_execute_node`` on them says whether this pass will actually deliver a parameter gradient:
    False under ``torch.autograd.grad(loss, z)``, True under ``loss.backward()``."""
    return [torch.autograd.graph.get_gradient_edge(p).node for p in params if p.requires_grad]


def _params_wanted(nodes) -> bool:
    return any(torch._C._will_engine_execute_node(n) for n in nodes)


def _flow_params(net):
    """Per step the twelve tensors of the flat gradient layout (``Plan.flow_grad_layout``), None where absent."""
    return [p for st in net.revnet2d_s[0].revnet2d_step_s for p in flow_step_params(st)]


class _GeneratorFn(torch.autograd.Function):
    """x_hat = G(z) on the kernels; inputs (net, z [B,nz], *conv weights and biases in ``gen`` order)."""

    @staticmethod
    def forward(ctx, net, z, *params):
        plan = net._plan(z.shape[0], z.device)
        plan.ensure_generator(net)
        x_hat = plan.generator_forward(z)
        # saving the parameters makes torch raise if they are modified in place before the backward
        ctx.save_for_backward(z, *params)
        ctx.net, ctx.plan, ctx.epoch = net, plan, plan.act_epoch
        ctx.nodes = _gradient_nodes(params)
        return x_hat

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_x_hat):
        z, *params = ctx.saved_tensors
        net = ctx.net
        want_z = ctx.needs_input_grad[1]
        want_params = _params_wanted(ctx.nodes)
        if want_params:
            # the weight gradients need a training plan's buffers; its workspace holds no activations of this z yet
            plan = net._plan(z.shape[0], z.device, train=True)
            plan.ensure_generator(net)
            plan.generator_forward(z)
        else:
            plan = ctx.plan
            plan.ensure_generator(net)
            if plan.act_epoch != ctx.epoch:   # another call overwrote this forward pass's activations
                plan.generator_forward(z)
        grad_z, flat = plan.generator_vjp(grad_x_hat.contiguous(), want_z=want_z, want_params=want_params)
        grads = [None] * len(params)
        if want_params:
            grads = [flat[off:off + size].view_as(p) for (off, size), p in zip(plan.generator_grad_layout(), params)]
        return (None, grad_z, *grads)


class _FlowFn(torch.autograd.Function):
    """(z_out, logdet) of the forward flow on the kernels; inputs (net, z [B,nz], *flow parameters in the order of
    ``Plan.flow_grad_layout`` without the absent ones)."""

    @staticmethod
    def forward(ctx, net, z, *params):
        plan = net._plan(z.shape[0], z.device)
        plan.ensure_flow(net)
        z_out, logdet, _logp, _ = plan.flow_forward(z)
        ctx.save_for_backward(z, *params)
        ctx.net, ctx.plan = net, plan
        ctx.nodes = _gradient_nodes(params)
        ctx.set_materialize_grads(False)   # an unused output passes a null seed instead of a tensor of zeros
        return z_out, logdet

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_z_out, grad_logdet):
        z, *params = ctx.saved_tensors
        want_z = ctx.needs_input_grad[1]
        want_params = _params_wanted(ctx.nodes)
        plan = ctx.plan
        plan.ensure_flow(ctx.net, need_inverse=want_params)   # d log|det W| / dW = W^-T
        grad_z, flat = plan.flow_vjp(z, None if grad_z_out is None else grad_z_out.contiguous(),
                                     None if grad_logdet is None else grad_logdet.contiguous(),
                                     want_z=want_z, want_params=want_params)
        grads = [None] * len(params)
        if want_params:
            layout = [ls for ls, p in zip(plan.flow_grad_layout(), _flow_params(ctx.net)) if p is not None]
            grads = [flat[off:off + size].view_as(p) for (off, size), p in zip(layout, params)]
        return (None, grad_z, *grads)


def generator_apply(net, z):
    """netG(z) for z [B,nz,1,1] or [B,nz] through ``_GeneratorFn``."""
    b = z.shape[0]
    convs = [m for m in net.gen if isinstance(m, torch.nn.ConvTranspose2d)]
    params = [p for m in convs for p in (m.weight, m.bias)]
    return _GeneratorFn.apply(net, z.reshape(b, net.nz).contiguous(), *params)


def flow_apply(net, z):
    """(z_out, logdet) of netF's forward direction for z [B,nz] through ``_FlowFn``."""
    params = [p for p in _flow_params(net) if p is not None]
    return _FlowFn.apply(net, z.contiguous(), *params)
