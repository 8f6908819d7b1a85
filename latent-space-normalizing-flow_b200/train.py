"""One training iteration of the reference (train.py:376-415) on the CUDA path, with data parallelism over the
latent batch: Langevin posterior inference (``lsnf_langevin_run``), the generator parameter update
(``generator_update``: ``lsnf_generator_param_grads`` -- forward, data-gradient chain, weight-gradient tap-GEMMs -- +
fused Adam; SURVEY.md section 8f rank 1) and the flow parameter update (``flow_update``: ``lsnf_flow_param_grads`` +
fused Adam; rank 2), all on ONE plan.  Each rank infers the latents of its shard (no collective) and computes its share
of the parameter gradients into one flat buffer per network; the buffers are summed across ranks (NCCL over NVLink) --
the generator's layer by layer on a comm stream, overlapping the remaining gradient kernels -- before the fused Adam
steps.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from .langevin import sample_langevin_post_z_with_flow
from .optim import FusedAdam
from .plan import as_mask, flow_step_params


def make_optimizers(netG, netF, args):
    """train.py:294-295: Adam for both networks.  ``FusedAdam`` is a ``torch.optim.Adam`` (same state_dict, same
    ``step()``) that the fused update kernels can drive directly."""
    g = lambda k, d: args.get(k, d) if isinstance(args, dict) else getattr(args, k, d)
    optG = FusedAdam(netG.parameters(), lr=g("g_lr", 0.0004), weight_decay=g("g_decay", 0),
                     betas=(g("g_beta1", 0.5), g("g_beta2", 0.999)))
    optF = FusedAdam(netF.parameters(), lr=g("f_lr", 0.0004), weight_decay=g("f_decay", 0),
                     betas=(g("f_beta1", 0.5), g("f_beta2", 0.999)))
    return optG, optF


_comm_streams = {}


def _comm_stream(device):
    """One side stream per device on which the gradient all-reduces are issued, so that they overlap the kernels the
    main stream keeps launching (the remaining layers' weight gradients, the flow update)."""
    key = (device.type, device.index)
    if key not in _comm_streams:
        _comm_streams[key] = torch.cuda.Stream(device=device)
    return _comm_streams[key]


def _gen_plan_and_buffers(netG, z_k, x, plan, mask=None):
    b = z_k.shape[0]
    z2 = z_k.detach().reshape(b, netG.nz).contiguous().float()
    xx = x.detach().contiguous().float()
    m = as_mask(mask, xx) if mask is not None else None
    if plan is None:
        plan = netG._plan(b, z2.device, train=True)
    plan.ensure_generator(netG)
    flat = getattr(plan, "_ggrad_flat", None)
    if flat is None:
        flat = plan._ggrad_flat = torch.zeros(int(plan.lib.lsnf_generator_grad_floats(plan.handle)),
                                              dtype=torch.float32, device=z2.device)
    convs = [m for m in netG.gen if isinstance(m, torch.nn.ConvTranspose2d)]
    params = [p for m in convs for p in (m.weight, m.bias)]
    layout = plan.generator_grad_layout()
    pairs = [(p, flat[off:off + size].view_as(p)) for (off, size), p in zip(layout, params)]
    return plan, z2, xx, m, flat, layout, pairs


def generator_gradients(netG, z_k, x, global_batch, plan=None, *, mask=None):
    """(flat gradient buffer, [(parameter, gradient view)], this rank's share of loss_g) of
    loss_g = mse_sum(G(z_k), x) / global_batch (train.py:392-394) through ``lsnf_generator_param_grads``: forward,
    data-gradient chain and one weight-gradient tap-GEMM per layer on the tensor cores.  With ``mask`` (per-pixel
    weight m, ``plan.as_mask``) loss_g = sum m (G(z_k) - x)^2 / global_batch."""
    plan, z2, xx, m, flat, layout, pairs = _gen_plan_and_buffers(netG, z_k, x, plan, mask)
    flat, loss = plan.generator_param_grads(z2, xx, global_batch, flat, mask=m)
    return flat, pairs, loss


class _PendingGeneratorUpdate:
    """Gradients computed, all-reduces in flight on the comm stream; ``finish()`` waits for them and applies Adam."""

    def __init__(self, netG, optG, args, flat, pairs, loss, handles):
        self.netG, self.optG, self.args = netG, optG, args
        self.flat, self.pairs, self.loss, self.handles = flat, pairs, loss, handles

    def finish(self):
        g = lambda k, d: self.args.get(k, d) if isinstance(self.args, dict) else getattr(self.args, k, d)
        for h in self.handles:
            h.wait()   # the CURRENT stream waits for the collective; the host does not block
        scale = None
        if g("g_is_grad_clamp", False):   # train.py:396-397 (upstream names an undefined `opt` there; intended semantics)
            scale = torch.clamp(float(g("g_max_norm", 100)) / (torch.linalg.vector_norm(self.flat) + 1e-6), max=1.0)
        params, grads = [p for p, _ in self.pairs], [v for _, v in self.pairs]
        if isinstance(self.optG, FusedAdam):
            self.optG.fused_step(params, grads, grad_scale=scale)
        else:
            for p, v in self.pairs:
                p.grad = v.clone() if scale is None else v * scale
            self.optG.step()
        return self.loss


def generator_update_begin(netG, optG, z_k, x, args, *, global_batch=None, group=None, world=1, plan=None, mask=None):
    """First half of the generator step of train.py:390-398: gradients, and with several ranks their all-reduce
    started layer by layer (bucket = one layer's weight + bias gradient, last layer first) on a comm stream while the
    main stream computes the next layer's weight gradient.  ``.finish()`` completes the step.  ``mask``: per-pixel
    weight of the loss, as in ``generator_gradients``."""
    b_global = z_k.shape[0] if global_batch is None else int(global_batch)
    plan, z2, xx, m, flat, layout, pairs = _gen_plan_and_buffers(netG, z_k, x, plan, mask)
    if world <= 1:
        flat, loss = plan.generator_param_grads(z2, xx, b_global, flat, mask=m)
        return _PendingGeneratorUpdate(netG, optG, args, flat, pairs, loss, [])
    comm = _comm_stream(z2.device)
    main = torch.cuda.current_stream(z2.device)
    handles = []
    flat, loss = plan.generator_param_grads(z2, xx, b_global, flat, part=-2, mask=m)

    def reduce_async(t):
        ev = torch.cuda.Event()
        ev.record(main)
        with torch.cuda.stream(comm):
            comm.wait_event(ev)
            handles.append(dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=True))

    reduce_async(loss)
    n_layers = len(layout) // 2
    for l in reversed(range(n_layers)):
        plan.generator_param_grads(z2, xx, b_global, flat, part=l, loss=loss)
        lo = layout[2 * l][0]
        hi = layout[2 * l + 1][0] + layout[2 * l + 1][1]
        reduce_async(flat[lo:hi])
    return _PendingGeneratorUpdate(netG, optG, args, flat, pairs, loss, handles)


def generator_update(netG, optG, z_k, x, args, *, global_batch=None, group=None, world=1, plan=None, mask=None):
    """The generator step of train.py:390-398 without autograd.  Returns loss_g."""
    return generator_update_begin(netG, optG, z_k, x, args, global_batch=global_batch, group=group, world=world,
                                  plan=plan, mask=mask).finish()


def flow_params_in_order(netF):
    """The flow parameters in the order of the flat gradient buffer (``Plan.flow_grad_layout``): per step, the twelve
    tensors of ``_FLOW_PARAM_ORDER``; ``None`` where a step has no such parameter (shuffle permutation)."""
    out = []
    for st in netF.revnet2d_s[0].revnet2d_step_s:
        out += flow_step_params(st)
    return out


def flow_gradients(netF, z_k, global_batch, plan=None):
    """(flat gradient buffer, [(parameter, gradient view)], this rank's share of loss_f) of
    loss_f = -(1/global_batch) sum_b log p(z_b) (train.py:403-410) through ``lsnf_flow_param_grads``."""
    b = z_k.shape[0]
    z2 = z_k.detach().reshape(b, netF.nz).contiguous().float()
    if plan is None:
        plan = netF._plan(b, z2.device)
    plan.ensure_flow(netF, need_inverse=True)
    flat = getattr(plan, "_fgrad_flat", None)
    if flat is None:
        flat = plan._fgrad_flat = torch.zeros(int(plan.lib.lsnf_flow_grad_floats(plan.handle)), dtype=torch.float32,
                                              device=z2.device)
    flat, loss = plan.flow_param_grads(z2, global_batch, flat)
    pairs = [(p, flat[off:off + size].view_as(p)) for (off, size), p in zip(plan.flow_grad_layout(),
                                                                            flow_params_in_order(netF)) if p is not None]
    return flat, pairs, loss


def flow_update(netF, optF, z_k, args, *, global_batch=None, group=None, world=1, plan=None):
    """The flow step of train.py:403-415 without autograd: gradients by the fused flow kernel + batch reductions,
    one all-reduce of the flat buffer across ranks, optional norm clipping, fused Adam.  Returns loss_f."""
    g = lambda k, d: args.get(k, d) if isinstance(args, dict) else getattr(args, k, d)
    b_global = z_k.shape[0] if global_batch is None else int(global_batch)
    flat, pairs, loss = flow_gradients(netF, z_k, b_global, plan=plan)
    if world > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=group)
    scale = None
    if g("f_is_grad_clamp", False):   # train.py:411-412, clip_grad_norm_ semantics
        scale = torch.clamp(float(g("f_max_norm", 100)) / (torch.linalg.vector_norm(flat) + 1e-6), max=1.0)
    params, grads = [p for p, _ in pairs], [v for _, v in pairs]
    if isinstance(optF, FusedAdam):
        optF.fused_step(params, grads, grad_scale=scale)
    else:   # any other torch optimizer: hand it the same gradients
        for p, v in pairs:
            p.grad = v.clone() if scale is None else v * scale
        optF.step()
    return loss


_iter_counter = [0]


def training_iteration(x, netG, netF, optG, optF, args, *, global_batch=None, sample_offset=None, seed=None,
                       z0=None, group=None, data_parallel=None, mask=None):
    """x: this rank's shard [B_local, nc, H, W] on the GPU.  Returns (loss_g, loss_f, |grad_g|, |grad_f|, z_k).
    ``mask``: this rank's shard of a per-pixel likelihood weight (any shape that broadcasts to x's, ``plan.as_mask``)
    for training on partly observed images: both the Langevin energy and loss_g weight (G(z) - x)^2 by it.

    Mirrors train.py:378-415: z_0 ~ N(0, I); z_k = Langevin(z_0, x); generator step on mse_sum(G(z_k), x) / B;
    flow step on -mean log p(z_k) (with the f_is_grad_clamp / f_max_norm clipping of train.py:411-412).  With several
    ranks the losses are normalised by the GLOBAL batch, so the summed gradients equal the single-process ones.

    Data parallelism: every rank must draw DIFFERENT chains.  ``sample_offset`` (index of this shard's first sample in
    the global batch) defaults to the contiguous sharding of ``dist.shard_range``; the Philox noise is keyed by
    (seed, global sample index, step) and z_0 is the rank's slice of ONE global draw from a generator seeded with
    ``seed``, so an N-rank iteration reproduces the single-process one.  ``seed`` defaults to
    (args.seed << 32) ^ iteration counter -- identical on every rank, as it must be."""
    b_local = x.shape[0]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if data_parallel is False:
        world = 1   # e.g. a single-process reference run inside an initialised process group
    g = lambda k, d: args.get(k, d) if isinstance(args, dict) else getattr(args, k, d)
    if seed is None:
        seed = (int(g("seed", 1)) << 32) ^ _iter_counter[0]
    _iter_counter[0] += 1
    if world > 1:
        rank = dist.get_rank(group)
        if global_batch is None:
            sizes = torch.tensor([b_local], device=x.device)
            dist.all_reduce(sizes, group=group)
            global_batch = int(sizes.item())
        if sample_offset is None:
            from .dist import shard_range
            a, b = shard_range(int(global_batch), rank, world)
            if b - a != b_local:
                raise ValueError(f"rank {rank} holds {b_local} samples but the contiguous sharding of a global batch of "
                                 f"{global_batch} gives it {b - a}; pass sample_offset explicitly")
            sample_offset = a
    b_global = b_local if global_batch is None else int(global_batch)
    sample_offset = 0 if sample_offset is None else int(sample_offset)
    netG.train()
    netF.train()
    if z0 is None:                                                                       # train.py:384
        gen = torch.Generator(x.device).manual_seed(int(seed) & (2 ** 63 - 1))
        z0 = torch.randn(b_global, netG.nz, 1, 1, device=x.device, generator=gen)[sample_offset:sample_offset + b_local]
    z_k, gn, fn = sample_langevin_post_z_with_flow(z0, x, netG, netF, args, seed=seed,
                                                   sample_offset=sample_offset, train=True, mask=mask)   # train.py:387
    from .langevin import langevin_plan
    from .plan import default_bwd_passes
    plan = langevin_plan(netG, netF, b_local, x.device, default_bwd_passes(), train=True)  # the plan that call used
    # generator update (train.py:390-398): weight-gradient tap-GEMMs, per-layer all-reduces on the comm stream ...
    masked = {} if mask is None else {"mask": mask}   # an unmasked iteration makes exactly the unmasked call
    pending = generator_update_begin(netG, optG, z_k, x, args, global_batch=b_global, group=group, world=world,
                                     plan=plan, **masked)
    # ... overlapped with the flow update (train.py:403-415): gradient kernels + one flat all-reduce + fused Adam.
    # The two updates are independent (neither reads the other network's parameters), so finishing the generator's
    # Adam step after the flow's changes nothing.
    loss_f = flow_update(netF, optF, z_k, args, global_batch=b_global, group=group, world=world, plan=plan)
    loss_g = pending.finish()
    return loss_g.detach(), loss_f.detach(), gn, fn, z_k
