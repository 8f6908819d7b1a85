"""Data-parallel plumbing (SURVEY.md section 8e): the latent batch is sharded contiguously across ranks, one
process per GPU; Langevin chains are independent per sample so the loop itself needs no collective.  The only
exchange is the parameter-gradient all-reduce of the training-mode G / F updates (train.py:394, :411)."""
from __future__ import annotations

from typing import Iterable, Tuple

import torch
import torch.distributed as dist


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous [start, stop) of rank's rows; the first ``n % world`` ranks get one extra row."""
    base, rem = divmod(n, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def shard_batch(t: torch.Tensor, rank: int, world: int) -> torch.Tensor:
    a, b = shard_range(t.shape[0], rank, world)
    return t[a:b]


def langevin_sharded(z_global, x_global, netG, netF, args, *, seed: int, rank: int = None, world: int = None,
                     gather: bool = False, mask=None, **kw):
    """Run this rank's shard of a global batch.  Noise is keyed by the GLOBAL sample index, so every rank draws
    exactly the noise the single-GPU run draws for its samples (the latents then agree up to fp32 summation order:
    split-K / stream-K cut points depend on the tile count).  Returns (z_shard or gathered z, |grad_g|, |grad_f|)
    with the two diagnostics averaged over the global batch when ``gather``.  ``mask`` (per-pixel likelihood weight of
    the global batch, ``plan.as_mask``) is sharded like x; a mask without a batch axis of the global batch's size
    (e.g. [1,1,H,W] or [H,W]) is shared by every sample and passed to each rank whole."""
    from .langevin import sample_langevin_post_z_with_flow
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    a, b = shard_range(z_global.shape[0], rank, world)
    if mask is not None and mask.dim() == x_global.dim() and mask.shape[0] == x_global.shape[0]:
        mask = mask[a:b]
    z, gn, fn = sample_langevin_post_z_with_flow(z_global[a:b], x_global[a:b], netG, netF, args, seed=seed,
                                                 sample_offset=a, mask=mask, **kw)
    if not gather:
        return z, gn, fn
    sizes = [shard_range(z_global.shape[0], r, world) for r in range(world)]
    parts = [torch.empty((e - s,) + tuple(z.shape[1:]), dtype=z.dtype, device=z.device) for s, e in sizes]
    dist.all_gather(parts, z.contiguous())
    w = torch.stack([gn, fn]) * float(b - a)
    dist.all_reduce(w)
    w = w / float(z_global.shape[0])
    return torch.cat(parts, 0), w[0], w[1]


def allreduce_grads(params: Iterable[torch.nn.Parameter], scale: float = 1.0, group=None) -> int:
    """Sum the .grad of every parameter across ranks with ONE flat all-reduce (NCCL over NVLink on the GPU box,
    gloo in the CPU tests), then multiply by ``scale``.  With the losses of train.py:393 / :410 computed on the
    local shard -- mse_sum / B_local and -mean over B_local -- ``scale = B_local / B_global`` reproduces the
    single-process gradient when shards are equal (scale = 1/world).  Returns the number of bytes reduced."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if scale != 1.0:
        flat.mul_(scale)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n
    return flat.numel() * flat.element_size()
