"""CPU emulation of the tensor-core operand splits of the generator stages (DIAGNOSTIC; no GPU, no product code).

Question (DESIGN.md section 4.1, SURVEY.md section 8f "what comes next"): the Langevin loop runs every generator
GEMM as THREE tcgen05 passes (hi*hi + hi*lo + lo*hi of a 16-bit hi|lo operand split), which caps the loop at 0.30 of
the one-pass tensor roofline.  Which cheaper operand formats for the two cross terms would still hold north_star's
1e-4 on z_T?  This script replays the full noisy chain (train.py:307-335 as restated by oracle/refpath.py, injected
noise) on the CPU with the generator's forward and data-gradient contractions replaced by emulations of each scheme:
operands are rounded to the scheme's formats, the partial products are summed in fp32 (fp16 x fp16 and fp8 x fp8
products are exact in fp32, as they are in the tensor core's fp32 accumulator), activations are stored between layers
as the fp16 hi|lo pair / the gradients as the bf16 hi|lo pair the kernels write, and LeakyReLU' takes the sign of the
EMULATED forward activation (DESIGN.md section 2, "LeakyReLU kinks").  z_T of every scheme is compared with the plain
fp32 oracle.

Calibration: three of the schemes have been measured on a B200 (profiles/r2_parity_cifar10_b100_t40.json,
profiles/r2_fwd2pass_ab.json); the emulation is only trusted for the unmeasured ones as far as it reproduces those.

    python tools/precision_emulation.py --batch 16 --seeds 1 2 3 --out profiles/r2_precision_emulation_cpu.json
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lsnf_b200.synth as synth  # noqa: E402  (numpy only: deterministic synthetic parameters)
from oracle import refpath  # noqa: E402

F8 = torch.float8_e4m3fn


def pow2_floor(v: float) -> float:
    return 2.0 ** math.floor(math.log2(v)) if v > 0 else 1.0


def fp8_scale_exp(m: float) -> int:
    """k with m * 2^k in [128, 256), clamped to [-40, 40]; 0 for m = 0 (csrc/lsnf_internal.cuh fp8_scale_exp)."""
    if not m > 0:
        return 0
    return max(-40, min(40, 8 - math.frexp(m)[1]))


def split(t: torch.Tensor, dt: torch.dtype):
    """t ~= hi + lo with both halves representable in ``dt`` (what split_z / the stage epilogues store)."""
    hi = t.to(dt).float()
    lo = (t - hi).to(dt).float()
    return hi, lo


def q8_tensor(t: torch.Tensor) -> torch.Tensor:
    """e4m3 with ONE power-of-two scale per tensor (max |t| -> [128, 256))."""
    m = float(t.abs().max())
    if m == 0.0:
        return t
    s = 128.0 / pow2_floor(m)
    return (t * s).to(F8).float() / s


def q8_block(t: torch.Tensor, axis: int, block: int = 32) -> torch.Tensor:
    """e4m3 with one power-of-two scale per ``block`` consecutive elements along the contraction axis -- the operand
    format of tcgen05.mma kind::mxf8f6f4 (UE8M0 scale per 32 K elements)."""
    t = t.movedim(axis, -1)
    shp = t.shape
    n = shp[-1]
    pad = (-n) % block
    if pad:
        t = F.pad(t, (0, pad))
    g = t.reshape(-1, block)
    m = g.abs().amax(dim=1, keepdim=True).clamp_min(1e-38)
    s = 128.0 / torch.exp2(torch.floor(torch.log2(m)))
    q = (g * s).to(F8).float() / s
    q = q.reshape(*shp[:-1], n + pad)[..., :n]
    return q.movedim(-1, axis)


class Scheme:
    """hi*hi in ``base`` (torch.float16 / torch.bfloat16 / None = plain fp32) plus the listed cross terms.

    cross: subset of {"a_hi*w_lo", "a_lo*w_hi"} computed in ``cross_fmt``:
       "16"  - the 16-bit halves themselves (the shipped 3-pass kernels)
       "f8t" - both operands of the cross term re-rounded to e4m3, one scale per tensor
       "f8b" - e4m3 with a power-of-two scale per 32 elements along K (kind::mxf8f6f4)
       "f8x" - what the wide data-gradient stages build: each operand times its power-of-two scale 2^k
               (max |tensor| * 2^k in [128, 256)) split into fp16 halves, hi*hi in fp16, both cross terms in
               e4m3 (round to nearest) with the lo halves lifted by 2^11; ``base`` is ignored
    passes: tensor-pipe cost in units of one 16-bit pass (fp8 runs at twice the 16-bit rate)."""

    def __init__(self, name, base, cross=(), cross_fmt="16", scale_w=True):
        self.name, self.base, self.cross, self.cross_fmt, self.scale_w = name, base, tuple(cross), cross_fmt, scale_w
        self.passes = 0.0 if base is None else 1.0 + len(self.cross) * (1.0 if cross_fmt == "16" else 0.5)

    def contract(self, a, w, op, a_axis, w_axis):
        """op(a, w) is bilinear; a_axis / w_axis are the contraction (channel) axes of the two operands."""
        if self.base is None:
            return op(a, w)
        k = 1.0
        if self.cross_fmt == "f8x":
            sa, sw = 2.0 ** fp8_scale_exp(float(a.abs().max())), 2.0 ** fp8_scale_exp(float(w.abs().max()))
            ah, al = split(a * sa, F16)
            wh, wl = split(w * sw, F16)
            e = lambda t: t.to(F8).float()   # noqa: E731
            lift = 2.0 ** 11
            return (op(ah, wh) + (op(e(ah), e(wl * lift)) + op(e(al * lift), e(wh))) / lift) / (sa * sw)
        if self.scale_w:   # per-layer power-of-two weight scale (max |w| -> [1, 2)), undone exactly afterwards
            k = 1.0 / pow2_floor(float(w.abs().max()))
        ah, al = split(a, self.base)
        wh, wl = split(w * k, self.base)
        out = op(ah, wh)

        def q(t, axis):
            if self.cross_fmt == "16":
                return t
            return q8_tensor(t) if self.cross_fmt == "f8t" else q8_block(t, axis)

        if "a_hi*w_lo" in self.cross:
            out = out + op(q(ah, a_axis), q(wl, w_axis))
        if "a_lo*w_hi" in self.cross:
            out = out + op(q(al, a_axis), q(wh, w_axis))
        return out / k


class EmuConvT(torch.autograd.Function):
    """ConvTranspose2d whose forward contraction follows ``fwd`` and whose data gradient follows ``bwd``."""

    @staticmethod
    def forward(ctx, a, w, b, stride, pad, fwd, bwd):
        ctx.save_for_backward(w)
        ctx.cfg = (stride, pad, bwd)
        y = fwd.contract(a, w, lambda A, W: F.conv_transpose2d(A, W, None, stride, pad), 1, 0)
        return y + b.view(1, -1, 1, 1)

    @staticmethod
    def backward(ctx, g):
        (w,) = ctx.saved_tensors
        stride, pad, bwd = ctx.cfg
        # data gradient of conv_transpose2d = conv2d(g, W, stride, pad) (SURVEY.md section 8a, A2'); K = C_out * taps
        ga = bwd.contract(g, w, lambda G, W: F.conv2d(G, W, None, stride, pad), 1, 1)
        return ga, None, None, None, None, None, None


class Store(torch.autograd.Function):
    """What lives in HBM between two stages: the activation as an fp16 hi|lo pair on the way forward, the gradient
    as a bf16 hi|lo pair on the way back (DESIGN.md section 3).  Identity for the fp32 scheme."""

    @staticmethod
    def forward(ctx, a, fwd, bwd):
        ctx.bwd = bwd
        if fwd.base is None:
            return a
        hi, lo = split(a, fwd.base)
        return hi + lo

    @staticmethod
    def backward(ctx, g):
        if ctx.bwd.base is None:
            return g, None, None
        if not ctx.bwd.cross:   # the single-pass data gradient carries ONE 16-bit tensor end to end
            return g.to(ctx.bwd.base).float(), None, None
        hi, lo = split(g, ctx.bwd.base)
        return hi + lo, None, None


def generator_forward_emulated(gp, z, layers, leak, fwd: Scheme, bwd: Scheme):
    h = Store.apply(z, fwd, bwd)
    last = len(layers) - 1
    for i, (_ci, _co, _k, s, p) in enumerate(layers):
        h = EmuConvT.apply(h, gp[f"gen.{3 * i}.weight"], gp[f"gen.{3 * i}.bias"], s, p, fwd, bwd)
        if i == last:
            h = torch.tanh(h)
        else:
            h = Store.apply(F.leaky_relu(h, leak), fwd, bwd)
    return h


def langevin_emulated(z0, x, gp, fp, layers, *, depth, steps, step_size, sigma, eps, leak, fwd, bwd):
    """refpath.langevin (train.py:307-335) with the generator term going through the emulated contractions; the flow
    prior stays plain fp32 (the flow kernel computes in fp32)."""
    z = z0.clone().detach().requires_grad_(True)
    bsz = z.shape[0]
    for t in range(steps):
        x_hat = generator_forward_emulated(gp, z, layers, leak, fwd, bwd)
        g_log_lkhd = 1.0 / (2.0 * sigma * sigma) * F.mse_loss(x_hat, x, reduction="sum")
        z_grad_g = torch.autograd.grad(g_log_lkhd, z)[0]
        ll, _z1, _ld = refpath.log_prior(fp, z.reshape(bsz, -1), depth)
        z_grad_f = torch.autograd.grad(-ll.sum(), z)[0]
        z.data = z.data - 0.5 * step_size * step_size * (z_grad_g + z_grad_f)
        z.data += step_size * eps[t]
    return z.detach()


def rel_l2(a, b):
    return float(torch.linalg.vector_norm(a.double() - b.double()) / torch.linalg.vector_norm(b.double()))


F16, BF16 = torch.float16, torch.bfloat16
BOTH = ("a_hi*w_lo", "a_lo*w_hi")
FWD = {
    "fp32": Scheme("fp32", None),
    "f16x3": Scheme("fp16 hi|lo, 3 passes (shipped)", F16, BOTH),
    "f16x2_drop_w_lo": Scheme("fp16, weights' lo half dropped (2 passes)", F16, ("a_lo*w_hi",)),
    "f16x2_drop_a_lo": Scheme("fp16, activations' lo half dropped (2 passes)", F16, ("a_hi*w_lo",)),
    "f16x1": Scheme("fp16 single pass", F16, ()),
    "f16+f8t": Scheme("fp16 hi*hi + both cross terms in e4m3, per-tensor scale (2 pass-equivalents)", F16, BOTH, "f8t"),
    "f16+f8b": Scheme("fp16 hi*hi + both cross terms in e4m3, scale per 32 K (kind::mxf8f6f4; 2 pass-equivalents)",
                      F16, BOTH, "f8b"),
}
BWD = {
    "fp32": Scheme("fp32", None),
    "bf16x3": Scheme("bf16 hi|lo, 3 passes (shipped default)", BF16, BOTH, scale_w=False),
    "f16x1": Scheme("fp16 single pass (shipped opt-in)", F16, (), scale_w=False),
    "f16+f8t": Scheme("fp16 hi*hi + cross terms in e4m3, per-tensor scale", F16, BOTH, "f8t"),
    "f16+f8b": Scheme("fp16 hi*hi + cross terms in e4m3, scale per 32 K", F16, BOTH, "f8b"),
    "f16+f8x": Scheme("fp16 hi*hi + cross terms as one e4m3 stream, power-of-two scale per tensor (shipped on the "
                      "wide stages)", F16, BOTH, "f8x", scale_w=False),
}
# (forward, data gradient, z_T error measured on a B200 at B=100 or None)
COMBOS = [
    ("f16x3", "bf16x3", "4.5e-5 .. 4.8e-5 (profiles/r2_parity_cifar10_b100_t40.json)"),
    ("f16x3", "f16x1", "5.2e-5 .. 5.6e-5 (same file)"),
    ("f16x2_drop_w_lo", "bf16x3", "1.47e-4 .. 1.53e-4 (profiles/r2_fwd2pass_ab.json)"),
    ("f16x2_drop_a_lo", "bf16x3", "1.47e-4 .. 1.53e-4 (profiles/r2_fwd2pass_ab.json)"),
    ("f16x1", "f16x1", None),
    ("f16+f8t", "bf16x3", None),
    ("f16+f8b", "bf16x3", None),
    ("f16+f8b", "f16+f8b", None),
    ("f16+f8t", "f16+f8t", None),
    ("f16+f8b", "f16x1", None),
    ("f16x3", "f16+f8b", None),
    ("f16x3", "f16+f8t", None),
    ("f16x3", "f16+f8x", None),
]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dataset", default="cifar10")
    ap.add_argument("--nz", type=int, default=128)
    ap.add_argument("--ngf", type=int, default=128)
    ap.add_argument("--f-width", type=int, default=64)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--sigma", type=float, default=0.3)
    ap.add_argument("--seeds", type=int, nargs="+", default=[1, 2, 3])
    ap.add_argument("--combos", type=int, nargs="*", default=None, help="indices into COMBOS (default: all)")
    ap.add_argument("--yardstick", action="store_true", help="also measure the reference against ITSELF: fp32 vs fp64, "
                    "and fp32 with one CPU thread vs all of them (another summation order)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    torch.manual_seed(0)
    layers = synth.generator_layers(a.dataset, a.nz, a.ngf)
    img = synth.image_size(a.dataset)
    combos = COMBOS if a.combos is None else [COMBOS[i] for i in a.combos]
    rows = {f"{f} / {b}": {"forward": FWD[f].name, "data_gradient": BWD[b].name,
                           "passes_per_iteration_of_6": FWD[f].passes + BWD[b].passes, "measured_on_b200": m,
                           "z_T_rel_l2_vs_fp32_oracle": []} for f, b, m in combos}
    t_all = time.time()
    yard = {}
    for seed in a.seeds:
        to_t = lambda sd: {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}
        gp = to_t(synth.generator_state(a.dataset, a.nz, a.ngf, seed=seed))
        fp = to_t(synth.flow_state(a.nz, a.f_width, seed=seed))
        x, z0, eps = (torch.from_numpy(v) for v in synth.inputs(a.batch, a.nz, 3, img, a.steps, seed=seed))
        kw = dict(depth=5, steps=a.steps, step_size=0.1, sigma=a.sigma, leak=0.2)
        t0 = time.time()
        ref, _, _ = refpath.langevin(z0, x, gp, fp, layers, eps=eps, **kw)
        print(f"seed {seed}: fp32 oracle {time.time() - t0:.1f} s", flush=True)
        if a.yardstick:
            d = lambda sd: {k: v.double() for k, v in sd.items()}
            r64, _, _ = refpath.langevin(z0.double(), x.double(), d(gp), d(fp), layers, eps=eps.double(), **kw)
            nthr = torch.get_num_threads()
            torch.set_num_threads(1)
            r1, _, _ = refpath.langevin(z0, x, gp, fp, layers, eps=eps, **kw)
            torch.set_num_threads(nthr)
            y = yard.setdefault("fp32 oracle vs its own fp64 run", [])
            y.append(rel_l2(ref, r64))
            y = yard.setdefault(f"fp32 oracle, 1 thread vs {nthr} threads", [])
            y.append(rel_l2(r1, ref))
            print(f"  reference against itself: fp32 vs fp64 {rel_l2(ref, r64):.3e}; 1 vs {nthr} threads "
                  f"{rel_l2(r1, ref):.3e}", flush=True)
        for f, b, _m in combos:
            t0 = time.time()
            zt = langevin_emulated(z0, x, gp, fp, layers, eps=eps, fwd=FWD[f], bwd=BWD[b], **kw)
            err = rel_l2(zt, ref)
            rows[f"{f} / {b}"]["z_T_rel_l2_vs_fp32_oracle"].append(err)
            print(f"  {f:>16} / {b:<8} z_T rel-l2 {err:.3e}   ({time.time() - t0:.1f} s)", flush=True)
    out = {"what": "CPU emulation of operand-split schemes for the generator GEMMs of the Langevin loop; z_T after the "
                   "full noisy chain against the plain fp32 oracle (oracle/refpath.py), injected noise",
           "config": {"dataset": a.dataset, "nz": a.nz, "ngf": a.ngf, "f_width": a.f_width, "batch": a.batch,
                      "steps": a.steps, "sigma": a.sigma, "seeds": a.seeds},
           "budget": 1e-4, "reference_against_itself": yard, "schemes": rows, "torch": torch.__version__, "wall_s": time.time() - t_all,
           "not_a_gpu_measurement": True}
    if a.out:
        json.dump(out, open(a.out, "w"), indent=1)
    print(json.dumps({k: [f"{e:.2e}" for e in v["z_T_rel_l2_vs_fp32_oracle"]] for k, v in rows.items()}, indent=1))


if __name__ == "__main__":
    main()
