"""The fused flow-prior kernels against fp64 autograd on the oracle across the configurations lsnf_plan_create accepts,
with invertible 1x1 matrices that are NOT orthogonal.

Every other flow test loads ``synth.flow_state``, whose 1x1 matrices are the Q of a QR decomposition: log|det W| = 0 and
W^-1 = W^T there, so a log-det that is never added, or a transpose in place of the inverse, passes them.  Here each W
is Q1 diag(d) Q2 with |d| log-uniform in [0.5, 2] -- log|det W| of order one per step, negative determinants, one
direction shrunk 64-fold in some steps (condition number ~1e2), and in others a block layout with a zero diagonal that
forces a row interchange at every pivot.  The cases walk the shape-dependent code paths of the kernels: the column
groups and K split of the mat-vecs (nz, f_width not multiples of 32), every samples-per-CTA tier with a ragged last CTA
(B = 1, 31, 33, 65, 1203) and the fallback to a smaller tier where the preferred one does not fit, a matrix ring that
holds the whole pass, wraps around or holds one matrix at a time, the library's Gauss-Jordan log-det / inverse up to
its largest size (nz = 160) and the torch det / inv path above it."""
import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import autograd_fns, synth
from oracle import refpath
from helpers import REL_TOL, record, rel_err, rel_l2, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_TOL = 1e-5      # rel-l2 of gradients, as tests/test_gpu_kernel_autograd.py
DEEP = 16            # from this depth on the bound is 4x the fp32 oracle's own distance from fp64, if that is larger


def _w_kind(i, nz, depth):
    kind = (i + nz // 4) % 4   # 0 plain, 1 negative determinant, 2 ill-conditioned, 3 zero diagonal
    # a 64-fold shrink in every fourth step of a deep flow compounds beyond what fp32 can follow (the fp32 oracle
    # itself loses the inverse); deep flows get the other three kinds
    return 0 if kind == 2 and depth >= DEEP else kind


def general_w(rng, nz, kind, depth):
    """Q1 diag(d) Q2 with |d| log-uniform in [0.5, 2], recentred so that log|det W| = sum log|d| is +-(0.5 ... 1.5)
    per block: of order one whatever nz, as in a trained flow (see the module docstring for the four kinds).  A
    product of `depth` such matrices spreads its singular values by about exp(depth * mean(log^2 d) / 3); deep flows
    narrow the range of log|d| by sqrt(5 / depth) so that the whole flow stays as well conditioned as one of the
    reference's depth 5, and fp32 can follow it."""
    def q(n):
        return np.linalg.qr(rng.standard_normal((n, n)))[0]

    def block(n, sign):
        u = rng.uniform(-np.log(2.0), np.log(2.0), n) * min(1.0, np.sqrt(5 / depth))
        c = rng.uniform(0.5, 1.5) * rng.choice([-1.0, 1.0])
        d = np.exp(u - u.mean() + c / n)
        if kind == 2:
            d[rng.integers(n)] = 1.0 / 64
        d[0] *= sign
        return q(n) @ np.diag(d) @ q(n)

    if kind == 3:   # [[0, M2], [M1, 0]]: every diagonal element is zero
        h = nz // 2
        w = np.zeros((nz, nz))
        w[:h, h:], w[h:, :h] = block(h, -1.0), block(h, 1.0)
    else:
        w = block(nz, -1.0 if kind == 1 else 1.0)
    return w.astype(np.float32)


def general_flow_state(nz, width, depth, coupling, perm, seed=3, zero_logs=False):
    sd = synth.flow_state(nz, width, depth, coupling, perm, seed=seed)
    rng = np.random.default_rng(1000 + seed)
    for i in range(depth):
        pre = f"revnet2d_s.0.revnet2d_step_s.{i}."
        if perm == 2:
            sd[pre + "invertible_1x1_conv.w"] = general_w(rng, nz, _w_kind(i, nz, depth), depth)
        if zero_logs:   # log-det of the actnorm layers = 0: what remains of an additive flow's log-det is sum log|det W|
            sd[pre + "actnorm.logs"] = np.zeros_like(sd[pre + "actnorm.logs"])
    return sd


def _net(nz, width, depth, coupling, perm, sd):
    args = lsnf_b200.make_args(nz=nz, f_width=width, f_depth=depth, f_flow_coupling=coupling, f_flow_permutation=perm)
    netF = lsnf_b200._netF(args, nz=nz).to(DEV)
    netF.load_state_dict(to_torch(sd))
    return netF


def _params(sd, dtype):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dtype) if v.dtype.kind == "f" else torch.from_numpy(v)
            for k, v in sd.items()}


def _inverse_input(sd, eps, depth, coupling, perm):
    """eps for the inverse pass: standard normal, except for deep flows.  A deep flow contracts volume by up to e^-900
    (its log-det), so its inverse overflows at most normal points even in fp64; there it is evaluated on the forward
    image (fp64) of a normal batch."""
    if depth < DEEP:
        return eps
    zero = torch.zeros(eps.shape[0], dtype=torch.float64)
    return refpath.flow_forward(_params(sd, torch.float64), eps.double(), zero, depth, coupling, perm)[0].float()


def _grad_names(netF, plan, flat):
    named = {id(p): k for k, p in netF.named_parameters()}
    out = {}
    for (off, size), p in zip(plan.flow_grad_layout(), autograd_fns._flow_params(netF)):
        if p is not None:
            out[named[id(p)]] = flat[off:off + size].view_as(p).cpu()
    return out


def oracle(sd, keys, z, eps, seeds, depth, coupling, perm, dtype):
    """Everything the kernels are compared with, from the oracle in `dtype`: forward, reverse, and the gradients of
    -sum_b log p(z_b) and of the VJP losses sum(z_out * g) + sum(logdet * l) w.r.t. z and the parameters `keys`."""
    fp = _params(sd, dtype)
    B = z.shape[0]
    out = {}

    def run(loss_of):
        leaves = {k: fp[k].clone().requires_grad_(True) for k in keys}
        zz = z.to(dtype).clone().requires_grad_(True)
        ll, zo, ld = refpath.log_prior({**fp, **leaves}, zz, depth, coupling, perm)
        loss_of(ll, zo, ld).backward()
        # what the loss does not depend on (an additive flow's log-det on z and the shifts) has the gradient zero
        grad = lambda t: t.grad if t.grad is not None else torch.zeros_like(t)
        return ll.detach(), zo.detach(), ld.detach(), grad(zz), {k: grad(leaves[k]) for k in keys}

    ll, zo, ld, gz, gp = run(lambda ll, zo, ld: -ll.sum())
    out.update(logp=ll, z_out=zo, logdet=ld, grad_z=gz, param={k: v / B for k, v in gp.items()})
    for name, (sg, sl) in seeds.items():
        def vjp_loss(ll, zo, ld, sg=sg, sl=sl):
            loss = 0.0
            if sg is not None:
                loss = loss + (zo * sg.to(dtype)).sum()
            if sl is not None:
                loss = loss + (ld * sl.to(dtype)).sum()
            return loss
        _, _, _, gz, gp = run(vjp_loss)
        out["vjp_" + name] = (gz, gp)
    with torch.no_grad():
        zr, obj = refpath.flow_reverse(fp, eps.to(dtype), torch.zeros(B, dtype=dtype), depth, coupling, perm)
        out["inv_z"], out["inv_negobj"] = zr, -obj
        out["roundtrip"] = refpath.flow_reverse(fp, zo, torch.zeros(B, dtype=dtype), depth, coupling, perm)[0]
    return out


def near_kinks(sd, z, depth, coupling, perm):
    """{step: number of (sample, unit) pairs of its coupling MLP whose ReLU input is within 1e-5 of the layer's
    largest of zero}, in fp64.  An fp32 forward pass may take the other branch there, which moves the gradients of that
    step's fc_1 / fc_2 parameters by up to that sample's share of the batch sum (DESIGN.md section 2, kinks)."""
    fp = _params(sd, torch.float64)
    x, n, out = z.double(), z.shape[1], {}
    for i in range(depth):
        pre = f"revnet2d_s.0.revnet2d_step_s.{i}."
        x = (x + fp[pre + "actnorm.b"]) * torch.exp(3.0 * fp[pre + "actnorm.logs"])
        x = x @ fp[pre + "invertible_1x1_conv.w"] if perm == 2 else x[:, fp[pre + "shuffle_features.indices"].long()]
        x1, x2 = x[:, : n // 2], x[:, n // 2:]
        p1 = (x1 @ fp[pre + "f.fc_1.w"] + fp[pre + "f.fc_1.actnorm.b"]) * torch.exp(3.0 * fp[pre + "f.fc_1.actnorm.logs"])
        p2 = (torch.relu(p1) @ fp[pre + "f.fc_2.w"] + fp[pre + "f.fc_2.actnorm.b"]) * torch.exp(
            3.0 * fp[pre + "f.fc_2.actnorm.logs"])
        out[i] = sum(int((p.abs() <= 1e-5 * p.abs().max()).sum()) for p in (p1, p2))
        h = refpath.coupling_mlp(fp, pre, x1)
        x2 = (x2 + h[:, 0::2]) * torch.sigmoid(h[:, 1::2] + 2.0) if coupling == 1 else x2 + h
        x = torch.cat([x1, x2], 1)
    return out


def _flatten(o):
    """name -> tensor of every compared quantity"""
    flat = {k: o[k] for k in ("z_out", "logdet", "logp", "grad_z", "inv_z", "inv_negobj")}
    flat.update({"dparam/" + k: v for k, v in o["param"].items()})
    for k in o:
        if k.startswith("vjp_"):
            gz, gp = o[k]
            flat[k + "/z"] = gz
            flat.update({f"{k}/{n}": v for n, v in gp.items()})
    return flat


def _err(name, got, want):
    # values: the suite's max-relative REL_TOL metric; gradients: rel-l2 as tests/test_gpu_kernel_autograd.py
    if name in ("z_out", "logdet", "logp", "inv_z", "inv_negobj", "roundtrip"):
        return rel_err(got, want), REL_TOL
    return rel_l2(got, want), GRAD_TOL


#       nz, f_width, f_depth, coupling, permutation, B        samples per CTA; matrix ring; log|det W| / W^-1
CASES = [
    (4, 36, 2, 1, 2, 1),         # S=1; whole pass resident; Gauss-Jordan
    (4, 232, 1, 0, 2, 33),       # widest flow: falls back from S=2 to S=1; ring holds one matrix at a time
    (36, 100, 16, 0, 2, 31),     # S=1, deep
    (36, 4, 32, 1, 2, 65),       # S=4, deepest, narrowest
    (100, 36, 2, 1, 2, 1203),    # S=8, ragged last CTA
    (100, 100, 16, 1, 2, 33),    # S=2, deep; ring wraps
    (160, 36, 1, 1, 2, 65),      # S=4; largest Gauss-Jordan size
    (160, 100, 2, 0, 2, 1203),   # S=8; ring wraps
    (164, 36, 2, 1, 2, 31),      # S=1; torch det / inv
    (164, 100, 1, 1, 2, 65),     # S=4; torch det / inv
    (200, 36, 2, 1, 2, 1203),    # falls back from S=8 to S=4; W alone fills most of the ring
    (200, 4, 16, 0, 2, 33),      # S=2, deep; torch det / inv
    (128, 64, 32, 1, 2, 1250),   # falls back from S=8 to S=4 (config 4's batch, deepest flow)
    (4, 4, 1, 1, 1, 1),          # shuffle: S=1, smallest everything
    (4, 232, 2, 0, 1, 65),       # shuffle, widest flow: falls back from S=4 to S=1
    (36, 36, 32, 1, 1, 1203),    # shuffle: S=8, deepest
    (100, 100, 16, 1, 1, 31),    # shuffle: S=1, deep
    (160, 36, 16, 0, 1, 65),     # shuffle: S=4
    (164, 100, 2, 1, 1, 33),     # shuffle: S=2
    (200, 100, 1, 1, 1, 1203),   # shuffle: S=8
    (256, 64, 5, 1, 1, 100),     # shuffle at the largest nz (no nz^2 in the footprint)
]


@pytest.mark.parametrize("nz,w,depth,coupling,perm,B", CASES)
def test_flow_kernels_against_fp64_autograd(nz, w, depth, coupling, perm, B):
    sd = general_flow_state(nz, w, depth, coupling, perm)
    netF = _net(nz, w, depth, coupling, perm, sd)
    plan = netF._plan(B, DEV)
    plan.ensure_flow(netF, need_inverse=True)
    gen = torch.Generator().manual_seed(nz * 1000 + B)
    z = torch.randn(B, nz, generator=gen)
    eps = _inverse_input(sd, torch.randn(B, nz, generator=gen), depth, coupling, perm)
    gzo, gld = torch.randn(B, nz, generator=gen), torch.randn(B, generator=gen)
    seeds = {"both": (gzo, gld), "z_out": (gzo, None), "logdet": (None, gld)}
    zd = z.to(DEV)
    # ---- the kernels ----
    z_out, logdet, logp, grad_z = plan.flow_forward(zd, want_grad=True)
    inv_z, inv_negobj = plan.flow_inverse(eps.to(DEV))
    roundtrip, _ = plan.flow_inverse(z_out)
    flat, loss = plan.flow_param_grads(zd, B)
    got = {"z_out": z_out, "logdet": logdet, "logp": logp, "grad_z": grad_z, "inv_z": inv_z, "inv_negobj": inv_negobj}
    got.update({"dparam/" + k: v for k, v in _grad_names(netF, plan, flat).items()})
    for name, (sg, sl) in seeds.items():
        gz, flat_v = plan.flow_vjp(zd, None if sg is None else sg.to(DEV), None if sl is None else sl.to(DEV),
                                   want_params=True)
        got[f"vjp_{name}/z"] = gz
        got.update({f"vjp_{name}/{k}": v for k, v in _grad_names(netF, plan, flat_v).items()})
    got = {k: v.cpu() for k, v in got.items()}
    keys = sorted(k.split("/", 1)[1] for k in got if k.startswith("dparam/"))
    assert len(keys) == depth * (12 if perm == 2 else 11)
    # ---- the oracle in fp64, and in fp32 for the deep flows' bound ----
    want = oracle(sd, keys, z, eps, seeds, depth, coupling, perm, torch.float64)
    want_flat = _flatten(want)
    assert set(want_flat) == set(got), set(want_flat) ^ set(got)
    o32 = _flatten(oracle(sd, keys, z, eps, seeds, depth, coupling, perm, torch.float32)) if depth >= DEEP else {}
    assert abs(loss.item() - float(-want["logp"].mean())) <= REL_TOL * abs(float(want["logp"].mean()))
    kinks = near_kinks(sd, z, depth, coupling, perm)
    rows = []
    for name in sorted(got):
        e, tol = _err(name, got[name], want_flat[name])
        floor = _err(name, o32[name], want_flat[name])[0] if o32 else 0.0
        bound = max(tol, 4 * floor)
        step = name.split("revnet2d_step_s.")[-1].split(".")[0] if ".f.fc_1." in name or ".f.fc_2." in name else None
        if step is not None:
            bound = max(bound, kinks[int(step)] / B)
        rows.append((name, e, bound, floor))
    e_rt = rel_err(roundtrip.cpu(), z)
    floor_rt = rel_err(refpath.flow_reverse(_params(sd, torch.float32), want["z_out"].float(), torch.zeros(B), depth,
                                            coupling, perm)[0], z) if o32 else 0.0
    rows.append(("roundtrip", e_rt, max(REL_TOL, 4 * floor_rt), floor_rt))
    worst = max(rows, key=lambda r: r[1] / r[2])
    lad = 0.0
    if perm == 2:
        lad = max(abs(float(np.linalg.slogdet(sd[f"revnet2d_s.0.revnet2d_step_s.{i}.invertible_1x1_conv.w"]
                                              .astype(np.float64))[1])) for i in range(depth))
    print(f"flow nz={nz} w={w} depth={depth} coupling={coupling} perm={perm} B={B} (max |log det W| {lad:.2f}): "
          f"{len(rows)} quantities, worst {worst[0]} {worst[1]:.2e} (bound {worst[2]:.1e}, fp32 oracle {worst[3]:.1e}); "
          f"{sum(kinks.values())} ReLU inputs within 1e-5 of zero")
    record(f"r4_flow_shapes_nz{nz}_w{w}_d{depth}_c{coupling}_p{perm}_b{B}.json",
           {"case": dict(nz=nz, f_width=w, f_depth=depth, coupling=coupling, permutation=perm, B=B),
            "worst": {"name": worst[0], "err": worst[1], "bound": worst[2], "fp32_oracle": worst[3]},
            "max_abs_log_det_w": lad, "near_kinks": sum(kinks.values())})
    for name, e, bound, _ in rows:
        assert e <= bound, (name, e, bound)


@pytest.mark.parametrize("nz", [4, 36, 132, 160, 164])
def test_log_det_and_inverse_of_general_1x1_matrices(nz):
    # Additive coupling and zero actnorm log-scales: the flow's log-det is exactly sum_L log|det W_L|, so it must agree
    # with slogdet in fp64 to 1e-5 per step.  nz <= 160: the library's Gauss-Jordan kernel; 164: torch det / inv.
    depth, B = 4, 33    # one W of each kind
    sd = general_flow_state(nz, 36, depth, 0, 2, seed=5, zero_logs=True)
    ws = [sd[f"revnet2d_s.0.revnet2d_step_s.{i}.invertible_1x1_conv.w"].astype(np.float64) for i in range(depth)]
    signs, lads = zip(*(np.linalg.slogdet(w) for w in ws))
    assert min(signs) < 0 < max(signs) and max(abs(l) for l in lads) > 0.5
    assert any(np.all(np.diag(w) == 0) for w in ws)
    netF = _net(nz, 36, depth, 0, 2, sd)
    plan = netF._plan(B, DEV)
    plan.ensure_flow(netF, need_inverse=True)
    gen = torch.Generator().manual_seed(nz)
    z, eps = torch.randn(B, nz, generator=gen), torch.randn(B, nz, generator=gen)
    _, logdet, _, _ = plan.flow_forward(z.to(DEV))
    e_ld = float((logdet.cpu().double() - sum(lads)).abs().max())
    fp = _params(sd, torch.float64)
    zr, obj = refpath.flow_reverse(fp, eps.double(), torch.zeros(B, dtype=torch.float64), depth, 0, 2)
    inv_z, negobj = plan.flow_inverse(eps.to(DEV))
    e_inv, e_obj = rel_err(inv_z.cpu(), zr), float((negobj.cpu().double() + obj).abs().max())
    print(f"nz={nz}: sum log|det W| = {sum(lads):+.4f} (signs {signs}), kernel log-det off by {e_ld:.1e}; "
          f"inverse pass rel err {e_inv:.1e}, -objective off by {e_obj:.1e}")
    record(f"r4_flow_linalg_nz{nz}.json", {"nz": nz, "sum_log_abs_det": sum(lads), "logdet_abs_err": e_ld,
                                           "inverse_rel_err": e_inv, "negobj_abs_err": e_obj})
    assert e_ld <= 1e-5 * depth, e_ld
    assert e_obj <= 1e-5 * depth, e_obj
    assert e_inv <= REL_TOL, e_inv
