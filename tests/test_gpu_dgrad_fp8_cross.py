"""The wide data-gradient stages with their cross terms in e4m3 (DESIGN.md section 4.1): the operand conversion equals
torch's float8_e4m3fn rounding bit for bit, each such stage's output equals an fp64 contraction of the very operands
it read (which pins the instruction and shared-memory descriptors, the K order of the e4m3 row and the scales), and
repeated calls and graph replays give identical bits."""
import ctypes as C

import numpy as np
import pytest
import torch

import lsnf_b200
from lsnf_b200 import _cabi, synth
from helpers import build_nets

pytestmark = pytest.mark.gpu

CONFIGS = [dict(dataset="cifar10", nz=128, ngf=128), dict(dataset="svhn", nz=100, ngf=64)]
B = 100


def _plan(c):
    dev = torch.device("cuda:0")
    _, netG, netF = build_nets(c)
    plan = lsnf_b200.langevin_plan(netG, netF, B, dev, 3)
    plan.ensure_generator(netG)
    plan.ensure_flow(netF)
    x_np, z_np, _ = synth.inputs(B, c["nz"], 3, plan.img, 1, seed=5)
    x = torch.from_numpy(x_np).to(dev)
    z = torch.from_numpy(z_np).to(dev).reshape(B, c["nz"]).contiguous()
    return plan, netG, x, z


def _cross_stages(plan):
    sms = torch.cuda.get_device_properties(plan.device).multi_processor_count
    out = []
    for i in range(len(plan.stages())):
        rec = _cabi.LaunchInfo()
        _cabi.check(plan.lib.lsnf_plan_stage_launch_info(plan.handle, i, sms, C.byref(rec)), "launch_info")
        if rec.cross_fp8:
            assert rec.kernel == _cabi.KERNEL_PAIR
            out.append(i)
    return out


def _ws(plan):
    return plan._ws[plan._ws_ptr - plan._ws.data_ptr():]


def _bf16(ws, off, n):
    return ws[off:off + 2 * n].view(torch.bfloat16)


def _fp8_scale_exp(m):
    """csrc/lsnf_internal.cuh fp8_scale_exp: k with m * 2^k in [128, 256)."""
    if not m > 0:
        return 0
    return max(-40, min(40, 8 - int(np.frexp(np.float32(m))[1])))


def _operands(ws, off, rows, K):
    """(fp16 hi, the first and the second e4m3 half of each 128-byte row) of a converted / packed operand
    [rows][fp16 x K | e4m3 row pairs], as float64."""
    buf = ws[off:off + rows * 4 * K].view(rows, 4 * K)
    hi16 = buf[:, :2 * K].contiguous().view(torch.float16).double()
    x8 = buf[:, 2 * K:].reshape(rows, K // 64, 2, 64).contiguous().view(torch.float8_e4m3fn).double()
    return hi16, x8[:, :, 0].reshape(rows, K), x8[:, :, 1].reshape(rows, K)


@pytest.mark.parametrize("c", CONFIGS, ids=[c["dataset"] for c in CONFIGS])
def test_cross_stages_match_an_fp64_contraction_of_their_operands(c):
    plan, netG, x, z = _plan(c)
    stages = plan.stages()
    cross = _cross_stages(plan)
    if c["dataset"] == "cifar10":
        assert cross == [5, 6]
    assert cross, "no stage runs its cross terms in e4m3"
    plan.generator_forward(z)
    plan.generator_dgrad(x, 0.3)
    torch.cuda.synchronize()
    ws = _ws(plan)
    leak = 0.2
    for i in cross:
        s, prod = stages[i], stages[i - 1]
        K, H = s.k_per_tap, s.grid_h
        rows_a = B * s.a_planes * s.a_h * s.a_w
        # ---- the conversion of the producer's bf16 hi|lo output, bit for bit ----
        g = _bf16(ws, prod.out_offset, rows_a * 2 * K).view(rows_a, 2 * K)
        v = g[:, :K].float() + g[:, K:].float()                   # exact in fp32
        ka = _fp8_scale_exp(float(v.abs().max()))
        v = v * 2.0 ** ka
        h = v.to(torch.float16).float()
        conv = ws[s.a_offset:s.a_offset + rows_a * 4 * K].view(rows_a, 4 * K)
        want_hi16 = (h * 32.0).to(torch.float16).contiguous().view(torch.uint8)
        assert torch.equal(conv[:, :2 * K].contiguous(), want_hi16.view(rows_a, 2 * K)), (i, "hi16")
        x8 = conv[:, 2 * K:].reshape(rows_a, K // 64, 2, 64)
        want_h8 = h.to(torch.float8_e4m3fn).view(torch.uint8).reshape(rows_a, K // 64, 64)
        want_l8 = ((v - h) * 2048.0).to(torch.float8_e4m3fn).view(torch.uint8).reshape(rows_a, K // 64, 64)
        assert torch.equal(x8[:, :, 0], want_h8), (i, "hi8")
        assert torch.equal(x8[:, :, 1], want_l8), (i, "lo8")
        # ---- the stage's output against fp64 over the same operands ----
        a_hs, a_h8, a_l8 = _operands(ws, s.a_offset, rows_a, K)
        a_cat = torch.cat([a_hs, a_h8, a_l8], 1).view(s.a_planes, B, s.a_h, s.a_w, 3 * K)
        w_hs, w_l8, w_h8 = _operands(ws, s.b_offset, s.b_rows, K)
        w_cat = torch.cat([w_hs, w_l8, w_h8], 1)                 # pairs a_hi8 with w_lo8 and a_lo8 with w_hi8
        kw = _fp8_scale_exp(float(netG.state_dict()[f"gen.{3 * s.layer}.weight"].abs().max()))
        N = s.n_pad
        acc = torch.zeros(B, H, H, N, dtype=torch.float64, device=ws.device)
        padded = torch.nn.functional.pad(a_cat, (0, 0, 1, 1, 1, 1))   # |dy|, |dx| <= 1: zero fill as TMA does
        for t in range(s.n_taps[0]):
            tp = s.taps[0][t]
            a_t = padded[tp.plane, :, 1 + tp.dy:1 + tp.dy + H, 1 + tp.dx:1 + tp.dx + H]
            acc += a_t @ w_cat[tp.brow:tp.brow + N].T
        ref = acc * 2.0 ** -(ka + kw + 11)
        # LeakyReLU' from the sign of the saved forward activation act[l-1] (fp16 hi|lo, [B][H][H][2N])
        act_off = stages[s.layer - 1].out_offset
        act = ws[act_off:act_off + B * H * H * 2 * N * 2].view(torch.float16).view(B, H, H, 2 * N)
        neg = torch.signbit(act[..., :N])
        ref = torch.where(neg, ref * leak, ref)
        out = _bf16(ws, s.out_offset, B * H * H * 2 * N)
        if s.out_phase_split:
            out = out.view(2, 2, B, H // 2, H // 2, 2 * N).permute(2, 3, 0, 4, 1, 5).reshape(B, H, H, 2 * N)
        else:
            out = out.view(B, H, H, 2 * N)
        got = out[..., :N].double() + out[..., N:].double()
        err = float((got - ref).norm() / ref.norm())
        worst = float(((got - ref).abs() / ref.abs().max()).max())
        print(f"{c['dataset']} stage {i}: ka {ka} kw {kw} rel-l2 {err:.2e} worst {worst:.2e}")
        # fp32 accumulation plus the 16-bit hi|lo output (about 2^-17 relative); a wrong K order, pairing or scale
        # leaves errors of 2^-8 and more
        assert err < 2e-5, (i, err)
        assert worst < 1e-4, (i, worst)


@pytest.mark.parametrize("c", CONFIGS, ids=[c["dataset"] for c in CONFIGS])
def test_repeated_calls_and_graph_replays_are_bit_identical(c):
    plan, _netG, x, z = _plan(c)
    plan.generator_forward(z)
    g1 = plan.generator_dgrad(x, 0.3).clone()
    g2 = plan.generator_dgrad(x, 0.3).clone()
    assert torch.equal(g1, g2)
    # stages run alone (the producers of the e4m3 stages included) leave the scales of the next call alone
    for i in range(len(plan.stages()) // 2, len(plan.stages()) - 1):
        plan.run_stage(i)
    plan.generator_forward(z * 4.0)
    for i in range(len(plan.stages()) // 2, len(plan.stages()) - 1):
        plan.run_stage(i)
    plan.generator_forward(z)
    assert torch.equal(plan.generator_dgrad(x, 0.3), g1)
    runs = [plan.langevin_run(z, x, 45, 0.1, 0.3, True, seed=11)[0].clone() for _ in range(3)]   # eager, then replays
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[1], runs[2])
