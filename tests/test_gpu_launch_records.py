"""The launch record lsnf_plan_stage_launch_info reports is the launch each tap-GEMM stage makes: every stage of a
CIFAR-10 and an SVHN plan runs alone under torch.profiler, and the kernel's name, grid, block and shared memory in the
trace must equal the record for the device's SM count."""
import ctypes as C
import json
import os
import re
import tempfile

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import lsnf_b200
from lsnf_b200 import _cabi, synth
from helpers import build_nets, record

pytestmark = pytest.mark.gpu

# The trace reports static plus dynamic shared memory.  The tap-GEMM kernels declare only dynamic shared memory, and
# on a B200 their static share in the trace is 0 (the 1 KiB per CTA the system reserves is not counted).
STATIC_SMEM = 0


def _kernel_events(trace_path):
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    return sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])


@pytest.mark.parametrize("bwd_passes", [1, 3])
@pytest.mark.parametrize("c", [dict(dataset="cifar10", nz=128, ngf=128), dict(dataset="svhn", nz=100, ngf=64)])
def test_each_stage_launches_as_its_record_says(c, bwd_passes):
    dev = torch.device("cuda:0")
    B = 100
    _, netG, netF = build_nets(c)
    plan = lsnf_b200.langevin_plan(netG, netF, B, dev, bwd_passes)
    plan.ensure_generator(netG)
    x_np, z_np, _ = synth.inputs(B, c["nz"], 3, plan.img, 1, seed=3)
    plan.generator_forward(torch.from_numpy(z_np).to(dev).reshape(B, c["nz"]).contiguous())
    plan.generator_dgrad(torch.from_numpy(x_np).to(dev), 0.3)
    n = len(plan.stages())
    for i in range(n):   # module loading and first-launch work stay out of the trace
        plan.run_stage(i)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            plan.run_stage(i)
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        kernels = _kernel_events(path)
    assert len(kernels) == n, [k["name"] for k in kernels]

    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    seen = []
    for i, k in enumerate(kernels):
        rec = _cabi.LaunchInfo()
        _cabi.check(plan.lib.lsnf_plan_stage_launch_info(plan.handle, i, sms, C.byref(rec)), "launch_info")
        info = plan.stages()[i]
        if rec.kernel == _cabi.KERNEL_PAIR:
            want = r"tapgemm_tc2_kernel<"
        else:
            want = rf"tapgemm_tc_kernel<{info.block_n}>"
        args = k["args"]
        seen.append({"stage": i, "name": k["name"], "grid": args["grid"], "block": args["block"],
                     "shared memory": args["shared memory"], "record smem": rec.smem_bytes})
        assert re.search(want, k["name"]), (i, k["name"], want)
        assert list(args["grid"]) == [rec.grid_x, rec.grid_y, rec.grid_z], (i, args["grid"])
        assert list(args["block"]) == [rec.block, 1, 1], (i, args["block"])
        assert args["shared memory"] == rec.smem_bytes + STATIC_SMEM, (i, args["shared memory"], rec.smem_bytes)
    record(f"launch_records_{c['dataset']}_bwd{bwd_passes}.json", {"sms": sms, "stages": seen})
