"""Which data-gradient stages run their cross terms in e4m3 (tc_cross_fp8): the 3-pass stages of the CTA-pair kernel
with at least 8 M tiles, at every benchmark workload; the weight-streaming stages of CelebA-HQ256 at B=8 (1 and 4 M
tiles) keep three 16-bit passes.  Host only."""
import ctypes as C

import pytest

from lsnf_b200 import _cabi


def _records(arch, nz, ngf, batch, bwd_passes=0):
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=3, f_depth=5, f_width=64,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=bwd_passes)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "create")
    out = []
    for i in range(lib.lsnf_plan_num_stages(h)):
        s, li = _cabi.StageInfo(), _cabi.LaunchInfo()
        _cabi.check(lib.lsnf_plan_stage_info(h, i, C.byref(s)), "info")
        _cabi.check(lib.lsnf_plan_stage_launch_info(h, i, 148, C.byref(li)), "launch")
        out.append((s, li))
    lib.lsnf_plan_destroy(h)
    return out


@pytest.mark.parametrize("arch,nz,ngf,batch,want", [
    ("cifar10", 128, 128, 100, [5, 6]),
    ("svhn", 100, 64, 100, [6]),
    ("celeba_crop", 100, 128, 100, [6, 7, 8]),
    ("celeba_hq256", 100, 128, 8, [10]),
])
def test_e4m3_cross_stages_of_the_benchmark_workloads(arch, nz, ngf, batch, want):
    recs = _records(arch, nz, ngf, batch)
    assert [i for i, (_s, li) in enumerate(recs) if li.cross_fp8] == want
    for s, li in recs:
        if li.cross_fp8:
            assert s.kind == 1 and li.kernel == _cabi.KERNEL_PAIR and s.passes == 3
            assert batch * s.grid_h * s.grid_w >= 8 * 128


def test_single_pass_data_gradient_keeps_its_format():
    assert not any(li.cross_fp8 for _s, li in _records("cifar10", 128, 128, 100, bwd_passes=1))
