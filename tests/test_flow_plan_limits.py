"""Plan creation refuses exactly the flow configurations whose fused flow kernels cannot launch (no GPU needed).

The forward kernel keeps its per-step activations and a ring of the streamed matrices in the 227 KB of shared memory
one CTA may opt in to; lsnf_plan_create checks that footprint at one sample per CTA with the function the launchers
use, and the launchers drop to a smaller samples-per-CTA tier where the preferred one does not fit, so whether a
configuration runs does not depend on the batch.  tests/test_gpu_flow_shapes.py runs the accepted ones."""
import ctypes as C

import pytest

from lsnf_b200 import _cabi


def _create(**kw):
    lib = _cabi.load()
    base = dict(arch=_cabi.ARCH["none"], batch=100, nz=100, ngf=0, nc=3, f_depth=5, f_width=64, f_permutation=2,
                f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=3, train=0)
    base.update(kw)
    h = C.c_void_p()
    rc = lib.lsnf_plan_create(C.byref(_cabi.Config(**base)), C.byref(h))
    msg = lib.lsnf_last_error()
    if rc == 0:
        lib.lsnf_plan_destroy(h)
    return rc, msg


@pytest.mark.parametrize("kw", [
    dict(f_width=256),                                   # f_width^2 alone is 256 KB
    dict(f_width=240, nz=4, f_depth=1),                  # 225 KB of matrix plus the fixed part
    dict(f_width=236, nz=4, f_depth=1),                  # the first width past the bound
    dict(nz=256, f_permutation=2),                       # nz^2 of the invertible 1x1 matrix
    dict(nz=232, f_permutation=2, f_width=4, f_depth=1),
    dict(nz=208, f_permutation=2, f_depth=32),           # W plus the activation stash of 32 steps
    dict(nz=256, f_permutation=1, f_width=200, f_depth=1),
    dict(nz=100, f_width=196, f_depth=32),
])
def test_plan_creation_refuses_flows_that_cannot_launch(kw):
    rc, msg = _create(**kw)
    assert rc == -1, (kw, rc)
    assert b"shared memory" in msg and b"f_width" in msg, msg


@pytest.mark.parametrize("kw", [
    dict(nz=256, f_permutation=1, f_width=64),           # the shuffle has no matrix: nz^2 does not count
    dict(nz=128, f_width=64, f_depth=32, batch=1250),    # fits at S = 4 (not at its preferred S = 8)
    dict(nz=100, f_width=128, f_depth=32, batch=1250),   # the CelebA-HQ256 flow, deep, at config 4's batch
    dict(nz=4, f_width=232, f_depth=1, batch=33),        # the widest flow that fits
    dict(nz=228, f_permutation=2, f_width=4, f_depth=1),  # the largest W that fits
    dict(nz=204, f_permutation=2, f_depth=32),
    dict(nz=256, f_permutation=1, f_width=196, f_depth=1),
    dict(nz=100, f_width=192, f_depth=32),
    dict(nz=200, f_width=100, f_depth=1, f_permutation=1, batch=1203),
])
def test_plan_creation_accepts_flows_that_fit_at_one_sample_per_cta(kw):
    rc, msg = _create(**kw)
    assert rc == 0, (kw, msg)


@pytest.mark.parametrize("arch,ngf", [("svhn", 64), ("cifar10", 128)])
@pytest.mark.parametrize("train", [False, True])
def test_generator_plans_get_their_plan_at_the_largest_nz(arch, ngf, train, monkeypatch):
    # _netG._plan carries a placeholder flow the generator never runs; it must not be what refuses the plan
    import lsnf_b200
    from lsnf_b200 import model
    seen = {}
    monkeypatch.setattr(model, "get_plan", lambda **kw: seen.update(kw))
    netG = lsnf_b200._netG(lsnf_b200.make_args(dataset=arch, nz=256, ngf=ngf))
    netG._plan(100, "cuda:0", train=train)
    cfg = {k: seen[k] for k in ("batch", "nz", "ngf", "nc", "f_depth", "f_width", "f_permutation", "f_coupling", "leak")}
    rc, msg = _create(arch=_cabi.ARCH[arch], train=int(train), **cfg)
    assert rc == 0, msg
    # the invertible 1x1 placeholder would have been refused: nz^2 = 256 KB
    assert _create(arch=_cabi.ARCH[arch], **dict(cfg, f_permutation=2))[0] == -1
