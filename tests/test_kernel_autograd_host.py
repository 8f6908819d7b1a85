"""Host logic of ``lsnf_b200.kernel_autograd`` on the CPU, with the plan stubbed: the switch defaults to off, CPU tensors
stay on the eager branch, the generator's backward asks the library for parameter gradients only when autograd will
accumulate them, and a backward whose activations were overwritten re-runs its forward pass first.  The kernels behind
the plan are covered by tests/test_gpu_kernel_autograd.py; the new C entry points' error paths are checked here."""
import ctypes as C

import pytest
import torch

import lsnf_b200
from lsnf_b200 import _cabi, autograd_fns


class FakePlan:
    """Records what the Functions ask of a plan; the 'kernels' are cheap CPU stand-ins with the right shapes."""

    def __init__(self, net, batch, train):
        self.net, self.batch, self.train = net, batch, train
        self.act_epoch = 0
        self.forwards, self.vjps = [], []

    def ensure_generator(self, net):
        pass

    def ensure_flow(self, net, need_inverse=False):
        pass

    def generator_forward(self, z):
        self.act_epoch += 1
        self.forwards.append(z.clone())
        return torch.tanh(z.sum(1)).reshape(-1, 1, 1, 1).expand(-1, 3, 32, 32).contiguous()

    def generator_grad_layout(self):
        sizes = [p.numel() for m in self.net.gen if isinstance(m, torch.nn.ConvTranspose2d) for p in (m.weight, m.bias)]
        offs = [sum(sizes[:i]) for i in range(len(sizes))]
        return list(zip(offs, sizes))

    def generator_vjp(self, grad_x_hat, want_z=True, want_params=False):
        self.vjps.append(dict(want_z=want_z, want_params=want_params, z=self.forwards[-1].clone()))
        n = sum(s for _, s in self.generator_grad_layout())
        return (torch.ones(self.batch, self.net.nz) if want_z else None,
                torch.ones(n) if want_params else None)

    def flow_forward(self, z, want_grad=False):
        return z.clone(), torch.zeros(z.shape[0]), torch.zeros(z.shape[0]), None

    def flow_grad_layout(self):
        sizes = [p.numel() if p is not None else 1 for p in autograd_fns._flow_params(self.net)]
        return [(sum(sizes[:i]), s) for i, s in enumerate(sizes)]

    def flow_vjp(self, z, grad_z_out, grad_logdet, want_z=True, want_params=False):
        self.vjps.append(dict(want_z=want_z, want_params=want_params, seed_g=grad_z_out is not None,
                              seed_ld=grad_logdet is not None))
        n = sum(s for _, s in self.flow_grad_layout())
        return (torch.ones_like(z) if want_z else None, torch.ones(n) if want_params else None)


@pytest.fixture
def nets(monkeypatch):
    args = lsnf_b200.make_args(dataset="svhn", nz=100, ngf=8)
    netG, netF = lsnf_b200._netG(args), lsnf_b200._netF(args, nz=100)
    plans = {}

    def fake_plan(net):
        def make(batch, device, train=False):
            key = (id(net), batch, train)
            if key not in plans:
                plans[key] = FakePlan(net, batch, train)
            return plans[key]
        return make

    monkeypatch.setattr(netG, "_plan", fake_plan(netG))
    monkeypatch.setattr(netF, "_plan", fake_plan(netF))
    return netG, netF, plans


def test_the_switch_defaults_to_off_and_works_as_a_call_and_as_a_context_manager():
    assert autograd_fns.is_enabled() is False
    with lsnf_b200.kernel_autograd():
        assert autograd_fns.is_enabled()
        with lsnf_b200.kernel_autograd(False):
            assert not autograd_fns.is_enabled()
        assert autograd_fns.is_enabled()
    assert not autograd_fns.is_enabled()
    lsnf_b200.kernel_autograd(True)
    try:
        assert autograd_fns.is_enabled()
    finally:
        lsnf_b200.kernel_autograd(False)
    assert not autograd_fns.is_enabled()


def test_cpu_tensors_take_the_eager_branch_with_the_switch_on(nets):
    netG, netF, plans = nets
    z = torch.randn(4, 100, 1, 1, requires_grad=True)
    with lsnf_b200.kernel_autograd():
        x = netG(z)
        zo, obj, extra = netF(z.reshape(4, 100), torch.zeros(4))
        zr = netF(zo, obj, reverse=True)
    for t in (x, zo, obj, zr):
        assert "_GeneratorFn" not in type(t.grad_fn).__name__ and "_FlowFn" not in type(t.grad_fn).__name__
    assert extra == [] and plans == {}        # no plan was asked for anything
    g = torch.autograd.grad(x.sum() + obj.sum(), z)[0]
    assert g.shape == z.shape


def _gen(netG, z):
    return autograd_fns.generator_apply(netG, z)


def test_autograd_grad_wrt_z_asks_for_no_parameter_gradients_and_backward_does(nets):
    netG, _, plans = nets
    x = torch.zeros(4, 3, 32, 32)
    z = torch.randn(4, 100, 1, 1, requires_grad=True)
    # the reference closure (train.py:313-314): parameters still require grad, only dL/dz is asked for
    xh = _gen(netG, z)
    gz = torch.autograd.grad(((xh - x) ** 2).sum(), z)[0]
    assert gz.shape == z.shape
    (plan,) = plans.values()
    assert not plan.train and plan.vjps[-1] == dict(want_z=True, want_params=False, z=plan.vjps[-1]["z"])
    assert all(p.grad is None for p in netG.parameters())
    # the reference's generator update (train.py:390-394): z detached, loss.backward() fills every parameter's .grad
    xh = _gen(netG, z.detach())
    ((xh - x) ** 2).sum().backward()
    train_plans = [p for p in plans.values() if p.train]
    assert len(train_plans) == 1
    tp = train_plans[0]
    assert tp.vjps[-1]["want_params"] and not tp.vjps[-1]["want_z"]
    assert len(tp.forwards) == 1                          # the training plan ran the forward pass of this z itself
    assert all(p.grad is not None and torch.all(p.grad == 1) for p in netG.parameters())


def test_a_second_forward_on_the_plan_makes_the_first_backward_rerun_its_forward(nets):
    netG, _, plans = nets
    z1 = torch.randn(4, 100, requires_grad=True)
    z2 = torch.randn(4, 100, requires_grad=True)
    y1 = _gen(netG, z1)
    (plan,) = plans.values()
    y2 = _gen(netG, z2)
    assert len(plan.forwards) == 2
    torch.autograd.grad(y1.sum(), z1)
    assert len(plan.forwards) == 3 and torch.equal(plan.vjps[-1]["z"], z1.detach())   # re-ran at z1
    torch.autograd.grad(y2.sum(), z2)
    assert len(plan.forwards) == 4 and torch.equal(plan.vjps[-1]["z"], z2.detach())
    y3 = _gen(netG, z1)
    torch.autograd.grad(y3.sum(), z1)
    assert len(plan.forwards) == 5                        # nothing in between: no re-run


def test_flow_backward_passes_null_seeds_for_unused_outputs_and_parameter_gradients_on_backward(nets):
    _, netF, plans = nets
    z = torch.randn(4, 100, requires_grad=True)
    zo, logdet = autograd_fns.flow_apply(netF, z)
    torch.autograd.grad(logdet.sum(), z)
    (plan,) = plans.values()
    assert plan.vjps[-1] == dict(want_z=True, want_params=False, seed_g=False, seed_ld=True)
    zo, logdet = autograd_fns.flow_apply(netF, z.detach())
    (0.5 * (zo ** 2).sum() - logdet.sum()).backward()
    assert plan.vjps[-1] == dict(want_z=False, want_params=True, seed_g=True, seed_ld=True)
    assert netF.revnet2d_s[0].revnet2d_step_s[0].actnorm.logs.grad is not None


def test_the_backward_is_once_differentiable(nets):
    netG, _, _ = nets
    z = torch.randn(4, 100, requires_grad=True)
    g = torch.autograd.grad((_gen(netG, z) ** 2).sum(), z, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.sum().backward()


def test_vjp_entry_points_fail_with_a_status_and_a_message_on_an_unbound_plan():
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH["cifar10"], batch=4, nz=128, ngf=128, nc=3, f_depth=5, f_width=64,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=_cabi.GEMM_TCGEN05, bwd_passes=0, train=1)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "lsnf_plan_create")
    try:
        buf = (C.c_float * 16)()
        for rc in (lib.lsnf_generator_vjp(h, buf, buf, buf, None),
                   lib.lsnf_flow_vjp(h, buf, buf, buf, buf, buf, None)):
            assert rc == -3                                   # LSNF_ERR_STATE
            assert b"lsnf_plan_bind" in lib.lsnf_last_error()
        assert lib.lsnf_generator_vjp(None, buf, buf, buf, None) == -1
    finally:
        lib.lsnf_plan_destroy(h)
