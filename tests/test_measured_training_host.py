"""Host side of training from linear measurements y = A vec(G(z)) + sigma noise, on the CPU: the measured parameter
update of the oracle (fp64 autograd; the masked update for identity rows), the plan of a config with ``train`` and
``meas_rows`` (its workspace is the training plan's plus the measured regions, its stage and launch records are those
of the measured inference plan), and the Python plumbing with the plan stubbed: argument errors, the unmeasured call
unchanged, and a world-size-2 gloo run that shards y, hands A whole to each rank and normalises by the global batch.
The kernels are covered by tests/test_gpu_measured_training.py."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import lsnf_b200
from lsnf_b200 import _cabi, dist as ldist, langevin as llang, synth, train as ltrain
from oracle import refpath
import masked_oracle
import measured_oracle as MO
import measured_training_oracle as MTO
from helpers import rel_l2, to_torch
from test_plan_tables import BASELINE_CONFIGS, launch_infos, stage_infos

B, NC, IMG = 4, 3, 32
N = NC * IMG * IMG


# ---- the oracle ------------------------------------------------------------------------------------------------------
def _oracle_setup(seed=3, ngf=16, dtype=torch.float32):
    gp = to_torch(synth.generator_state("svhn", 100, ngf, 3, seed=seed), dtype=dtype)
    fp = to_torch(synth.flow_state(100, 64, 5, 1, 2, seed=seed), dtype=dtype)
    layers = refpath.generator_layers("svhn", 100, ngf)
    x_np, z0_np, _ = synth.inputs(B, 100, 3, 32, 1, seed=seed)
    return gp, fp, layers, torch.from_numpy(x_np), torch.from_numpy(z0_np).reshape(B, 100, 1, 1)


def _leaves(gp, fp):
    gl = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    fl = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in fp.items()}
    og = torch.optim.Adam(list(gl.values()), lr=1e-4, betas=(0.5, 0.999))
    of = torch.optim.Adam([fl[k] for k in refpath.trainable_flow_keys(fl)], lr=1e-4, betas=(0.5, 0.999))
    return gl, fl, og, of


def test_measured_parameter_update_is_fp64_autograd_of_the_measured_loss():
    gp, fp, layers, x, z0 = _oracle_setup(dtype=torch.float64)
    A = torch.from_numpy(MO.gaussian_operator(N // 8, N, seed=1)).double()
    y = x.double().reshape(B, -1) @ A.t() + 0.05
    gl, fl, og, of = _leaves(gp, fp)
    loss_g, _ = MTO.parameter_updates(gl, fl, z0.double(), y, A, layers, og, of, depth=5)
    # fp64, written out independently of the oracle's helpers: the loss and the gradients the Adam step was given
    leaves = {k: v.clone().requires_grad_(True) for k, v in gp.items()}
    xh = refpath.generator_forward(leaves, z0.double(), layers)
    r = xh.reshape(B, -1) @ A.t() - y
    want = (r * r).sum() / B
    want.backward()
    assert loss_g.item() == pytest.approx(want.item(), rel=1e-12)
    for k in gl:
        assert torch.allclose(gl[k].grad, leaves[k].grad, rtol=1e-10, atol=0), k
    # the fp32 oracle agrees with fp64
    g32 = _oracle_setup()[0]
    l32 = MTO.generator_loss(g32, z0, y.float(), A.float(), layers)
    assert abs(l32.item() - want.item()) < 1e-5 * want.item()


def test_identity_rows_of_a_mask_give_the_masked_parameter_update():
    gp, fp, layers, x, z0 = _oracle_setup()
    mask = np.ones((NC, IMG, IMG), np.float32)
    mask[:, 8:20, 4:30] = 0.0
    mask[1, ::3] = 0.0
    A = torch.from_numpy(MO.identity_rows(mask))
    y = x.reshape(B, -1)[:, torch.from_numpy(mask.reshape(-1) > 0)]
    gm, fm, ogm, ofm = _leaves(gp, fp)
    gk, fk, ogk, ofk = _leaves(gp, fp)
    lm, lfm = MTO.parameter_updates(gm, fm, z0, y, A, layers, ogm, ofm, depth=5)
    lk, lfk = masked_oracle.parameter_updates(gk, fk, z0, x, torch.from_numpy(mask).expand(B, NC, IMG, IMG), layers,
                                              ogk, ofk, depth=5)
    assert lm.item() == pytest.approx(lk.item(), rel=1e-5) and lfm.item() == lfk.item()
    for k in gm:
        assert rel_l2(gm[k].detach(), gk[k].detach()) < 1e-6, k


# ---- the plan of a config with train and meas_rows -------------------------------------------------------------------
def _create(arch, nz, ngf, batch, meas_rows, train):
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=3, f_depth=5, f_width=64,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=0, train=int(train),
                       meas_rows=meas_rows)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "create")
    return h


def _grad_layout(lib, h, L):
    off, size = (C.c_int64 * (2 * L))(), (C.c_int64 * (2 * L))()
    _cabi.check(lib.lsnf_generator_grad_layout(h, off, size), "layout")
    return list(off), list(size)


def _shifted(info, delta):
    """A copy of a stage record with its three workspace offsets moved by delta bytes."""
    s = _cabi.StageInfo.from_buffer_copy(bytes(info))
    s.a_offset += delta
    s.b_offset += delta
    s.out_offset += delta
    return bytes(s)


@pytest.mark.parametrize("arch,nz,ngf,batch", BASELINE_CONFIGS)
def test_training_plan_with_an_operator_is_the_training_plan_plus_the_measured_regions(arch, nz, ngf, batch):
    lib = _cabi.load()
    n = 3 * synth.image_size(arch) ** 2
    plain, train = _create(arch, nz, ngf, batch, 0, False), _create(arch, nz, ngf, batch, 0, True)
    ws_plain, ws_train = lib.lsnf_workspace_bytes(plain), lib.lsnf_workspace_bytes(train)
    s_plain, s_train = stage_infos(lib, plain), stage_infos(lib, train)
    L = len(s_plain) // 2
    # meas_rows = 0: the training plan's stages are the inference plan's, its extra regions come after them
    assert [bytes(x) for x in s_train] == [bytes(x) for x in s_plain]
    assert ws_train > ws_plain
    grads = lib.lsnf_generator_grad_floats(train)
    layout = _grad_layout(lib, train, L)
    for m in (1, 257, n // 4, n):
        meas, both = _create(arch, nz, ngf, batch, m, False), _create(arch, nz, ngf, batch, m, True)
        regions = lib.lsnf_workspace_bytes(meas) - ws_plain
        assert regions >= 8 * m * n
        assert lib.lsnf_workspace_bytes(both) == ws_train + regions
        s_meas, s_both = stage_infos(lib, meas), stage_infos(lib, both)
        assert len(s_both) == len(s_meas) == 2 * L + 2
        # the generator's stages are those of both plans without an operator, the operator's sit after the training
        # regions, shifted by exactly their size
        assert [bytes(x) for x in s_both[:2 * L]] == [bytes(x) for x in s_plain]
        assert [bytes(x) for x in s_both[2 * L:]] == [_shifted(x, ws_train - ws_plain) for x in s_meas[2 * L:]]
        for st in s_both[2 * L:]:
            assert min(st.a_offset, st.b_offset, st.out_offset) >= ws_train
        assert [bytes(x) for x in launch_infos(lib, both)] == [bytes(x) for x in launch_infos(lib, meas)]
        assert lib.lsnf_generator_grad_floats(both) == grads and _grad_layout(lib, both, L) == layout
        assert lib.lsnf_langevin_launch_count(both, 20) == lib.lsnf_langevin_launch_count(train, 20)
        lib.lsnf_plan_destroy(meas)
        lib.lsnf_plan_destroy(both)
    lib.lsnf_plan_destroy(plain)
    lib.lsnf_plan_destroy(train)


def test_measured_parameter_gradients_on_an_unbound_plan_fail_cleanly():
    lib = _cabi.load()
    h = _create("svhn", 100, 64, 4, 16, True)
    flat = (C.c_float * 4)()
    assert lib.lsnf_generator_param_grads_measured(h, flat, flat, 4, flat, None, -1, None) == -3
    assert lib.lsnf_generator_param_grads_measured(None, flat, flat, 4, flat, None, -1, None) == -1
    lib.lsnf_plan_destroy(h)


# ---- Python plumbing with the plan stubbed ---------------------------------------------------------------------------
class _RecordingPlan:
    """Stands in for a training plan: records every parameter-gradient call and every operator it is handed."""

    def __init__(self, netG):
        self.convs = [m for m in netG.gen if isinstance(m, torch.nn.ConvTranspose2d)]
        self.calls = []
        self.operators = []

    def ensure_generator(self, netG):
        pass

    def ensure_operator(self, A):
        self.operators.append(A)

    def generator_grad_layout(self):
        sizes = [p.numel() for m in self.convs for p in (m.weight, m.bias)]
        return [(sum(sizes[:i]), s) for i, s in enumerate(sizes)]

    def generator_param_grads(self, z, x, global_batch, flat, part=-1, loss=None, **kw):
        self.calls.append(("unmeasured", part, global_batch, tuple(x.shape), kw))
        return flat, torch.zeros(())

    def generator_param_grads_measured(self, z, y, global_batch, flat=None, part=-1, loss=None):
        self.calls.append(("measured", part, global_batch, tuple(y.shape), {}))
        return flat, torch.zeros(())


def _nets(ngf=4):
    args = lsnf_b200.make_args(dataset="svhn", nz=100, ngf=ngf, seed=5)
    return args, lsnf_b200._netG(args), lsnf_b200._netF(args, nz=100)


def _stub_plan(netG):
    plan = _RecordingPlan(netG)
    plan._ggrad_flat = torch.zeros(sum(s for _, s in plan.generator_grad_layout()))
    return plan


def test_generator_update_with_an_operator_makes_the_measured_calls(monkeypatch):
    args, netG, _ = _nets()
    plan = _stub_plan(netG)
    # meta tensors: the argument logic is device-independent
    z = torch.empty(6, 100, 1, 1, device="meta")
    A, y = torch.empty(40, N, device="meta"), torch.empty(6, 40, device="meta")
    ltrain.generator_update_begin(netG, None, z, y, args, plan=plan, operator=A, global_batch=11)
    assert plan.calls == [("measured", -1, 11, (6, 40), {})] and plan.operators == [A]
    # several ranks: the prologue, then each layer from the last down, all at the global batch
    plan.calls.clear()
    reduced = []
    monkeypatch.setattr(ltrain.torch.cuda, "current_stream", lambda dev: None)

    class _Ev:
        def record(self, s):
            pass

    class _Ctx:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    monkeypatch.setattr(ltrain.torch.cuda, "Event", _Ev)
    monkeypatch.setattr(ltrain.torch.cuda, "stream", lambda s: _Ctx())
    monkeypatch.setattr(ltrain.dist, "all_reduce", lambda t, **kw: reduced.append(t.shape) or object())

    class _Comm:
        def wait_event(self, ev):
            pass

    monkeypatch.setattr(ltrain, "_comm_stream", lambda dev: _Comm())
    ltrain.generator_update_begin(netG, None, z, y, args, plan=plan, operator=A, global_batch=11, world=2)
    assert [c[:3] for c in plan.calls] == [("measured", -2, 11), ("measured", 3, 11), ("measured", 2, 11),
                                          ("measured", 1, 11), ("measured", 0, 11)]
    assert len(reduced) == 5


def test_unmeasured_generator_update_passes_no_new_keyword():
    args, netG, _ = _nets()
    plan = _stub_plan(netG)
    z, x = torch.empty(6, 100, 1, 1, device="meta"), torch.empty(6, 3, 32, 32, device="meta")
    ltrain.generator_update_begin(netG, None, z, x, args, plan=plan)
    assert plan.calls == [("unmeasured", -1, 6, (6, 3, 32, 32), {"mask": None})] and plan.operators == []


@pytest.mark.parametrize("A_shape,y_shape,exc", [
    ((40, N + 1), (6, 40), ValueError), ((40,), (6, 40), ValueError), ((0, N), (6, 0), ValueError),
    ((40, N), (6, 41), ValueError), ((40, N), (5, 40), ValueError), ((40, N), (6, 40, 1), ValueError)])
def test_operator_and_measurement_shape_errors(A_shape, y_shape, exc):
    args, netG, _ = _nets()
    plan = _stub_plan(netG)
    z = torch.empty(6, 100, 1, 1, device="meta")
    with pytest.raises(exc):
        ltrain.generator_update_begin(netG, None, z, torch.empty(y_shape, device="meta"), args, plan=plan,
                                      operator=torch.empty(A_shape, device="meta"))
    with pytest.raises(TypeError):
        ltrain.generator_gradients(netG, z, torch.empty(6, 40, device="meta"), 6, plan=plan, operator=np.zeros((40, N)))
    assert plan.calls == []


def test_mask_and_operator_together_raise_value_error():
    args, netG, netF = _nets()
    plan = _stub_plan(netG)
    z = torch.empty(6, 100, 1, 1, device="meta")
    A, y = torch.empty(40, N, device="meta"), torch.empty(6, 40, device="meta")
    for fn in (lambda: ltrain.generator_update_begin(netG, None, z, y, args, plan=plan, operator=A, mask=y),
               lambda: ltrain.generator_gradients(netG, z, y, 6, plan=plan, operator=A, mask=y),
               lambda: lsnf_b200.training_iteration(y, netG, netF, None, None, args, operator=A, mask=y)):
        with pytest.raises(ValueError, match="not both"):
            fn()
    assert plan.calls == []


def _install_recorders(setattr_, log):
    def fake_langevin(z, x, netG, netF, args, verbose=False, **kw):
        log["langevin"] = dict(x=x, kw={k: v for k, v in kw.items() if k not in ("seed",)})
        return z.clone(), torch.tensor(1.0), torch.tensor(2.0)

    class Pending:
        def finish(self):
            return torch.tensor(3.0)

    def fake_gen_begin(netG, optG, z_k, x, args, **kw):
        log["gen"] = dict(x=x, kw=kw)
        return Pending()

    def fake_plan(*a, **kw):
        log["plan"] = kw
        return "plan"

    setattr_(ltrain, "sample_langevin_post_z_with_flow", fake_langevin)
    setattr_(ltrain, "generator_update_begin", fake_gen_begin)
    setattr_(ltrain, "flow_update", lambda netF, optF, z_k, args, **kw: log.__setitem__("flow", kw) or torch.tensor(4.0))
    setattr_(llang, "langevin_plan", fake_plan)


def test_training_iteration_passes_the_operator_to_inference_the_plan_and_the_update(monkeypatch):
    log = {}
    _install_recorders(monkeypatch.setattr, log)
    args, netG, netF = _nets()
    y, A = torch.zeros(6, 40), torch.zeros(40, N)
    lsnf_b200.training_iteration(y, netG, netF, None, None, args, seed=1, operator=A)
    assert log["langevin"]["x"] is y and log["langevin"]["kw"]["operator"] is A and log["langevin"]["kw"]["mask"] is None
    assert log["plan"] == {"train": True, "meas_rows": 40}
    assert log["gen"]["x"] is y and log["gen"]["kw"]["operator"] is A and "mask" not in log["gen"]["kw"]
    assert log["gen"]["kw"]["plan"] == "plan" and log["gen"]["kw"]["global_batch"] == 6
    assert "operator" not in log["flow"]
    # without an operator the calls carry no new keyword
    x = torch.zeros(6, 3, 32, 32)
    lsnf_b200.training_iteration(x, netG, netF, None, None, args, seed=1)
    assert "operator" not in log["langevin"]["kw"] and log["plan"] == {"train": True}
    assert set(log["gen"]["kw"]) == {"global_batch", "group", "world", "plan"}


# ---- data parallel: a world-size-2 gloo run --------------------------------------------------------------------------
def _worker(rank, world, port, tmp, sizes):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    log = {}
    _install_recorders(lambda obj, name, val: setattr(obj, name, val), log)
    args, netG, netF = _nets()
    Bg, m = sum(sizes), 24
    y_global = torch.arange(Bg * m, dtype=torch.float32).reshape(Bg, m)
    A = torch.ones(m, N)
    a, b = ldist.shard_range(Bg, rank, world)
    lsnf_b200.training_iteration(y_global[a:b], netG, netF, None, None, args, operator=A)
    out = dict(start=a, stop=b, lang_x=log["langevin"]["x"], lang_A=log["langevin"]["kw"]["operator"] is A,
               offset=log["langevin"]["kw"]["sample_offset"], gen_x=log["gen"]["x"],
               gen_A=log["gen"]["kw"]["operator"] is A, gen_batch=log["gen"]["kw"]["global_batch"],
               gen_world=log["gen"]["kw"]["world"], flow_batch=log["flow"]["global_batch"], plan=log["plan"])
    torch.save(out, f"{tmp}.{rank}")
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("sizes", [(6, 6), (7, 6)])
def test_data_parallel_iteration_shards_y_and_hands_each_rank_the_whole_operator(tmp_path, sizes):
    port = 33600 + (os.getpid() + sum(sizes)) % 2000
    tmp = str(tmp_path / "dp")
    mp.spawn(_worker, args=(2, port, tmp, sizes), nprocs=2, join=True)
    Bg, m = sum(sizes), 24
    y_global = torch.arange(Bg * m, dtype=torch.float32).reshape(Bg, m)
    for k in range(2):
        r = torch.load(f"{tmp}.{k}", weights_only=False)
        a, b = r["start"], r["stop"]
        assert b - a == sizes[k] and r["offset"] == a
        assert torch.equal(r["lang_x"], y_global[a:b]) and torch.equal(r["gen_x"], y_global[a:b])
        assert r["lang_A"] and r["gen_A"]
        assert r["gen_batch"] == r["flow_batch"] == Bg and r["gen_world"] == 2
        assert r["plan"] == {"train": True, "meas_rows": m}
