"""Host logic of the C library, no GPU: the stage tables (taps, phases, packed-weight index map) that drive the
tensor-core tap-GEMMs are emulated in numpy and compared with torch's conv_transpose2d and its data gradient."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from lsnf_b200 import _cabi, synth


def make_plan(arch, nz, ngf, batch, f_width=64):
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=3, f_depth=5, f_width=f_width,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "create")
    return lib, h


def stage_infos(lib, h):
    out = []
    for i in range(lib.lsnf_plan_num_stages(h)):
        s = _cabi.StageInfo()
        _cabi.check(lib.lsnf_plan_stage_info(h, i, C.byref(s)), "info")
        out.append(s)
    return out


def packed_matrix(lib, h, idx, info, w):
    """Packed hi-half operand [b_rows, b_k] of stage idx built through lsnf_plan_pack_index."""
    ci_n, co_n, k, _ = w.shape
    m = np.zeros((info.b_rows, info.b_k))
    r, c = C.c_int64(), C.c_int64()
    for ci in range(ci_n):
        for co in range(co_n):
            for ky in range(k):
                for kx in range(k):
                    _cabi.check(lib.lsnf_plan_pack_index(h, idx, ci, co, ky, kx, C.byref(r), C.byref(c)), "pack_index")
                    assert m[r.value, c.value] == 0.0, "two weights map to the same packed element"
                    m[r.value, c.value] = w[ci, co, ky, kx]
    return m


def taps_of(info, phase):
    if info.tap_gen_k:
        k = info.tap_gen_k
        return [(t // k, t % k, 0, 0, t * info.k_per_tap) for t in range(k * k)]
    return [(t.dy, t.dx, t.plane, t.brow, 0) for t in list(info.taps[phase])[: info.n_taps[phase]]]


def emulate(info, a, bm):
    """a: [planes, B, a_h, a_w, k_per_tap]; returns D [phase][B, grid_h, grid_w, n_pad]."""
    P, B, ah, aw, ka = a.shape
    gh, gw = info.grid_h, info.grid_w
    out = []
    for ph in range(info.n_phases):
        d = np.zeros((B, gh, gw, info.n_pad))
        for dy, dx, plane, brow, bcol in taps_of(info, ph):
            sh = np.zeros((B, gh, gw, ka))
            for m in range(gh):
                for n in range(gw):
                    y, x = m + dy, n + dx
                    if 0 <= y < ah and 0 <= x < aw:
                        sh[:, m, n, :] = a[plane, :, y, x, :]
            d += sh @ bm[brow:brow + info.n_pad, bcol:bcol + ka].T
        out.append(d)
    return out


@pytest.mark.parametrize("arch,nz,ngf", [("svhn", 100, 32), ("cifar10", 128, 32)])
def test_stage_tables_reproduce_conv_transpose_and_its_data_gradient(arch, nz, ngf):
    B = 2
    lib, h = make_plan(arch, nz, ngf, B)
    infos = stage_infos(lib, h)
    layers = synth.generator_layers(arch, nz, ngf)
    L = len(layers)
    assert len(infos) == 2 * L
    rng = np.random.default_rng(0)
    hin = 1
    for l, (ci, co, k, s, p) in enumerate(layers):
        hout = (hin - 1) * s - 2 * p + k
        w = rng.standard_normal((ci, co, k, k))
        x = rng.standard_normal((B, ci, hin, hin))
        xt = torch.from_numpy(x).requires_grad_(True)
        y = F.conv_transpose2d(xt, torch.from_numpy(w), stride=s, padding=p)
        g = rng.standard_normal(tuple(y.shape))
        gin = torch.autograd.grad(y, xt, torch.from_numpy(g))[0].numpy()
        # ---------- forward stage ----------
        fi = infos[l]
        assert fi.kind == 0 and fi.layer == l and fi.box_b * fi.box_h * fi.box_w == 128
        bm = packed_matrix(lib, h, l, fi, w)
        a = np.zeros((1, B, fi.a_h, fi.a_w, fi.k_per_tap))
        a[0, :, :, :, :ci] = x.transpose(0, 2, 3, 1)
        d = emulate(fi, a, bm)
        got = np.zeros((B, hout, hout, co))
        if l == 0:
            got = d[0][:, 0, 0, : fi.n_valid].reshape(B, k, k, co)
        elif l == L - 1:
            # direct product + gather (last_gather_tanh_kernel): every output pixel sums the taps that land on it
            assert fi.epilogue == 3 and fi.n_phases == 1 and fi.n_valid == k * k * co and fi.n_pad in (32, 64)
            dd = d[0]
            for oy in range(hout):
                for ox in range(hout):
                    for ky in range(k):
                        ty = oy + p - ky
                        if ty < 0 or ty % s or ty // s >= hin:
                            continue
                        for kx in range(k):
                            tx = ox + p - kx
                            if tx < 0 or tx % s or tx // s >= hin:
                                continue
                            t = ky * k + kx
                            got[:, oy, ox, :] += dd[:, ty // s, tx // s, t * co:(t + 1) * co]
        else:
            for ph in range(fi.n_phases):
                got[:, fi.out_off_y[ph]::fi.out_mul, fi.out_off_x[ph]::fi.out_mul, :] = d[ph][..., :co]
        np.testing.assert_allclose(got, y.detach().numpy().transpose(0, 2, 3, 1), rtol=1e-9, atol=1e-9)
        # ---------- data-gradient stage ----------
        bidx = L + (L - 1 - l)
        bi = infos[bidx]
        assert bi.kind == 1 and bi.layer == l
        bmb = packed_matrix(lib, h, bidx, bi, w)
        g_nhwc = g.transpose(0, 2, 3, 1)
        if l == L - 1:      # explicit im2col operand written by recon_grad_im2col_kernel
            a = np.zeros((1, B, hin, hin, 64))
            for iy in range(hin):
                for ix in range(hin):
                    for t in range(k * k):
                        oy, ox = iy * s - p + t // k, ix * s - p + t % k
                        if 0 <= oy < hout and 0 <= ox < hout:
                            a[0, :, iy, ix, t * co:(t + 1) * co] = g_nhwc[:, oy, ox, :]
        elif l == 0:        # plain NHWC; generated taps walk the k x k positions
            a = g_nhwc[None]
        else:               # phase-split planes
            a = np.stack([g_nhwc[:, py::2, px::2, :] for py in (0, 1) for px in (0, 1)])
            assert bi.a_planes == 4
        dg = emulate(bi, a, bmb)[0]
        want = gin.transpose(0, 2, 3, 1)
        np.testing.assert_allclose(dg[..., :ci], want, rtol=1e-9, atol=1e-9)
        if bi.n_pad > ci:
            assert np.all(dg[..., ci:] == 0)
        # consumer/producer layout agreement: a hidden data-gradient stage writes phase-split iff its consumer is stride 2
        if 0 < l:
            assert bi.out_phase_split == (1 if l - 1 > 0 else 0)
        hin = hout
    lib.lsnf_plan_destroy(h)


def test_plan_rejects_what_the_reference_rejects():
    lib = _cabi.load()
    h = C.c_void_p()

    def rc(**kw):
        base = dict(arch=0, batch=4, nz=100, ngf=64, nc=3, f_depth=5, f_width=64, f_permutation=2, f_coupling=1,
                    leak=0.2, gemm_impl=0)
        base.update(kw)
        return lib.lsnf_plan_create(C.byref(_cabi.Config(**base)), C.byref(h))

    assert rc() == 0
    lib.lsnf_plan_destroy(h)
    assert rc(nz=101) == -1 and b"even" in lib.lsnf_last_error()          # model.py:383
    assert rc(f_permutation=0) == -4                                      # model.py:372-379
    assert rc(f_coupling=2) == -4
    assert rc(arch=7) == -1                                               # model.py:154
    assert rc(ngf=8) == -1 and b"multiples of 64" in lib.lsnf_last_error()
    assert rc(batch=0) == -1


def test_compute_entry_points_fail_loudly_without_binding():
    lib, h = make_plan("svhn", 100, 32, 4)
    assert lib.lsnf_generator_forward(h, None, None, None) == -3          # LSNF_ERR_STATE: not bound
    assert b"bind" in lib.lsnf_last_error()
    assert lib.lsnf_workspace_bytes(h) > 0
    # split_z + per iteration (4 forward + fused last-layer kernel + 4 data-gradient + flow + update) + one
    # set-dyn kernel per replayed graph chunk of 40 iterations
    assert lib.lsnf_langevin_launch_count(h, 20) == 1 + 20 * (2 * 4 + 3) + 1
    assert lib.lsnf_langevin_launch_count(h, 8000) == 1 + 8000 * (2 * 4 + 3) + 200
    lib.lsnf_plan_destroy(h)


# ---- launch geometry of the tcgen05 path (host decisions: which kernel, ring, shared memory, occupancy) --------
import bench  # noqa: E402  (the BASELINE.json configurations live in bench.WORKLOADS)

BASELINE_CONFIGS = [(w["dataset"], w["nz"], w["ngf"], w["B"]) for w in bench.WORKLOADS.values()]
SMEM_MAX = 232448      # 227 KiB per CTA on sm_100
SMEM_PER_SM = 233472   # 228 KiB per SM, 1 KiB reserved per resident CTA


def launch_infos(lib, h, num_sms=148, bwd_passes=None):
    out = []
    for i in range(lib.lsnf_plan_num_stages(h)):
        li = _cabi.LaunchInfo()
        _cabi.check(lib.lsnf_plan_stage_launch_info(h, i, num_sms, C.byref(li)), "launch_info")
        out.append(li)
    return out


@pytest.mark.parametrize("bwd_passes", [1, 3])
@pytest.mark.parametrize("arch,nz,ngf,batch", BASELINE_CONFIGS)
def test_launch_geometry_respects_the_hardware_limits(arch, nz, ngf, batch, bwd_passes):
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=3, f_depth=5, f_width=64,
                       f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=bwd_passes)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "create")
    infos, launches = stage_infos(lib, h), launch_infos(lib, h)
    for s, li in zip(infos, launches):
        total = (s.tap_gen_k ** 2 if s.tap_gen_k else s.n_taps[0]) * (s.k_per_tap // 64)   # K blocks per tile
        assert li.block == 320 and li.grid_x >= 1 and li.grid_y >= 1 and li.grid_z >= 1
        assert li.smem_bytes <= SMEM_MAX
        assert li.ring_stages >= 1 and li.ring_stages * li.stage_bytes + 1280 <= li.smem_bytes
        # the CTAs one SM can hold must fit its shared memory and its 512 TMEM columns
        assert li.ctas_per_sm >= 1
        assert li.ctas_per_sm * (li.smem_bytes + 1024) <= SMEM_PER_SM
        assert li.ctas_per_sm * li.tmem_columns <= 512
        if li.kernel == _cabi.KERNEL_PAIR:
            # persistent CTA pairs: 256-wide N tiles, no split-K, a K loop worth pipelining, one pair per SM pair
            assert s.block_n == 256 and s.n_pad % 256 == 0 and s.k_splits == 1 and total >= 3
            assert li.grid_x % 2 == 0 and li.grid_x <= 148 and li.ctas_per_sm == 1 and li.tmem_columns == 512
            assert li.ring_stages * li.stage_bytes == 3 * 65536
            assert (li.ring_stages == 6) == (s.passes == 1)
            if li.stream_k:
                assert li.grid_x == 148 and total >= 8
        else:
            assert (li.grid_x, li.grid_y) == (-(-batch * s.grid_h * s.grid_w // 128), s.n_pad // s.block_n)
            assert li.grid_z == s.n_phases * s.k_splits and not li.stream_k
            if total <= 2 or (s.k_splits == 1 and total <= 4):
                assert li.ctas_per_sm >= 2, "short K loops must leave room for a second CTA per SM"
        if li.tma_store:
            # 16-bit outputs of wide tiles only, and 32 KiB of staging must exist
            assert s.epilogue in (0, 2) and s.block_n >= 128 and s.k_splits == 1
            if li.kernel == _cabi.KERNEL_SINGLE:
                assert li.ring_stages * li.stage_bytes >= 32768
    # the headline configuration: both wide forward layers and their data gradients run on the pair kernel
    if arch == "cifar10":
        kinds = [li.kernel for li in launches]
        assert kinds == [0, 1, 1, 0, 0, 1, 1, 0]
    lib.lsnf_plan_destroy(h)


def test_launch_geometry_scales_with_the_sm_count():
    lib, h = make_plan("cifar10", 128, 128, 100)
    for sms in (148, 132, 64):
        for li in launch_infos(lib, h, sms):
            if li.kernel == _cabi.KERNEL_PAIR:
                assert li.grid_x <= sms - sms % 2
    li = _cabi.LaunchInfo()
    assert lib.lsnf_plan_stage_launch_info(h, 99, 148, C.byref(li)) == -1
    assert lib.lsnf_plan_stage_launch_info(h, 0, 1, C.byref(li)) == -1
    lib.lsnf_plan_destroy(h)


def baseline_launch_records():
    """Every field of lsnf_plan_stage_launch_info, per stage of every BASELINE configuration."""
    recs = []
    for arch, nz, ngf, batch in BASELINE_CONFIGS:
        lib, h = make_plan(arch, nz, ngf, batch)
        recs.append([[getattr(li, f) for f, _ in li._fields_ if f != "reserved"] for li in launch_infos(lib, h)])
        lib.lsnf_plan_destroy(h)
    return recs


def test_launch_records_do_not_depend_on_the_environment():
    # How a stage launches depends on the stage and the SM count alone: variables that once forced the 1-CTA
    # kernel, per-thread epilogue stores or no stream-K change no record.
    import json
    import os
    import subprocess
    import sys
    tests = os.path.dirname(os.path.abspath(__file__))
    script = (f"import sys, json; sys.path[:0] = [{os.path.dirname(tests)!r}, {tests!r}]; import test_plan_tables as t; "
              "print(json.dumps(t.baseline_launch_records()))")
    env = dict(os.environ, LSNF_NO_PAIR="1", LSNF_NO_TMA_STORE="1", LSNF_STREAMK="0")
    out = subprocess.run([sys.executable, "-c", script], env=env, check=True, capture_output=True, text=True,
                         timeout=600).stdout
    assert json.loads(out.splitlines()[-1]) == baseline_launch_records()


def test_multiply_high_division_of_the_fused_last_layer_kernel_is_exact():
    # gen_aux.cu FastDiv: x / d == umulhi(x, floor((2^32 - 1) / d) + 1) whenever x * d < 2^32; the kernel divides
    # tile-local indices (< 2^16) by tile extents (< 2^11)
    rng = np.random.default_rng(0)
    for d in list(range(2, 70)) + [96, 128, 258, 660, 1020, 1980, 2047]:
        m = (0xFFFFFFFF // d) + 1
        xs = np.concatenate([np.arange(0, 4096), rng.integers(0, min(2 ** 32 // d, 2 ** 20), 4096)]).astype(np.uint64)
        assert np.array_equal((xs * np.uint64(m)) >> np.uint64(32), xs // np.uint64(d)), d
