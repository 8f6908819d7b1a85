"""Python owner of one ``lsnf_plan`` (include/lsnf.h): workspace allocation through torch, parameter packing with
change tracking, and thin typed wrappers over the C-ABI entry points.  PyTorch is used for device memory and
streams only."""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Dict, Optional, Tuple

import torch

from . import _cabi

_FLOW_PARAM_ORDER = ("actnorm.b", "actnorm.logs", "invertible_1x1_conv.w", "f.fc_1.w", "f.fc_1.actnorm.b",
                     "f.fc_1.actnorm.logs", "f.fc_2.w", "f.fc_2.actnorm.b", "f.fc_2.actnorm.logs", "f.fc_zeros.w",
                     "f.fc_zeros.b", "f.fc_zeros.logs")


def flow_step_params(st):
    """The twelve parameter tensors of one ``revnet2d_step`` in the order of ``_FLOW_PARAM_ORDER`` (plain attribute
    access: this runs once per training iteration); ``None`` for the 1x1 matrix of a shuffle step."""
    f = st.f
    w = st.invertible_1x1_conv.w if st.invertible_1x1_conv is not None else None
    return [st.actnorm.b, st.actnorm.logs, w, f.fc_1.w, f.fc_1.actnorm.b, f.fc_1.actnorm.logs, f.fc_2.w,
            f.fc_2.actnorm.b, f.fc_2.actnorm.logs, f.fc_zeros.w, f.fc_zeros.b, f.fc_zeros.logs]


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _check_tensor(t: torch.Tensor, name: str, device, shape=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the Langevin path has no CPU fallback")
    if t.device != device:
        raise RuntimeError(f"{name} is on {t.device}, plan is on {device}")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32 (got {t.dtype})")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise RuntimeError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")


def as_mask(mask, x: torch.Tensor) -> torch.Tensor:
    """The per-pixel likelihood weight ``mask`` of a masked reconstruction loss as the library reads it: an fp32
    contiguous tensor of x's shape [B,nc,H,W] on x's device.  ``mask`` may have any shape that broadcasts to x's
    ([B,1,H,W], [1,1,H,W], [H,W], ...) and any real or bool dtype (True = 1 = observed, 0 = missing; fractional weights
    in [0, 1] are allowed).  A mask on the CPU raises RuntimeError, as x does; a shape that does not broadcast to x's
    raises ValueError."""
    if not isinstance(mask, torch.Tensor):
        raise TypeError("mask must be a torch.Tensor")
    try:
        shape = torch.broadcast_shapes(tuple(mask.shape), tuple(x.shape))
    except RuntimeError:
        shape = None
    if shape != tuple(x.shape):
        raise ValueError(f"mask of shape {tuple(mask.shape)} does not broadcast to x's shape {tuple(x.shape)}")
    if mask.device.type == "cpu":
        raise RuntimeError("mask must be a CUDA tensor: the Langevin path has no CPU fallback")
    if mask.device != x.device:
        raise RuntimeError(f"mask is on {mask.device}, x is on {x.device}")
    if mask.is_complex():
        raise ValueError("mask must be real")
    return mask.detach().to(torch.float32).expand(x.shape).contiguous()


def as_operator(A, x_shape) -> torch.Tensor:
    """The dense linear measurement operator ``A`` [m, n] of y = A vec(x) + noise as the library reads it: a contiguous
    fp32 CUDA matrix whose columns match the images, n = nc*H*W for x of shape ``x_shape`` ([B,nc,H,W] or [nc,H,W];
    vec is x.view(B, -1), NCHW order).  Raises TypeError for a non-tensor, ValueError for a matrix that is not 2-D, has
    the wrong column count, a dtype that does not cast to fp32 (complex) or a non-finite value, and RuntimeError for a
    CPU tensor.  Heteroscedastic noise: scale row i of A and of y by sigma / sigma_i."""
    if not isinstance(A, torch.Tensor):
        raise TypeError("operator must be a torch.Tensor")
    n = 1
    for d in tuple(x_shape)[-3:]:
        n *= int(d)
    if A.dim() != 2:
        raise ValueError(f"operator must be a 2-D matrix [m, n] (got shape {tuple(A.shape)})")
    if A.shape[1] != n or A.shape[0] < 1:
        raise ValueError(f"operator of shape {tuple(A.shape)} does not act on images of {n} = nc*H*W values")
    if A.is_complex() or A.dtype == torch.bool:
        raise ValueError(f"operator of dtype {A.dtype} does not cast to float32")
    if A.device.type != "meta" and not bool(torch.isfinite(A).all()):
        raise ValueError("operator has non-finite values")
    if A.device.type == "cpu":
        raise RuntimeError("operator must be a CUDA tensor: the Langevin path has no CPU fallback")
    return A.detach().to(torch.float32).contiguous()


def as_measurements(y, A: torch.Tensor, batch: int) -> torch.Tensor:
    """``y`` [batch, m] for the operator A [m, n] as an fp32 contiguous tensor; ValueError for another shape."""
    if not isinstance(y, torch.Tensor):
        raise TypeError("y must be a torch.Tensor")
    if tuple(y.shape) != (int(batch), int(A.shape[0])):
        raise ValueError(f"y has shape {tuple(y.shape)}, expected [B, m] = {(int(batch), int(A.shape[0]))}")
    return y.detach().to(torch.float32).contiguous()


class Plan:
    def __init__(self, *, arch: str, batch: int, nz: int, ngf: int, nc: int, f_depth: int, f_width: int,
                 f_permutation: int, f_coupling: int, leak: float, device, gemm_impl: int = _cabi.GEMM_TCGEN05,
                 bwd_passes: int = 0, train: bool = False, meas_rows: int = 0):
        self.lib = _cabi.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("lsnf_b200 plans live on a CUDA device; there is no CPU fallback")
        self.cfg = _cabi.Config(arch=_cabi.ARCH[arch], batch=batch, nz=nz, ngf=ngf, nc=nc, f_depth=f_depth,
                                f_width=f_width, f_permutation=f_permutation, f_coupling=f_coupling, leak=leak,
                                gemm_impl=gemm_impl, bwd_passes=bwd_passes, train=int(bool(train)),
                                meas_rows=int(meas_rows))
        self.arch, self.batch, self.nz, self.nc = arch, batch, nz, nc
        self.train = bool(train)
        self.meas_rows = int(meas_rows)
        self.f_depth, self.f_permutation = f_depth, f_permutation
        handle = C.c_void_p()
        _cabi.check(self.lib.lsnf_plan_create(C.byref(self.cfg), C.byref(handle)), "lsnf_plan_create")
        self.handle = handle
        self.ws_bytes = self.lib.lsnf_workspace_bytes(self.handle)
        with torch.cuda.device(self.device):
            self._ws = torch.zeros(self.ws_bytes + 1024, dtype=torch.uint8, device=self.device)
            base = self._ws.data_ptr()
            self._ws_ptr = (base + 1023) // 1024 * 1024
            _cabi.check(self.lib.lsnf_plan_bind(self.handle, C.c_void_p(self._ws_ptr), self.ws_bytes), "lsnf_plan_bind")
        self._g_sig = None
        self._f_sig = None
        self._f_has_inv = False
        self._a_sig = None
        self._keep = []  # tensors referenced by in-flight pack kernels
        # bumped by every call that overwrites the generator activations in the workspace (and by a re-pack, which
        # makes them stale): a backward pass that finds it moved re-runs its forward pass before lsnf_generator_vjp
        self.act_epoch = 0
        from .synth import image_size
        self.img = image_size(arch) if arch != "none" else 0

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.lsnf_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---- introspection -------------------------------------------------------------------------------
    def stages(self):
        out = []
        for i in range(self.lib.lsnf_plan_num_stages(self.handle)):
            info = _cabi.StageInfo()
            _cabi.check(self.lib.lsnf_plan_stage_info(self.handle, i, C.byref(info)), "lsnf_plan_stage_info")
            out.append(info)
        return out

    def run_stage(self, index: int) -> None:
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_plan_run_stage(self.handle, int(index), _stream(self.device)), "lsnf_plan_run_stage")

    def launch_count(self, steps: int) -> int:
        return int(self.lib.lsnf_langevin_launch_count(self.handle, steps))

    # ---- parameters ----------------------------------------------------------------------------------
    @staticmethod
    def _sig(tensors):
        """What the packed copies were made from: the Parameter OBJECTS (weakly referenced), their storage and their
        version counters.  Storage address + version alone is not an identity: the caching allocator hands the
        addresses of a freed model to the next one, whose freshly loaded parameters carry the same versions -- a
        second model built after the first one was dropped would silently run on the first one's packed weights."""
        return tuple((weakref.ref(t), t.data_ptr(), t._version) for t in tensors)

    @staticmethod
    def _same(sig, tensors) -> bool:
        return sig is not None and len(sig) == len(tensors) and all(
            r() is t and ptr == t.data_ptr() and ver == t._version for (r, ptr, ver), t in zip(sig, tensors))

    def invalidate(self) -> None:
        """Forget the packed parameters: the next call re-packs the generator and flow weights (and re-evaluates the
        hoisted log|det W| / W^-1).  Packed copies are keyed on (data_ptr, Parameter._version); in-place edits through
        ``.data`` (``p.data.copy_()``, EMA swaps, manual init -- the idiom the reference itself uses) do not bump the
        version counter, so call this (or ``lsnf_b200.invalidate_plans()``) after such an edit."""
        self._g_sig = None
        self._f_sig = None
        self._f_has_inv = False

    def ensure_generator(self, netG) -> None:
        convs = [m for m in netG.gen if isinstance(m, torch.nn.ConvTranspose2d)]
        ws = [m.weight for m in convs]
        bs = [m.bias for m in convs]
        if self._same(self._g_sig, ws + bs):
            return
        sig = self._sig(ws + bs)
        for i, (w, b) in enumerate(zip(ws, bs)):
            _check_tensor(w.data, f"gen.{3 * i}.weight", self.device)
            _check_tensor(b.data, f"gen.{3 * i}.bias", self.device)
        wp = _cabi.ptr_array([w.data_ptr() for w in ws])
        bp = _cabi.ptr_array([b.data_ptr() for b in bs])
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_pack_generator_weights(self.handle, wp, bp, len(ws), C.c_void_p(_stream(self.device))),
                        "lsnf_pack_generator_weights")
        self._g_sig = sig
        self.act_epoch += 1

    def ensure_flow(self, netF, need_inverse: bool = False) -> None:
        steps = netF.revnet2d_s[0].revnet2d_step_s
        named = []
        for st in steps:
            ps = flow_step_params(st)
            if ps[2] is None:
                ps[2] = ps[0]  # placeholder pointer for the absent 1x1 matrix, ignored by the library
            named += ps
        if self._same(self._f_sig, named) and (self._f_has_inv or not need_inverse):
            return
        sig = self._sig(named)
        for t in named:
            _check_tensor(t.data, "flow parameter", self.device)
        with torch.cuda.device(self.device), torch.no_grad():
            params = _cabi.ptr_array([t.data_ptr() for t in named])
            keep = []
            perm = perm_inv = lad_ptr = winv = None
            if self.f_permutation == 2 and self.nz <= 160:
                # log|det W| (fp64, model.py:182) and W^-1 (model.py:193) by the library's own kernel: one launch
                # instead of two batched torch LU factorisations (~1 ms of small kernels per parameter version)
                need_inverse = True
            elif self.f_permutation == 2:
                w_all = torch.stack([st.invertible_1x1_conv.w.detach() for st in steps])
                # model.py:182 -- determinant in fp64, cast back to fp32; hoisted out of the loop
                lad = torch.log(torch.abs(torch.linalg.det(w_all.double()))).float().contiguous()
                keep.append(lad)
                lad_ptr = C.c_void_p(lad.data_ptr())
                if need_inverse:
                    # model.py:193 (fp32).  inv_ex: torch.linalg.inv reads cuSOLVER's status on the HOST (a device
                    # synchronisation per call, i.e. per training iteration); a singular W gives inf/NaN latents instead
                    inv = torch.linalg.inv_ex(w_all, check_errors=False).inverse.contiguous()
                    keep.append(inv)
                    winv = _cabi.ptr_array([inv[i].data_ptr() for i in range(len(steps))])
            else:
                idx = [st.shuffle_features.indices.data.contiguous() for st in steps]
                idv = [st.shuffle_features.indices_inverse.data.contiguous() for st in steps]
                keep += idx + idv
                perm = _cabi.ptr_array([t.data_ptr() for t in idx])
                perm_inv = _cabi.ptr_array([t.data_ptr() for t in idv])
            _cabi.check(self.lib.lsnf_pack_flow_weights(self.handle, params, perm, perm_inv, lad_ptr, winv,
                                                        C.c_void_p(_stream(self.device))), "lsnf_pack_flow_weights")
            self._keep = keep
        self._f_sig = sig
        self._f_has_inv = need_inverse or self.f_permutation != 2

    def ensure_operator(self, A: torch.Tensor) -> None:
        """Pack the measurement operator A [meas_rows, nc*H*W] (``as_operator``) unless this very tensor, at the same
        storage and version, is already packed: an in-place edit of A (which bumps its version) is repacked."""
        if self._same(self._a_sig, [A]):
            return
        sig = self._sig([A])
        a = as_operator(A, (self.nc, self.img, self.img))
        if a.shape[0] != self.meas_rows or a.device != self.device:
            raise ValueError(f"operator of shape {tuple(a.shape)} on {a.device} does not fit this plan "
                             f"(meas_rows {self.meas_rows}, {self.device})")
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_pack_measurement(self.handle, a.data_ptr(), C.c_void_p(_stream(self.device))),
                        "lsnf_pack_measurement")
        self._keep_a = a   # read by the pack kernels in flight
        self._a_sig = sig

    # ---- compute -------------------------------------------------------------------------------------
    def generator_forward(self, z: torch.Tensor) -> torch.Tensor:
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        out = torch.empty(self.batch, self.nc, self.img, self.img, dtype=torch.float32, device=self.device)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_forward(self.handle, z.data_ptr(), out.data_ptr(), _stream(self.device)),
                        "lsnf_generator_forward")
        return out

    def generator_dgrad(self, x: torch.Tensor, sigma: float, *, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """d/dz [1/(2 sigma^2) sum m (G(z) - x)^2] at the z of the last ``generator_forward``; m = ``mask`` (see
        ``as_mask``), or 1 without one."""
        _check_tensor(x, "x", self.device, (self.batch, self.nc, self.img, self.img))
        m = as_mask(mask, x) if mask is not None else None
        g = torch.empty(self.batch, self.nz, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_dgrad_masked(self.handle, x.data_ptr(), m.data_ptr() if m is not None
                                                             else None, float(sigma), g.data_ptr(), _stream(self.device)),
                        "lsnf_generator_dgrad_masked")
        return g

    def generator_vjp(self, grad_x_hat: torch.Tensor, want_z: bool = True, want_params: bool = False):
        """(dL/dz [B,nz] or None, flat parameter-gradient buffer or None) for upstream dL/dx_hat, at the z of the last
        ``generator_forward`` on this plan (``act_epoch`` tells whether that is still the one in the workspace).
        ``want_params`` needs ``train=True``; the buffer has the layout of ``generator_grad_layout``."""
        _check_tensor(grad_x_hat, "grad_x_hat", self.device, (self.batch, self.nc, self.img, self.img))
        g = torch.empty(self.batch, self.nz, dtype=torch.float32, device=self.device) if want_z else None
        flat = None
        if want_params:
            flat = torch.empty(int(self.lib.lsnf_generator_grad_floats(self.handle)), dtype=torch.float32,
                               device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_vjp(self.handle, grad_x_hat.data_ptr(), g.data_ptr() if want_z else None,
                                                    flat.data_ptr() if want_params else None, _stream(self.device)),
                        "lsnf_generator_vjp")
        return g, flat

    def flow_vjp(self, z: torch.Tensor, grad_z_out: Optional[torch.Tensor], grad_logdet: Optional[torch.Tensor],
                 want_z: bool = True, want_params: bool = False):
        """(dL/dz [B,nz] or None, flat parameter-gradient buffer or None) of the forward flow at z for upstream
        dL/dz_out [B,nz] and dL/dlogdet [B] (either None = 0).  The buffer has the layout of ``flow_grad_layout``;
        ``want_params`` needs ``ensure_flow(netF, need_inverse=True)``."""
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        if grad_z_out is not None:
            _check_tensor(grad_z_out, "grad_z_out", self.device, (self.batch, self.nz))
        if grad_logdet is not None:
            _check_tensor(grad_logdet, "grad_logdet", self.device, (self.batch,))
        g = torch.empty_like(z) if want_z else None
        flat = None
        if want_params:
            flat = torch.zeros(int(self.lib.lsnf_flow_grad_floats(self.handle)), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_flow_vjp(
                self.handle, z.data_ptr(), grad_z_out.data_ptr() if grad_z_out is not None else None,
                grad_logdet.data_ptr() if grad_logdet is not None else None, g.data_ptr() if want_z else None,
                flat.data_ptr() if want_params else None, _stream(self.device)), "lsnf_flow_vjp")
        return g, flat

    def flow_forward(self, z: torch.Tensor, want_grad: bool = False):
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        z_out = torch.empty_like(z)
        logdet = torch.empty(self.batch, dtype=torch.float32, device=self.device)
        logp = torch.empty_like(logdet)
        grad = torch.empty_like(z) if want_grad else None
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_flow_forward(self.handle, z.data_ptr(), z_out.data_ptr(), logdet.data_ptr(),
                                                   logp.data_ptr(), grad.data_ptr() if want_grad else None,
                                                   _stream(self.device)), "lsnf_flow_forward")
        return z_out, logdet, logp, grad

    def flow_inverse(self, eps: torch.Tensor):
        _check_tensor(eps, "eps", self.device, (self.batch, self.nz))
        z = torch.empty_like(eps)
        negobj = torch.empty(self.batch, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_flow_inverse(self.handle, eps.data_ptr(), z.data_ptr(), negobj.data_ptr(),
                                                   _stream(self.device)), "lsnf_flow_inverse")
        return z, negobj

    def sample_prior(self, eps: torch.Tensor, to_unit_range: bool = True, want_z: bool = False):
        """eps [B,nz] -> x = clamp((G(F^-1(eps)) + 1) / 2, 0, 1) in one C-ABI call (train.py:565-576)."""
        _check_tensor(eps, "eps", self.device, (self.batch, self.nz))
        x = torch.empty(self.batch, self.nc, self.img, self.img, dtype=torch.float32, device=self.device)
        z = torch.empty_like(eps) if want_z else None
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_sample_prior(self.handle, eps.data_ptr(), x.data_ptr(),
                                                   z.data_ptr() if want_z else None, int(bool(to_unit_range)),
                                                   _stream(self.device)), "lsnf_sample_prior")
        return (x, z) if want_z else x

    # ---- generator parameter update (train.py:390-398) -----------------------------------------------
    def generator_grad_layout(self):
        """[(offset, size)] inside the flat gradient buffer: layer l's weight gradient (the parameter's own
        [C_in, C_out, k, k] layout) at index 2l, its bias gradient at 2l+1 (lsnf_generator_grad_layout)."""
        n = 2 * len([s for s in self.stages() if s.kind == 0])
        off, size = (C.c_int64 * n)(), (C.c_int64 * n)()
        _cabi.check(self.lib.lsnf_generator_grad_layout(self.handle, off, size), "lsnf_generator_grad_layout")
        return [(int(off[i]), int(size[i])) for i in range(n)]

    def generator_param_grads(self, z: torch.Tensor, x: torch.Tensor, global_batch: int,
                              flat: Optional[torch.Tensor] = None, part: int = -1, loss: Optional[torch.Tensor] = None,
                              *, mask: Optional[torch.Tensor] = None):
        """Gradients of loss_g = mse_sum(G(z), x) / global_batch w.r.t. every generator weight and bias into one
        flat fp32 buffer (returned with this rank's share of loss_g).  Needs ``train=True`` at plan creation and
        ``ensure_generator`` on the current parameters.  ``part``: -1 everything; -2 forward + loss + data-gradient
        chain only; l >= 0 only layer l's gradients (include/lsnf.h).  ``mask`` (see ``as_mask``) weights the loss
        per pixel, loss_g = sum m (G(z) - x)^2 / global_batch; only the part -1 and -2 calls read it."""
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        _check_tensor(x, "x", self.device, (self.batch, self.nc, self.img, self.img))
        m = as_mask(mask, x) if mask is not None else None
        n = int(self.lib.lsnf_generator_grad_floats(self.handle))
        if flat is None:
            flat = torch.zeros(n, dtype=torch.float32, device=self.device)
        _check_tensor(flat, "flat gradient buffer", self.device, (n,))
        if loss is None:
            loss = torch.empty((), dtype=torch.float32, device=self.device)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_param_grads_masked(
                self.handle, z.data_ptr(), x.data_ptr(), m.data_ptr() if m is not None else None, int(global_batch),
                flat.data_ptr(), loss.data_ptr(), int(part), _stream(self.device)), "lsnf_generator_param_grads_masked")
        return flat, loss

    def generator_param_grads_measured(self, z: torch.Tensor, y: torch.Tensor, global_batch: int,
                                       flat: Optional[torch.Tensor] = None, part: int = -1,
                                       loss: Optional[torch.Tensor] = None):
        """``generator_param_grads`` for the measured loss loss_g = |A vec(G(z)) - y|^2 / global_batch with the operator
        of the last ``ensure_operator``; y [B, meas_rows].  Needs ``train=True`` and ``meas_rows`` > 0 at plan
        creation; only the part -1 and -2 calls read y."""
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        _check_tensor(y, "y", self.device, (self.batch, self.meas_rows))
        n = int(self.lib.lsnf_generator_grad_floats(self.handle))
        if flat is None:
            flat = torch.zeros(n, dtype=torch.float32, device=self.device)
        _check_tensor(flat, "flat gradient buffer", self.device, (n,))
        if loss is None:
            loss = torch.empty((), dtype=torch.float32, device=self.device)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_param_grads_measured(
                self.handle, z.data_ptr(), y.data_ptr(), int(global_batch), flat.data_ptr(), loss.data_ptr(), int(part),
                _stream(self.device)), "lsnf_generator_param_grads_measured")
        return flat, loss

    # ---- flow parameter update (train.py:403-415) ----------------------------------------------------
    def flow_grad_layout(self):
        """[(offset, size)] of every flow parameter gradient inside the flat buffer, step-major, in the order of
        ``_FLOW_PARAM_ORDER`` (include/lsnf.h: lsnf_flow_grad_layout)."""
        n = self.f_depth * _cabi.FLOW_PTRS_PER_STEP
        off, size = (C.c_int64 * n)(), (C.c_int64 * n)()
        _cabi.check(self.lib.lsnf_flow_grad_layout(self.handle, off, size), "lsnf_flow_grad_layout")
        return [(int(off[i]), int(size[i])) for i in range(n)]

    def flow_param_grads(self, z: torch.Tensor, global_batch: int, flat: Optional[torch.Tensor] = None):
        """Gradients of loss_f = -(1/global_batch) sum_b log p(z_b) w.r.t. every flow parameter, into one flat
        fp32 buffer (returned with this rank's share of loss_f as a 0-d tensor).  ``ensure_flow(netF,
        need_inverse=True)`` must have packed the current parameters."""
        _check_tensor(z, "z", self.device, (self.batch, self.nz))
        n = int(self.lib.lsnf_flow_grad_floats(self.handle))
        if flat is None:
            flat = torch.zeros(n, dtype=torch.float32, device=self.device)
        _check_tensor(flat, "flat gradient buffer", self.device, (n,))
        loss = torch.empty((), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_flow_param_grads(self.handle, z.data_ptr(), int(global_batch), flat.data_ptr(),
                                                       loss.data_ptr(), _stream(self.device)), "lsnf_flow_param_grads")
        return flat, loss

    def langevin_update(self, z, grad_g, grad_f, step_size, eps=None, with_noise=True, seed=0, sample_offset=0,
                        step=0, want_norms=True):
        for t, n in ((z, "z"), (grad_g, "grad_g"), (grad_f, "grad_f")):
            _check_tensor(t, n, self.device, (self.batch, self.nz))
        if eps is not None:
            _check_tensor(eps, "eps", self.device, (self.batch, self.nz))
        norms = torch.empty(2, dtype=torch.float32, device=self.device) if want_norms else None
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_langevin_update(
                self.handle, z.data_ptr(), grad_g.data_ptr(), grad_f.data_ptr(), float(step_size),
                eps.data_ptr() if eps is not None else None, int(bool(with_noise)), int(seed), int(sample_offset),
                int(step), norms.data_ptr() if want_norms else None, _stream(self.device)), "lsnf_langevin_update")
        return norms

    def langevin_run(self, z0, x, steps, step_size, sigma, with_noise=True, eps=None, seed=0, sample_offset=0,
                     out: Optional[torch.Tensor] = None, norms: Optional[torch.Tensor] = None, *,
                     mask: Optional[torch.Tensor] = None):
        """``steps`` Langevin iterations from z0 on the energy 1/(2 sigma^2) sum m (G(z) - x)^2 - log p(z), with
        m = ``mask`` (see ``as_mask``) or 1 without one.  Returns (z_T, [mean |grad_g|, mean |grad_f|])."""
        _check_tensor(z0, "z", self.device, (self.batch, self.nz))
        _check_tensor(x, "x", self.device, (self.batch, self.nc, self.img, self.img))
        m = as_mask(mask, x) if mask is not None else None
        if eps is not None:
            _check_tensor(eps, "eps", self.device, (steps, self.batch, self.nz))
        if out is None:
            out = torch.empty_like(z0)
        if norms is None:
            norms = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_langevin_run_masked(
                self.handle, z0.data_ptr(), x.data_ptr(), m.data_ptr() if m is not None else None, int(steps),
                float(step_size), float(sigma), int(bool(with_noise)), eps.data_ptr() if eps is not None else None,
                int(seed) & (2 ** 64 - 1), int(sample_offset), out.data_ptr(), norms.data_ptr(), _stream(self.device)),
                "lsnf_langevin_run_masked")
        return out, norms

    def langevin_run_measured(self, z0, y, steps, step_size, sigma, with_noise=True, eps=None, seed=0,
                              sample_offset=0):
        """``steps`` Langevin iterations from z0 on |A vec(G(z)) - y|^2 / (2 sigma^2) - log p(z) with the operator of
        the last ``ensure_operator``; y [B, meas_rows].  Returns (z_T, [mean |grad_g|, mean |grad_f|])."""
        _check_tensor(z0, "z", self.device, (self.batch, self.nz))
        _check_tensor(y, "y", self.device, (self.batch, self.meas_rows))
        if eps is not None:
            _check_tensor(eps, "eps", self.device, (steps, self.batch, self.nz))
        out = torch.empty_like(z0)
        norms = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_langevin_run_measured(
                self.handle, z0.data_ptr(), y.data_ptr(), int(steps), float(step_size), float(sigma),
                int(bool(with_noise)), eps.data_ptr() if eps is not None else None, int(seed) & (2 ** 64 - 1),
                int(sample_offset), out.data_ptr(), norms.data_ptr(), _stream(self.device)),
                "lsnf_langevin_run_measured")
        return out, norms

    def generator_dgrad_measured(self, y: torch.Tensor, sigma: float) -> torch.Tensor:
        """d/dz [|A vec(G(z)) - y|^2 / (2 sigma^2)] at the z of the last ``generator_forward``."""
        _check_tensor(y, "y", self.device, (self.batch, self.meas_rows))
        g = torch.empty(self.batch, self.nz, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_generator_dgrad_measured(self.handle, y.data_ptr(), float(sigma), g.data_ptr(),
                                                               _stream(self.device)), "lsnf_generator_dgrad_measured")
        return g

    def ais_run(self, z0, x, betas, steps, step_size, sigma, *, target_accept: float = 0.0,
                mask: Optional[torch.Tensor] = None, eps: Optional[torch.Tensor] = None,
                u: Optional[torch.Tensor] = None, seed: int = 0, sample_offset: int = 0):
        """Annealed importance sampling with MALA transitions from z0 along the schedule ``betas`` [steps+1] (fp32, on
        the plan's device) on pi_beta(z) ~ p(z) exp(-beta sum m (G(z) - x)^2 / (2 sigma^2)) (include/lsnf.h:
        lsnf_ais_run).  ``target_accept`` > 0 adapts each chain's step size, <= 0 keeps ``step_size``.  ``eps``
        [steps,B,nz] and ``u`` [steps,B] inject the noise.  Returns (z_T [B,nz], log w [B] without the likelihood's
        normalising constant, acceptance rate [B])."""
        _check_tensor(z0, "z", self.device, (self.batch, self.nz))
        _check_tensor(x, "x", self.device, (self.batch, self.nc, self.img, self.img))
        _check_tensor(betas, "betas", self.device, (int(steps) + 1,))
        m = as_mask(mask, x) if mask is not None else None
        if eps is not None:
            _check_tensor(eps, "eps", self.device, (steps, self.batch, self.nz))
        if u is not None:
            _check_tensor(u, "u", self.device, (steps, self.batch))
        z_out = torch.empty_like(z0)
        log_w = torch.empty(self.batch, dtype=torch.float32, device=self.device)
        rate = torch.empty_like(log_w)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_ais_run(
                self.handle, z0.data_ptr(), x.data_ptr(), m.data_ptr() if m is not None else None, betas.data_ptr(),
                int(steps), float(step_size), float(target_accept), float(sigma),
                eps.data_ptr() if eps is not None else None, u.data_ptr() if u is not None else None,
                int(seed) & (2 ** 64 - 1), int(sample_offset), z_out.data_ptr(), log_w.data_ptr(), rate.data_ptr(),
                _stream(self.device)), "lsnf_ais_run")
        return z_out, log_w, rate

    def ais_run_measured(self, z0, y, betas, steps, step_size, sigma, *, target_accept: float = 0.0,
                         eps: Optional[torch.Tensor] = None, u: Optional[torch.Tensor] = None, seed: int = 0,
                         sample_offset: int = 0):
        """``ais_run`` on pi_beta(z) ~ p(z) exp(-beta |A vec(G(z)) - y|^2 / (2 sigma^2)), y [B, meas_rows], with the
        operator of the last ``ensure_operator``.  log w is without -(m/2) log(2 pi sigma^2)."""
        _check_tensor(z0, "z", self.device, (self.batch, self.nz))
        _check_tensor(y, "y", self.device, (self.batch, self.meas_rows))
        _check_tensor(betas, "betas", self.device, (int(steps) + 1,))
        if eps is not None:
            _check_tensor(eps, "eps", self.device, (steps, self.batch, self.nz))
        if u is not None:
            _check_tensor(u, "u", self.device, (steps, self.batch))
        z_out = torch.empty_like(z0)
        log_w = torch.empty(self.batch, dtype=torch.float32, device=self.device)
        rate = torch.empty_like(log_w)
        self.act_epoch += 1
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.lsnf_ais_run_measured(
                self.handle, z0.data_ptr(), y.data_ptr(), betas.data_ptr(), int(steps), float(step_size),
                float(target_accept), float(sigma), eps.data_ptr() if eps is not None else None,
                u.data_ptr() if u is not None else None, int(seed) & (2 ** 64 - 1), int(sample_offset),
                z_out.data_ptr(), log_w.data_ptr(), rate.data_ptr(), _stream(self.device)), "lsnf_ais_run_measured")
        return z_out, log_w, rate


_PLANS: Dict[Tuple, Plan] = {}


def default_bwd_passes(noisy_chain: bool = False) -> int:
    """Tensor-core passes of the data-gradient stages (include/lsnf.h, DESIGN.md section 4.1).

    Always 3 (bf16 hi|lo split, 16 significant bits per operand: z_T at the reference's own fp32 noise floor) unless the caller opts
    in to the single fp16 pass with ``bwd_passes=1`` / ``LSNF_BWD_PASSES=1``: that mode is ~1.4x faster end to end
    but carries an 11-bit significand through the gradient (measured margins on z_T against the 1e-4 budget:
    profiles/r2_parity_cifar10_b100_t40.json).  ``noisy_chain`` is kept for call compatibility and ignored."""
    import os
    env = os.environ.get("LSNF_BWD_PASSES")
    if env:
        return int(env)
    return 3


def get_plan(*, arch, batch, nz, ngf, nc, f_depth, f_width, f_permutation, f_coupling, leak, device,
             gemm_impl=_cabi.GEMM_TCGEN05, bwd_passes=None, train=False, meas_rows=0) -> Plan:
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if bwd_passes is None:
        bwd_passes = default_bwd_passes()
    key = (str(device), arch, batch, nz, ngf, nc, f_depth, f_width, f_permutation, f_coupling, float(leak), gemm_impl,
           bwd_passes, bool(train), int(meas_rows))
    p = _PLANS.get(key)
    if p is None:
        if len(_PLANS) > 16:
            _PLANS.pop(next(iter(_PLANS)))
        p = Plan(arch=arch, batch=batch, nz=nz, ngf=ngf, nc=nc, f_depth=f_depth, f_width=f_width,
                 f_permutation=f_permutation, f_coupling=f_coupling, leak=leak, device=device, gemm_impl=gemm_impl,
                 bwd_passes=bwd_passes, train=train, meas_rows=meas_rows)
        _PLANS[key] = p
    return p


def clear_plans():
    _PLANS.clear()


def invalidate_plans():
    """Re-pack the parameters of every cached plan at its next use (see ``Plan.invalidate``)."""
    for p in _PLANS.values():
        p.invalidate()
