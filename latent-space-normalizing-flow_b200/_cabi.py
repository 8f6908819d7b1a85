"""ctypes binding of include/lsnf.h.  The library is built in-tree by ``__graft_entry__.build()``; there is no
fallback: if it is missing, or a call fails, a RuntimeError is raised."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LSNF_LIB: load another build of the same ABI (A/B timing of two library versions on one box)
LIB_PATH = os.environ.get("LSNF_LIB") or os.path.join(_HERE, "_lib", "liblsnf_b200.so")
_lib = None

LSNF_MAX_TAPS = 16
LSNF_MAX_PHASES = 4
FLOW_PTRS_PER_STEP = 12

ARCH = {"none": -1, "svhn": 0, "cifar10": 1, "celeba_crop": 2, "celeba_hq256": 3}
GEMM_TCGEN05, GEMM_SIMT = 0, 1


class Config(C.Structure):
    _fields_ = [("arch", C.c_int32), ("batch", C.c_int32), ("nz", C.c_int32), ("ngf", C.c_int32), ("nc", C.c_int32),
                ("f_depth", C.c_int32), ("f_width", C.c_int32), ("f_permutation", C.c_int32),
                ("f_coupling", C.c_int32), ("leak", C.c_float), ("gemm_impl", C.c_int32),
                ("bwd_passes", C.c_int32), ("train", C.c_int32), ("reserved", C.c_int32 * 3)]


class Tap(C.Structure):
    _fields_ = [("dy", C.c_int32), ("dx", C.c_int32), ("plane", C.c_int32), ("brow", C.c_int32)]


class StageInfo(C.Structure):
    _fields_ = [("kind", C.c_int32), ("layer", C.c_int32), ("grid_h", C.c_int32), ("grid_w", C.c_int32),
                ("box_b", C.c_int32), ("box_h", C.c_int32), ("box_w", C.c_int32), ("k_per_tap", C.c_int32),
                ("n_valid", C.c_int32), ("n_pad", C.c_int32), ("block_n", C.c_int32), ("n_phases", C.c_int32),
                ("n_taps", C.c_int32 * LSNF_MAX_PHASES), ("taps", (Tap * LSNF_MAX_TAPS) * LSNF_MAX_PHASES),
                ("out_mul", C.c_int32), ("out_off_y", C.c_int32 * LSNF_MAX_PHASES),
                ("out_off_x", C.c_int32 * LSNF_MAX_PHASES), ("out_phase_split", C.c_int32),
                ("out_channels", C.c_int32), ("epilogue", C.c_int32), ("k_splits", C.c_int32),
                ("a_planes", C.c_int32), ("a_h", C.c_int32), ("a_w", C.c_int32), ("tap_gen_k", C.c_int32),
                ("b_k", C.c_int32), ("b_rows", C.c_int32), ("operand_fp16", C.c_int32), ("passes", C.c_int32),
                ("a_offset", C.c_int64), ("b_offset", C.c_int64), ("out_offset", C.c_int64), ("flops", C.c_int64)]


class LaunchInfo(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("grid_x", C.c_int32), ("grid_y", C.c_int32), ("grid_z", C.c_int32),
                ("block", C.c_int32), ("ring_stages", C.c_int32), ("stage_bytes", C.c_int32),
                ("smem_bytes", C.c_int32), ("ctas_per_sm", C.c_int32), ("tmem_columns", C.c_int32),
                ("tma_store", C.c_int32), ("stream_k", C.c_int32), ("cross_fp8", C.c_int32),
                ("reserved", C.c_int32 * 3)]


KERNEL_SINGLE, KERNEL_PAIR = 0, 1

EXPORTS = {
    # name: (restype, argtypes)
    "lsnf_abi_version": (C.c_int, []),
    "lsnf_last_error": (C.c_char_p, []),
    "lsnf_plan_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "lsnf_plan_destroy": (None, [C.c_void_p]),
    "lsnf_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "lsnf_plan_bind": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "lsnf_pack_generator_weights": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int32,
                                              C.c_void_p]),
    "lsnf_pack_flow_weights": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                         C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]),
    "lsnf_generator_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_generator_dgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "lsnf_flow_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "lsnf_flow_inverse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_langevin_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                       C.c_int32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]),
    "lsnf_langevin_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_int32,
                                    C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_sample_prior": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "lsnf_generator_grad_floats": (C.c_size_t, [C.c_void_p]),
    "lsnf_generator_grad_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lsnf_generator_param_grads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_int32, C.c_void_p]),
    "lsnf_flow_grad_floats": (C.c_size_t, [C.c_void_p]),
    "lsnf_flow_grad_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lsnf_flow_param_grads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_langevin_run_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                           C.c_float, C.c_int32, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "lsnf_generator_dgrad_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "lsnf_generator_param_grads_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                    C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "lsnf_generator_vjp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_flow_vjp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_ais_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                               C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "lsnf_adam_step": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                 C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int32), C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                 C.c_int64, C.c_void_p, C.c_void_p]),
    "lsnf_plan_run_stage": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "lsnf_langevin_launch_count": (C.c_int, [C.c_void_p, C.c_int32]),
    "lsnf_plan_num_stages": (C.c_int, [C.c_void_p]),
    "lsnf_plan_stage_info": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(StageInfo)]),
    "lsnf_plan_pack_index": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lsnf_plan_stage_launch_info": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(LaunchInfo)]),
}


def load():
    """Load the shared library (once) and declare every prototype of include/lsnf.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"lsnf_b200: native library {LIB_PATH} is missing -- build it with "
            "`python __graft_entry__.py` (nvcc, sm_100a). There is no CPU or PyTorch fallback for the Langevin path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.lsnf_abi_version() != 1:
        raise RuntimeError("lsnf_b200: ABI version mismatch between _cabi.py and the built library")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().lsnf_last_error()
        raise RuntimeError(f"lsnf_b200: {what} failed ({rc}): {msg.decode() if msg else ''}")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(p) for p in ptrs])
    return arr
