"""ctypes binding of include/cfnerf_b200.h.  There is no fallback: a missing library is an ImportError."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

_i64, _i32, _f32p, _vp, _sz = C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t


class CfnConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("D", "W", "L_pos", "L_dir", "h_alpha", "h_rgb", "F", "K", "precision")]


# every symbol include/cfnerf_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "cfn_last_error": (C.c_char_p, []),
    "cfn_version": (_i32, []),
    "cfn_create": (_i32, [C.POINTER(CfnConfigC), C.POINTER(_vp)]),
    "cfn_destroy": (_i32, [_vp]),
    "cfn_set_deterministic": (_i32, [_vp, _i32]),
    "cfn_param_count": (_i32, [_vp]),
    "cfn_param_name": (C.c_char_p, [_vp, _i32]),
    "cfn_param_numel": (_i64, [_vp, _i32]),
    "cfn_pack_weights": (_i32, [_vp, C.POINTER(_vp), _i32, _vp]),
    "cfn_flow_param_width": (_i32, [_vp]),
    "cfn_zvals_f32": (_i32, [_f32p, _f32p, _f32p, _i32, _f32p, _i64, _i32, _vp]),
    "cfn_rays_from_pose_f32": (_i32, [_i32, _i32, C.c_double, C.POINTER(C.c_float), C.c_double, C.c_double, _i32, C.c_double,
                               _f32p, _vp]),
    "cfn_workspace_bytes": (_i32, [_vp, _i64, _i32, C.POINTER(_sz)]),
    "cfn_network_fwd": (_i32, [_vp, _f32p, _f32p, _f32p, _f32p, _i64, _i32, _f32p, _vp, _sz, _i32, _vp]),
    "cfn_network_bwd": (_i32, [_vp, _f32p, _i64, _i32, _vp, _sz, C.POINTER(_vp), _i32, _vp]),
    "cfn_flow_composite_fwd": (_i32, [_vp, _f32p, _f32p, _f32p, _i32, _f32p, _f32p, _i64, _i64, _i32, _i32, _f32p, _f32p,
                                      _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _i32, _vp]),
    "cfn_flow_composite_bwd": (_i32, [_vp, _f32p, _f32p, _f32p, _i32, _f32p, _f32p, _i64, _i64, _i32, _i32, _f32p, _f32p,
                                      C.c_float, C.c_float, _f32p, _i32, _f32p, _i32, _f32p, _f32p, _vp]),
    "cfn_flow_composite_bwd_dev": (_i32, [_vp, _f32p, _f32p, _f32p, _i32, _f32p, _f32p, _i64, _i64, _i32, _i32, _f32p,
                                          _f32p, _f32p, _f32p, _i32, _f32p, _i32, _f32p, _f32p, _vp]),
    "cfn_raw2outputs_f32": (_i32, [_f32p, _f32p, _f32p, _i32, _i32, _f32p, _f32p, _f32p, _f32p, _i64, _i32, _i32, _vp]),
    "cfn_sample_pdf_f32": (_i32, [_f32p, _f32p, _f32p, _f32p, _vp, _i64, _i32, _i32, _vp]),
    "cfn_merge_sorted_f32": (_i32, [_f32p, _f32p, _f32p, _i64, _i32, _i32, _vp]),
    "cfn_mean_over_k_f32": (_i32, [_f32p, _f32p, _i64, _i32, _vp]),
    "cfn_kde_nll_f32": (_i32, [_f32p, _f32p, _i64, _i32, C.c_float, _f32p, _f32p, _vp]),
    "cfn_trainer_loss_f32": (_i32, [_f32p, _f32p, _f32p, _f32p, _i64, _i64, _i32, C.c_float, C.c_float, _f32p, _f32p, _f32p,
                                    _vp]),
    "cfn_adam_step_f32": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64),
                          C.c_float, C.c_float, C.c_float, C.c_float, _i32, C.c_float, _vp]),
    "cfn_adam_step_dev_f32": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64),
                              _f32p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _vp]),
    "cfn_globals_grad_f32": (_i32, [_vp, _f32p, _i64, C.c_float, _f32p, _vp]),
    "cfn_debug_profile": (_i32, [_vp, _vp, _i32]),
    "cfn_gemm_bf16": (_i32, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i64,
                      _i32, _i32, _vp, _vp]),
    "cfn_gemm_f32": (_i32, [_i32, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _i32, _i64,
                     _i32, _i32, _i32, _i32, _vp]),
}

PREC = {"fp32": 0, "bf16": 1, "fp16": 2, "tf32": 3}

_lib = None


def load():
    """Load libcfnerf_b200.so (built in-tree by `python -m cfnerf_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library must be built first (python -m cfnerf_b200.build). "
            "cfnerf_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class CfnError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().cfn_last_error()
        raise CfnError(f"{what or 'cfnerf_b200'} failed (code {rc}): {msg.decode() if msg else '?'}")
