"""ctypes loader for lib/libska.so.  There is NO fallback: if the CUDA library is missing or a
call fails, the caller gets an exception (SkaError / RuntimeError), never a CPU path."""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

from . import _cabi

_LOCK = threading.Lock()
_LIB = None

# SKA_LIB_PATH selects an experimental build of the SAME CUDA library (tools/variants.py); never a CPU path
LIB_PATH = Path(os.environ.get("SKA_LIB_PATH") or (Path(__file__).resolve().parent / "lib" / "libska.so"))


class SkaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        self.code = code
        name = _cabi.ERRORS.get(code, f"cudaError {code}" if code > 0 else f"error {code}")
        super().__init__(f"libska: {name}: {msg}")


_vp = C.c_void_p
_SIGS = {
    "ska_abi_version": (C.c_int, []),
    "ska_last_error": (C.c_char_p, []),
    "ska_build_arch": (C.c_char_p, []),
    "ska_triangulate_reproject_f32": (
        C.c_int,
        [C.POINTER(_cabi.SkaCamera), C.c_int32, _vp, _vp, _vp, C.c_int64, C.c_int32, C.c_int32, C.c_uint32,
         _vp, _vp, _vp, _vp, _vp],
    ),
    "ska_tri_frames_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int64]),
    "ska_triangulate_reproject_frames_f32": (
        C.c_int,
        [C.POINTER(_cabi.SkaCamera), C.c_int32, _vp, _vp, _vp, C.c_int64, C.c_int32, C.c_int32, C.c_uint32,
         _vp, _vp, _vp, _vp, _vp, C.c_size_t, _vp],
    ),
    "ska_reproject_points_f32": (
        C.c_int, [C.POINTER(_cabi.SkaCamera), C.c_int32, _vp, _vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp]
    ),
    "ska_frame_stats_f32": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _vp, _vp]),
    "ska_post_triage_f32": (
        C.c_int,
        [C.POINTER(_cabi.SkaCamera), _vp, _vp, _vp, C.c_int64, C.c_int32, C.c_uint32, C.c_double, C.c_double, _vp, _vp, _vp, _vp],
    ),
    "ska_frame_flag_counts_u8": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, _vp]),
    "ska_savgol_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "ska_savgol_f32": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, C.c_size_t, _vp]),
    "ska_loss_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "ska_reg_workspace_bytes": (C.c_size_t, []),
    "ska_ba_red_doubles": (C.c_int32, [C.c_int32]),
    "ska_ba_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "ska_ba_sum_f32": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.c_size_t, _vp]),
    "ska_ba_linearize_f32": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_solve_f64": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), C.c_uint64, _vp]),
    "ska_ba_backsub_f32": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_control_f64": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_calib_red_doubles": (C.c_int32, [C.c_int32]),
    "ska_ba_calib_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "ska_ba_calib_linearize_f32": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_calib_solve_f64": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), C.c_uint64, _vp, _vp]),
    "ska_ba_calib_backsub_f32": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_calib_control_f64": (C.c_int, [C.POINTER(_cabi.SkaBaProblem), _vp]),
    "ska_ba_reg_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "ska_ba_reg_cost_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, _vp]),
    "ska_ba_reg_finish_cost_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, _vp]),
    "ska_ba_reg_linearize_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), _vp]),
    "ska_ba_reg_cg_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, _vp]),
    "ska_ba_reg_apply_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), _vp]),
    "ska_ba_reg_control_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), _vp]),
    "ska_ba_reg_cost_robust_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, C.c_int32, C.c_double, _vp]),
    "ska_ba_reg_linearize_robust_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, C.c_double, _vp]),
    "ska_ba_reg_cg_robust_f64": (C.c_int, [C.POINTER(_cabi.SkaBaRegProblem), C.c_int32, C.c_int32, C.c_double, _vp]),
    "ska_peer_region_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "ska_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "ska_peer_free": (C.c_int, [_vp]),
    "ska_peer_export": (C.c_int, [_vp, C.c_char_p]),
    "ska_peer_import": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "ska_peer_close": (C.c_int, [_vp]),
    "ska_peer_allreduce_f64": (C.c_int, [C.POINTER(_cabi.SkaPeerComm), _vp, C.c_int32, _vp]),
    "ska_peer_allgather_f64": (C.c_int, [C.POINTER(_cabi.SkaPeerComm), _vp, C.c_int32, _vp, _vp]),
    "ska_fuse_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "ska_fuse_frames_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_int32, C.POINTER(_cabi.SkaFuseParams), _vp, _vp, _vp, _vp, _vp, _vp,
                                       C.c_size_t, _vp]),
    "ska_rigid_fuse_f64": (C.c_int, [_vp, _vp, C.c_int64, C.c_int32, C.POINTER(C.c_int32), C.c_double, _vp, C.c_int32, _vp, _vp, C.c_int64, _vp, _vp,
                                     _vp, _vp, _vp]),
    "ska_ema_f64": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int64,
                              C.c_int32, _vp, _vp]),
}
_SIGS["ska_first_order_record_f64"] = (C.c_int, [_vp, _vp, _vp, C.c_int64, C.POINTER(C.c_void_p), _vp, C.POINTER(C.c_double), C.c_double,
                                                 C.c_double, C.c_double, _vp])
for _sfx in ("f32", "f64"):
    _i64, _i32 = C.c_int64, C.c_int32
    _SIGS[f"ska_project_points_{_sfx}"] = (C.c_int, [_vp, _i64, _i32, _i32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp])
    _SIGS[f"ska_reprojection_loss_{_sfx}"] = (
        C.c_int, [_vp, _i64, _i32, _i32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _vp]
    )
    _SIGS[f"ska_pose_temporal_{_sfx}"] = (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, C.c_size_t, _vp])
    _SIGS[f"ska_bone_length_{_sfx}"] = (
        C.c_int, [_vp, _i64, _i32, C.POINTER(_i32), C.POINTER(_i32), _i32, _vp, _vp, _vp, _vp, C.c_size_t, _vp]
    )
    _SIGS[f"ska_camera_centre_{_sfx}"] = (C.c_int, [_vp, _vp, _i64, _vp, _vp])
    _SIGS[f"ska_camera_smooth_{_sfx}"] = (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, C.c_size_t, _vp])
    _SIGS[f"ska_adam_step_{_sfx}"] = (C.c_int, [_vp, _vp, _vp, _vp, _i64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp])
    _SIGS[f"ska_adam_step_terms_{_sfx}"] = (C.c_int, [_vp, _vp, C.c_double, _vp, C.c_double, _vp, C.c_double, _vp, _vp, _i64, C.c_double, C.c_double,
                                                      C.c_double, _vp, _vp, _vp])
    _SIGS[f"ska_so3_tangent_grad_{_sfx}"] = (C.c_int, [_vp, _vp, _i64, _vp, _vp])
    _SIGS[f"ska_so3_retract_{_sfx}"] = (C.c_int, [_vp, _vp, _i64, _vp])
    _SIGS[f"ska_baseline_reg_{_sfx}"] = (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _vp])


def exported_symbols():
    """Every symbol include/ska.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGS)


def load():
    """Load libska.so once; build it first if it is missing or older than its sources (build.needs_build; needs nvcc -
    where nvcc is absent a stale prebuilt library is loaded with a warning).  Raises if it cannot be had - the product has
    no CPU path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        from . import build as _build

        default_lib = "SKA_LIB_PATH" not in os.environ
        stale = False
        if default_lib and LIB_PATH.exists():
            try:
                stale = _build.needs_build()  # a .cu / .cuh / ska.h newer than the library: never run old kernels silently
            except OSError:
                stale = False
        if not LIB_PATH.exists() or os.environ.get("SKA_REBUILD") == "1" or stale:
            try:
                _build.build(force=os.environ.get("SKA_REBUILD") == "1")
            except RuntimeError:
                if not (stale and LIB_PATH.exists()):
                    raise
                import warnings  # no nvcc on this machine (a deployment box): the prebuilt library is what there is

                warnings.warn(f"{LIB_PATH} is older than its sources and nvcc is not available to rebuild it")
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing and could not be built; there is no CPU fallback")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)  # AttributeError here = header / library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        if lib.ska_abi_version() != _cabi.ABI_VERSION:
            raise RuntimeError(f"libska ABI {lib.ska_abi_version()} != expected {_cabi.ABI_VERSION}")
        _LIB = lib
    return _LIB


def check(code: int):
    if code != 0:
        msg = load().ska_last_error()
        raise SkaError(code, msg.decode() if msg else "")
