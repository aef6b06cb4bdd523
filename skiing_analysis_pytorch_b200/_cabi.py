"""ctypes mirror of include/ska.h (structs, constants) - no compute here."""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 9
MAX_VIEWS = 8
MAX_BA_VIEWS = 8
MAX_BONES = 16

LAYOUT_VIEW_MAJOR = 0
LAYOUT_FRAME_MAJOR = 1

SOLVER_SECULAR = 0
SOLVER_JACOBI64 = 1
SOLVER_JACOBI32 = 2
WEIGHT_SQRT = 4
PINHOLE_REPROJ = 8

SOLVERS = {"secular": SOLVER_SECULAR, "jacobi64": SOLVER_JACOBI64, "jacobi32": SOLVER_JACOBI32}

BA_CAM_DOUBLES = 24
BA_CTRL_DOUBLES = 16
BA_HIST_DOUBLES = 8
BA_RED2_DOUBLES = 4
BA_CTRL_LAMBDA, BA_CTRL_NU, BA_CTRL_SUMCONF, BA_CTRL_CUR, BA_CTRL_ITER = 0, 1, 2, 3, 4
BA_CTRL_PREDCAM, BA_CTRL_OK = 5, 6  # written by the solve: camera part of the predicted decrease; 1 if the reduced system was positive definite
BA_CTRL_COST, BA_CTRL_ACCEPTED = 7, 8
BA_CTRL_PRIOR_CUR, BA_CTRL_PRIOR_TRIAL = 9, 10  # calibrating BA, written by the solve: intrinsics-prior cost at the current / trial cameras
BA_FORCE_WIDE = 1
BA_TENSOR_CORE = 2
BA_LOSS_L2, BA_LOSS_HUBER, BA_LOSS_CAUCHY = 0, 1, 2
BA_LOSSES = {"l2": BA_LOSS_L2, "huber": BA_LOSS_HUBER, "cauchy": BA_LOSS_CAUCHY}


def check_loss(loss, loss_scale):
    """A solver's `loss` / `loss_scale` arguments as the C ABI takes them: (SKA_BA_LOSS_* value, scale in pixels, 0.0 for
    "l2"), or ValueError."""
    if loss not in BA_LOSSES:
        raise ValueError(f"unknown loss {loss!r}; expected one of {tuple(BA_LOSSES)}")
    if loss == "l2":
        return BA_LOSS_L2, 0.0
    if loss_scale is None or not np.isfinite(float(loss_scale)) or float(loss_scale) <= 0.0:
        raise ValueError(f"loss={loss!r} needs a finite loss_scale > 0 (pixels), got {loss_scale!r}")
    return BA_LOSSES[loss], float(loss_scale)

ERRORS = {-1: "SKA_EINVAL", -2: "SKA_EUNSUPPORTED", -3: "SKA_EALIGN", -4: "SKA_EWORKSPACE"}
SKA_EWORKSPACE = -4


class SkaCamera(C.Structure):
    _fields_ = [
        ("K", C.c_double * 9),
        ("R", C.c_double * 9),
        ("t", C.c_double * 3),
        ("dist", C.c_double * 14),
    ]


class SkaBaProblem(C.Structure):
    _fields_ = [
        ("C", C.c_int32),
        ("J", C.c_int32),
        ("T", C.c_int64),
        ("layout", C.c_int32),
        ("flags", C.c_uint32),
        ("d_x2d", C.c_void_p),
        ("d_conf", C.c_void_p),
        ("d_Xpp", C.c_void_p),
        ("d_cams", C.c_void_p),
        ("d_ctrl", C.c_void_p),
        ("d_red", C.c_void_p),
        ("d_red2", C.c_void_p),
        ("d_delta", C.c_void_p),
        ("d_hist", C.c_void_p),
        ("d_workspace", C.c_void_p),
        ("ws_bytes", C.c_size_t),
        ("hist_rows", C.c_int64),
        ("peer", C.c_void_p),
        ("loss", C.c_int32),
        ("loss_scale", C.c_double),
    ]


BA_REG_NVEC, BA_REG_SUMS, BA_REG_SC_DOUBLES, BA_REG_HIST_DOUBLES = 7, 40, 64, 16
BA_REG_SC_CUR, BA_REG_SC_LAMBDA, BA_REG_SC_NU, BA_REG_SC_ITER, BA_REG_SC_COST, BA_REG_SC_ACCEPTED = 0, 1, 2, 3, 4, 7
BA_REG_SC_TOL2, BA_REG_SC_COEF, BA_REG_SC_T_GLOBAL, BA_REG_SC_DOT = 15, 16, 21, 47
BA_REG_CG_BEGIN, BA_REG_CG_INIT, BA_REG_CG_MATVEC, BA_REG_CG_ALPHA, BA_REG_CG_UPDATE, BA_REG_CG_BETA, BA_REG_CG_DIR = range(7)
BA_REG_FREE = {"pose_only": 0, "pose_cam_t": 0x38, "full": 0x3F}


class SkaBaRegProblem(C.Structure):
    _fields_ = [
        ("C", C.c_int32), ("J", C.c_int32), ("n_bones", C.c_int32), ("free_mask", C.c_uint32),
        ("T_local", C.c_int64), ("has_prev", C.c_int32), ("has_next", C.c_int32),
        ("bone_i", C.c_int32 * 16), ("bone_j", C.c_int32 * 16),
        ("d_x2d", C.c_void_p), ("d_conf", C.c_void_p), ("d_K", C.c_void_p), ("d_X", C.c_void_p), ("d_cams", C.c_void_p),
        ("d_vec", C.c_void_p), ("d_pinv", C.c_void_p), ("d_lfac", C.c_void_p), ("d_sc", C.c_void_p), ("d_sums", C.c_void_p),
        ("d_hist", C.c_void_p), ("hist_rows", C.c_int64), ("d_workspace", C.c_void_p), ("ws_bytes", C.c_size_t), ("peer", C.c_void_p),
    ]


MAX_PEERS = 8


class SkaPeerComm(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("slot_doubles", C.c_int32), ("poll_limit_log2", C.c_int32),
                ("recv", C.c_void_p * 8), ("flags", C.c_void_p * 8), ("d_state", C.c_void_p), ("d_skip", C.c_void_p)]


class SkaFuseParams(C.Structure):
    _fields_ = [
        ("sigma_px", C.c_double),
        ("sigma_3d", C.c_double),
        ("scale_mode", C.c_int32),
        ("min_points", C.c_int32),
        ("root", C.c_int32),
        ("lhip", C.c_int32),
        ("rhip", C.c_int32),
        ("lsho", C.c_int32),
        ("rsho", C.c_int32),
        ("pad_", C.c_int32),
    ]


FUSE_NO_ALIGN, FUSE_FIT_LEFT_FAILED, FUSE_FIT_RIGHT_FAILED = 1, 2, 4
FUSE_MAX_JOINTS = 96


def red_layout(n_cams: int) -> dict:
    """Offsets inside the packed reduced system d_red (include/ska.h)."""
    nc = n_cams - 1
    n = 6 * nc
    ns = n * (n + 1) // 2
    return dict(n=n, sw=0, bw=ns, gc=ns + n, hcc=ns + 2 * n, cost=ns + 2 * n + 21 * nc, clamp=ns + 2 * n + 21 * nc + 1,
                size=ns + 2 * n + 21 * nc + 2)


BA_CALIB_PARAMS = 15
BA_CALIB_INTRINSICS = 9
BA_CALIB_CAM_BLOCK = 160


def calib_red_layout(n_cams: int) -> dict:
    """Offsets inside the calibrating BA's packed reduced system (include/ska.h): Sw triangle over the n = 15 C - 6
    free-able parameters, then one 160-double block per camera (upper triangle of the 17 x 17 row products)."""
    n = BA_CALIB_PARAMS * n_cams - 6
    ns = n * (n + 1) // 2
    return dict(n=n, sw=0, cam=ns, size=ns + BA_CALIB_CAM_BLOCK * n_cams)


def calib_tri(r: int, s: int) -> int:
    """Index of entry (r, s), r <= s, in the row-major upper triangle of the 17 x 17 per-camera block."""
    return r * 17 - (r * (r - 1)) // 2 + (s - r)


def calib_col(c: int, r: int) -> int:
    """Column of parameter r of camera c in the reduced system (camera 0: r >= 6 only)."""
    return r - 6 if c == 0 else BA_CALIB_INTRINSICS + BA_CALIB_PARAMS * (c - 1) + r


def make_cameras(K, R, t, dist=None):
    """Pack V cameras into a ctypes SkaCamera array.

    K (3,3)|(V,3,3); R (V,3,3); t (V,3); dist None | (n,) shared | list of per-view (n,)|None.
    """
    R = np.asarray(R, np.float64)
    V = R.shape[0]
    t = np.asarray(t, np.float64).reshape(V, 3)
    K = np.asarray(K, np.float64)
    K = np.broadcast_to(K, (V, 3, 3)) if K.ndim == 2 else K.reshape(V, 3, 3)
    if dist is None:
        dists = [None] * V
    elif isinstance(dist, (list, tuple)) and len(dist) == V and any(d is None or np.ndim(d) >= 1 for d in dist):
        dists = list(dist)  # one entry (vector or None) per view
    else:
        try:
            arr = np.asarray(dist, np.float64)
        except (TypeError, ValueError):  # ragged / contains None: one entry per view
            arr = None
        if arr is not None and arr.ndim <= 1:
            dists = [arr.reshape(-1)] * V
        elif arr is not None and arr.ndim == 2 and arr.shape[0] != V and 1 in arr.shape:
            dists = [arr.reshape(-1)] * V  # (1,n) / (n,1) as OpenCV returns it
        else:
            dists = list(dist)
            if len(dists) != V:
                raise ValueError(f"need {V} distortion vectors, got {len(dists)}")
    cams = (SkaCamera * V)()
    for v in range(V):
        cams[v].K[:] = K[v].reshape(-1).tolist()
        cams[v].R[:] = R[v].reshape(-1).tolist()
        cams[v].t[:] = t[v].tolist()
        d = np.zeros(14)
        if dists[v] is not None:
            dv = np.asarray(dists[v], np.float64).reshape(-1)
            if dv.size not in (4, 5, 8, 12, 14):
                raise ValueError(f"distortion vector must have 4, 5, 8, 12 or 14 entries, got {dv.size}")
            d[: dv.size] = dv
        cams[v].dist[:] = d.tolist()
    return cams
