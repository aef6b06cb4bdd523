"""bundle_adjustment/loss.py on the GPU: same names, argument meaning, return conventions and error
behaviour as the reference module, with the arithmetic in libska.so (ska_project.cu / ska_losses.cu).

Every function takes CUDA tensors (float32 or float64; inputs are cast to ``X3d``'s dtype and device
like loss.py:27-32 does) and returns what the reference returns: ``project_points`` a (T,C,J,2)
tensor, the losses 0-dim tensors on the inputs' device.  All of them are differentiable: the
kernels return the value and the analytic gradient in one pass (what torch.autograd would derive
from the reference's broadcasting expressions), wrapped in ``torch.autograd.Function``.  There is
no CPU path: CPU tensors raise.

Reference: bundle_adjustment/loss.py:17-155 (file:line relative to the reference checkout).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _cabi, _lib

# bundle_adjustment/loss.py:118-131 - COCO-17 limb topology (applied blindly to any J, loss.py:137-139)
BONES = [(11, 13), (13, 15), (12, 14), (14, 16), (5, 7), (7, 9), (6, 8), (8, 10), (5, 6), (11, 12), (5, 11), (6, 12)]


def _sfx(dtype) -> str:
    if dtype == torch.float32:
        return "f32"
    if dtype == torch.float64:
        return "f64"
    raise TypeError(f"only float32 / float64 tensors are supported, got {dtype}")


def _cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: this package has no CPU path (got device {t.device})")


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


_WS: dict = {}


def _workspace(dev, nbytes: int) -> torch.Tensor:
    """Per-device scratch for the fixed-order reductions (stream-ordered reuse on the current stream)."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=dev)
        _WS[key] = ws
    return ws


def _normalise_cameras(X3d, R, t, K):
    """Shape handling of loss.py:34-52,74-79 -> contiguous tensors + frame strides (0 = shared)."""
    dev, dt = X3d.device, X3d.dtype
    K = K.to(device=dev, dtype=dt)
    R = R.to(device=dev, dtype=dt)
    t = t.to(device=dev, dtype=dt)
    if X3d.dim() == 2:
        X3d = X3d.unsqueeze(0)
    T, J, _ = X3d.shape
    if R.dim() == 3:
        Cn = R.shape[0]
        R_s = 0
        t_s = 0
        if t.dim() != 2:
            raise RuntimeError(f"t {tuple(t.shape)} cannot be broadcast with R {tuple(R.shape)}")
    elif R.dim() == 4:
        T_R, Cn = R.shape[:2]
        assert T_R == T
        R_s = 9 * Cn
        if t.dim() == 2:
            t_s = 0
        else:
            assert t.shape[:2] == (T, Cn)
            t_s = 3 * Cn
    else:
        raise ValueError(f"Unsupported R shape: {R.shape}")
    if K.dim() == 3:
        K_s = 0
    elif K.dim() == 4:
        K_s = 9 * Cn
        if K.shape[0] != T:
            raise RuntimeError(f"K {tuple(K.shape)} does not match T={T}")
    else:
        raise ValueError(f"Unsupported K shape: {K.shape}")
    if K.shape[-3] != Cn or t.shape[-2] != Cn:
        raise RuntimeError(f"camera count mismatch: R {tuple(R.shape)}, t {tuple(t.shape)}, K {tuple(K.shape)}")
    return X3d.contiguous(), R.contiguous(), t.contiguous(), K.contiguous(), T, J, Cn, R_s, t_s, K_s


class _ReprojectionSums(torch.autograd.Function):
    """sums = [sum conf |proj - x2d|^2, sum conf, #clamped, 0] (fp64) with the analytic gradient of
    sums[0] w.r.t. X3d, R, t, K computed in the same pass."""

    @staticmethod
    def forward(ctx, X3d, R, t, K, x2d, conf2d, dims):
        T, J, Cn, R_s, t_s, K_s = dims
        dev, dt = X3d.device, X3d.dtype
        lib = _lib.load()
        need = [ctx.needs_input_grad[i] for i in range(4)]
        gX = torch.empty_like(X3d) if need[0] else None
        gR = torch.empty_like(R) if need[1] else None
        gt = torch.empty_like(t) if need[2] else None
        gK = torch.empty_like(K) if need[3] else None
        sums = torch.zeros(4, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            nbytes = int(lib.ska_loss_workspace_bytes(Cn))
            ws = _workspace(dev, nbytes)
            fn = getattr(lib, f"ska_reprojection_loss_{_sfx(dt)}")
            _lib.check(fn(_p(X3d), T, J, Cn, _p(R), R_s, _p(t), t_s, _p(K), K_s, _p(x2d), _p(conf2d), _p(sums), _p(gX), _p(gR),
                          _p(gt), _p(gK), _p(ws), ws.numel(), _stream(dev)))
        ctx.grads = (gX, gR, gt, gK)
        return sums

    @staticmethod
    def backward(ctx, g):
        s = 2.0 * g[0]
        out = [None if gi is None else gi * s.to(gi.dtype) for gi in ctx.grads]
        return (*out, None, None, None)


def project_points(X3d: torch.Tensor, R: torch.Tensor, t: torch.Tensor, K: torch.Tensor) -> torch.Tensor:
    """loss.py:17-84.  X3d (T,J,3)|(J,3); R (T,C,3,3)|(C,3,3); t (T,C,3)|(C,3); K (C,3,3)|(T,C,3,3)
    -> (T,C,J,2) in X3d's dtype.  Z is clamped at 1e-6 (:67) and the full K is applied (:74-82).
    Differentiable w.r.t. X3d, R, t, K (via the reprojection adjoint kernel)."""
    _cuda(X3d, "X3d")
    return _ProjectPoints.apply(X3d, R, t, K)


class _ProjectPoints(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X3d, R, t, K):
        Xc, Rc, tc, Kc, T, J, Cn, R_s, t_s, K_s = _normalise_cameras(X3d, R, t, K)
        dev, dt = Xc.device, Xc.dtype
        out = torch.empty((T, Cn, J, 2), dtype=dt, device=dev)
        if T > 0:
            with torch.cuda.device(dev):
                fn = getattr(_lib.load(), f"ska_project_points_{_sfx(dt)}")
                _lib.check(fn(_p(Xc), T, J, Cn, _p(Rc), R_s, _p(tc), t_s, _p(Kc), K_s, _p(out), _stream(dev)))
        ctx.save_for_backward(Xc, Rc, tc, Kc)
        ctx.dims = (T, J, Cn, R_s, t_s, K_s)
        ctx.in_shapes = (X3d.shape, R.shape, t.shape, K.shape)
        ctx.in_dtypes = (X3d.dtype, R.dtype, t.dtype, K.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        # vector-Jacobian product: the loss adjoint kernel in cotangent mode (d_conf = NULL)
        Xc, Rc, tc, Kc = ctx.saved_tensors
        T, J, Cn, R_s, t_s, K_s = ctx.dims
        dev, dt = Xc.device, Xc.dtype
        need = ctx.needs_input_grad
        gX = torch.empty_like(Xc) if need[0] else None
        gR = torch.empty_like(Rc) if need[1] else None
        gt = torch.empty_like(tc) if need[2] else None
        gK = torch.empty_like(Kc) if need[3] else None
        sums = torch.zeros(4, dtype=torch.float64, device=dev)
        gc = g.to(dt).contiguous()
        lib = _lib.load()
        with torch.cuda.device(dev):
            ws = _workspace(dev, int(lib.ska_loss_workspace_bytes(Cn)))
            fn = getattr(lib, f"ska_reprojection_loss_{_sfx(dt)}")
            _lib.check(fn(_p(Xc), T, J, Cn, _p(Rc), R_s, _p(tc), t_s, _p(Kc), K_s, _p(gc), None, _p(sums), _p(gX), _p(gR),
                          _p(gt), _p(gK), _p(ws), ws.numel(), _stream(dev)))
        outs = []
        for gi, shp, dty in zip((gX, gR, gt, gK), ctx.in_shapes, ctx.in_dtypes):
            outs.append(None if gi is None else gi.reshape(shp).to(dty))
        return tuple(outs)


def reprojection_loss(X3d, R, t, K, x2d, conf2d, w=1.0) -> torch.Tensor:
    """loss.py:90-94: ``w * sum(conf * |proj - x2d|^2) / (sum(conf) + 1e-6)`` as a 0-dim tensor.
    One fused kernel pass computes the value and the gradient w.r.t. X3d, R, t, K; x2d / conf2d are
    data (a gradient request on them raises)."""
    _cuda(X3d, "X3d")
    if (torch.is_tensor(x2d) and x2d.requires_grad) or (torch.is_tensor(conf2d) and conf2d.requires_grad):
        raise NotImplementedError("reprojection_loss is differentiable w.r.t. X3d, R, t, K only (x2d / conf2d are observations)")
    Xc, Rc, tc, Kc, T, J, Cn, R_s, t_s, K_s = _normalise_cameras(X3d, R, t, K)
    dt, dev = Xc.dtype, Xc.device
    x2 = x2d.to(device=dev, dtype=dt).expand(T, Cn, J, 2).contiguous()
    cf = conf2d.to(device=dev, dtype=dt).expand(T, Cn, J).contiguous()
    sums = _ReprojectionSums.apply(Xc, Rc, tc, Kc, x2, cf, (T, J, Cn, R_s, t_s, K_s))
    return (w * sums[0] / (sums[1] + 1e-6)).to(dt)


# ---------------------------------------------------------------------------------------------
def camera_center_from_Rt(R, t):
    """loss.py:97-100: C = -R^T t, any leading dims -> (...,3)."""
    _cuda(R, "R")
    return _CameraCentre.apply(R, t)


class _CameraCentre(torch.autograd.Function):
    @staticmethod
    def forward(ctx, R, t):
        dt = torch.promote_types(R.dtype, t.dtype)
        lead = R.shape[:-2]
        Rc = R.to(dt).contiguous()
        tc = t.to(device=R.device, dtype=dt).expand(*lead, 3).contiguous()
        n = Rc.numel() // 9
        out = torch.empty((*lead, 3), dtype=dt, device=R.device)
        if n:
            with torch.cuda.device(R.device):
                fn = getattr(_lib.load(), f"ska_camera_centre_{_sfx(dt)}")
                _lib.check(fn(_p(Rc), _p(tc), n, _p(out), _stream(R.device)))
        ctx.save_for_backward(Rc, tc)
        ctx.in_meta = (R.shape, R.dtype, t.shape, t.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        # gR[i][k] = -t_i gC_k ; gt = -R gC  (tiny per-camera outer products: autograd plumbing)
        Rc, tc = ctx.saved_tensors
        Rs, Rd, ts, td = ctx.in_meta
        gR = -(tc.unsqueeze(-1) * g.unsqueeze(-2))
        gt = -(Rc @ g.unsqueeze(-1)).squeeze(-1)
        return gR.reshape(Rs).to(Rd), gt.sum_to_size(ts).to(td) if gt.shape != ts else gt.to(td)


def _mean(w, total, count, dt):
    """``w * total / count``; with no term (count 0) torch's mean of an empty tensor: nan, and a zero gradient."""
    if count == 0:
        return (w * total * 0.0 + float("nan")).to(dt)
    return (w * total / count).to(dt)


class _RawSum(torch.autograd.Function):
    """Generic wrapper: `launch(grads_wanted) -> (sum tensor (fp64, 0-dim), [unscaled grads])`."""

    @staticmethod
    def forward(ctx, launch, *tensors):
        need = [ctx.needs_input_grad[i + 1] for i in range(len(tensors))]
        total, grads = launch(need)
        ctx.grads = grads
        return total

    @staticmethod
    def backward(ctx, g):
        return (None, *[None if gi is None else gi * g.to(gi.dtype) for gi in ctx.grads])


def camera_smooth_loss(R, t, w=1e-2):
    """loss.py:103-106: ``w * mean((C[1:] - C[:-1])^2)`` over the leading (time) axis."""
    _cuda(R, "R")
    dt = torch.promote_types(R.dtype, t.dtype)
    dev = R.device
    Rc = R.to(dt).contiguous()
    tc = t.to(device=dev, dtype=dt).expand(*R.shape[:-2], 3).contiguous()
    D0 = Rc.shape[0]
    M = (Rc.numel() // 9) // max(D0, 1)
    count = max(D0 - 1, 0) * M * 3

    def launch(need):
        lib = _lib.load()
        gR = torch.empty_like(Rc) if need[0] else None
        gt = torch.empty_like(tc) if need[1] else None
        s = torch.zeros(1, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
            fn = getattr(lib, f"ska_camera_smooth_{_sfx(dt)}")
            _lib.check(fn(_p(Rc), _p(tc), D0, M, _p(s), _p(gR), _p(gt), _p(ws), ws.numel(), _stream(dev)))
        return s[0].clone(), [gR, gt]

    total = _RawSum.apply(launch, Rc, tc)
    return _mean(w, total, count, dt)


def baseline_reg_loss(R, t, w=1e-2):
    """loss.py:109-114: ``w * mean((|C0 - C1| - mean.detach())^2)``; 0 for a single camera."""
    _cuda(R, "R")
    if R.shape[1] < 2:
        return torch.tensor(0.0, device=R.device)
    dt = torch.promote_types(R.dtype, t.dtype)
    dev = R.device
    Rc = R.to(dt).contiguous()
    tc = t.to(device=dev, dtype=dt).expand(*R.shape[:-2], 3).contiguous()
    T, Cn = Rc.shape[0], Rc.shape[1]
    lib = _lib.load()
    fn = getattr(lib, f"ska_baseline_reg_{_sfx(dt)}")
    mean = torch.zeros(1, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        ws = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
        _lib.check(fn(_p(Rc), _p(tc), T, Cn, None, _p(mean), None, None, _p(ws), ws.numel(), _stream(dev)))
    mean = mean / T  # detached by construction (loss.py:114)

    def launch(need):
        gR = torch.empty_like(Rc) if need[0] else None
        gt = torch.empty_like(tc) if need[1] else None
        s = torch.zeros(1, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws2 = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
            _lib.check(fn(_p(Rc), _p(tc), T, Cn, _p(mean), _p(s), _p(gR), _p(gt), _p(ws2), ws2.numel(), _stream(dev)))
        return s[0].clone(), [gR, gt]

    total = _RawSum.apply(launch, Rc, tc)
    return (w * total / T).to(dt)


def bone_length_loss(X3d, ref_bone_len=None, w=1e-2):
    """loss.py:134-150: ``w * mean((|X_i - X_j| - ref)^2)`` over (T, bones); ref = per-bone mean over T
    (detached) or the given vector.  Bones with an index >= J are skipped (:137-139)."""
    _cuda(X3d, "X3d")
    T, J, _ = X3d.shape
    keep = [k for k, (i, j) in enumerate(BONES) if i < J and j < J]
    if not keep:
        return torch.tensor(0.0, device=X3d.device)
    dt, dev = X3d.dtype, X3d.device
    Xc = X3d.contiguous()
    nb = len(keep)
    bi = (C.c_int32 * nb)(*[BONES[k][0] for k in keep])
    bj = (C.c_int32 * nb)(*[BONES[k][1] for k in keep])
    lib = _lib.load()
    fn = getattr(lib, f"ska_bone_length_{_sfx(dt)}")
    if ref_bone_len is None:
        sums = torch.zeros(_cabi.MAX_BONES, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
            _lib.check(fn(_p(Xc), T, J, bi, bj, nb, None, _p(sums), None, _p(ws), ws.numel(), _stream(dev)))
        ref = (sums / T).contiguous()
    else:
        r = ref_bone_len.to(device=dev, dtype=torch.float64).reshape(-1)
        if r.numel() != nb:
            raise RuntimeError(f"ref_bone_len has {r.numel()} entries for {nb} bones")
        ref = torch.zeros(_cabi.MAX_BONES, dtype=torch.float64, device=dev)
        ref[:nb] = r

    def launch(need):
        gX = torch.empty_like(Xc) if need[0] else None
        s = torch.zeros(_cabi.MAX_BONES, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws2 = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
            _lib.check(fn(_p(Xc), T, J, bi, bj, nb, _p(ref), _p(s), _p(gX), _p(ws2), ws2.numel(), _stream(dev)))
        return s[0].clone(), [gX]

    total = _RawSum.apply(launch, Xc)
    return (w * total / (T * nb)).to(dt)


def pose_temporal_loss(X3d, w=1e-2):
    """loss.py:153-155: ``w * mean((X[1:] - X[:-1])^2)``."""
    _cuda(X3d, "X3d")
    T, J, _ = X3d.shape
    dt, dev = X3d.dtype, X3d.device
    Xc = X3d.contiguous()

    def launch(need):
        lib = _lib.load()
        gX = torch.empty_like(Xc) if need[0] else None
        s = torch.zeros(1, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws = _workspace(dev, int(lib.ska_reg_workspace_bytes()))
            fn = getattr(lib, f"ska_pose_temporal_{_sfx(dt)}")
            _lib.check(fn(_p(Xc), T, J, _p(s), _p(gX), _p(ws), ws.numel(), _stream(dev)))
        return s[0].clone(), [gX]

    total = _RawSum.apply(launch, Xc)
    return _mean(w, total, max(T - 1, 0) * J * 3, dt)
