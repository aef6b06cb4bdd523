"""Values and gradients of the loss.py kernels (csrc/ska_project.cu: reprojection_loss, project_points' backward;
csrc/ska_losses.cu: the four regularisers) against float64 autograd on the plain torch restatement oracle/torch_ref.py,
at clip sizes where every kernel runs more than one block: the fixed-order partial rows, the grid-stride loops, the
staged bone kernel's frame blocks and the pose-temporal chunking.  tests/test_losses_gpu.py checks the same functions on
golden G3/G4, where every kernel is a single block.

The launch geometry is recomputed here from the device's SM count with the rules of the launch code, and every case
asserts that it reaches the path it is named for: a change of those rules fails here instead of silently shrinking what
is covered.  float32 kernels are compared with the reference run in float64 on the same float32 inputs."""
import ctypes as C
import functools
import math

import numpy as np
import pytest
import torch

from oracle import first_order as FO
from oracle import torch_ref as TR
from skiing_analysis_pytorch_b200 import _cabi, _lib, ba, synth
from skiing_analysis_pytorch_b200 import losses as L

pytestmark = pytest.mark.gpu

DT = {"f64": torch.float64, "f32": torch.float32}
# float64: kernel and reference differ by summation order only (~1e-16 per term; sums over <= 1.7 M terms with
# little cancellation), so values to 1e-12 relative and gradients to 1e-10 of the tensor's largest entry.
# float32 reprojection: the values and gradient tolerances of tests/test_losses_gpu.py (pixel coordinates ~1e3 carry
# an ulp of 6e-5 px; the residuals are a few px).
# float32 regularisers: the kernels take differences of float32 coordinates in float32 (one rounding, 6e-8 relative)
# and sum in float64; the bone residual |len - ref| is ~1/20 of the length, which makes that ~1e-6 relative.
TOL = {
    "f64": dict(value=1e-12, grad=1e-10, reg_value=1e-12, reg_grad=1e-10),
    "f32": dict(value=1e-4, grad=2e-3, reg_value=1e-5, reg_grad=1e-4),
}
KLB = KPB = 256  # block size of the regulariser (kLB) and reprojection (kPB) kernels


# ---------------------------------------------------------------------------------------------------- launch geometry
def _cdiv(a, b):
    return -(-a // b)


def _max_grid():  # ska_ba.cu ba_max_grid: 8 resident 256-thread blocks per SM
    return 8 * torch.cuda.get_device_properties(0).multi_processor_count


def _small_grid(n):  # ska_losses.cu small_grid: camera_smooth, baseline_reg, bone_length's direct kernel
    return max(1, min(_max_grid() // 4, _cdiv(n, KLB)))


def _loss_grid(n):  # ska_project.cu loss_grid: loss_points_kernel, loss_cam_shared_kernel (x C)
    return max(1, min(_max_grid() // 2, _cdiv(n, KPB)))


def _passes(n, grid, block):
    return _cdiv(n, grid * block)


def _bone_plan(J, dt):
    """ska_losses.cu bone_length, gradient pass -> (staged kernel?, FB frames per block)."""
    es = torch.empty((), dtype=dt).element_size()
    rs = (3 * J) | 1
    fb = 128
    while fb > 32 and 2 * fb * rs * es > 96 * 1024:
        fb //= 2
    return 2 * fb * rs * es <= 200 * 1024, fb


def _pt_chunk(T, J):
    """ska_losses.cu pose_temporal -> (frames per thread, grid)."""
    M = 3 * J
    max_blocks = _max_grid() * _cabi.MAX_BONES
    chunk = 128
    while chunk > 8 and _cdiv(T, chunk) * M < 300000:
        chunk //= 2
    while _cdiv(_cdiv(T, chunk) * M, KLB) > max_blocks:
        chunk *= 2
    return chunk, max(1, _cdiv(_cdiv(T, chunk) * M, KLB))


# ------------------------------------------------------------------------------------------------------------ inputs
def _so3(w):
    """Rodrigues, (...,3) -> (...,3,3); w is never exactly 0 here."""
    th = w.norm(dim=-1)[..., None, None]
    W = torch.zeros(w.shape[:-1] + (3, 3), dtype=w.dtype, device=w.device)
    W[..., 0, 1], W[..., 0, 2], W[..., 1, 2] = -w[..., 2], w[..., 1], -w[..., 0]
    W = W - W.transpose(-1, -2)
    return torch.eye(3, dtype=w.dtype, device=w.device) + torch.sin(th) / th * W + (1 - torch.cos(th)) / th**2 * (W @ W)


@functools.lru_cache(maxsize=2)
def _clip(rig, T, J, seed):
    return synth.make_clip_device(rig, T, J, torch.device("cuda:0"), seed=seed, layout="TCJ2")


def _problem(rig, T, J, cams, dt, seed=0):
    """make_clip_device observations; X, R, t, K perturbed (seeded) so that residuals and gradients are far from 0;
    10 % of the confidences zero.  cams: "shared" R/t/K (C,..), "perframe" R/t/K (T,C,..), "perframeR" R (T,C,3,3)
    with t (C,3) and K (C,3,3).  Returns X, R, t, K in dt and x2d, conf (float32)."""
    d = _clip(rig, T, J, seed)
    dev = d["X"].device
    g = torch.Generator(device=dev).manual_seed(1000 + seed)
    f64 = dict(dtype=torch.float64, device=dev)
    rn = lambda *s: torch.randn(*s, generator=g, **f64)
    Cn = len(d["R"])
    R0, t0, K0 = (torch.tensor(d[k], **f64) for k in ("R", "t", "K"))
    K0[:, 0, 1] = 0.5  # a skew entry: the full K of loss.py:74-82
    lead = (T, Cn) if cams != "shared" else (Cn,)
    R = _so3(0.02 * rn(*lead, 3)) @ R0
    t = t0 + 0.05 * rn(*((T, Cn) if cams == "perframe" else (Cn,)), 3)
    K = K0
    if cams == "perframe":
        K = K0.expand(T, Cn, 3, 3).clone()
        K[..., :2, :] *= 1.0 + 0.01 * rn(T, Cn, 2, 1)
    X = d["X"] + 0.03 * rn(T, J, 3)
    conf = d["conf"].clone()
    conf[torch.rand(conf.shape, generator=g, device=dev) < 0.1] = 0.0
    return X.to(dt), R.to(dt), t.to(dt), K.to(dt), d["x2d"], conf


def _cams(rig, T, dt, seed):
    """Per-frame cameras (T,C,3,3) / (T,C,3): the rig with seeded per-frame jitter."""
    R0, t0 = synth.rig(rig)
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    f64 = dict(dtype=torch.float64, device="cuda:0")
    Cn = len(R0)
    R = _so3(0.02 * torch.randn(T, Cn, 3, generator=g, **f64)) @ torch.tensor(R0, **f64)
    t = torch.tensor(t0, **f64) + 0.05 * torch.randn(T, Cn, 3, generator=g, **f64)
    return R.to(dt), t.to(dt)


def _poses(T, J, dt, seed):
    """A skeleton (T,J,3) from make_clip_device's model without its observations (which the regularisers do not read)."""
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    f64 = dict(dtype=torch.float64, device="cuda:0")
    tt = torch.arange(T, **f64)
    root = torch.stack([1.5 * torch.sin(2 * np.pi * tt / 300), 0.3 * torch.sin(2 * np.pi * tt / 90), 10.0 + torch.cos(2 * np.pi * tt / 240)], -1)
    X = root[:, None] + 0.4 * torch.randn(J, 3, generator=g, **f64) + 0.02 * torch.randn(T, J, 3, generator=g, **f64)
    return X.to(dt)


# --------------------------------------------------------------------------------------------------------- comparison
def _grads(fn, tensors):
    leaves = [x.detach().clone().requires_grad_(True) for x in tensors]
    v = fn(*leaves)
    v.backward()
    return v.detach(), [x.grad for x in leaves]


def _compare(ours_fn, ref_fn, inputs, prec, value_key, grad_key, what):
    """ours on `inputs` (dtype of prec) against the float64 reference on the same numbers."""
    tol = TOL[prec]
    v, go = _grads(ours_fn, inputs)
    vr, gr = _grads(ref_fn, [x.double() for x in inputs])
    assert v.dtype == DT[prec], what
    if math.isnan(vr.item()):
        assert math.isnan(v.item()), what
    else:
        assert abs(v.item() - vr.item()) <= tol[value_key] * abs(vr.item()), (what, v.item(), vr.item())
    for k, (a, b) in enumerate(zip(go, gr)):
        assert a is not None and a.shape == b.shape and a.dtype == DT[prec], (what, k)
        assert bool(torch.isfinite(a).all()), (what, k)
        scale = b.abs().max().item()
        err = (a.double() - b).abs().max().item()
        assert err <= tol[grad_key] * scale or (scale == 0.0 and err == 0.0), (what, k, err, scale)
    return go


# ------------------------------------------------------------------------------------------------ 1. reprojection_loss
SHAPES = {  # rig (C = 8 / 2 / 3 / 8), T, J
    "one_block": ("8", 12, 17),  # T*J = 204 <= 256: the single-block control
    "blocks_J1": ("2b", 2000, 1),  # 2000 points: 8 blocks, no wrap
    "blocks_J70": ("3", 30, 70),  # 2100 points: 9 blocks, no wrap
    "wrap": ("8", 100_000, 17),  # 1.7 M points: the grid-stride loop wraps (12 times on 148 SMs)
}


def _check_reproj_geometry(shape, T, J):
    grid = _loss_grid(T * J)
    if shape == "one_block":
        assert grid == 1
    elif shape.startswith("blocks"):
        assert grid > 1 and _passes(T * J, grid, KPB) == 1
    else:
        assert _passes(T * J, grid, KPB) >= 2


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("cams", ["shared", "perframe", "perframeR"])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_reprojection_loss_value_and_gradients(cuda, shape, cams, prec):
    rig, T, J = SHAPES[shape]
    _check_reproj_geometry(shape, T, J)
    X, R, t, K, x2d, conf = _problem(rig, T, J, cams, DT[prec])
    assert (conf == 0).any() and (conf > 0).any()
    c64, x64 = conf.double(), x2d.double()
    _compare(lambda *a: L.reprojection_loss(*a, x2d, conf, w=0.7), lambda *a: TR.reprojection_loss(*a, x64, c64, w=0.7),
             [X, R, t, K], prec, "value", "grad", (shape, cams))


@pytest.mark.parametrize("cams", ["shared", "perframe"])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_reprojection_loss_behind_the_camera(cuda, cams, prec):
    """Points behind camera 0 divide by the 1e-6 depth clamp and get no depth derivative (autograd of clamp(min=1e-6),
    loss.py:67).  Kept apart from the cases above: one clamped point sets the scale of every gradient."""
    X, R, t, K, x2d, conf = _problem("2b", 6, 17, cams, DT[prec], seed=1)
    behind = [(0, 3), (2, 11), (5, 16)]
    for k, (f, j) in enumerate(behind):  # camera 0 sits at the origin looking down +z; these points are at z = -5
        X[f, j] = torch.tensor([0.02 * (k + 1), -0.01, -5.0], dtype=X.dtype)
        conf[f, 0, j] = 1.0
    c64, x64 = conf.double(), x2d.double()
    _compare(lambda *a: L.reprojection_loss(*a, x2d, conf), lambda *a: TR.reprojection_loss(*a, x64, c64),
             [X, R, t, K], prec, "value", "grad", ("clamp", cams))
    Rf = R.double() if R.dim() == 4 else R.double()[None].expand(6, 2, 3, 3)
    tf = t.double() if t.dim() == 3 else t.double()[None].expand(6, 2, 3)
    z = torch.einsum("tcb,tjb->tcj", Rf[..., 2, :], X.double()) + tf[..., 2:3]
    out = _abi_reprojection(X, R, t, K, x2d.to(X.dtype), conf.to(X.dtype))
    assert out["sums"][2].item() == float((z < 1e-6).sum()) == len(behind)


# ------------------------------------------------------------------------------------------ 2. project_points backward
@pytest.mark.parametrize("cams", ["shared", "perframe"])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_project_points_backward_at_scale(cuda, cams, prec):
    """Cotangent mode of the loss kernels (conf == NULL) over 1.7 M points x 3 cameras."""
    T, J = 100_000, 17
    assert _passes(T * J, _loss_grid(T * J), KPB) >= 2
    X, R, t, K, _, _ = _problem("3", T, J, cams, DT[prec], seed=2)
    cot = torch.randn(T, 3, J, 2, dtype=torch.float64, device=cuda, generator=torch.Generator(device=cuda).manual_seed(7))
    cot_s = cot.to(DT[prec])
    ours = lambda *a: (L.project_points(*a) * cot_s).sum()
    ref = lambda *a: (TR.project_points(*a) * cot).sum()
    # the value is a sum of 10 M signed terms in the caller's dtype (torch's own sum): not what this test is about
    go = _grads(ours, [X, R, t, K])[1]
    gr = _grads(ref, [X.double(), R.double(), t.double(), K.double()])[1]
    for k, (a, b) in enumerate(zip(go, gr)):
        assert a.dtype == DT[prec] and a.shape == b.shape
        assert (a.double() - b).abs().max().item() <= TOL[prec]["grad"] * b.abs().max().item(), (cams, k)


# --------------------------------------------------------------------------------------------------- 3. regularisers
BONE_CASES = {  # (prec, J): FB of the staged kernel, or 0 = the direct kernel (its shared-memory rows would not fit)
    ("f32", 17): 128, ("f64", 17): 64, ("f64", 70): 32, ("f32", 70): 32, ("f64", 150): 0, ("f32", 270): 0,
}


@pytest.mark.parametrize("prec,J,kind", [(p, j, "direct" if fb == 0 else "staged_walk") for (p, j), fb in BONE_CASES.items()]
                         + [("f64", 17, "one_block")])
def test_bone_length_paths(cuda, prec, J, kind):
    """The staged kernel with FB = 128 / 64 / 32 frames per block, each block walking three blocks of frames with a
    partial last one (and a clip shorter than one block); the direct kernel with a gradient in both precisions."""
    dt = DT[prec]
    staged, FB = _bone_plan(J, dt)
    assert (FB if staged else 0) == BONE_CASES[(prec, J)]
    if kind == "staged_walk":
        T = 2 * _max_grid() * FB + FB // 2 + 3
        assert T % FB != 0 and _cdiv(T, min(_max_grid(), _cdiv(T, FB)) * FB) == 3
    elif kind == "one_block":
        T = FB - 19
    else:
        T = _max_grid() // 4 * KLB + 1001 if prec == "f64" else 3001
        assert _small_grid(T) > 1
    X = _poses(T, J, dt, seed=10 + J)
    _compare(lambda X_: L.bone_length_loss(X_, w=0.2), lambda X_: TR.bone_length(X_, None, 0.2), [X], prec,
             "reg_value", "reg_grad", (prec, J, T))


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_bone_length_skipped_bones_given_reference_and_zero_length(cuda, prec):
    dt = DT[prec]
    # J = 12: the bones touching joints 12..16 are skipped (loss.py:137-139), six remain; a given ref_bone_len
    X = _poses(5001, 12, dt, seed=20)
    nb = sum(1 for i, j in L.BONES if i < 12 and j < 12)
    assert nb == 6
    ref = 0.5 + 0.1 * torch.rand(nb, dtype=torch.float64, device=cuda, generator=torch.Generator(device=cuda).manual_seed(3))
    _compare(lambda X_: L.bone_length_loss(X_, ref_bone_len=ref, w=0.3), lambda X_: TR.bone_length(X_, ref, 0.3), [X], prec,
             "reg_value", "reg_grad", "J=12")
    # two coinciding joints: a zero-length bone in every third frame, whose subgradient is 0 (torch.norm at 0)
    X = _poses(4001, 17, dt, seed=21)
    X[::3, 7] = X[::3, 5]
    _compare(lambda X_: L.bone_length_loss(X_, w=0.3), lambda X_: TR.bone_length(X_, None, 0.3), [X], prec, "reg_value", "reg_grad",
             "zero length")


@pytest.mark.parametrize("prec,T", [("f64", T) for T in (1, 2, 7, 8, 9, 129, 200_001)] + [("f32", T) for T in (1, 2, 9, 129, 200_001)])
def test_pose_temporal(cuda, prec, T):
    """Chunks of 8 frames per thread at short clips (T = 129: a last chunk of one frame), several frames per thread and
    many blocks at 200 k frames; T = 1 has no term (nan, zero gradient, like torch's mean of an empty tensor)."""
    J = 17
    chunk, grid = _pt_chunk(T, J)
    if T > 1000:
        assert chunk > 8 and grid > 1
    X = _poses(T, J, DT[prec], seed=30 + T)
    _compare(lambda X_: L.pose_temporal_loss(X_, w=0.2), lambda X_: TR.pose_temporal(X_, 0.2), [X], prec, "reg_value", "reg_grad",
             (prec, T))


def test_pose_temporal_chunk_doubling_f32(cuda):
    """A clip long enough that the per-block partials would overflow the workspace at 128 frames per thread: the chunk
    doubles (about 3 M frames x 70 joints on 148 SMs, 2.5 GB of float32)."""
    J = 70
    T = int(1.02 * 128 * KLB * _max_grid() * _cabi.MAX_BONES / (3 * J))
    chunk, _ = _pt_chunk(T, J)
    assert chunk >= 256
    g = torch.Generator(device=cuda).manual_seed(40)
    X = (10.0 + 0.01 * torch.randn(T, J, 3, device=cuda, generator=g)).float()
    tol = TOL["f32"]
    Xv = X.clone().requires_grad_(True)
    v = L.pose_temporal_loss(Xv, w=0.2)
    v.backward()
    Xr = X.double().requires_grad_(True)
    vr = TR.pose_temporal(Xr, 0.2)
    vr.backward()
    assert abs(v.item() - vr.item()) <= tol["reg_value"] * vr.item()
    assert (Xv.grad.double() - Xr.grad).abs().max().item() <= tol["reg_grad"] * Xr.grad.abs().max().item()


@pytest.mark.parametrize("layout", ["T33", "TC33"])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_camera_smooth(cuda, layout, prec):
    dt = DT[prec]
    n_wrap = 2 * _max_grid() // 4 * KLB + 77  # cameras: the grid-stride loop wraps three times
    for T in (1, 2, 33, n_wrap if layout == "T33" else n_wrap // 3):
        R, t = _cams("3", T, dt, seed=50 + T)
        if layout == "T33":
            R, t = R[:, 0].contiguous(), t[:, 0].contiguous()
        n = R.numel() // 9
        if T > 1000:
            assert _passes(n, _small_grid(n), KLB) == 3
        _compare(lambda R_, t_: L.camera_smooth_loss(R_, t_, w=0.1), lambda R_, t_: TR.camera_smooth(R_, t_, 0.1), [R, t], prec,
                 "reg_value", "reg_grad", (layout, T))


@pytest.mark.parametrize("rig", ["2b", "3", "8"])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_baseline_reg(cuda, rig, prec):
    dt = DT[prec]
    for T in (5, 2 * _max_grid() // 4 * KLB + 77):
        R, t = _cams(rig, T, dt, seed=60 + T)
        R[::5, 1], t[::5, 1] = R[::5, 0], t[::5, 0]  # two identical cameras: zero baseline, subgradient 0
        if T > 1000:
            assert _passes(T, _small_grid(T), KLB) == 3
        gR, gt = _compare(lambda R_, t_: L.baseline_reg_loss(R_, t_, w=0.3), lambda R_, t_: TR.baseline_reg(R_, t_, 0.3), [R, t],
                          prec, "reg_value", "reg_grad", (rig, T))
        assert bool((gR[:, 2:] == 0).all()) and bool((gt[:, 2:] == 0).all())  # only cameras 0 and 1 enter


# ------------------------------------------------------------------------------- 4. exact properties through the C ABI
_p = lambda a: None if a is None else C.c_void_p(a.data_ptr())
_WS = {}


def _ws():
    """One workspace for every call below, like losses.py's cache: the calls of different sizes reuse it."""
    if "ws" not in _WS:
        lib = _lib.load()
        n = max(int(lib.ska_loss_workspace_bytes(8)), int(lib.ska_reg_workspace_bytes()))
        _WS["ws"] = torch.empty(n, dtype=torch.uint8, device="cuda:0")
    return _WS["ws"]


def _nan(shape, dt):
    return torch.full(shape, float("nan"), dtype=dt, device="cuda:0")


def _sfx(dt):
    return "f32" if dt == torch.float32 else "f64"


def _abi_reprojection(X, R, t, K, x2d, conf):
    """ska_reprojection_loss_* with every output pre-filled with NaN.  R/t/K frame strides as losses.py derives them."""
    T, J, _ = X.shape
    Cn = R.shape[-3]
    dt = X.dtype
    out = dict(sums=_nan((4,), torch.float64), gX=_nan(X.shape, dt), gR=_nan(R.shape, dt), gt=_nan(t.shape, dt), gK=_nan(K.shape, dt))
    ws = _ws()
    fn = getattr(_lib.load(), f"ska_reprojection_loss_{_sfx(dt)}")
    _lib.check(fn(_p(X), T, J, Cn, _p(R), 9 * Cn if R.dim() == 4 else 0, _p(t), 3 * Cn if t.dim() == 3 else 0, _p(K),
                  9 * Cn if K.dim() == 4 else 0, _p(x2d), _p(conf), _p(out["sums"]), _p(out["gX"]), _p(out["gR"]), _p(out["gt"]),
                  _p(out["gK"]), _p(ws), ws.numel(), None))
    torch.cuda.synchronize()
    out["sums"] = out["sums"][:3]  # entry 3 is reserved and not written
    return out


def _abi_bone(X, ref):
    T, J, _ = X.shape
    keep = [(i, j) for i, j in L.BONES if i < J and j < J]
    bi = (C.c_int32 * len(keep))(*[i for i, _ in keep])
    bj = (C.c_int32 * len(keep))(*[j for _, j in keep])
    out = dict(sums=_nan((_cabi.MAX_BONES,), torch.float64), gX=_nan(X.shape, X.dtype) if ref is not None else None)
    ws = _ws()
    _lib.check(getattr(_lib.load(), f"ska_bone_length_{_sfx(X.dtype)}")(_p(X), T, J, bi, bj, len(keep), _p(ref), _p(out["sums"]),
                                                                         _p(out["gX"]), _p(ws), ws.numel(), None))
    torch.cuda.synchronize()
    return {k: v for k, v in out.items() if v is not None}


def _abi_pose_temporal(X):
    T, J, _ = X.shape
    out = dict(sum=_nan((1,), torch.float64), gX=_nan(X.shape, X.dtype))
    ws = _ws()
    _lib.check(getattr(_lib.load(), f"ska_pose_temporal_{_sfx(X.dtype)}")(_p(X), T, J, _p(out["sum"]), _p(out["gX"]), _p(ws), ws.numel(), None))
    torch.cuda.synchronize()
    return out


def _abi_camera_smooth(R, t):
    out = dict(sum=_nan((1,), torch.float64), gR=_nan(R.shape, R.dtype), gt=_nan(t.shape, t.dtype))
    ws = _ws()
    _lib.check(getattr(_lib.load(), f"ska_camera_smooth_{_sfx(R.dtype)}")(_p(R), _p(t), R.shape[0], R.shape[1], _p(out["sum"]), _p(out["gR"]),
                                                                           _p(out["gt"]), _p(ws), ws.numel(), None))
    torch.cuda.synchronize()
    return out


def _abi_baseline(R, t, mean):
    out = dict(sum=_nan((1,), torch.float64))
    if mean is not None:
        out.update(gR=_nan(R.shape, R.dtype), gt=_nan(t.shape, t.dtype))
    ws = _ws()
    _lib.check(getattr(_lib.load(), f"ska_baseline_reg_{_sfx(R.dtype)}")(_p(R), _p(t), R.shape[0], R.shape[1], _p(mean), _p(out["sum"]),
                                                                          _p(out.get("gR")), _p(out.get("gt")), _p(ws), ws.numel(), None))
    torch.cuda.synchronize()
    return out


def _all_written_and_equal(a, b, what):
    for k in a:
        assert not bool(torch.isnan(a[k]).any()), (what, k, "an output entry was never written")
        assert torch.equal(a[k], b[k]), (what, k, "not bit-identical")


def _abi_calls(dt, T, J, rig, seed):
    """Every C ABI loss entry point on one clip -> {name: outputs}."""
    res = {}
    for cams in ("shared", "perframe", "perframeR"):
        X, R, t, K, x2d, conf = _problem(rig, T, J, cams, dt, seed=seed)
        res[f"reproj_{cams}"] = _abi_reprojection(X, R, t, K, x2d.to(dt), conf.to(dt))
    res["bone_pass0"] = _abi_bone(X, None)
    res["bone_pass1"] = _abi_bone(X, res["bone_pass0"]["sums"] / T)
    res["pose_temporal"] = _abi_pose_temporal(X)
    Rf, tf = _cams(rig, T, dt, seed=seed)
    res["camera_smooth"] = _abi_camera_smooth(Rf, tf)
    res["baseline_pass0"] = _abi_baseline(Rf, tf, None)
    res["baseline_pass1"] = _abi_baseline(Rf, tf, res["baseline_pass0"]["sum"] / T)
    return res


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_abi_writes_every_output_and_repeats_bit_for_bit(cuda, prec):
    """Fixed-order reductions without atomics (DESIGN §3.4): the same call gives the same bits, also after a call of
    another size has reused the workspace in between; and every output entry is written."""
    dt = DT[prec]
    first = _abi_calls(dt, 20_000, 17, "3", seed=3)
    _abi_calls(dt, 1_001, 70, "8", seed=4)  # other grids, camera counts and partial-row layouts in the same workspace
    again = _abi_calls(dt, 20_000, 17, "3", seed=3)
    for name in first:
        _all_written_and_equal(first[name], again[name], name)


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_points_do_not_depend_on_the_rest_of_the_clip(cuda, prec):
    """Per-point gX of reprojection_loss and bone_length and the per-frame camera gradients (loss_cam_frames_kernel) of
    a frame range are bit-identical whether the range is the whole call or part of a larger clip (another grid, other
    block boundaries)."""
    dt = DT[prec]
    T, J, a, b = 20_000, 17, 777, 7_342
    for cams in ("shared", "perframe", "perframeR"):
        X, R, t, K, x2d, conf = _problem("3", T, J, cams, dt, seed=5)
        x2d, conf = x2d.to(dt), conf.to(dt)
        full = _abi_reprojection(X, R, t, K, x2d, conf)
        rows = lambda z, nd: z[a:b] if z.dim() == nd else z  # per-frame tensors: the range's rows; shared ones whole
        sub = _abi_reprojection(X[a:b], rows(R, 4), rows(t, 3), rows(K, 4), x2d[a:b], conf[a:b])
        assert torch.equal(full["gX"][a:b], sub["gX"]), (cams, "gX")
        for k, src, nd in (("gR", R, 4), ("gt", t, 3), ("gK", K, 4)):
            if src.dim() == nd:
                assert torch.equal(full[k][a:b], sub[k]), (cams, k)
    for J in (17, 70):
        X = _poses(T, J, dt, seed=6)
        nb = sum(1 for i, j in L.BONES if i < J and j < J)
        ref = torch.zeros(_cabi.MAX_BONES, dtype=torch.float64, device=cuda)
        ref[:nb] = 0.5
        assert a % _bone_plan(J, dt)[1] != 0
        assert torch.equal(_abi_bone(X, ref)["gX"][a:b], _abi_bone(X[a:b], ref)["gX"]), ("bone", J)


# ---------------------------------------------------------------------------------- 5. the first-order solve at scale
def test_first_order_solve_at_scale_matches_the_oracle(cuda):
    """ba.run_local_ba(optimizer="adam", mode="full") in float64 on 10 k frames x 17 joints x 2 per-frame cameras, where
    every loss kernel runs more than one block, against oracle/first_order.py on the CPU with the torch restatement as its
    loss module.  Tolerances of the golden-G9 trajectory test (tests/test_first_order_gpu.py)."""
    T, J = 10_000, 17
    assert _loss_grid(T * J) > 1
    staged, FB = _bone_plan(J, torch.float64)
    assert staged and _cdiv(T, FB) > 1 and _pt_chunk(T, J)[1] > 1 and _small_grid(T * 2) > 1 and _small_grid(T) > 1
    d = synth.make_clip_device("2b", T, J, cuda, seed=8)
    R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=2)
    g = torch.Generator(device=cuda).manual_seed(9)
    f64 = dict(dtype=torch.float64, device=cuda)
    R = _so3(0.002 * torch.randn(T, 2, 3, generator=g, **f64)) @ torch.tensor(R0, **f64)
    t = torch.tensor(t0, **f64) + 0.01 * torch.randn(T, 2, 3, generator=g, **f64)
    X0 = d["X"] + 0.05 * torch.randn(T, J, 3, generator=g, **f64)
    K = torch.tensor(d["K"])
    Ro, to, Xo, h = ba.run_local_ba(K, R, t, X0, d["x2d"], d["conf"], num_iters=5, lr=1e-2, device="cuda", mode="full", optimizer="adam")
    Rr, tr, Xr, hr = FO.run_adam(TR.ReferenceNames, K, R.cpu(), t.cpu(), X0.cpu(), d["x2d"].cpu(), d["conf"].cpu(), num_iters=5, lr=1e-2,
                                 mode="full")
    row = lambda r: [r["loss"]] + [r[k] for k in ba.FIRST_ORDER_TERMS]
    np.testing.assert_allclose([row(r) for r in h], [row(r) for r in hr], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(Xo.cpu().numpy(), Xr.numpy(), atol=1e-8)
    np.testing.assert_allclose(to.cpu().numpy(), tr.numpy(), atol=1e-8)
    np.testing.assert_allclose(Ro.cpu().numpy(), Rr.numpy(), atol=1e-9)
