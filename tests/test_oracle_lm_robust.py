"""The robust (Huber / Cauchy) extension of the Schur-LM specification (tests/oracle_robust.py) on the CPU, and the C ABI's
validation of the loss fields without a GPU."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import lm
from oracle import lm_calib as lc
from skiing_analysis_pytorch_b200 import synth
from tests import oracle_robust as orb

def _flat(clip, C):
    T, J = clip.X.shape[:2]
    x = clip.x_fm.astype(float).transpose(0, 2, 1, 3).reshape(T * J, C, 2)
    cf = clip.conf_fm.astype(float).transpose(0, 2, 1).reshape(T * J, C)
    return x, cf / (cf.sum() + 1e-6)


def _problem6(frac=0.2):
    """Small 2-camera problem with injected outliers and one point behind camera 1 (depth-clamped there)."""
    clip, R0, t0, X0 = lm.make_problem("2b", 6, 5, seed=3)
    synth.inject_outliers(clip.x_vm, 5, frac, seed=4)
    X = X0.reshape(-1, 3).copy()
    centre = -R0[1].T @ t0[1]
    X[7] = centre - 1.0 * R0[1][2]
    x, w = _flat(clip, 2)
    return X, R0, t0, clip.K, x, w


def _scale_between_branches(X, R, t, K, x, w):
    e, _, _, cl = lm.residual_blocks(X, R, t, K, x, w)
    s = (e**2).sum(-1)[~cl]
    return float(np.sqrt(np.median(s)))


def _torch_rho(s, loss, d):
    if loss == "huber":
        return torch.where(s <= d * d, s, 2 * d * torch.sqrt(s.clamp_min(d * d)) - d * d)
    return d * d * torch.log1p(s / (d * d))


def _skew(v):
    z = torch.zeros((), dtype=v.dtype)
    return torch.stack([torch.stack([z, -v[2], v[1]]), torch.stack([v[2], z, -v[0]]), torch.stack([-v[1], v[0], z])])


def _cam_update(R, t, dcam):
    Rn = torch.stack([torch.matrix_exp(_skew(dcam[c, :3])) @ R[c] for c in range(R.shape[0])])
    return Rn, t + dcam[:, 3:]


def _F6(X, dcam, R, t, K, x, w, loss, d):
    Rn, tn = _cam_update(R, t, dcam)
    Xc = torch.einsum("cab,nb->nca", Rn, X) + tn
    Z = Xc[..., 2].clamp_min(lm.ZMIN)
    xn, yn = Xc[..., 0] / Z, Xc[..., 1] / Z
    u = K[:, 0, 0] * xn + K[:, 0, 1] * yn + K[:, 0, 2]
    v = K[:, 1, 0] * xn + K[:, 1, 1] * yn + K[:, 1, 2]
    s = (u - x[..., 0]) ** 2 + (v - x[..., 1]) ** 2
    return (w * _torch_rho(s, loss, d)).sum()


def _Fcalib(X, dcam, th, R, t, x, w, loss, d):
    Rn, tn = _cam_update(R, t, dcam[:, :6])
    th = th + dcam[:, 6:]
    Xc = torch.einsum("cab,nb->nca", Rn, X) + tn
    z = Xc[..., 2]
    keep = z >= lm.ZMIN
    Z = z.clamp_min(lm.ZMIN)
    xn, yn = Xc[..., 0] / Z, Xc[..., 1] / Z
    fx, fy, cx, cy, k1, k2, p1, p2, k3 = th.unbind(-1)
    r2 = xn * xn + yn * yn
    rad = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
    xd = xn * rad + 2 * p1 * xn * yn + p2 * (r2 + 2 * xn * xn)
    yd = yn * rad + p1 * (r2 + 2 * yn * yn) + 2 * p2 * xn * yn
    s = (fx * xd + cx - x[..., 0]) ** 2 + (fy * yd + cy - x[..., 1]) ** 2
    s = torch.where(keep, s, torch.zeros_like(s))
    return (w * _torch_rho(s, loss, d)).sum()


def _rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_robust_weights_and_the_huber_inlier_branch():
    s = np.array([0.0, 0.25, 4.0, 4.0 + 1e-9, 100.0, 1e12])
    rho, om = orb.robust(s, "huber", 2.0)
    assert np.array_equal(rho[:4], s[:4]) and np.array_equal(om[:3], np.ones(3))
    np.testing.assert_allclose(rho[4:], 2 * 2.0 * np.sqrt(s[4:]) - 4.0, rtol=1e-15)
    np.testing.assert_allclose(om[3:], 2.0 / np.sqrt(s[3:]), rtol=1e-15)
    rho, om = orb.robust(s, "cauchy", 2.0)
    np.testing.assert_allclose(rho, 4.0 * np.log1p(s / 4.0), rtol=1e-15)
    np.testing.assert_allclose(om, 1.0 / (1.0 + s / 4.0), rtol=1e-15)
    for loss in ("huber", "cauchy"):  # omega = rho'(s)
        h = 1e-6
        r1, _ = orb.robust(s[2:5] + h, loss, 2.0)
        r0, _ = orb.robust(s[2:5] - h, loss, 2.0)
        _, o = orb.robust(s[2:5], loss, 2.0)
        np.testing.assert_allclose((r1 - r0) / (2 * h), o, rtol=1e-6)
    with pytest.raises(ValueError):
        orb.robust(s, "tukey", 1.0)
    with pytest.raises(ValueError):
        orb.robust(s, "huber", 0.0)


@pytest.mark.parametrize("loss", ["huber", "cauchy"])
def test_gradient_is_half_the_autograd_gradient_6param(loss):
    X, R, t, K, x, w = _problem6()
    d = _scale_between_branches(X, R, t, K, x, w)
    e, _, _, cl = lm.residual_blocks(X, R, t, K, x, w)
    s = (e**2).sum(-1)
    assert cl.sum() == 1 and (s[~cl] <= d * d).any() and (s[~cl] > d * d).any()
    lin = orb.linearise(X, R, t, K, x, w, 1e-3, keep_points=True, loss=loss, scale=d)
    T = lambda a: torch.tensor(a, dtype=torch.float64)
    Xt = T(X).requires_grad_(True)
    dc = torch.zeros((2, 6), dtype=torch.float64, requires_grad=True)
    F = _F6(Xt, dc, T(R), T(t), T(K), T(x), T(w), loss, d)
    F.backward()
    assert abs(lin.cost - F.item()) <= 1e-12 * F.item()
    assert _rel(lin.gp, 0.5 * Xt.grad.numpy()) < 1e-10
    assert _rel(lin.gc, 0.5 * dc.grad.numpy()) < 1e-10
    assert orb.cost_only(X, R, t, K, x, w, loss, d)[0] == pytest.approx(F.item(), rel=1e-12)


@pytest.mark.parametrize("loss", ["huber", "cauchy"])
def test_gradient_is_half_the_autograd_gradient_calib(loss):
    clip, R0, t0, th, X0 = lc.make_problem("2b", 6, 5, seed=3)
    synth.inject_outliers(clip.x_vm, 5, 0.2, seed=4)
    X = X0.reshape(-1, 3).copy()
    X[7] = -R0[1].T @ t0[1] - 1.0 * R0[1][2]  # behind camera 1: excluded there
    x, w = _flat(clip, 2)
    e, _, _, cl = lc.residual_blocks(X, R0, t0, th, x)
    s = (e**2).sum(-1)[~cl]
    d = float(np.sqrt(np.median(s)))
    assert cl.sum() == 1 and (s <= d * d).any() and (s > d * d).any()
    lin = orb.calib_linearise(X, R0, t0, th, x, w, 1e-3, loss, d)
    T = lambda a: torch.tensor(a, dtype=torch.float64)
    Xt = T(X).requires_grad_(True)
    dc = torch.zeros((2, 15), dtype=torch.float64, requires_grad=True)
    F = _Fcalib(Xt, dc, T(th), T(R0), T(t0), T(x), T(w), loss, d)
    F.backward()
    assert abs(lin.cost - F.item()) <= 1e-12 * F.item()
    assert _rel(lin.gc, 0.5 * dc.grad.numpy()) < 1e-10
    # the point gradient: sum over the observations of w omega A^T e
    _, om, _ = orb.calib_weights(X, R0, t0, th, x, w, loss, d)
    _, A, _, _ = lc.residual_blocks(X, R0, t0, th, x)
    gp = np.einsum("ncij,nci->nj", A * (w * om)[..., None, None], e)
    assert _rel(gp, 0.5 * Xt.grad.numpy()) < 1e-10
    assert orb.calib_cost_only(X, R0, t0, th, x, w, loss, d)[0] == pytest.approx(F.item(), rel=1e-12)


@pytest.mark.parametrize("loss", ["huber", "cauchy"])
def test_schur_step_equals_the_dense_step(loss):
    X, R, t, K, x, w = _problem6()
    d = _scale_between_branches(X, R, t, K, x, w)
    lam, free = 1e-2, lm.free_mask(2, "full")
    lin = orb.linearise(X, R, t, K, x, w, lam, loss=loss, scale=d)
    dc, _, ok = lm.solve_reduced(lin, lam, free)
    dp, _ = orb.back_substitute(X, R, t, K, x, w, lam, dc, loss, d)
    dc_ref, dp_ref = orb.dense_step(X, R, t, K, x, w, lam, free, loss, d)
    assert ok
    assert _rel(dc, dc_ref) < 1e-8 and _rel(dp, dp_ref) < 1e-8

    clip, R0, t0, th, X0 = lc.make_problem("2b", 4, 5, seed=3)
    synth.inject_outliers(clip.x_vm, 5, 0.2, seed=4)
    Xf = X0.reshape(-1, 3)
    x, w = _flat(clip, 2)
    freec, rp = lc.free_mask(2), np.broadcast_to(lc.PRIOR_RHO, (2, lc.NI)).copy()
    lin = orb.calib_linearise(Xf, R0, t0, th, x, w, lam, loss, d)
    dc, _, ok = lc.solve_reduced(lin, lam, freec, th, th, rp)
    dp, _ = orb.calib_back_substitute(Xf, R0, t0, th, x, w, lam, dc, loss, d)
    dc_ref, dp_ref = orb.calib_dense_step(Xf, R0, t0, th, x, w, lam, freec, th, rp, loss, d)
    assert ok
    assert _rel(dc, dc_ref) < 1e-7 and _rel(dp, dp_ref) < 1e-7


def _hist_equal(a, b):
    assert len(a) == len(b)
    for ra, rb in zip(a, b):
        assert ra == rb, (ra, rb)


def test_l2_default_and_huber_inside_scale_reproduce_the_l2_oracle_exactly():
    clip, R0, t0, X0 = lm.make_problem("2b", 30, 17)
    ref = lm.run_lm(X0, R0, t0, clip.K, clip.x_fm, clip.conf_fm, num_iters=6)
    x, w = _flat(clip, 2)
    e, _, _, _ = lm.residual_blocks(X0.reshape(-1, 3), R0, t0, clip.K, x, w)
    big = 10.0 * float(np.sqrt((e**2).sum(-1).max()))
    for kw in (dict(), dict(loss="huber", scale=big)):
        got = orb.run_lm(X0, R0, t0, clip.K, clip.x_fm, clip.conf_fm, num_iters=6, **kw)
        _hist_equal(got[3], ref[3])
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])

    clip, R0, t0, th, X0 = lc.make_problem("2b", 30, 17)
    kw0 = dict(num_iters=5, prior_rho=lc.PRIOR_RHO, prior_theta=synth.theta_from_K(clip.K))
    ref = lc.run_lm(X0, R0, t0, th, clip.x_fm, clip.conf_fm, **kw0)
    for kw in (dict(), dict(loss="huber", scale=big)):
        got = orb.calib_run_lm(X0, R0, t0, th, clip.x_fm, clip.conf_fm, **kw0, **kw)
        _hist_equal(got[4], ref[4])
        for a, b in zip(got[:4], ref[:4]):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("loss,scale,trials", [("huber", 3.0, 110), ("cauchy", 3.0, 40)])
def test_robust_lm_reaches_the_minimum_of_F(loss, scale, trials):
    """The robust LM's final cost equals an independent minimiser's (L-BFGS-B on the same F with its autograd gradient);
    costs are compared, not parameters: the global scale is a null direction.  Reweighting converges linearly where
    Huber's kink is active, so Huber gets more trials (measured: converged after ~100; Cauchy after ~30)."""
    from scipy.optimize import minimize

    T, J = 10, 17
    clip, R0, t0, X0 = lm.make_problem("2b", T, J, seed=0)
    synth.inject_outliers(clip.x_vm, J, 0.10, seed=1)
    R, t, X, hist = orb.run_lm(X0, R0, t0, clip.K, clip.x_fm, clip.conf_fm, num_iters=trials, loss=loss, scale=scale)
    x, w = _flat(clip, 2)
    F_lm = orb.cost_only(X.reshape(-1, 3), R, t, clip.K, x, w, loss, scale)[0]
    g0 = orb.linearise(X0.reshape(-1, 3), R0, t0, clip.K, x, w, 0.0, keep_points=True, loss=loss, scale=scale)
    g1 = orb.linearise(X.reshape(-1, 3), R, t, clip.K, x, w, 0.0, keep_points=True, loss=loss, scale=scale)
    n0 = np.sqrt((g0.gp**2).sum() + (g0.gc[1:] ** 2).sum())
    n1 = np.sqrt((g1.gp**2).sum() + (g1.gc[1:] ** 2).sum())
    assert n1 < 1e-6 * n0, (n1, n0)

    Tt = lambda a: torch.tensor(a, dtype=torch.float64)
    Rt, tt, Kt, xt, wt = Tt(R0), Tt(t0), Tt(clip.K), Tt(x), Tt(w)
    N = T * J

    def fg(p):
        pt = torch.tensor(p, dtype=torch.float64, requires_grad=True)
        dcam = torch.cat([torch.zeros(1, 6, dtype=torch.float64), pt[3 * N:].view(1, 6)])
        F = _F6(pt[: 3 * N].view(N, 3), dcam, Rt, tt, Kt, xt, wt, loss, scale)
        F.backward()
        return F.item(), pt.grad.numpy().copy()

    p0 = np.concatenate([X0.reshape(-1), np.zeros(6)])
    res = minimize(fg, p0, jac=True, method="L-BFGS-B", options=dict(maxiter=50000, maxfun=100000, ftol=1e-16, gtol=1e-13, maxcor=50))
    assert abs(F_lm - res.fun) <= 1e-6 * res.fun, (F_lm, res.fun, res.message)
    assert hist[0]["cost"] > 1.5 * F_lm


# ------------------------------------------------------------------------------------------ C ABI, no GPU needed
def _problem_struct(C_, loss, scale, flags=0):
    from skiing_analysis_pytorch_b200 import _cabi

    fake = 1 << 20  # aligned, never dereferenced: validation returns before any CUDA call
    return _cabi.SkaBaProblem(C=C_, J=17, T=10, layout=_cabi.LAYOUT_FRAME_MAJOR, flags=flags, d_x2d=fake, d_conf=fake, d_Xpp=fake,
                              d_cams=fake, d_ctrl=fake, d_red=fake, d_red2=fake, d_delta=fake, d_hist=None, d_workspace=fake,
                              ws_bytes=1 << 20, hist_rows=0, peer=None, loss=loss, loss_scale=scale)


def test_abi_rejects_bad_losses_before_any_cuda_call():
    import re
    from pathlib import Path

    from skiing_analysis_pytorch_b200 import _cabi, _lib

    hdr = (Path(__file__).resolve().parent.parent / "include" / "ska.h").read_text()
    assert int(re.search(r"#define SKA_ABI_VERSION (\d+)", hdr).group(1)) == _cabi.ABI_VERSION == 9
    for name, val in (("L2", 0), ("HUBER", 1), ("CAUCHY", 2)):
        assert int(re.search(rf"#define SKA_BA_LOSS_{name} (\d+)", hdr).group(1)) == val == getattr(_cabi, f"BA_LOSS_{name}")
    assert C.sizeof(_cabi.SkaBaProblem) == 144  # the two loss fields appended after `peer`
    lib = _lib.load()
    assert lib.ska_abi_version() == _cabi.ABI_VERSION
    einval, eunsup = -1, -2
    lin = (lib.ska_ba_linearize_f32, lib.ska_ba_backsub_f32, lib.ska_ba_calib_linearize_f32, lib.ska_ba_calib_backsub_f32)
    for fn in lin:
        for loss, scale in ((3, 1.0), (-1, 1.0), (1, 0.0), (1, -2.0), (1, float("nan")), (2, float("inf")), (2, 0.0), (2, 1e-30)):
            p = _problem_struct(2, loss, scale)
            assert fn(C.byref(p), None) == einval, (fn, loss, scale)
    p = _problem_struct(8, _cabi.BA_LOSS_HUBER, 2.0, flags=_cabi.BA_TENSOR_CORE)
    assert lib.ska_ba_linearize_f32(C.byref(p), None) == eunsup
    assert b"tensor-core" in lib.ska_last_error()


def test_python_rejects_bad_losses():
    from skiing_analysis_pytorch_b200 import ba

    x = torch.zeros((1, 2, 1, 2))
    for kw in (dict(loss="tukey"), dict(loss="huber"), dict(loss="cauchy", loss_scale=0.0), dict(loss="huber", loss_scale=float("nan")),
               dict(loss="huber", loss_scale=2.0, tensor_core=True)):
        with pytest.raises((ValueError, RuntimeError)) as ei:
            ba.BundleAdjuster(x, x[..., 0], np.eye(3), np.stack([np.eye(3)] * 2), np.zeros((2, 3)), x[:, 0, :, :1].expand(1, 1, 3), **kw)
        assert ei.type is ValueError, (kw, ei.value)


def test_inject_outliers_model():
    clip = synth.make_clip("2b", 50, 17, seed=0)
    x0, c0 = clip.x_fm.copy(), clip.conf_fm.copy()
    x = x0.copy()
    m = synth.inject_outliers(x, 17, 0.05, seed=2)
    assert m.shape == (50, 2, 17) and m.sum() == round(0.05 * m.size)
    assert np.array_equal(x[~m], x0[~m])
    moved = np.linalg.norm(x[m] - x0[m], axis=-1)
    assert (moved > 0).all()
    rows = np.argwhere(m)
    swaps = [any(np.array_equal(x[tuple(r)], x0[r[0], r[1], j]) for j in range(17) if j != r[2]) for r in rows]
    assert sum(swaps) >= m.sum() // 2
    shift = moved[~np.array(swaps)]
    assert ((shift >= 50 - 1e-3) & (shift <= 300 + 1e-3)).all()
    assert np.array_equal(clip.conf_fm, c0)
    x2 = x0.copy()
    assert np.array_equal(synth.inject_outliers(x2, 17, 0.05, seed=2), m) and np.array_equal(x2, x)
