"""The Schur-LM bundle-adjustment kernels piece by piece against a float64 reference, at clip sizes where every
multi-tile path runs: the 6-parameter engine (csrc/ska_ba.cu, csrc/ska_ba_wide.cu) and the calibrating engine
(csrc/ska_ba_calib.cu).  tests/test_ba_gpu.py and tests/test_ba_calib_gpu.py compare the linearisation with the numpy
oracle only where each CTA handles one tile, and the rest of a trial only through the cost history.

One trial is driven a launch at a time (linearize, solve, backsub, control) and the engine's device state is read in
between:
  linearize  every entry of the packed reduced system, the cost, the clamp count and the sum of confidences;
  solve      delta against a dense float64 Cholesky solve of the system assembled from the GPU's own `red`, for every
             free mask; the trial cameras against exp([d_omega]x) R, t + d_t (and theta + d_theta);
  backsub    every trial point against X - Hd^-1 (gp + W delta) with the GPU's own delta; red2 (trial cost,
             predicted point decrease, clamp count);
  control    the gain ratio, the decision, the Nielsen update and the history row recomputed from the GPU's inputs.
The reference is oracle/lm.py / oracle/lm_calib.py restated in float64 torch (pinned to the numpy oracle below) and run
on the GPU in point chunks.  It reads what the kernels read: the float32 points of Xpp[cur] and the cameras rounded to
float32 the way load_cam / load_cam_calib round them, so what remains is the kernels' own arithmetic.

Each large case derives its shape from the device's SM count and an UPPER bound on resident CTAs per SM, and asserts
the grid-stride passes or tiles per CTA it needs, whatever the occupancy query returns.  The kernel constants the
geometry uses are mirrored here and checked against the sources."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import lm, lm_calib as lc
from skiing_analysis_pytorch_b200 import _cabi, api, ba, synth
from tests.test_ba_calib_gpu import _unpack as _unpack_calib
from tests.test_ba_gpu import _unpack as _unpack6

pytestmark = pytest.mark.gpu

CSRC = Path(__file__).resolve().parent.parent / "skiing_analysis_pytorch_b200" / "csrc"

# ------------------------------------------------------------------------------------- kernel constants (mirrored)
K_BA_BLOCK = 256      # ska_ba.cuh: kBaBlock - ba_linearize_reg, ba_backsub_kernel, ba_calib_backsub_kernel
WIDE_WARPS = 12       # ska_ba_wide.cu: SKA_BA_WIDE_WARPS - a tile is 12 warps x 32 = 384 points
CALIB_WARPS = 12      # ska_ba_calib.cu: SKA_BA_CALIB_WARPS
K_FLUSH = 16          # ska_ba.cuh: kFlush - wide / calib fp32 window, in tiles
K_Y_STRIDE = 100      # ska_ba.cuh: kYStride - staged floats per column (shared memory per warp)
K_TC_PTS = 48         # ska_ba_wide.cu: kTcPts = 4 * kTcWarps
K_TC_FLUSH = 32       # ska_ba_wide.cu: kTcFlush - tensor-core fp32 window, in tiles
SIZEOF_CAMF, SIZEOF_CAMC = 72, 84  # ska_ba.cuh CamF (18 floats), ska_ba_calib.cuh CamC (21 floats)

# ---------------------------------------------------------------------------------------------------- tolerances
# Measured on one NVIDIA B200 (1000 W power limit, 148 SMs) with about a 3x margin; each comment gives the largest error
# measured over the cases below.  The small-size bounds of tests/test_ba_gpu.py / test_ba_calib_gpu.py (2e-5 / 3e-5 of
# block scale) were the starting point: at these sizes every path stays far inside them, the tensor-core form included.
TOL = dict(
    lin=2.5e-6,     # Sw / bw / gc / Hcc entries, of their block's largest entry (7.5e-7: Sw, wide kernel at C = 8)
    lin_tc=5e-5,    # the same with Sw accumulated by tcgen05.mma: 32-tile fp32 windows in tensor memory (1.5e-5 at C = 8)
    lin_calib=2.5e-6,  # calibrating engine, entries scaled by sqrt(H_rr H_ss) (8.4e-7: camera 1's Hcc)
    cost=3e-7,      # linearisation cost, relative (1.0e-7: register path)
    sumconf=6e-9,   # ba_sum_kernel (fp32 runs of <= 64 terms, fp64 beyond), relative (2.1e-9)
    solve=3.5e-12,  # fp64 Cholesky against fp64 Cholesky: |d - d_ref| / |d_ref|_inf (1.1e-12 at n = 42)
    pred_cam=6e-15,  # camera part of the predicted decrease, relative (2.0e-15)
    cams=4e-16,     # trial R (absolute), t and theta (of the largest entry): fp64 update of fp64 state (1.1e-16)
    dp=5e-4,        # per trial point: |X_trial - X - dp_ref| - 1 ulp(X), over |dp_ref|_inf of that point (1.5e-4)
    trial=7e-7,     # trial cost, relative (2.2e-7)
    # predicted point decrease, of sum_points |term|: the point terms dp . (lam D dp - gp) take both signs and cancel
    # (sum |term| / |sum| up to 162 at C = 8), so fp32 per-point rounding is bounded by the terms' total, not the sum
    # (2.0e-7; relative to |sum|: 3.3e-5 at C = 8, unchanged when the per-thread fp32 sums are folded into fp64)
    pred_pts=6e-7,
)
CTRL_TOL = 1e-14    # control: the same fp64 operations as the kernel (to fp64 rounding)


def _err(got, ref, scale):
    got, ref = np.asarray(got, float), np.asarray(ref, float)
    return float(np.abs(got - ref).max() / scale) if got.size else 0.0


def _within(name, err, tol):
    print(f"    {name:<28s} {err:.3e}  (tol {tol:.1e})")
    assert err <= tol, (name, err, tol)


# ---------------------------------------------------------------------------------- float64 reference (torch port)
ZMIN = lm.ZMIN


def _rb6(X, R, t, K, x):
    """oracle/lm.py residual_blocks: X (N,3), R (C,3,3), t (C,3), K (C,3,3), x (N,C,2) -> e, A, B (N,C,2,6), clamped."""
    Xc = torch.einsum("cab,nb->nca", R, X) + t
    z = Xc[..., 2]
    clamped = z < ZMIN
    iz = 1.0 / z.clamp_min(ZMIN)
    xn, yn = Xc[..., 0] * iz, Xc[..., 1] * iz
    k00, k01, k02, k10, k11, k12 = (K[:, i, j] for i in range(2) for j in range(3))
    fu, fv = k00 * xn + k01 * yn, k10 * xn + k11 * yn
    e = torch.stack([fu + k02, fv + k12], -1) - x
    live = (~clamped).to(X.dtype)
    ju = torch.stack([k00 * iz, k01 * iz, -fu * iz * live], -1)
    jv = torch.stack([k10 * iz, k11 * iz, -fv * iz * live], -1)
    Jx = torch.stack([ju, jv], -2)
    A = torch.einsum("ncij,cjk->ncik", Jx, R)
    p = (Xc - t)[..., None, :].expand_as(Jx)
    return e, A, torch.cat([torch.linalg.cross(p, Jx, dim=-1), Jx], -1), clamped


def _rbc(X, R, t, th, x):
    """oracle/lm_calib.py residual_blocks: th (C,9) -> e, A, B (N,C,2,15), clamped; clamped observations excluded."""
    Xc = torch.einsum("cab,nb->nca", R, X) + t
    z = Xc[..., 2]
    clamped = z < ZMIN
    live = (~clamped).to(X.dtype)
    iz = 1.0 / z.clamp_min(ZMIN)
    xn, yn = Xc[..., 0] * iz, Xc[..., 1] * iz
    fx, fy, cx, cy, k1, k2, p1, p2, k3 = th.unbind(-1)
    r2 = xn * xn + yn * yn
    rad = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
    drad = k1 + r2 * (2 * k2 + 3 * k3 * r2)
    xd = xn * rad + 2 * p1 * xn * yn + p2 * (r2 + 2 * xn * xn)
    yd = yn * rad + p1 * (r2 + 2 * yn * yn) + 2 * p2 * xn * yn
    e = torch.stack([fx * xd + cx, fy * yd + cy], -1) - x
    a11 = rad + 2 * xn * xn * drad + 2 * p1 * yn + 6 * p2 * xn
    a12 = 2 * xn * yn * drad + 2 * p1 * xn + 2 * p2 * yn
    a22 = rad + 2 * yn * yn * drad + 6 * p1 * yn + 2 * p2 * xn
    ju = torch.stack([fx * a11 * iz, fx * a12 * iz, -fx * (a11 * xn + a12 * yn) * iz * live], -1)
    jv = torch.stack([fy * a12 * iz, fy * a22 * iz, -fy * (a12 * xn + a22 * yn) * iz * live], -1)
    Jx = torch.stack([ju, jv], -2)
    A = torch.einsum("ncij,cjk->ncik", Jx, R)
    p = (Xc - t)[..., None, :].expand_as(Jx)
    zero, one = torch.zeros_like(xn), torch.ones_like(xn)
    r4, r6 = r2 * r2, r2 * r2 * r2
    Bu = torch.stack([xd, zero, one, zero, fx * xn * r2, fx * xn * r4, fx * 2 * xn * yn, fx * (r2 + 2 * xn * xn), fx * xn * r6], -1)
    Bv = torch.stack([zero, yd, zero, one, fy * yn * r2, fy * yn * r4, fy * (r2 + 2 * yn * yn), fy * 2 * xn * yn, fy * yn * r6], -1)
    B = torch.cat([torch.linalg.cross(p, Jx, dim=-1), Jx, torch.stack([Bu, Bv], -2)], -1)
    keep = ~clamped
    return (torch.where(keep[..., None], e, 0.0), torch.where(keep[..., None, None], A, 0.0), torch.where(keep[..., None, None], B, 0.0),
            clamped)


def _safe_inv(Hd):
    """oracle/lm.py _safe_inverse for a batch of 3x3 blocks: the inverse, or ZERO where the block is not positive
    definite (its Cholesky pivots, the test of ska_ba.cuh chol3)."""
    h = lambda i, j: Hd[:, i, j]
    a = h(0, 0).sqrt()
    b, d = h(0, 1) / a, h(0, 2) / a
    d1 = h(1, 1) - b * b
    c = d1.sqrt()
    e = (h(1, 2) - d * b) / c
    d2 = h(2, 2) - d * d - e * e
    f = d2.sqrt()
    ok = (h(0, 0) > 0) & (d1 > 0) & (d2 > 0) & torch.isfinite(Hd).flatten(1).all(1)
    z = torch.zeros_like(a)
    M = torch.stack([torch.stack([1 / a, z, z], -1), torch.stack([-b / (a * c), 1 / c, z], -1),
                     torch.stack([(b * e - c * d) / (a * c * f), -e / (c * f), 1 / f], -1)], -2)  # L^-1
    return torch.where(ok[:, None, None], M.transpose(1, 2) @ M, 0.0)


def _damped(Hpp, lam):
    return Hpp + lam * torch.diag_embed(Hpp.diagonal(dim1=1, dim2=2))


def _linearise(e, A, B, w, lam):
    """oracle linearise -> (Hcc (C,P,P), gc (C,P), Sw (PC,PC), bw (PC,), cost)."""
    N, C, _, P = B.shape
    wA, wB = A * w[..., None, None], B * w[..., None, None]
    Hpp = torch.einsum("ncij,ncik->njk", wA, A)
    gp = torch.einsum("ncij,nci->nj", wA, e)
    W = torch.einsum("ncij,ncik->njck", wA, B).reshape(N, 3, P * C)
    Hinv = _safe_inv(_damped(Hpp, lam))
    Sw = torch.einsum("nik,nil->kl", W, Hinv @ W)
    bw = torch.einsum("nik,ni->k", W, (Hinv @ gp[..., None])[..., 0])
    return (torch.einsum("ncij,ncik->cjk", wB, B), torch.einsum("ncij,nci->cj", wB, e), Sw, bw, (w[..., None] * e**2).sum())


def _back_substitute(e, A, B, w, lam, delta):
    """oracle back_substitute: dp = -Hd^-1 (gp + W delta) (N,3) and each point's part of the predicted decrease (N,)."""
    wA = A * w[..., None, None]
    Hpp = torch.einsum("ncij,ncik->njk", wA, A)
    gp = torch.einsum("ncij,nci->nj", wA, e)
    rhs = torch.einsum("ncij,nci->nj", wA, e + torch.einsum("ncik,ck->nci", B, delta))
    diag = Hpp.diagonal(dim1=1, dim2=2)
    dp = -(_safe_inv(_damped(Hpp, lam)) @ rhs[..., None])[..., 0]
    return dp, (dp * (lam * diag * dp - gp)).sum(1)


def _so3_exp_left(w, R):
    """ska_ba.cuh so3_exp_left in float64 numpy: exp([w]x) R."""
    th2 = float(w @ w)
    if th2 < 1e-8:
        A_, B_ = 1.0 - th2 / 6.0, 0.5 - th2 / 24.0
    else:
        th = np.sqrt(th2)
        A_, B_ = np.sin(th) / th, (1.0 - np.cos(th)) / th2
    W = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    return (np.eye(3) + A_ * W + B_ * (W @ W)) @ R


# -------------------------------------------------------------------------------------- the port against the oracle
@pytest.mark.parametrize("rig,T,J", [("2b", 600, 17), ("3", 300, 17), ("8", 200, 70), ("calib", 600, 17)])
def test_reference_port_matches_numpy_oracle(cuda, rig, T, J):
    """The float64 torch port equals oracle/lm.py / oracle/lm_calib.py to 1e-12 relative (linearise, back_substitute,
    cost) at <= 20 k points, with zero-confidence points, points behind camera 0 and a non-zero camera step."""
    calib = rig == "calib"
    if calib:
        clip, R0, t0, th, X0 = lc.make_problem("2b", T, J)
        cam = th
    else:
        clip, R0, t0, X0 = lm.make_problem(rig, T, J)
        cam = clip.K
    C = len(R0)
    X0 = X0.reshape(-1, 3).copy()
    X0[5], X0[777] = [0.0, 0.0, -5.0], [0.3, -0.2, -1.0]
    x = clip.x_fm.astype(float).transpose(0, 2, 1, 3).reshape(-1, C, 2)
    w = clip.conf_fm.astype(float).transpose(0, 2, 1).reshape(-1, C)
    w[11], w[1234] = 0.0, 0.0
    if not calib:  # as in the large cases: no weight on a clamped observation (its 1e9 px/m Jacobian sets every scale)
        w[np.einsum("cb,nb->nc", R0[:, 2], X0) + t0[:, 2] < lm.ZMIN] = 0.0
    rng = np.random.default_rng(3)
    P = 15 if calib else 6
    delta = rng.normal(0.0, 1e-3, (C, P))
    delta[0, :6] = 0.0
    lam = 1e-3
    if calib:
        ref = lc.linearise(X0, R0, t0, th, x, w, lam)
        dp_o, pp_o = lc.back_substitute(X0, R0, t0, th, x, w, lam, delta)
        c_o, n_o = lc.cost_only(X0, R0, t0, th, x, w)
    else:
        ref = lm.linearise(X0, R0, t0, clip.K, x, w, lam)
        dp_o, pp_o = lm.back_substitute(X0, R0, t0, clip.K, x, w, lam, delta)
        c_o, n_o = lm.cost_only(X0, R0, t0, clip.K, x, w)
    g = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(cuda)
    e, A, B, cl = (_rbc if calib else _rb6)(g(X0), g(R0), g(t0), g(cam), g(x))
    Hcc, gc, Sw, bw, cost = (v.cpu().numpy() for v in _linearise(e, A, B, g(w), lam))
    dp, pp = _back_substitute(e, A, B, g(w), lam, g(delta))
    assert int(cl.sum()) == ref.n_clamped == n_o > 0
    for got, want in ((Hcc, ref.Hcc), (gc, ref.gc), (Sw, ref.Sw), (bw, ref.bw), (dp.cpu().numpy(), dp_o)):
        assert _err(got, want, np.abs(want).max()) <= 1e-12
    for got, want in ((float(cost), ref.cost), (float((g(w)[..., None] * e**2).sum()), c_o), (float(pp.sum()), pp_o)):
        assert abs(got - want) <= 1e-12 * abs(want)
    assert np.all(dp.cpu().numpy()[[11, 1234]] == 0.0) and np.all(dp_o[[11, 1234]] == 0.0)


# ------------------------------------------------------------------------------- the reference over an engine's state
def _chunks(eng, slot, pts=1 << 20):
    """(point slice, X (n,3), x (n,C,2), conf (n,C)) in float64 over frame chunks of the engine's own device buffers."""
    T, J, C = eng.T, eng.J, eng.C
    step = max(1, pts // J)
    fm = eng.layout == _cabi.LAYOUT_FRAME_MAJOR
    for a in range(0, T, step):
        b = min(T, a + step)
        if fm:
            x, w = eng.x2d[a:b].permute(0, 2, 1, 3), eng.conf[a:b].permute(0, 2, 1)
        else:
            x, w = eng.x2d[:, a:b].permute(1, 2, 0, 3), eng.conf[:, a:b].permute(1, 2, 0)
        yield (slice(a * J, b * J), eng.Xpp[slot, a * J: b * J].double(), x.reshape(-1, C, 2).double(), w.reshape(-1, C).double())


def _cams(eng, slot, calib):
    """Camera slot `slot` as the kernels hold it: R, t (and theta) rounded to float32; K / k22 rounded (load_cam)."""
    cm, C = eng.cams[slot], eng.C
    r32 = lambda v: v.float().double()
    R, t = r32(cm[:, 0:9]).reshape(C, 3, 3), r32(cm[:, 9:12])
    if calib:
        return R, t, r32(cm[:, 12:21])
    K = torch.zeros((C, 3, 3), dtype=torch.float64, device=cm.device)
    K[:, :2, :] = r32(cm[:, 12:18] / cm[:, 20:21]).reshape(C, 2, 3)
    K[:, 2, 2] = 1.0
    return R, t, K


def _ref_linearise(eng, calib):
    rb = _rbc if calib else _rb6
    cur, lam = int(eng.ctrl[_cabi.BA_CTRL_CUR]), float(np.float32(eng.ctrl[_cabi.BA_CTRL_LAMBDA].item()))
    cams = _cams(eng, 0, calib)
    tot, ncl = None, 0
    for _, X, x, w in _chunks(eng, cur):
        e, A, B, cl = rb(X, *cams, x)
        part = _linearise(e, A, B, w, lam)
        tot = part if tot is None else [u + v for u, v in zip(tot, part)]
        ncl += int(cl.sum())
    Hcc, gc, Sw, bw, cost = (v.cpu().numpy() for v in tot)
    return Hcc, gc, Sw, bw, float(cost), ncl


# ------------------------------------------------------------------------------------------------- per-piece checks
def _s(eng):
    return 1.0 / (float(eng.ctrl[_cabi.BA_CTRL_SUMCONF]) + 1e-6)


def _check_linearise(eng, calib, tc=False):
    red = eng.red.cpu().numpy()
    Hcc_r, gc_r, Sw_r, bw_r, cost_r, ncl_r = _ref_linearise(eng, calib)
    if calib:
        Hcc, gc, bw, Sw, cost, ncl = _unpack_calib(red, 2)
        tol = TOL["lin_calib"]
        for c in range(2):  # natural scale of a parameter pair: sqrt(H_rr H_ss) (px/px focal and px/unit distortion columns)
            sc = np.sqrt(np.diag(Hcc_r[c]))
            _within(f"Hcc[{c}]", _err(Hcc[c] / np.outer(sc, sc), Hcc_r[c] / np.outer(sc, sc), 1.0), tol)
            _within(f"gc[{c}]", _err(gc[c] / sc, gc_r[c] / sc, np.abs(gc_r[c] / sc).max()), tol)
        free = np.ones(30, bool)
        free[:6] = False  # camera 0's extrinsics are the gauge: not in the reduced system
        sc = np.sqrt(np.concatenate([np.diag(Hcc_r[0]), np.diag(Hcc_r[1])]))
        _within("Sw", _err((Sw / np.outer(sc, sc))[np.ix_(free, free)], (Sw_r / np.outer(sc, sc))[np.ix_(free, free)], 1.0), tol)
        _within("bw", _err((bw / sc)[free], (bw_r / sc)[free], max(np.abs(bw_r / sc).max(), np.abs(gc_r.reshape(-1) / sc).max())), tol)
    else:
        Sw, bw, gc, Hcc, cost, ncl = _unpack6(red, eng.C)
        n, tol = 6 * (eng.C - 1), TOL["lin"]
        _within("Hcc", _err(Hcc, Hcc_r[1:], np.abs(Hcc_r[1:]).max()), tol)
        _within("gc", _err(gc, gc_r[1:].reshape(n), np.abs(gc_r).max()), tol)
        _within("Sw", _err(Sw, Sw_r[6:, 6:], np.abs(Sw_r[6:, 6:]).max()), TOL["lin_tc"] if tc else tol)
        _within("bw", _err(bw, bw_r[6:], max(np.abs(bw_r[6:]).max(), np.abs(gc_r).max())), tol)
    _within("cost", abs(cost - cost_r) / cost_r, TOL["cost"])
    assert ncl == ncl_r, (ncl, ncl_r)
    return ncl_r


def _solve_ref6(red, C, lam, s, mask):
    Sw, bw, gc, Hcc, _, _ = _unpack6(red, C)
    n = 6 * (C - 1)
    H = np.zeros((n, n))
    for c in range(C - 1):
        H[6 * c: 6 * c + 6, 6 * c: 6 * c + 6] = Hcc[c]
    hd = np.diag(H).copy()
    S = s * (H + lam * np.diag(hd) - Sw)
    b = s * (bw - gc)
    f = np.array([(mask >> (6 + i)) & 1 for i in range(n)], bool)
    return _masked_cholesky_solve(S, b, f), s * hd, s * gc, f


def _solve_ref_calib(red, lam, s, mask, theta, prior):
    """oracle/lm_calib.py solve_reduced on the GPU's packed system (camera 0's extrinsics dropped)."""
    Hcc, gc, bw, Sw, _, _ = _unpack_calib(red, 2)
    P = _cabi.BA_CALIB_PARAMS
    cols = [(c, r) for c in range(2) for r in range(P) if not (c == 0 and r < 6)]
    idx = np.array([P * c + r for c, r in cols])
    n = len(cols)
    pr, pg = np.zeros(n), np.zeros(n)
    if prior is not None:
        for i, (c, r) in enumerate(cols):
            if r >= 6:
                pr[i] = prior[c, 1, r - 6]
                pg[i] = pr[i] * (theta[c, r - 6] - prior[c, 0, r - 6])
    hd = np.array([s * Hcc[c, r, r] for c, r in cols]) + pr
    g = np.array([s * gc[c, r] for c, r in cols]) + pg
    S = -s * Sw[np.ix_(idx, idx)]
    for i, (ci, ri) in enumerate(cols):
        for j, (cj, rj) in enumerate(cols):
            if ci == cj:
                S[i, j] += s * Hcc[ci, ri, rj]
    S[np.diag_indices(n)] = hd * (1.0 + lam) - s * np.diag(Sw)[idx]
    b = s * bw[idx] - g
    f = np.array([(mask >> (P * c + r)) & 1 for c, r in cols], bool)
    return _masked_cholesky_solve(S, b, f), hd, g, f


def _masked_cholesky_solve(S, b, f):
    S = S.copy()
    S[~f, :] = 0.0
    S[:, ~f] = 0.0
    S[~f, ~f] = 1.0
    L = np.linalg.cholesky(S)
    return np.linalg.solve(L.T, np.linalg.solve(L, np.where(f, b, 0.0)))


def _check_solve(eng, calib, modes):
    """Every free mask in turn; the last one stays in place for the rest of the trial."""
    red, C = eng.red.cpu().numpy(), eng.C
    lam, s = float(eng.ctrl[_cabi.BA_CTRL_LAMBDA]), _s(eng)
    cams0 = eng.cams[0].cpu().numpy()
    prior = eng.prior.cpu().numpy() if calib and eng.prior is not None else None
    for mode in modes:
        eng.mask = ba.calib_free_mask(C, mode) if calib else ba.free_mask(C, mode)
        eng.solve()
        ctrl, delta, cams1 = eng.ctrl.cpu().numpy(), eng.delta.cpu().numpy(), eng.cams[1].cpu().numpy()
        assert ctrl[_cabi.BA_CTRL_OK] == 1.0, mode
        if calib:
            d_ref, hd, g, f = _solve_ref_calib(red, lam, s, eng.mask, cams0[:, 12:21], prior)
            dc = delta.reshape(C, 15)
            assert np.all(dc[0, :6] == 0.0)
            d = np.array([dc[c, r] for c in range(C) for r in range(15) if not (c == 0 and r < 6)])
        else:
            d_ref, hd, g, f = _solve_ref6(red, C, lam, s, eng.mask)
            assert np.all(delta[:6] == 0.0)
            d = delta[6:]
        pred_ref = float(np.sum(f * d_ref * (lam * hd * d_ref - g)))
        if not f.any():  # pose_only: no camera parameter, an identity system
            assert np.all(d == 0.0) and ctrl[_cabi.BA_CTRL_PREDCAM] == 0.0
        else:
            assert np.all(d[~f] == 0.0)
            _within(f"solve {mode} delta", _err(d, d_ref, np.abs(d_ref).max()), TOL["solve"])
            _within(f"solve {mode} pred_cam", abs(ctrl[_cabi.BA_CTRL_PREDCAM] - pred_ref) / abs(pred_ref), TOL["pred_cam"])
        # trial cameras: camera 0 unchanged bit for bit; R <- exp([d_omega]x) R, t <- t + d_t (, theta <- theta + d_theta)
        dc = delta.reshape(C, -1)
        if not calib:
            assert np.array_equal(cams1[0], cams0[0]) and np.array_equal(cams1[:, 12:], cams0[:, 12:]), mode
        else:
            assert np.array_equal(cams1[0, :12], cams0[0, :12]) and np.array_equal(cams1[:, 21:], cams0[:, 21:]), mode
            _within(f"solve {mode} theta", _err(cams1[:, 12:21], cams0[:, 12:21] + dc[:, 6:15], np.abs(cams0[:, 12:21]).max()), TOL["cams"])
        R1 = np.stack([_so3_exp_left(dc[c, :3], cams0[c, :9].reshape(3, 3)) for c in range(C)])
        _within(f"solve {mode} R", _err(cams1[:, :9], R1.reshape(C, 9), 1.0), TOL["cams"])
        _within(f"solve {mode} t", _err(cams1[:, 9:12], cams0[:, 9:12] + dc[:, 3:6], np.abs(cams0[:, 9:12]).max()), TOL["cams"])
        if calib and prior is not None:  # prior part of the cost at the current and the trial intrinsics
            for slot, cm in ((_cabi.BA_CTRL_PRIOR_CUR, cams0), (_cabi.BA_CTRL_PRIOR_TRIAL, cams1)):
                ref = float((prior[:, 1] * (cm[:, 12:21] - prior[:, 0]) ** 2).sum())
                assert abs(ctrl[slot] - ref) <= 1e-12 * ref, (slot, ctrl[slot], ref)


def _check_backsub(eng, calib):
    """Every trial point against the reference step from the GPU's own delta (rounded to float32 as the kernel reads
    it); red2 against the trial cost at the GPU's trial points and cameras."""
    rb = _rbc if calib else _rb6
    cur, lam = int(eng.ctrl[_cabi.BA_CTRL_CUR]), float(np.float32(eng.ctrl[_cabi.BA_CTRL_LAMBDA].item()))
    cams, trial = _cams(eng, 0, calib), _cams(eng, 1, calib)
    delta = eng.delta.float().double().reshape(eng.C, -1)
    worst, Ft, pred, pred_abs, ncl, n_still = 0.0, 0.0, 0.0, 0.0, 0, 0
    for sl, X, x, w in _chunks(eng, cur):
        e, A, B, _ = rb(X, *cams, x)
        dp, pp = _back_substitute(e, A, B, w, lam, delta)
        pred += float(pp.sum())
        pred_abs += float(pp.abs().sum())
        Xn32 = eng.Xpp[1 - cur, sl]
        Xn = Xn32.double()
        still = (dp == 0).all(1)  # no factor (nobody observes the point): X kept bit for bit
        assert torch.equal(Xn32[still], eng.Xpp[cur, sl][still])
        n_still += int(still.sum())
        ulp = torch.maximum(X.abs(), Xn.abs()).amax(1) * 2.0**-23
        err = ((Xn - X - dp).abs().amax(1) - ulp).clamp_min(0.0) / dp.abs().amax(1).clamp_min(1e-30)
        worst = max(worst, float(err[~still].max()) if (~still).any() else 0.0)
        e2, _, _, cl2 = rb(Xn, *trial, x)
        Ft += float((w[..., None] * e2**2).sum())
        ncl += int(cl2.sum())
    red2 = eng.red2.cpu().numpy()
    _within("backsub points", worst, TOL["dp"])
    _within("backsub trial cost", abs(red2[0] - Ft) / Ft, TOL["trial"])
    _within("backsub pred points", abs(red2[1] - pred) / pred_abs, TOL["pred_pts"])
    assert red2[2] == ncl, (red2[2], ncl)
    return n_still


def _expected_control(eng, calib):
    """ctrl and the history row that ba_control_kernel / ba_calib_control_kernel must produce from the current state."""
    C = eng.C
    red, red2, ctrl = eng.red.cpu().numpy(), eng.red2.cpu().numpy(), eng.ctrl.cpu().numpy()
    s = 1.0 / (ctrl[_cabi.BA_CTRL_SUMCONF] + 1e-6)
    if calib:
        L = _cabi.calib_red_layout(C)
        blk = [red[L["cam"] + _cabi.BA_CALIB_CAM_BLOCK * c: L["cam"] + _cabi.BA_CALIB_CAM_BLOCK * (c + 1)] for c in range(C)]
        data = sum(float(b[_cabi.calib_tri(15, 15)]) for b in blk)
        n_cl = sum(float(b[153]) for b in blk)
        F, Ft = s * data + ctrl[_cabi.BA_CTRL_PRIOR_CUR], s * red2[0] + ctrl[_cabi.BA_CTRL_PRIOR_TRIAL]
    else:
        L = _cabi.red_layout(C)
        F, Ft, n_cl = s * red[L["cost"]], s * red2[0], red[L["clamp"]]
    pred = ctrl[_cabi.BA_CTRL_PREDCAM] + s * red2[1]
    lam, nu = float(ctrl[_cabi.BA_CTRL_LAMBDA]), float(ctrl[_cabi.BA_CTRL_NU])
    rho = (F - Ft) / pred if pred > 0.0 else 0.0
    accepted = bool(ctrl[_cabi.BA_CTRL_OK] > 0.5 and np.isfinite(Ft) and Ft < F)
    lam1, nu1 = lm.nielsen_update(lam, nu, rho, accepted)
    it = int(ctrl[_cabi.BA_CTRL_ITER])
    row = np.array([it, F, Ft, lam, rho, float(accepted), n_cl, pred])
    after = ctrl.copy()
    after[_cabi.BA_CTRL_LAMBDA], after[_cabi.BA_CTRL_NU] = lam1, nu1
    after[_cabi.BA_CTRL_CUR] = 1.0 - ctrl[_cabi.BA_CTRL_CUR] if accepted else ctrl[_cabi.BA_CTRL_CUR]
    after[_cabi.BA_CTRL_COST] = Ft if accepted else F
    after[_cabi.BA_CTRL_ACCEPTED] = float(accepted)
    after[_cabi.BA_CTRL_ITER] = it + 1
    return after, row, accepted


def _check_control(eng, calib):
    after, row, accepted = _expected_control(eng, calib)
    cams = eng.cams.cpu().numpy()
    eng.control()
    ctrl, hist = eng.ctrl.cpu().numpy(), eng.hist.cpu().numpy()
    np.testing.assert_allclose(ctrl, after, rtol=CTRL_TOL, atol=0)
    np.testing.assert_allclose(hist[int(row[0])], row, rtol=CTRL_TOL, atol=0, equal_nan=True)
    assert np.array_equal(eng.cams[0].cpu().numpy(), cams[1] if accepted else cams[0])  # accept commits the trial cameras
    return accepted


# ------------------------------------------------------------------------------------------------- launch geometry
def _props():
    return torch.cuda.get_device_properties(0)


def _sms():
    return _props().multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


def _ctas_per_sm_ub(threads, smem=0):
    """Upper bound on resident CTAs per SM from the thread and shared-memory limits (registers can only lower it)."""
    p = _props()
    ub = p.max_threads_per_multi_processor // threads
    return min(ub, p.shared_memory_per_multiprocessor // smem) if smem else ub


def _wide_smem(C):  # ska_ba_wide.cu Wide<C>::smem
    n = 6 * (C - 1)
    size = _cabi.red_layout(C)["size"]
    return WIDE_WARPS * n * K_Y_STRIDE * 4 + size * 8 + C * SIZEOF_CAMF


def _calib_smem(C):  # ska_ba_calib.cu Calib<C>::smem
    L = _cabi.calib_red_layout(C)
    return CALIB_WARPS * L["n"] * K_Y_STRIDE * 4 + L["size"] * 8 + C * SIZEOF_CAMC


def _plan(kind, C):
    """kind -> (points per unit, largest grid): a unit is a grid-stride pass of one thread (256-thread kernels) or a
    tile of one CTA (384-point wide / calib tiles, 48-point tensor-core tiles)."""
    sms = _sms()
    if kind == "reg":          # ba_linearize_reg<2>: grid_for, at most 8 resident 256-thread CTAs per SM
        return K_BA_BLOCK, sms * _ctas_per_sm_ub(K_BA_BLOCK)
    if kind == "wide":         # launch_wide: SMs x occupancy of a 384-thread CTA
        return 32 * WIDE_WARPS, sms * _ctas_per_sm_ub(32 * WIDE_WARPS, _wide_smem(C))
    if kind == "tc":           # launch_tc: one CTA per SM
        return K_TC_PTS, sms
    if kind == "calib":        # ba_calib_linearize: SMs x occupancy of a 384-thread CTA
        return 32 * CALIB_WARPS, sms * _ctas_per_sm_ub(32 * CALIB_WARPS, _calib_smem(C))
    raise ValueError(kind)


def _min_units(kind, C, N):
    """The fewest grid-stride passes (threads) or tiles (CTAs) any thread / CTA of the linearisation gets."""
    per, grid = _plan(kind, C)
    units = _cdiv(N, per)
    return units // min(grid, units) if kind != "reg" else N // (min(grid, units) * per)


def _frames_for(kind, C, J, need):
    """Frames so that every thread / CTA gets >= `need` units, with a ragged last tile."""
    per, grid = _plan(kind, C)
    T = _cdiv(need * grid * per, J)
    while (T * J) % per == 0:
        T += 1
    return T


def test_mirrored_kernel_constants_match_the_sources():
    src = {f: (CSRC / f).read_text() for f in ("ska_ba.cuh", "ska_ba_wide.cu", "ska_ba_calib.cu", "ska_ba_calib.cuh")}
    want = [("ska_ba.cuh", r"constexpr int kBaBlock = (\d+);", K_BA_BLOCK), ("ska_ba.cuh", r"constexpr int kFlush = (\d+);", K_FLUSH),
            ("ska_ba.cuh", r"constexpr int kYStride = (\d+);", K_Y_STRIDE),
            ("ska_ba_wide.cu", r"#define SKA_BA_WIDE_WARPS (\d+)", WIDE_WARPS),
            ("ska_ba_wide.cu", r"constexpr int kTcWarps = (\d+);", K_TC_PTS // 4),
            ("ska_ba_wide.cu", r"constexpr int kTcPts = 4 \* kTcWarps;", None),
            ("ska_ba_wide.cu", r"constexpr int kTcFlush = (\d+);", K_TC_FLUSH),
            ("ska_ba_calib.cu", r"#define SKA_BA_CALIB_WARPS (\d+)", CALIB_WARPS),
            ("ska_ba.cuh", r"float R\[9\], t\[3\];\s*float k00, k01, k02, k10, k11, k12;", None),
            ("ska_ba_calib.cuh", r"float R\[9\], t\[3\];\s*float fx, fy, cx, cy, k1, k2, p1, p2, k3;", None)]
    for f, pat, val in want:
        m = re.search(pat, src[f])
        assert m is not None, (f, pat)
        if val is not None:
            assert int(m.group(1)) == val, (f, pat, m.group(1), val)
    # the launch rules the geometry below mirrors
    ba_cu = (CSRC / "ska_ba.cu").read_text()
    for kern in ("ba_linearize_reg", "ba_backsub_kernel"):
        assert f"__launch_bounds__(kBaBlock, 2) {kern}" in ba_cu, kern
    assert "__launch_bounds__(kBaBlock, 2) ba_calib_backsub_kernel" in src["ska_ba_calib.cu"]
    assert "int64_t grid = sms;  // one CTA per SM" in src["ska_ba_wide.cu"]
    assert "if (++since == kFlush || last)" in src["ska_ba_wide.cu"] and "if (++since == kFlush || last)" in src["ska_ba_calib.cu"]


# ------------------------------------------------------------------------------------------------------ large cases
# name -> (rig, J, layout, kind, linearisation units needed (None: the config 3 shape, T = 100 000), engine options)
CASES = {
    "reg_config3": ("2b", 17, "TCJ2", "reg", None, {}),
    "reg_56_per_thread": ("2b", 17, "CTJ2", "reg", 56, {}),
    "wide_c2_two_folds": ("2b", 17, "TCJ2", "wide", K_FLUSH + 1, dict(force_wide=True)),
    "wide_c3": ("3", 17, "TCJ2", "wide", 2 * K_FLUSH + 1, {}),
    "wide_c8": ("8", 70, "TCJ2", "wide", 2 * K_FLUSH + 1, {}),
    "tc_c5": ("5", 17, "TCJ2", "tc", 2 * K_TC_FLUSH + 1, dict(tensor_core=True)),
    "tc_c8": ("8", 70, "TCJ2", "tc", 2 * K_TC_FLUSH + 1, dict(tensor_core=True)),
    "calib_config3": ("2b", 17, "TCJ2", "calib", None, {}),
}


def _edge_points(T, J):
    """(frame, joint) of a few points nobody observes and a few points behind camera 0, the last frame included."""
    nofactor = [(1, 0), (T // 3, 5 % J), (T - 1, J - 1)]
    behind = [(2, 1 % J), (T // 2, 3 % J), (T - 1, 0)]
    return nofactor, behind


def _large_engine(name, cuda):
    rig, J, layout, kind, need, opts = CASES[name]
    calib = kind == "calib"
    C = len(synth.rig(rig)[0])
    T = 100_000 if need is None else _frames_for(kind, C, J, need)
    d = synth.make_clip_device(rig, T, J, cuda, seed=7, layout=layout)
    R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
    K, kw = d["K"], {}
    if calib:
        th = lc.perturb_intrinsics(d["K"])
        K, dist = synth.theta_to_K_dist(th)
        kw = dict(dist=dist, prior_rho=lc.PRIOR_RHO, prior_theta=lc.intr_from_K(d["K"]))
    xvm = d["x2d"] if layout == "CTJ2" else d["x2d"].permute(1, 0, 2, 3).contiguous()
    X0 = api.triangulate_reproject(xvm, K, R0, t0, want=("X",)).X.float().contiguous()
    del xvm
    conf = d["conf"]
    cv = (lambda f, j: conf[f, :, j]) if layout == "TCJ2" else (lambda f, j: conf[:, f, j])
    nofactor, behind = _edge_points(T, J)
    for f, j in nofactor:
        cv(f, j).zero_()
    for f, j in behind:
        X0[f, j] = torch.tensor([0.0, 0.0, -5.0])  # z = -5 in camera 0: loss.py's depth clamp
        if not calib:
            # the 6-parameter engine keeps a clamped observation in the cost with a 1e9 px/m Jacobian that would set the
            # scale of every block compared here: the camera does not see it (conf 0), the clamp is still counted.
            # The calibrating engine excludes clamped observations itself.
            z = torch.from_numpy(R0[:, 2] @ np.array([0.0, 0.0, -5.0]) + t0[:, 2])
            conf_fj = cv(f, j)
            conf_fj[z.to(conf.device) < 0] = 0.0
    eng_cls = ba.CalibratingBundleAdjuster if calib else ba.BundleAdjuster
    eng = eng_cls(d["x2d"], conf, K, R0, t0, X0, layout=layout, max_iters=4, **kw, **opts)
    del d, X0
    return eng, kind, need, calib


@pytest.mark.parametrize("name", list(CASES))
def test_lm_trial_pieces_at_scale(cuda, name):
    eng, kind, need, calib = _large_engine(name, cuda)
    try:
        N, C = eng.N, eng.C
        per, _ = _plan(kind, C)
        units = _min_units(kind, C, N)
        back = N // (min(_plan("reg", C)[1], _cdiv(N, K_BA_BLOCK)) * K_BA_BLOCK)  # backsub: the register path's grid rule
        unit = "points per thread" if kind == "reg" else "tiles per CTA"
        print(f"\n[{name}] N = {N} points ({eng.T} x {eng.J}, C = {C}): >= {units} {unit}, >= {back} backsub points per thread")
        assert N % per != 0  # a ragged last tile
        assert units >= (need or 2)  # the path the case is named for
        if kind == "calib":
            assert units >= K_FLUSH + 1  # at least one intermediate fold
        assert back >= (1 if kind == "tc" else 2)  # the tensor-core cases are too small for a second backsub pass
        # sum of confidences (ba_sum_kernel, at construction)
        sc = float(eng.conf.double().sum())
        _within("sum conf", abs(float(eng.ctrl[_cabi.BA_CTRL_SUMCONF]) - sc) / sc, TOL["sumconf"])
        eng.linearize()
        ncl = _check_linearise(eng, calib, tc=kind == "tc")
        assert ncl >= 3  # the points behind camera 0
        modes = ("intr_only", "extr_focal", "full") if calib else ("pose_only", "pose_cam_t", "full")
        _check_solve(eng, calib, modes)
        eng.backsub()
        assert _check_backsub(eng, calib) >= 3  # the points nobody observes
        assert _check_control(eng, calib)  # the first trial from a perturbed start is accepted
    finally:
        del eng
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------- small crafted problems
def _small_engine(calib, cuda):
    if calib:
        clip, R0, t0, th, X0 = lc.make_problem("2b", 60, 17)
        K, dist = synth.theta_to_K_dist(th)
        kw = dict(dist=dist, prior_rho=lc.PRIOR_RHO, prior_theta=lc.intr_from_K(clip.K))
        cls = ba.CalibratingBundleAdjuster
    else:
        clip, R0, t0, X0 = lm.make_problem("3", 60, 17)
        K, kw, cls = clip.K, {}, ba.BundleAdjuster
    x, c = torch.from_numpy(clip.x_fm).to(cuda), torch.from_numpy(clip.conf_fm).to(cuda)
    return cls(x, c, K, R0, t0, torch.from_numpy(X0).to(cuda), max_iters=4, **kw)


@pytest.mark.parametrize("calib", [False, True], ids=["six_param", "calib"])
def test_indefinite_reduced_system_gives_no_step_and_a_rejection(cuda, calib):
    """A reduced system that is not positive definite (crafted `red`: one negative camera diagonal): ctrl[kCtrlOk] = 0,
    delta all zeros, trial cameras = current cameras, and the controller rejects the trial although the points alone
    lower the cost."""
    eng = _small_engine(calib, cuda)
    eng.linearize()
    if calib:
        o = _cabi.calib_red_layout(2)["cam"] + _cabi.calib_tri(6, 6)  # camera 0's fx diagonal: parameter 0
    else:
        o = _cabi.red_layout(eng.C)["hcc"]  # camera 1's first diagonal entry
    eng.red[o] = -1e3 * eng.red[o].abs()
    eng.solve()
    assert float(eng.ctrl[_cabi.BA_CTRL_OK]) == 0.0
    assert torch.all(eng.delta == 0.0)
    assert torch.equal(eng.cams[1], eng.cams[0])
    eng.backsub()
    after, row, accepted = _expected_control(eng, calib)
    assert not accepted and row[2] < row[1]  # the trial cost is lower: only the ok flag rejects it
    assert not _check_control(eng, calib)
    assert float(eng.ctrl[_cabi.BA_CTRL_LAMBDA]) == 2.0 * 1e-3


@pytest.mark.parametrize("calib", [False, True], ids=["six_param", "calib"])
def test_control_branches(cuda, calib):
    """ba_control_kernel / ba_calib_control_kernel on crafted red2 / ctrl from one real trial: accept, reject (higher
    trial cost, non-finite trial cost, failed solve), and a predicted decrease <= 0 (rho = 0) with either decision."""
    eng = _small_engine(calib, cuda)
    eng.linearize()
    eng.solve()
    eng.backsub()
    s = _s(eng)
    snap = [t.clone() for t in (eng.ctrl, eng.cams, eng.hist, eng.red2)]
    F_raw = float(eng.red2[0])  # raw trial cost (sum conf x err^2)
    if calib:
        L = _cabi.calib_red_layout(2)
        data = sum(float(eng.red[L["cam"] + _cabi.BA_CALIB_CAM_BLOCK * c + _cabi.calib_tri(15, 15)]) for c in range(2))
    else:
        data = float(eng.red[_cabi.red_layout(eng.C)["cost"]])
    neg_pred = -(float(eng.ctrl[_cabi.BA_CTRL_PREDCAM]) + 1.0) / s  # point part that makes the total -1
    crafted = {
        "accept": ({}, {}, True),
        "higher trial cost": ({0: 2.0 * data + 1.0}, {}, False),
        "nan trial cost": ({0: float("nan")}, {}, False),
        "failed solve": ({}, {_cabi.BA_CTRL_OK: 0.0}, False),
        "pred <= 0, accepted": ({1: neg_pred}, {}, True),
        "pred <= 0, rejected": ({0: 2.0 * data + 1.0, 1: neg_pred}, {}, False),
    }
    assert F_raw < data
    for what, (r2, ct, want) in crafted.items():
        for t, v in zip((eng.ctrl, eng.cams, eng.hist, eng.red2), snap):
            t.copy_(v)
        for k, v in r2.items():
            eng.red2[k] = v
        for k, v in ct.items():
            eng.ctrl[k] = v
        after, row, accepted = _expected_control(eng, calib)
        assert accepted == want, what
        if what.startswith("pred"):
            assert row[7] <= 0.0 and row[4] == 0.0, what
        assert _check_control(eng, calib) == want, what
