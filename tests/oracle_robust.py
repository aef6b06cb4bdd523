"""fp64 specification of the ROBUST Schur-LM bundle adjustments (Huber / Cauchy), built on oracle/lm.py and
oracle/lm_calib.py, which stay the specification of the L2 solvers and are not changed.

With s = e_u^2 + e_v^2 (px^2), d > 0 the scale in pixels and w = conf / (sum conf + 1e-6):
    loss     rho(s)                                   omega(s) = rho'(s)
    l2       s                                        1
    huber    s (s <= d^2), 2 d sqrt(s) - d^2          1 (s <= d^2), d / sqrt(s)
    cauchy   d^2 ln(1 + s / d^2)                      1 / (1 + s / d^2)
Cost      F = sum w rho(s)  (+ the intrinsics prior in the calibrating form).
Step      iteratively reweighted Gauss-Newton: every sum of the L2 step (Hpp, gp, W, Hcc, gc, Sw, bw) uses w omega(s),
          omega evaluated at the current state and not differentiated, so g = grad(F) / 2 holds exactly and the Nielsen
          gain ratio, its predicted decrease and the accept rule keep their meaning.
Trial     sum w rho(s_trial).
Clamped   6-parameter form: loss.py's depth clamp; a clamped observation is weighted by omega of its (huge) error.
          Calibrating form: still excluded (zero residual, rho(0) = 0).
The cost is evaluated as sum (w omega) s + sum w (rho - omega s) - the split of the calibrating kernel's slot 154 - so
that Huber with every residual inside d reproduces the L2 numbers bit for bit (rho = s and omega = 1 exactly).
"""
from __future__ import annotations

import numpy as np

from oracle import lm
from oracle import lm_calib as lc

LOSSES = ("l2", "huber", "cauchy")


def robust(s, loss="l2", scale=None):
    """(rho, omega) of squared pixel errors s (any shape)."""
    s = np.asarray(s, float)
    if loss == "l2":
        return s, np.ones_like(s)
    if loss not in LOSSES:
        raise ValueError(f"unknown loss {loss!r}")
    d = float(scale)
    if not d > 0:
        raise ValueError("a robust loss needs scale > 0")
    if loss == "huber":
        inl = s <= d * d
        root = np.sqrt(np.where(inl, 1.0, s))
        return np.where(inl, s, 2.0 * d * root - d * d), np.where(inl, 1.0, d / root)
    q = s / (d * d)
    return d * d * np.log1p(q), 1.0 / (1.0 + q)


def _split_cost(w, om, rho, s):
    """sum (w omega) s + sum w (rho - omega s), with s (N,C) and the L2 summation order of the first term."""
    return float(((w * om) * s).sum() + (w * (rho - om * s)).sum())


# ------------------------------------------------------------------------------------------- 6-parameter (oracle/lm.py)
def weights(X, R, t, K, x2d, w, loss="l2", scale=None):
    """(rho, omega, e) at the current state."""
    e, _, _, _ = lm.residual_blocks(X, R, t, K, x2d, w)
    s = (e**2).sum(-1)
    rho, om = robust(s, loss, scale)
    return rho, om, e


def linearise(X, R, t, K, x2d, w, lam, keep_points=False, loss="l2", scale=None) -> lm.Linearisation:
    rho, om, e = weights(X, R, t, K, x2d, w, loss, scale)
    lin = lm.linearise(X, R, t, K, x2d, w * om, lam, keep_points)
    lin.cost = float(((w * om)[..., None] * e**2).sum() + (w * (rho - om * (e**2).sum(-1))).sum())
    return lin


def back_substitute(X, R, t, K, x2d, w, lam, delta_c, loss="l2", scale=None):
    _, om, _ = weights(X, R, t, K, x2d, w, loss, scale)
    return lm.back_substitute(X, R, t, K, x2d, w * om, lam, delta_c)


def cost_only(X, R, t, K, x2d, w, loss="l2", scale=None):
    Xc = np.einsum("cab,nb->nca", R, X) + t[None]
    Z = np.maximum(Xc[..., 2], lm.ZMIN)
    x, y = Xc[..., 0] / Z, Xc[..., 1] / Z
    Kb = K[None]
    u = Kb[..., 0, 0] * x + Kb[..., 0, 1] * y + Kb[..., 0, 2]
    v = Kb[..., 1, 0] * x + Kb[..., 1, 1] * y + Kb[..., 1, 2]
    d = (u - x2d[..., 0]) ** 2 + (v - x2d[..., 1]) ** 2
    rho, om = robust(d, loss, scale)
    return _split_cost(w, om, rho, d), int((Xc[..., 2] < lm.ZMIN).sum())


def dense_step(X, R, t, K, x2d, w, lam, free, loss="l2", scale=None):
    _, om, _ = weights(X, R, t, K, x2d, w, loss, scale)
    return lm.dense_step(X, R, t, K, x2d, w * om, lam, free)


def run_lm(X0, R0, t0, K, x2d, conf, num_iters=20, mode="full", lam0=lm.LAMBDA0, shards=1, loss="l2", scale=None):
    """oracle/lm.py run_lm with the robust cost and step (same arguments, same history rows)."""
    T, J, _ = X0.shape
    C = R0.shape[0]
    X = np.asarray(X0, float).reshape(T * J, 3).copy()
    R, t = np.asarray(R0, float).copy(), np.asarray(t0, float).copy()
    K = np.asarray(K, float)
    x = np.asarray(x2d, float).transpose(0, 2, 1, 3).reshape(T * J, C, 2)
    cf = np.asarray(conf, float).transpose(0, 2, 1).reshape(T * J, C)
    w = cf / (cf.sum() + 1e-6)
    free = lm.free_mask(C, mode)
    bounds = np.linspace(0, T, shards + 1).astype(int) * J
    parts = [slice(bounds[i], bounds[i + 1]) for i in range(shards)]
    lam, nu = float(lam0), 2.0
    history = []
    for it in range(num_iters):
        lin = None
        for s in parts:
            li = linearise(X[s], R, t, K, x[s], w[s], lam, loss=loss, scale=scale)
            lin = li if lin is None else lin + li
        dc, pred_cam, ok = lm.solve_reduced(lin, lam, free)
        Rn, tn = lm.apply_camera_step(R, t, dc)
        Xn = X.copy()
        pred, Ft = pred_cam, 0.0
        for s in parts:
            dp, pp = back_substitute(X[s], R, t, K, x[s], w[s], lam, dc, loss, scale)
            Xn[s] = X[s] + dp
            pred += pp
            Ft += cost_only(Xn[s], Rn, tn, K, x[s], w[s], loss, scale)[0]
        F = lin.cost
        rho = (F - Ft) / pred if pred > 0 else 0.0
        accepted = bool(ok and np.isfinite(Ft) and Ft < F)
        history.append(dict(iter=it, cost=F, trial_cost=Ft, lam=lam, rho=rho, accepted=accepted, n_clamped=lin.n_clamped, pred=pred))
        lam, nu = lm.nielsen_update(lam, nu, rho, accepted)
        if accepted:
            X, R, t = Xn, Rn, tn
    return R, t, X.reshape(T, J, 3), history


# ------------------------------------------------------------------------------------ calibrating (oracle/lm_calib.py)
def calib_weights(X, R, t, th, x2d, w, loss="l2", scale=None):
    e, _, _, _ = lc.residual_blocks(X, R, t, th, x2d)  # excluded observations: e = 0, rho(0) = 0
    s = (e**2).sum(-1)
    rho, om = robust(s, loss, scale)
    return rho, om, e


def calib_linearise(X, R, t, th, x2d, w, lam, loss="l2", scale=None) -> lc.Linearisation:
    rho, om, e = calib_weights(X, R, t, th, x2d, w, loss, scale)
    lin = lc.linearise(X, R, t, th, x2d, w * om, lam)
    lin.cost = float(((w * om)[..., None] * e**2).sum() + (w * (rho - om * (e**2).sum(-1))).sum())
    return lin


def calib_back_substitute(X, R, t, th, x2d, w, lam, delta, loss="l2", scale=None):
    _, om, _ = calib_weights(X, R, t, th, x2d, w, loss, scale)
    return lc.back_substitute(X, R, t, th, x2d, w * om, lam, delta)


def calib_cost_only(X, R, t, th, x2d, w, loss="l2", scale=None):
    uv, clamped = lc.project(X, R, t, th)
    dv = np.where(clamped[..., None], 0.0, uv - x2d)
    d = (dv**2).sum(-1)
    rho, om = robust(d, loss, scale)
    return float(((w * om)[..., None] * dv**2).sum() + (w * (rho - om * d)).sum()), int(clamped.sum())


def calib_dense_step(X, R, t, th, x2d, w, lam, free, th0, rho_prior, loss="l2", scale=None):
    _, om, _ = calib_weights(X, R, t, th, x2d, w, loss, scale)
    return lc.dense_step(X, R, t, th, x2d, w * om, lam, free, th0, rho_prior)


def calib_run_lm(X0, R0, t0, th0, x2d, conf, num_iters=20, free=None, lam0=lm.LAMBDA0, prior_theta=None, prior_rho=None, shards=1,
                 loss="l2", scale=None):
    """oracle/lm_calib.py run_lm with the robust cost and step (same arguments, same history rows)."""
    T, J, _ = X0.shape
    C = R0.shape[0]
    X = np.asarray(X0, float).reshape(T * J, 3).copy()
    R, t, th = np.asarray(R0, float).copy(), np.asarray(t0, float).copy(), np.asarray(th0, float).copy()
    x = np.asarray(x2d, float).transpose(0, 2, 1, 3).reshape(T * J, C, 2)
    cf = np.asarray(conf, float).transpose(0, 2, 1).reshape(T * J, C)
    w = cf / (cf.sum() + 1e-6)
    free = lc.free_mask(C) if free is None else np.asarray(free, bool).copy()
    free[0, :6] = False
    pth = th.copy() if prior_theta is None else np.asarray(prior_theta, float)
    rp = np.zeros((C, lc.NI)) if prior_rho is None else np.broadcast_to(np.asarray(prior_rho, float), (C, lc.NI)).copy()
    bounds = np.linspace(0, T, shards + 1).astype(int) * J
    parts = [slice(bounds[i], bounds[i + 1]) for i in range(shards)]
    lam, nu = float(lam0), 2.0
    history = []
    for it in range(num_iters):
        lin = None
        for s in parts:
            li = calib_linearise(X[s], R, t, th, x[s], w[s], lam, loss, scale)
            lin = li if lin is None else lin + li
        dc, pred_cam, ok = lc.solve_reduced(lin, lam, free, th, pth, rp)
        Rn, tn, thn = lc.apply_camera_step(R, t, th, dc)
        Xn = X.copy()
        pred, Ft = pred_cam, 0.0
        for s in parts:
            dp, pp = calib_back_substitute(X[s], R, t, th, x[s], w[s], lam, dc, loss, scale)
            Xn[s] = X[s] + dp
            pred += pp
            Ft += calib_cost_only(Xn[s], Rn, tn, thn, x[s], w[s], loss, scale)[0]
        F = lin.cost + lc.prior_cost(th, pth, rp)
        Ft += lc.prior_cost(thn, pth, rp)
        gain = (F - Ft) / pred if pred > 0 else 0.0
        accepted = bool(ok and np.isfinite(Ft) and Ft < F)
        history.append(dict(iter=it, cost=F, trial_cost=Ft, lam=lam, rho=gain, accepted=accepted, n_clamped=lin.n_clamped, pred=pred))
        lam, nu = lm.nielsen_update(lam, nu, gain, accepted)
        if accepted:
            X, R, t, th = Xn, Rn, tn, thn
    return R, t, th, X.reshape(T, J, 3), history
