"""fp64 specification of the ROBUST regularised LM (Huber / Cauchy on the reprojection group), built on oracle/lm_reg.py,
which stays the specification of the L2 solver and is not changed, with the rho / omega of tests/oracle_robust.py.

The loss applies to the reprojection group only.  Its term is c_r sum conf rho(s), s = |pi(R X + t) - x|^2, with
c_r = w_r / (sum conf + 1e-6) from the raw confidences; bone length, pose temporal, smoothness and baseline stay squared.
The step is lm_reg's with every reprojection row weighted by conf omega(s), omega at the current point and not
differentiated (lm_reg.jacobian puts conf into those rows only), so g = grad(F) / 2 with the bone / baseline means
detached, and the predicted decrease, the gain ratio and the accept rule keep their meaning.  Depth-clamped observations
keep their residual, as in lm_reg, and are weighted by omega of it.  With "l2" (omega = 1, rho = s exactly), and with Huber
whose every residual lies inside d, run_lm_reg reproduces lm_reg.run_lm bit for bit.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import lm_reg
from tests.oracle_robust import robust


def reg_weights(X, R, t, K, x2d, loss="l2", scale=None):
    """(rho, omega, s) of every observation (T,C,J) at one point, s = |pi(R X + t) - x|^2 as lm_reg.cost_terms computes it."""
    _, uv, _, _ = lm_reg.project(X, R, t, K)
    s = ((uv - x2d) ** 2).sum(-1)
    rho, om = robust(s, loss, scale)
    return rho, om, s


def reg_cost_terms(X, R, t, K, x2d, conf, coef, loss="l2", scale=None):
    """lm_reg.cost_terms with the reprojection term c_r sum conf rho(s)."""
    terms, ncl = lm_reg.cost_terms(X, R, t, K, x2d, conf, coef)
    rho, _, _ = reg_weights(X, R, t, K, x2d, loss, scale)
    terms["reproj"] = coef["reproj"] * float((conf * rho).sum())
    return terms, ncl


def reg_normal_system(X, R, t, K, x2d, conf, coef, mode, loss="l2", scale=None):
    """lm_reg.normal_system with the reprojection rows weighted by conf omega (coef stays that of the raw confidences)."""
    _, om, _ = reg_weights(X, R, t, K, x2d, loss, scale)
    return lm_reg.normal_system(X, R, t, K, x2d, conf * om, coef, mode)


def run_lm_reg(X0, R0, t0, K, x2d, conf, num_iters=10, mode="pose_only", weights=None, lam0=lm_reg.LAMBDA0, loss="l2", scale=None,
               solver="direct", cg_tol=1e-8, cg_max_iter=500):
    """oracle/lm_reg.py run_lm with the robust reprojection cost and step (same arguments, same history rows)."""
    if mode not in lm_reg.MODES:
        raise ValueError(f"unknown mode {mode!r}")
    X = np.asarray(X0, float).copy()
    T, J, _ = X.shape
    R = np.asarray(R0, float)
    t = np.asarray(t0, float)
    if R.ndim == 3:
        R, t = np.broadcast_to(R, (T,) + R.shape).copy(), np.broadcast_to(t, (T,) + t.shape).copy()
    R, t = R.copy(), t.copy()
    C = R.shape[1]
    K = np.broadcast_to(np.asarray(K, float), (C, 3, 3))
    x2d, conf = np.asarray(x2d, float), np.asarray(conf, float)
    coef = lm_reg.coefficients(T, J, C, float(conf.sum()), weights)
    lam, nu = float(lam0), 2.0
    hist = []
    blocks = lm_reg.jacobi_blocks(T, J, C, mode) if solver == "pcg" else None
    for it in range(num_iters):
        terms, ncl = reg_cost_terms(X, R, t, K, x2d, conf, coef, loss, scale)
        F = sum(terms.values())
        H, g, free, r2 = reg_normal_system(X, R, t, K, x2d, conf, coef, mode, loss, scale)
        D = H.diagonal()
        if solver == "direct":
            d_free = spla.splu((H + lam * sp.diags(D)).tocsc()).solve(-g)
            cg_iters = 0
        else:
            d_free, cg_iters = lm_reg.pcg(H, D, lam, g, blocks, cg_tol, cg_max_iter)
        delta = np.zeros(free.shape[0])
        delta[free] = d_free
        pred = float(d_free @ (lam * D * d_free - g))
        Xn, Rn, tn = lm_reg.apply_step(X, R, t, delta, mode)
        tterms, _ = reg_cost_terms(Xn, Rn, tn, K, x2d, conf, coef, loss, scale)
        Ft = sum(tterms.values())
        rho = (F - Ft) / pred if pred > 0 else 0.0
        accepted = bool(np.isfinite(Ft) and Ft < F)
        row = dict(iter=it, cost=F, trial_cost=Ft, lam=lam, rho=rho, accepted=accepted, pred=pred, n_clamped=ncl, cg_iters=cg_iters, r2=r2)
        row.update(terms)
        hist.append(row)
        if accepted:
            lam, nu = lam * max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3), 2.0
            X, R, t = Xn, Rn, tn
        else:
            lam, nu = lam * nu, 2.0 * nu
    return R, t, X, hist
