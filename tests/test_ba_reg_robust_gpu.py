"""GPU parity of the robust (Huber / Cauchy) regularised LM kernels (csrc/ska_ba_reg.cu through
ska_ba_reg_{cost,linearize,cg}_robust_f64) against the fp64 specification (tests/oracle_robust_reg.py run_lm_reg):

  pieces       one trial a launch at a time at the sizes where the grid-stride loops wrap, against
               tests/test_ba_reg_scale_gpu.py's float64 reference fed conf * omega at the current point (that file's
               tolerances), and the cost against c_r sum conf rho;
  trajectories against run_lm_reg at G12-like sizes with 5 % outliers (tests/test_ba_reg_gpu.py's tolerance);
  bit identity Huber with every residual inside d equals L2, the robust entry points with SKA_BA_LOSS_L2 equal the L2
               entry points, graph replay equals eager;
  shards       a frame-sharded robust solve emulated on one GPU follows the unsharded trajectory;
  outliers     per-frame cameras of the config-3 rig under 5 % gross 2D outliers."""
import pytest
import torch

from oracle import lm_reg
from skiing_analysis_pytorch_b200 import _cabi, ba_reg, synth
from tests import oracle_robust_reg as orb
from tests.test_ba_reg_gpu import COST_TOL, _check
from tests.test_ba_reg_scale_gpu import (CASES, SC_DONE, SC_NCL, SC_TERM, SUM_CLAMP, SUM_PRED, SUM_REPROJ, TOL, TRAJ_X_TOL, ZMIN,
                                         _FREE, _allreduce, _bounds, _cost, _err, _interior, _lockstep_trial, _point, _pt_passes,
                                         _solver, _term_err, _term_tol, _warp_passes, RegRef, clips)  # noqa: F401  (fixture)
from tests.test_oracle_lm_reg_robust import OUTLIER_ITERS, OUTLIER_SPEC, cam1_errors, outlier_problem

pytestmark = pytest.mark.gpu

ROBUST = [("huber", 3.0), ("cauchy", 3.0)]
SHARD_TRAJ_TOL = 1e-14  # lockstep trials against the unsharded solve: cost and trial cost, relative
# The pieces use tests/test_ba_reg_scale_gpu.py's TOL except for four entries measured against a normaliser that the robust
# weights shrink while the absolute rounding stays: the largest |g|, |D| and |y| (under L2 the large residuals of the
# drifting frames set them; here they are down-weighted) and each damped point block's largest entry (a point whose
# observations are down-weighted is held mostly by the bone and temporal terms).  Largest errors measured on one NVIDIA
# B200 (1000 W power limit) over the six cases: g 1.7e-14, D 4.9e-15, y 3.5e-15 (all pose_only), pinv 2.3e-14; the bounds
# keep the scale test's ~3x margin.  The other pieces stay well inside the L2 bounds (z <= 4.8e-12, r.z / p.y <= 1.6e-16).
PIECE_TOL = dict(TOL, g=5e-14, D=1.5e-14, y=1e-14, pinv=7e-14)


def _sq_errors(X, R, t, K, x2d):
    """s = |pi(R X + t) - x|^2 of every observation (T,C,J)."""
    Xc = torch.einsum("tcab,tjb->tcja", R, X) + t[:, :, None]
    iz = 1.0 / Xc[..., 2].clamp_min(ZMIN)
    xn, yn = Xc[..., 0] * iz, Xc[..., 1] * iz
    k = K[None, :, None]
    du = k[..., 0, 0] * xn + k[..., 0, 1] * yn + k[..., 0, 2] - x2d[..., 0]
    dv = k[..., 1, 0] * xn + k[..., 1, 1] * yn + k[..., 1, 2] - x2d[..., 1]
    return du * du + dv * dv


def _robust_state(s, loss, d):
    """(omega, rho) of squared errors s with the kernels' expressions: Huber d rsqrt(s), Cauchy 1 / (1 + s (1/d^2))."""
    if loss == "huber":
        inl = s <= d * d
        return torch.where(inl, 1.0, d * torch.rsqrt(s)), torch.where(inl, s, 2.0 * d * s.sqrt() - d * d)
    q = s * (1.0 / (d * d))
    return 1.0 / (1.0 + q), d * d * torch.log1p(q)


# ------------------------------------------------------------------------------------------------------ pieces
@pytest.mark.parametrize("loss", ["huber", "cauchy"])
@pytest.mark.parametrize("name", ["A_full_3_warp_passes", "B_pose_cam_t", "C_pose_only_3_point_passes"])
def test_lm_trial_pieces_at_scale(cuda, clips, name, loss):
    """d is the median residual of the start: half of the observations are down-weighted, Huber runs both branches."""
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    C = clip["R"].shape[1]
    K, x2d, conf = clip["K"], clip["x2d"].double(), clip["conf"].double()
    sq = _sq_errors(clip["X0"], clip["R"], clip["t"], torch.as_tensor(K, dtype=torch.float64, device=cuda).view(C, 3, 3), x2d)
    d = float(sq.median().sqrt())
    s = _solver(clip, mode, loss=loss, loss_scale=d)
    assert (_pt_passes(T, J) >= 2) if mode == "pose_only" else (_warp_passes(T) >= 2)
    k = _cabi
    lam = float(s.sc[k.BA_REG_SC_LAMBDA])
    X, R, t = _point(s)
    K = s.K.view(C, 3, 3)
    coef = lm_reg.coefficients(T, J, C, float(conf.sum()), None)  # c_r from the raw confidences
    om, rho = _robust_state(_sq_errors(X, R, t, K, x2d), loss, d)
    frac = float((om < 1.0).double().mean())
    print(f"\n[{name}, {loss} d = {d:.3f} px] T = {T}, {mode}: omega < 1 for {100 * frac:.1f} % of the observations")
    over = []

    def _within(what, err, tol):  # every piece is measured before the test fails
        print(f"    {what:<30s} {err:.3e}  (tol {tol:.1e})")
        if not err <= tol:
            over.append((what, err, tol))

    if loss == "huber":
        assert 0.3 < frac < 0.7
    ref = RegRef(X, R, t, K, x2d, conf * om, coef, mode)
    # ---- cost(0): the reprojection term is c_r sum conf rho; every other sum is the L2 solver's
    s.cost(0)
    s.finish_cost(0)
    terms, raw, ncl = _cost(X, R, t, K, x2d, conf, coef)
    raw[SUM_REPROJ] = (conf * rho).sum()
    terms["reproj"] = coef["reproj"] * float(raw[SUM_REPROJ])
    cols = [c for c in range(_cabi.BA_REG_SUMS) if c not in (SUM_PRED, 7)]
    got, want = s.sums[0, cols], raw[cols]
    assert torch.all(got[want == 0.0] == 0.0)
    _within("cost(0) raw sums", float(((got - want).abs() / want.abs().clamp_min(1e-300)).max()), PIECE_TOL["sums"])
    for i, term in enumerate(lm_reg.TERMS):
        _within(f"cost(0) {term}", _term_err(float(s.sc[SC_TERM + i]), term, terms, raw, coef), PIECE_TOL[_term_tol(term)])
    F = sum(terms.values())
    _within("cost(0) F", abs(s.cost_value - F) / F, PIECE_TOL["cost"])
    assert int(s.sc[SC_NCL].item()) == ncl == int(s.sums[0, SUM_CLAMP].item())
    # ---- linearize: g, D
    s.linearize()
    g_ref, D_ref = ref.gradient(), ref.diag()
    _within("linearize g", _err(_interior(s, 0), g_ref, g_ref.abs().max()), PIECE_TOL["g"])
    _within("linearize D", _err(_interior(s, 1), D_ref, D_ref.abs().max()), PIECE_TOL["D"])
    pinv_ref = ref.point_inverses(lam)
    _within("linearize pinv", float(((s.pinv - pinv_ref).abs() / pinv_ref.abs().amax(-1, keepdim=True)).max()), PIECE_TOL["pinv"])
    # ---- CG_BEGIN: z = M^-1 r (the preconditioner recomputes omega from the observations)
    s.cg(k.BA_REG_CG_BEGIN)
    r = _interior(s, 3)
    z_ref = ref.precond(r, lam)
    _within("BEGIN z", _err(_interior(s, 4), z_ref, z_ref.abs().max()), PIECE_TOL["z"])
    rz = float((r * z_ref).sum())
    _within("BEGIN r.z", abs(float(s.dot) - rz) / abs(rz), PIECE_TOL["dot"])
    # ---- CG_MATVEC with a seeded p
    gen = torch.Generator(device=cuda).manual_seed(5)
    fmask = torch.cat([torch.ones(3 * J, dtype=torch.bool, device=cuda), torch.tensor(_FREE[mode], device=cuda).repeat(C)])
    p = torch.randn(T, 3 * J + 6 * C, generator=gen, device=cuda, dtype=torch.float64) * fmask
    s.vec[5, 1:-1] = p
    s.sc[SC_DONE] = 0.0
    s.cg(k.BA_REG_CG_MATVEC)
    y_ref = ref.matvec(p, lam)
    _within("MATVEC y", _err(_interior(s, 6), y_ref, y_ref.abs().max()), PIECE_TOL["y"])
    py = float((p * y_ref).sum())
    _within("MATVEC p.y", abs(float(s.dot) - py) / abs(py), PIECE_TOL["dot"])
    assert not over, over


# ------------------------------------------------------------------------------------------------------ trajectories
def _g12_outliers(name, frac=0.05):
    rig, T, J, mode = lm_reg.G12_CASES[name]
    clip, R, t, X0 = lm_reg.make_problem(rig, T, J, cam_jitter=0.01)
    if frac:
        synth.inject_outliers(clip.x_vm, J, frac, seed=7)
    return clip, R, t, X0, mode


def _gpu_solver(clip, R, t, X0, mode, cuda, **kw):
    return ba_reg.RegularisedBundleAdjuster(torch.from_numpy(clip.x_fm).to(cuda), torch.from_numpy(clip.conf_fm).to(cuda), clip.K, R, t, X0,
                                            mode=mode, max_iters=16, cg_iters=80, **kw)


@pytest.mark.parametrize("loss,d", ROBUST)
@pytest.mark.parametrize("name", ["c3_pose", "c3_full", "c4_full"])
def test_trajectory_matches_spec(cuda, name, loss, d):
    clip, R, t, X0, mode = _g12_outliers(name)
    s = _gpu_solver(clip, R, t, X0, mode, cuda, loss=loss, loss_scale=d)
    n = 6
    s.run(n)
    hist = s.history
    ref = orb.run_lm_reg(X0, R, t, clip.K, clip.x_fm.astype(float), clip.conf_fm.astype(float), num_iters=n, mode=mode, loss=loss,
                         scale=d)[3]
    n_cmp = _check(hist, ref, n)
    assert n_cmp >= 3
    for k in range(n_cmp):
        for term in lm_reg.TERMS:
            assert abs(hist[k][term] - ref[k][term]) <= COST_TOL * max(ref[k]["cost"] * 1e-3, abs(ref[k][term])), (k, term)


# ------------------------------------------------------------------------------------------------------ bit identity
def _buffers(s):
    return [v.clone() for v in (s.Xh, s.Ch, s.vec, s.pinv, s.sc, s.sums, s.hist) + ((s.lfac,) if s.lfac is not None else ())]


@pytest.mark.parametrize("name", ["c3_pose", "c3_full"])
def test_huber_inside_scale_is_bit_identical_to_l2(cuda, name):
    clip, R, t, X0, mode = _g12_outliers(name, frac=0.0)
    a = _gpu_solver(clip, R, t, X0, mode, cuda)
    b = _gpu_solver(clip, R, t, X0, mode, cuda, loss="huber", loss_scale=1e4)  # every residual of this clip is < 1e3 px
    a.run(5)
    b.run(5)
    assert a.history == b.history
    for u, v in zip(_buffers(a), _buffers(b)):
        assert torch.equal(u, v)


class _L2EntryPoints(ba_reg.RegularisedBundleAdjuster):
    """The solver driven through ska_ba_reg_cost_f64 / _linearize_f64 / _cg_f64, the L2 solver's entry points."""

    def cost(self, which):
        self._call(self.lib.ska_ba_reg_cost_f64, which)

    def linearize(self):
        self._call(self.lib.ska_ba_reg_linearize_f64)

    def cg(self, op):
        self._call(self.lib.ska_ba_reg_cg_f64, op)


@pytest.mark.parametrize("name", ["c3_pose", "c3_full"])
def test_robust_entry_points_with_l2_equal_the_l2_entry_points(cuda, name):
    clip, R, t, X0, mode = _g12_outliers(name)
    a = _gpu_solver(clip, R, t, X0, mode, cuda)
    assert a.loss_id == _cabi.BA_LOSS_L2
    b = _L2EntryPoints(torch.from_numpy(clip.x_fm).to(cuda), torch.from_numpy(clip.conf_fm).to(cuda), clip.K, R, t, X0, mode=mode, max_iters=16,
                       cg_iters=80)
    a.run(4)
    b.run(4)
    assert a.history == b.history
    for u, v in zip(_buffers(a), _buffers(b)):
        assert torch.equal(u, v)


@pytest.mark.parametrize("loss,d", ROBUST)
def test_graph_replay_equals_eager(cuda, loss, d):
    clip, R, t, X0, mode = _g12_outliers("c3_full")
    runs = [_gpu_solver(clip, R, t, X0, mode, cuda, loss=loss, loss_scale=d) for _ in range(3)]
    runs[0].run(5)
    runs[1].run(5, graph=True)
    runs[2].run(5, graph=True)
    assert runs[0].history == runs[1].history == runs[2].history
    for u, v, w in zip(*(_buffers(r) for r in runs)):
        assert torch.equal(u, v) and torch.equal(v, w)


# ------------------------------------------------------------------------------------------------------ shards
def _sharded(clip, mode, full, **kw):
    """tests/test_ba_reg_scale_gpu.py's three shards (the middle one a single frame) of a robust solve, with the unsharded
    solver's scalars and state, halo rows included."""
    T = clip["X0"].shape[0]
    shards = []
    for a, b in _bounds(T):
        s = _solver(clip, mode, a, b, local_only=True, **kw)
        s.prob.has_prev, s.prob.has_next = int(a > 0), int(b < T)
        s.sc.copy_(full.sc)
        s.Xh.copy_(full.Xh[:, a: b + 2])
        s.Ch.copy_(full.Ch[:, a: b + 2])
        s.vec.copy_(full.vec[:, a: b + 2])
        shards.append(s)
    return shards


@pytest.mark.parametrize("name,loss,d", [("A_full_3_warp_passes", "huber", 3.0), ("A_full_3_warp_passes", "cauchy", 3.0),
                                         ("C_pose_only_3_point_passes", "cauchy", 3.0)])
def test_lockstep_shards_follow_the_unsharded_trajectory(cuda, clips, name, loss, d):
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    n = 4
    full = _solver(clip, mode, loss=loss, loss_scale=d)
    shards = _sharded(clip, mode, full, loss=loss, loss_scale=d)
    assert [s.Tl for s in shards][1] == 1
    for s in shards:
        s.cost(0)
    _allreduce([s.sums[0] for s in shards])
    for s in shards:
        s.finish_cost(0)
    assert float(shards[0].sc[_cabi.BA_REG_SC_COST]) == pytest.approx(full.cost_value, rel=SHARD_TRAJ_TOL, abs=0.0)
    full.run(n)
    for _ in range(n):
        _lockstep_trial(shards)
    for s in shards:
        s.iters_done = n
    hf, hs = full.history, shards[0].history
    for s in shards[1:]:
        assert s.history == hs
    for i in range(n):
        dev = abs(hs[i]["trial_cost"] - hf[i]["trial_cost"]) / hf[i]["trial_cost"]
        print(f"    trial {i}: trial cost {hf[i]['trial_cost']:.9f}  dev {dev:.2e}  cg {hs[i]['cg_iters']} / {hf[i]['cg_iters']}  "
              f"accepted {hs[i]['accepted']} / {hf[i]['accepted']}")
        assert dev <= SHARD_TRAJ_TOL and abs(hs[i]["cost"] - hf[i]["cost"]) <= SHARD_TRAJ_TOL * hf[i]["cost"]
        assert hs[i]["accepted"] == hf[i]["accepted"] and hs[i]["cg_iters"] == hf[i]["cg_iters"], i
    assert sum(h["accepted"] for h in hf) >= 2
    dx = float((torch.cat([s.X for s in shards]) - full.X).abs().max())
    print(f"    max |X_sharded - X| {dx:.2e}")
    assert dx <= TRAJ_X_TOL


# ------------------------------------------------------------------------------------------------------ outliers
def test_robust_loss_keeps_per_frame_cameras_under_outliers(cuda):
    """tests/test_oracle_lm_reg_robust.py's seeded problem (config-3 rig, "full", 5 % outliers, 10 trials): the mean
    per-frame camera-1 errors must order L2 > Huber > Cauchy, the robust ones within 10 % above the fp64 specification's
    (OUTLIER_SPEC) and L2's no more than 10 % below it."""
    clip, R, t, X0 = outlier_problem()
    err = {}
    for loss, d in [("l2", None)] + ROBUST:
        s = _gpu_solver(clip, R, t, X0, "full", cuda, loss=loss, loss_scale=d)
        s.run(OUTLIER_ITERS)
        err[loss] = tuple(float(e.mean()) for e in cam1_errors(s.R.cpu().numpy(), s.t.cpu().numpy(), clip.R, clip.t))
    print(err)
    for k in range(2):
        assert err["l2"][k] > err["huber"][k] > err["cauchy"][k], err
        assert err["l2"][k] >= 0.9 * OUTLIER_SPEC["l2"][k], err
        for loss in ("huber", "cauchy"):
            assert err[loss][k] <= 1.1 * OUTLIER_SPEC[loss][k], (loss, err)
