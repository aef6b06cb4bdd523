"""Freeze outputs of the REFERENCE's own functions as golden vectors (authoring container only).

    python -m oracle.make_golden            # writes tests/golden/*.npz

The reference has no tests or fixtures for this path (SURVEY.md section 4), so parity is pinned by
running its functions here on the deterministic synthetic inputs of skiing_analysis_pytorch_b200/
synth.py and committing inputs + outputs.  /root/reference does not exist on the GPU box; the
tests only ever read the .npz files.  Golden sets (SURVEY.md section 8c):
  G1  triangulation.triangulate.triangulate_joints, triangulation.reproject.reproject_points /
      reproject_and_visualize statistics on the config-1 rig (FIXED pose, two_view.py:209-221)
  G2  vggt.triangulate.make_P / triangulate_point / triangulate_one_frame and
      bundle_adjustment.reproject.reproject_points mode A on two non-identity cameras (quirk Q3)
  G3  bundle_adjustment.loss.project_points / reprojection_loss for every accepted shape, f32+f64
  G4  camera_smooth / baseline_reg / bone_length / pose_temporal scalars
  G7  triangulation.postprocess.post_triage_sequence / post_triage_single / smooth_skeleton (row N2)
  G8  fuse.main_raw / fuse.confidence / fuse.fuse: rigid alignment, weak-perspective and cross-view confidences,
      softmax fusion, adaptive EMA (row N3)
  G10 on-disk schemas (row N4): .pt keypoint dicts, SAM-3D-Body npz, fuse / triangulation writers - fixture files under
      tests/golden/io/ and the reference loaders' outputs for them
  G11 bundle_adjustment/fuse/fuse.py rigid_transform_3D (Umeyama on the torso joints + threshold fusion, row N3)
  G9  oracle/first_order.py (Adam on the full configured objective) driven by the reference's bundle_adjustment/loss.py
  G6  LM history of oracle/lm.py on BASELINE configs 3 and 5 at reduced T, with the REFERENCE's
      reprojection_loss evaluated at the initial and final state of each solve (pins the cost the
      LM minimises; the trajectory itself has no reference implementation - "parity unpinned")
  reference_signatures.json  parameter names and scalar defaults of the reference functions the drop-in shims
      stand in for (--only-signatures)
"""
from __future__ import annotations

import logging
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import ref_import  # noqa: E402
from skiing_analysis_pytorch_b200 import synth  # noqa: E402

OUT = ROOT / "tests" / "golden"


def g1():
    tri = ref_import.load("triangulation.triangulate")
    rep = ref_import.load("triangulation.reproject")
    clip = synth.make_clip("2a", T=48, J=17, seed=0)
    K = clip.K[0]
    R, t = clip.R[1], clip.t[1]  # cam2 w.r.t. cam1 (cam1 = identity on this rig)
    assert np.allclose(clip.R[0], np.eye(3)) and np.allclose(clip.t[0], 0)
    assert np.array_equal(tri.K_dist, synth.DIST_CALIB)
    kL, kR = clip.x_vm[0], clip.x_vm[1]
    X32 = np.stack([tri.triangulate_joints(kL[i], kR[i], K, R, t) for i in range(len(kL))])
    X64 = np.stack([tri.triangulate_joints(kL[i].astype(np.float64), kR[i].astype(np.float64), K, R, t.reshape(3, 1)) for i in range(len(kL))])
    assert X32.dtype == np.float32 and X64.dtype == np.float64
    projL_d, projR_d, projL_p, projR_p = [], [], [], []
    for i in range(len(kL)):
        pd = rep.reproject_points(X32[i], K, tri.K_dist, K, tri.K_dist, R, t)
        pp = rep.reproject_points(X32[i], K, None, K, None, R, t)
        projL_d.append(pd["proj_L"]); projR_d.append(pd["proj_R"])
        projL_p.append(pp["proj_L"]); projR_p.append(pp["proj_R"])
    img = np.zeros((108, 192, 3), np.uint8)
    stats = []
    keys = ["rmse_L", "rmse_R", "mean_err_L", "mean_err_R", "median_err_L", "median_err_R", "max_err_L", "max_err_R"]
    errL, errR = [], []
    with tempfile.TemporaryDirectory() as td:
        for i in range(8):
            res = rep.reproject_and_visualize(img, img, X32[i], kL[i], kR[i], K, tri.K_dist, K, tri.K_dist, R, t,
                                              out_path=str(Path(td) / "p.jpg"))
            stats.append([res[k] for k in keys])
            errL.append(res["err_L"]); errR.append(res["err_R"])
    np.savez_compressed(
        OUT / "g1_two_view_fixed_rig.npz", K=K, R=R, t=t, dist=tri.K_dist, kptL=kL, kptR=kR, X_f32=X32, X_f64=X64,
        projL_dist=np.stack(projL_d), projR_dist=np.stack(projR_d), projL_pin=np.stack(projL_p), projR_pin=np.stack(projR_p),
        stats=np.array(stats), stats_keys=np.array(keys), errL=np.stack(errL), errR=np.stack(errR),
    )


def g2():
    vt = ref_import.load("vggt.triangulate")
    brp = ref_import.load("bundle_adjustment.reproject")
    vrp = ref_import.load("vggt.reproject")
    rng = np.random.default_rng(7)
    clip = synth.make_clip("2b", T=16, J=17, seed=3)
    # move the world frame so that NEITHER camera is the identity (quirk Q3 needs this)
    Rw = synth.so3_exp(np.array([0.1, -0.3, 0.05]))
    tw = np.array([0.4, -0.2, 1.5])
    R = np.stack([clip.R[c] @ Rw for c in range(2)])
    t = np.stack([clip.R[c] @ tw + clip.t[c] for c in range(2)])
    K = np.stack([clip.K[0], clip.K[1] * np.array([[1.02, 1, 0.99], [1, 0.98, 1.01], [1, 1, 1]])])
    P = np.stack([vt.make_P(K[c], R[c], t[c]) for c in range(2)])
    kL, kR = clip.x_vm[0], clip.x_vm[1]
    Xpt = np.array([[vt.triangulate_point(P[0], P[1], kL[i, j], kR[i, j]) for j in range(17)] for i in range(len(kL))])
    img = np.zeros((108, 192, 3), np.uint8)
    X_frame, means = [], []
    logging.disable(logging.CRITICAL)
    with tempfile.TemporaryDirectory() as td:
        for i in range(4):
            X3d, res = vt.triangulate_one_frame(K, R, t, kL[i], kR[i], img, img, save_dir=Path(td), dist=None)
            X_frame.append(X3d); means.append([res["mean_err_L"], res["mean_err_R"]])
    pa = [brp.reproject_points(Xpt[i], K[0], None, K[1], None, R, t) for i in range(len(kL))]
    pa_d = [vrp.reproject_points(Xpt[i], K[0], synth.DIST_CALIB, K[1], synth.DIST_CALIB, list(R), list(t)) for i in range(len(kL))]
    R_rel = R[1] @ R[0].T
    t_rel = t[1] - R_rel @ t[0]
    pb = [brp.reproject_points(Xpt[i], K[0], None, K[1], None, R_rel, t_rel.reshape(3, 1)) for i in range(len(kL))]
    np.savez_compressed(
        OUT / "g2_vggt_two_cameras.npz", K=K, R=R, t=t, P=P, kptL=kL, kptR=kR, X_point=Xpt, X_frame=np.stack(X_frame),
        frame_mean_err=np.array(means), modeA_L=np.stack([p["proj_L"] for p in pa]), modeA_R=np.stack([p["proj_R"] for p in pa]),
        modeA_dist_L=np.stack([p["proj_L"] for p in pa_d]), modeA_dist_R=np.stack([p["proj_R"] for p in pa_d]),
        modeB_L=np.stack([p["proj_L"] for p in pb]), modeB_R=np.stack([p["proj_R"] for p in pb]), dist=synth.DIST_CALIB,
    )
    del rng


def g3_g4():
    import torch

    loss = ref_import.load("bundle_adjustment.loss")
    clip = synth.make_clip("4", T=12, J=17, seed=5)
    T, C, J = 12, 4, 17
    rng = np.random.default_rng(11)
    X = clip.X + rng.normal(0, 0.01, clip.X.shape)
    Kc = clip.K.copy()
    Kc[:, 0, 1] = [0.0, 0.7, -0.4, 0.2]  # skew is honoured by loss.py:74-82
    Rt = np.stack([np.stack([synth.so3_exp(rng.normal(0, 0.01, 3)) @ clip.R[c] for c in range(C)]) for _ in range(T)])
    tt = clip.t[None] + rng.normal(0, 0.02, (T, C, 3))
    Kt = Kc[None] * (1 + rng.normal(0, 1e-3, (T, C, 1, 1)))
    Kt[..., 2, :] = [0, 0, 1]
    x2d, conf = clip.x_fm, clip.conf_fm
    out = dict(X=X, K_c=Kc, R_c=clip.R, t_c=clip.t, R_t=Rt, t_t=tt, K_t=Kt, x2d=x2d, conf=conf)
    tt_ = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt)
    for name, dt in (("f64", torch.float64), ("f32", torch.float32)):
        Xt = tt_(X, dt)
        out[f"proj_static_{name}"] = loss.project_points(Xt, tt_(clip.R, dt), tt_(clip.t, dt), tt_(Kc, dt)).numpy()
        out[f"proj_perframe_{name}"] = loss.project_points(Xt, tt_(Rt, dt), tt_(tt, dt), tt_(Kt, dt)).numpy()
        out[f"proj_perframeR_statict_{name}"] = loss.project_points(Xt, tt_(Rt, dt), tt_(clip.t, dt), tt_(Kc, dt)).numpy()
        out[f"proj_single_{name}"] = loss.project_points(Xt[0], tt_(clip.R, dt), tt_(clip.t, dt), tt_(Kc, dt)).numpy()
        out[f"loss_static_{name}"] = loss.reprojection_loss(Xt, tt_(clip.R, dt), tt_(clip.t, dt), tt_(Kc, dt), tt_(x2d, dt), tt_(conf, dt)).item()
        out[f"loss_perframe_w_{name}"] = loss.reprojection_loss(Xt, tt_(Rt, dt), tt_(tt, dt), tt_(Kt, dt), tt_(x2d, dt), tt_(conf, dt), w=0.5).item()
        # a point behind a camera exercises Z.clamp(min=1e-6) (loss.py:67)
        Xb = Xt.clone()
        Xb[0, 0] = torch.tensor([0.0, 0.0, -5.0], dtype=dt)
        out[f"proj_clamped_{name}"] = loss.project_points(Xb, tt_(clip.R, dt), tt_(clip.t, dt), tt_(Kc, dt)).numpy()
    d = torch.float64
    out["camera_center"] = loss.camera_center_from_Rt(tt_(Rt, d), tt_(tt, d)).numpy()
    out["camera_smooth"] = loss.camera_smooth_loss(tt_(Rt, d), tt_(tt, d), w=0.1).item()
    out["baseline_reg"] = loss.baseline_reg_loss(tt_(Rt, d), tt_(tt, d), w=0.01).item()
    out["bone_length"] = loss.bone_length_loss(tt_(X, d), w=0.1).item()
    ref_len = np.linspace(0.2, 0.6, len(loss.BONES))
    out["bone_length_ref"] = loss.bone_length_loss(tt_(X, d), ref_bone_len=tt_(ref_len, d), w=0.1).item()
    out["ref_len"] = ref_len
    out["pose_temporal"] = loss.pose_temporal_loss(tt_(X, d), w=0.1).item()
    out["bones"] = np.array(loss.BONES)
    # J=70 (MHR skeleton): indices are applied blindly
    X70 = synth.make_clip("2b", T=6, J=70, seed=9).X
    out["X70"] = X70
    out["bone_length_70"] = loss.bone_length_loss(tt_(X70, d), w=0.1).item()
    np.savez_compressed(OUT / "g3_g4_loss.npz", **out)




def g6():
    import torch

    from oracle import lm

    loss = ref_import.load("bundle_adjustment.loss")
    out = {}
    for name, (rig, T, J, mode) in lm.G6_CASES.items():
        clip, R0, t0, X0 = lm.make_problem(rig, T, J)
        R, t, X, hist = lm.run_lm(X0, R0, t0, clip.K, clip.x_fm, clip.conf_fm, num_iters=10, mode=mode)
        tt_ = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(torch.float64)
        ref0 = loss.reprojection_loss(tt_(X0), tt_(R0), tt_(t0), tt_(clip.K), tt_(clip.x_fm), tt_(clip.conf_fm)).item()
        ref1 = loss.reprojection_loss(tt_(X), tt_(R), tt_(t), tt_(clip.K), tt_(clip.x_fm), tt_(clip.conf_fm)).item()
        out[f"{name}_hist"] = np.array([[h["iter"], h["cost"], h["trial_cost"], h["lam"], h["rho"], h["accepted"], h["n_clamped"], h["pred"]] for h in hist])
        out[f"{name}_R"] = R
        out[f"{name}_t"] = t
        out[f"{name}_X_head"] = X[:4]
        out[f"{name}_ref_loss_init"] = ref0
        out[f"{name}_ref_loss_final"] = ref1
    np.savez_compressed(OUT / "g6_lm_history.npz", **out)


def g7():
    """triangulation.postprocess.post_triage_sequence / smooth_skeleton of the reference (row N2)."""
    import warnings

    from oracle import geometry as G

    pp = ref_import.load("triangulation.postprocess")
    clip = synth.make_clip("2b", 80, 17, seed=21)
    K, R, t = clip.K[0], clip.R[1], clip.t[1]
    P = np.stack([G.make_P(K, np.eye(3), np.zeros(3)), G.make_P(K, R, t)])
    X = G.dlt_triangulate(P, clip.x_vm.reshape(2, -1, 2)).reshape(80, 17, 3).astype(np.float32)
    X[3, 4] = np.nan                     # a joint the triangulation lost
    X[10, 2] = [0.0, 0.0, -3.0]          # behind the cameras
    kL, kR = clip.x_vm[0].copy(), clip.x_vm[1].copy()
    kL[20, 5] += 40.0                    # a gross outlier
    out = dict(X=X, kptL=kL, kptR=kR, K=K, R=R, t=t, dist=synth.DIST_CALIB, confL=clip.conf_vm[0], confR=clip.conf_vm[1])
    cases = {"plain": dict(), "dist": dict(dist1=synth.DIST_CALIB, dist2=synth.DIST_CALIB),
             "conf_smooth": dict(confL=clip.conf_vm[0], confR=clip.conf_vm[1], smooth=True),
             "tight_smooth6": dict(err_thresh_px=1.0, smooth=True, sg_win=6, sg_poly=3)}
    keys = ["rmse_px", "median_err_px", "pos_depth_ratio", "kept_ratio", "kept_count"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name, kw in cases.items():
            Xc, st = pp.post_triage_sequence(X, kL, kR, K, K, R, t, **kw)
            out[f"{name}_X"] = Xc
            out[f"{name}_stats"] = np.array([[s[k] for k in keys] for s in st])
        Xc1, rep1, keep1 = pp.post_triage_single(X[20], kL[20], kR[20], K, K, R, t, confL=clip.conf_vm[0][20], confR=clip.conf_vm[1][20],
                                                 return_masks=True)
        out["single_X"], out["single_keep"], out["single_stats"] = Xc1, keep1, np.array([rep1[k] for k in keys])
        rng = np.random.default_rng(5)
        Xs = (synth.skeleton_clip(64, 5, rng)).astype(np.float32)
        Xs[rng.uniform(size=Xs.shape[:2]) < 0.15] = np.nan
        Xs[:, 4] = np.nan
        Xs[:60, 3] = np.nan              # fewer finite samples than the window: left alone
        out["smooth_in"] = Xs
        out["smooth_out_9_2"] = pp.smooth_skeleton(Xs, win=9, poly=2)
        out["smooth_out_8_3"] = pp.smooth_skeleton(Xs, win=8, poly=3)
    np.savez_compressed(OUT / "g7_post_triage.npz", **out)


def g8():
    """fuse/main_raw.py's per-frame pipeline + fuse/fuse.py's EMA, run through the reference's own dict-based functions
    (row N3): _align_right_to_left, weakpersp_reproj_confidence, crossview_consistency_confidence, fuse_frame_3d,
    temporal_smooth_ema (adaptive and fixed alpha)."""
    mr = ref_import.load("fuse.main_raw")
    cf = ref_import.load("fuse.confidence")
    ff = ref_import.load("fuse.fuse")
    T, J = 60, 70
    d = synth.make_fusion_clip(T, J, seed=3, nan_frac=0.05)
    ids = list(range(J))
    to_dict = lambda A: {j: A[j].copy() for j in ids}                 # loaders keep every joint id (NaN rows included)
    fused = np.full((T, J, 3), np.nan)
    ql, qr, aligned = np.zeros((T, J)), np.zeros((T, J)), np.full((T, J, 3), np.nan)
    c1l_all, c2_all = np.zeros((T, J)), np.zeros((T, J))
    seq = []
    for t in range(T):
        Xl, Xr, Ul, Ur = (to_dict(d[k][t]) for k in ("Xl", "Xr", "Ul", "Ur"))
        Xa = mr._align_right_to_left(Xl, Xr, ids)
        c1l, _, _, _ = cf.weakpersp_reproj_confidence(Xl, Ul, sigma_px=12.0)
        c1r, _, _, _ = cf.weakpersp_reproj_confidence(Xr, Ur, sigma_px=12.0)
        c2, _, _, _, _ = cf.crossview_consistency_confidence(
            Xl, Xr, root_idx=mr.IDX_PELVIS, left_hip_idx=mr.IDX_LHIP, right_hip_idx=mr.IDX_RHIP, left_shoulder_idx=mr.IDX_LSHO,
            right_shoulder_idx=mr.IDX_RSHO, sigma_3d=0.08, scale_mode="hip")
        ql[t], qr[t] = np.sqrt(c1l * c2), np.sqrt(c1r * c2)
        c1l_all[t], c2_all[t] = c1l, c2
        fd = ff.fuse_frame_3d(Xl, Xa, ql[t], qr[t], ids)
        seq.append(fd)
        for j in ids:
            if j in Xa:
                aligned[t, j] = Xa[j]
            if j in fd:
                fused[t, j] = fd[j]
    # a second sequence with 25 % of the joints missing (runs of NaN: the hold / reset branches of fuse.py:400-404)
    rng = np.random.default_rng(8)
    sparse = fused.copy()
    sparse[rng.random((T, J)) < 0.25] = np.nan
    sparse[10:14, :8] = np.nan
    seq_sparse = [{j: sparse[t, j].copy() for j in ids if np.isfinite(sparse[t, j]).all()} for t in range(T)]

    def ema(src=None, **kw):
        out = ff.temporal_smooth_ema(seq if src is None else src, ids, **kw)
        Y = np.full((T, J, 3), np.nan)
        for t in range(T):
            for j, v in out[t].items():
                Y[t, j] = v
        return Y
    # fuse/main_unity.py:_fuse_pair (:96-132): the same pipeline WITHOUT the rigid alignment on the 15 Unity target joints
    # (the key indices 14, 11, 12, 5, 6 are then POSITIONS in the 15-joint array, as the reference uses them)
    mu = ref_import.load("fuse.main_unity")
    du = synth.make_fusion_clip(40, 15, seed=5, nan_frac=0.04)
    du["Xr"] = du["Xl"] + np.random.default_rng(6).normal(0.0, 0.03, du["Xl"].shape)   # both views in one coordinate system
    mk = lambda A: {jid: A[k] for k, jid in enumerate(mu.TARGET_IDS)}
    seq_a = [{"p2d": mk(du["Ul"][t]), "p3d": mk(du["Xl"][t])} for t in range(40)]
    seq_b = [{"p2d": mk(du["Ur"][t]), "p3d": mk(du["Xr"][t])} for t in range(40)]
    fu = mu._fuse_pair(seq_a, seq_b, sigma_px=12.0, sigma_3d=0.08)
    unity = np.full((40, 15, 3), np.nan)
    for t in range(40):
        for k, jid in enumerate(mu.TARGET_IDS):
            if jid in fu[t]:
                unity[t, k] = fu[t][jid]
    su = ff.temporal_smooth_ema(fu, mu.TARGET_IDS, alpha=0.7, adaptive=True, alpha_min=0.45, alpha_max=0.92, speed_gain=0.25)
    unity_s = np.full((40, 15, 3), np.nan)
    for t in range(40):
        for k, jid in enumerate(mu.TARGET_IDS):
            if jid in su[t]:
                unity_s[t, k] = su[t][jid]
    np.savez_compressed(
        OUT / "g8_fusion.npz", unity_Xl=du["Xl"], unity_Xr=du["Xr"], unity_Ul=du["Ul"], unity_Ur=du["Ur"], unity_fused=unity,
        unity_smooth=unity_s, unity_ids=np.array(mu.TARGET_IDS), Xl=d["Xl"], Xr=d["Xr"], Ul=d["Ul"], Ur=d["Ur"], fused=fused, q_l=ql, q_r=qr, aligned=aligned,
        conf1_l=c1l_all, conf2=c2_all, ema_adaptive=ema(alpha=0.7, adaptive=True, alpha_min=0.45, alpha_max=0.92, speed_gain=0.25),
        ema_fixed=ema(alpha=0.7, adaptive=False), fused_sparse=sparse,
        ema_sparse=ema(seq_sparse, alpha=0.7, adaptive=True, alpha_min=0.45, alpha_max=0.92, speed_gain=0.25), ema_gain=ema(alpha=0.6, adaptive=True, alpha_min=0.3, alpha_max=0.95, speed_gain=2.0))
    print("g8 written: missing fused joints", int(np.isnan(fused[..., 0]).sum()), "of", T * J)


def first_order_problem(T=24, J=17, seed=0):
    """Per-frame cameras as vggt/multi_view_process.py:546-551 passes them: the perturbed rig of oracle/lm.py plus a small
    per-frame jitter (so camera_smooth / baseline_reg have something to do)."""
    from oracle import lm

    clip, R0, t0, X0 = lm.make_problem("2b", T, J, seed)
    rng = np.random.default_rng(seed + 7)
    R = np.stack([[synth.so3_exp(rng.normal(0.0, 2e-3, 3)) @ R0[c] for c in range(2)] for _ in range(T)])
    t = np.broadcast_to(t0[None], (T, 2, 3)) + rng.normal(0.0, 0.01, (T, 2, 3))
    return clip, R, t, X0


def g9():
    """Adam on the reference's full configured objective (oracle/first_order.py) with the loss VALUES computed by the
    reference's own bundle_adjustment/loss.py (row N1, first-order form)."""
    import torch

    from oracle import first_order as FO

    L = ref_import.load("bundle_adjustment.loss")
    clip, R, t, X0 = first_order_problem()
    out = dict(R0=R, t0=t, X0=X0, K=clip.K, x2d=clip.x_fm, conf=clip.conf_fm)
    for mode in FO.MODES:
        Ro, to, Xo, hist = FO.run_adam(L, clip.K, R, t, X0, clip.x_fm, clip.conf_fm, num_iters=25, lr=1e-2, mode=mode)
        out[f"{mode}_hist"] = np.array([[h["loss"]] + [h[k] for k in FO.TERMS] for h in hist])
        out[f"{mode}_R"], out[f"{mode}_t"], out[f"{mode}_X"] = Ro.numpy(), to.numpy(), Xo.numpy()
    np.savez_compressed(OUT / "g9_first_order.npz", **out)
    print("g9 written:", {m: (out[f"{m}_hist"][0, 0], out[f"{m}_hist"][-1, 0]) for m in FO.MODES})


def g10():
    """On-disk schemas either side of the path (row N4): fixture files written in the reference's formats - by the
    reference's own writers where it has one - and what the reference's own loaders return for them."""
    import json
    import shutil

    import torch
    import torchvision.io

    if not hasattr(torchvision.io, "read_video"):  # removed in torchvision 0.26; triangulation/load.py:9 imports it
        torchvision.io.read_video = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("no video decoding in the golden generator"))
    io_dir = OUT / "io"
    if io_dir.exists():
        shutil.rmtree(io_dir)
    io_dir.mkdir(parents=True)
    rng = np.random.default_rng(10)
    T, K = 9, 17
    H, W = 1080, 1920
    out = {}
    # ---- .pt dicts in the schema of prepare_dataset/process/preprocess.py:157-181
    tl = ref_import.load("triangulation.load")
    for side in ("left", "right"):
        px = np.concatenate([rng.uniform(0, W, (T, K, 1)), rng.uniform(0, H, (T, K, 1)), rng.uniform(0.2, 1, (T, K, 1))], -1).astype(np.float32)
        nrm = px.copy()
        nrm[..., 0] /= W
        nrm[..., 1] /= H
        pt = {"img_shape": (H, W), "none_index": [],
              "YOLO": {"bbox": torch.zeros(T, 4), "keypoints": torch.from_numpy(nrm), "keypoints_score": torch.from_numpy(rng.uniform(0, 1, (T, K)).astype(np.float32))},
              "detectron2": {"bbox": torch.tensor(rng.uniform(0, 1000, (T, 4)).astype(np.float32)), "keypoints": torch.from_numpy(px)}}
        torch.save(pt, io_dir / f"{side}.pt")
        xy, sc, _ = tl.load_keypoints_from_yolo_pt(str(io_dir / f"{side}.pt"))
        out[f"{side}_yolo_xy"], out[f"{side}_yolo_score"] = xy, sc
        xy, sc, *_ = tl.load_kpt_and_bbox_from_d2_pt(str(io_dir / f"{side}.pt"))
        out[f"{side}_d2_xy"], out[f"{side}_d2_score"] = xy, sc
    # ---- SAM-3D-Body outputs: one npz with the frame list (left), a directory of per-frame files (right, one frame longer)
    lr = ref_import.load("fuse.load.load_raw")
    d = synth.make_fusion_clip(7, 70, seed=12, dtype=np.float32)
    frames_l = [{"pred_keypoints_2d": d["Ul"][t], "pred_keypoints_3d": d["Xl"][t], "pred_cam_t": np.zeros(3, np.float32), "focal_length": np.float32(1100)} for t in range(6)]
    np.savez(io_dir / "osmo_2_sam_3d_body_outputs.npz", outputs=np.array(frames_l, dtype=object))
    (io_dir / "right").mkdir()
    for t in range(7):
        fr = {"pred_keypoints_2d": d["Ur"][t], "pred_keypoints_3d": d["Xr"][t], "pred_cam_t": np.zeros(3, np.float32), "focal_length": np.float32(1100)}
        np.savez(io_dir / "right" / f"frame_{t:04d}_sam_3d_body_outputs.npz", outputs=np.array([fr], dtype=object))
    res = lr.load_raw({"sam_l": str(io_dir / "osmo_2_sam_3d_body_outputs.npz"), "sam_r": str(io_dir / "right")})
    arr = lambda key, dim: np.stack([np.stack([np.asarray(res[t][key]["pred"][j], np.float64) for j in range(70)]) for t in sorted(res)])
    out.update(sam_Xl=arr("L_3D", 3), sam_Xr=arr("R_3D", 3), sam_Ul=arr("L_2D", 2), sam_Ur=arr("R_2D", 2))
    # ---- writers: the reference's own files
    fs = ref_import.load("fuse.save")
    seq = out["sam_Xl"].copy()
    seq[2, 5] = np.nan
    seq_dicts = [{j: seq[t, j] for j in range(70) if np.isfinite(seq[t, j]).all()} for t in range(len(seq))]
    fs.save_smoothed_results(seq_dicts, list(range(70)), str(io_dir / "ref_out" / "person_smoothed.npy"))
    out["seq_to_save"] = seq
    ts = ref_import.load("triangulation.save")
    X = rng.normal(size=(3, 17, 3)).astype(np.float32)
    Rr = [np.eye(3) * (1 + i) for i in range(3)]
    Tt = [np.arange(3.0).reshape(3, 1) + i for i in range(3)]
    vp = {"left": "/data/left.mp4", "right": Path("/data/right.mp4")}
    for fmt in ("npy", "csv", "json"):
        for i in range(3):
            ts.save_3d_joints(X[i], str(io_dir / "ref_out" / "joints"), 40 + i, Rr[i], Tt[i], vp, fmt=fmt)
    out.update(joints_X=X, joints_R=np.stack(Rr), joints_T=np.stack(Tt))
    np.savez_compressed(OUT / "g10_io.npz", **out)
    print("g10 written:", sorted(p.name for p in (io_dir / "ref_out" / "joints").iterdir())[:4], "...")


def g11():
    """bundle_adjustment/fuse/fuse.py:rigid_transform_3D (Umeyama alignment on the 5 torso joints + threshold fusion),
    the fusion the bundle_adjustment / fuse.side / front_side.side pipelines call (second half of row N3)."""
    bf = ref_import.load("bundle_adjustment.fuse.fuse")
    T, J = 40, 70
    d = synth.make_fusion_clip(T, J, seed=21, nan_frac=0.05)
    L, R = d["Xl"].copy(), d["Xr"].copy()
    full = synth.make_fusion_clip(12, J, seed=23, nan_frac=0.0)   # 12 complete frames: finite diagnostics (plain means)
    L[:12], R[:12] = full["Xl"], full["Xr"]
    rng = np.random.default_rng(22)
    wL, wR = rng.uniform(0.2, 1.0, (T, J)), rng.uniform(0.2, 1.0, (T, J))
    out = dict(L=L, R=R, wL=wL, wR=wR)
    for name, kw in (("plain", dict()), ("weighted", dict(wL=wL, wR=wR, tau=0.05)), ("scaled", dict(allow_scale=True, wL=wL[0], wR=wR[0]))):
        ok = np.array([np.isfinite(L[t][list(bf.TORSO_IDX)]).all(1).__and__(np.isfinite(R[t][list(bf.TORSO_IDX)]).all(1)).sum() >= 3 for t in range(T)])
        fused, diag = bf.rigid_transform_3D(L[ok], R[ok], return_diagnostics=True, **kw)
        out[f"{name}_ok"] = ok
        out[f"{name}_fused"] = fused
        out[f"{name}_R"] = np.stack([p["R"] for p in diag["per_frame"]])
        out[f"{name}_t"] = np.stack([p["t"] for p in diag["per_frame"]])
        out[f"{name}_s"] = np.array([p["s"] for p in diag["per_frame"]])
        out[f"{name}_diag"] = np.array([[p["LR_before"], p["Fused_vs_L"], p["Fused_vs_R"], p["gain"]] for p in diag["per_frame"]])
        out[f"{name}_mean_gain"] = diag["mean_gain"]
        out[f"{name}_bad"] = np.array(diag["bad_frames"], dtype=np.int64)
    f1, d1 = bf.rigid_transform_3D(L[0], R[0])   # single frame (J,3) in, (J,3) out
    out["single_fused"] = f1
    np.savez_compressed(OUT / "g11_rigid_fuse.npz", **out)
    print("g11 written: frames ok", int(out["plain_ok"].sum()), "of", T, "mean gain", out["plain_mean_gain"])


def g12():
    """Regularised LM (oracle/lm_reg.py, row N1 second-order form): the cost history of the exact-solve oracle, and the
    reference's OWN bundle_adjustment/loss.py evaluated at the oracle's first and final iterates - what pins `cost`."""
    import torch

    from oracle import first_order as FO
    from oracle import lm_reg

    L = ref_import.load("bundle_adjustment.loss")
    out = {}
    tt = lambda a: torch.from_numpy(np.asarray(a, float))
    for name, (rig, T, J, mode) in lm_reg.G12_CASES.items():
        clip, R, t, X0 = lm_reg.make_problem(rig, T, J, cam_jitter=0.01)
        x2d, conf = clip.x_fm.astype(float), clip.conf_fm.astype(float)
        Ro, to, Xo, hist = lm_reg.run_lm(X0, R, t, clip.K, x2d, conf, num_iters=8, mode=mode)
        out[f"{name}_cost"] = np.array([h["cost"] for h in hist])
        out[f"{name}_trial_cost"] = np.array([h["trial_cost"] for h in hist])
        out[f"{name}_accepted"] = np.array([h["accepted"] for h in hist])
        coef = lm_reg.coefficients(T, J, R.shape[1], conf.sum(), None)
        out[f"{name}_final_cost"] = sum(lm_reg.cost_terms(Xo, Ro, to, clip.K, x2d, conf, coef)[0].values())
        ref0, _ = FO.total_loss(L, tt(X0), tt(R), tt(t), tt(clip.K), tt(x2d), tt(conf), FO.DEFAULT_WEIGHTS)
        ref1, _ = FO.total_loss(L, tt(Xo), tt(Ro), tt(to), tt(clip.K), tt(x2d), tt(conf), FO.DEFAULT_WEIGHTS)
        out[f"{name}_ref_loss_first"], out[f"{name}_ref_loss_final"] = float(ref0), float(ref1)
        out[f"{name}_X"] = Xo
        assert abs(float(ref0) - hist[0]["cost"]) <= 1e-12 * hist[0]["cost"], (name, float(ref0), hist[0]["cost"])
    np.savez_compressed(OUT / "g12_lm_reg.npz", **out)
    print("g12 written:", {n: (out[f"{n}_cost"][0], out[f"{n}_final_cost"], out[f"{n}_ref_loss_final"]) for n in lm_reg.G12_CASES})


def signatures():
    """Parameter names and scalar defaults of every reference function listed in reference_signatures.json, re-read
    from the checkout (tests/test_dropin_cpu.py holds the drop-in shims to them)."""
    import json

    f = OUT / "reference_signatures.json"
    rec = json.loads(f.read_text())
    for module, funcs in rec.items():
        ref = ref_import.load(module)
        for fn in funcs:
            funcs[fn] = ref_import.signature_record(getattr(ref, fn))
    f.write_text(json.dumps(rec, indent=1) + "\n")


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    if "--only-signatures" in sys.argv:
        return signatures()
    if "--only-g12" in sys.argv:
        return g12()
    if "--only-g11" in sys.argv:
        return g11()
    if "--only-g10" in sys.argv:
        return g10()
    if "--only-g8" in sys.argv:
        return g8()
    if "--only-g9" in sys.argv:
        return g9()
    g9()
    g8()
    g7()
    g1()
    g2()
    g3_g4()
    g6()
    signatures()
    for f in sorted(OUT.glob("*.npz")):
        print(f.name, f.stat().st_size)


if __name__ == "__main__":
    main()
