"""Deterministic synthetic rigs, skeleton clips and observations (SURVEY.md section 8d).

There is no dataset in the reference (and no network): every test and benchmark runs on these.
Conventions: world->camera ``x_c = R x_w + t``; ``R_y(theta) = [[c,0,s],[0,1,0],[-s,0,c]]``
(two_view.py:209-211); look-at placement ``C_v = centre - d * R_v^T e_z``, ``t_v = -R_v C_v``.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

# camera_calibration/calibration_parameters.npz (camera_matrix / dist_coeffs), also hard-coded at
# triangulation/main.py:51-63 and triangulation/triangulate.py:39-56 of the reference.
K_CALIB = np.array(
    [
        [1116.9289548941917, 0.0, 955.77175993563799],
        [0.0, 1117.3341496962166, 538.91061167202145],
        [0.0, 0.0, 1.0],
    ]
)
DIST_CALIB = np.array(
    [
        -1.1940477842823853,
        -15.440461757486913,
        0.00013163161053023783,
        0.00019082529328353381,
        98.843073622415901,
        -1.3588290520381034,
        -14.555841222727574,
        96.219667412855202,
        0.0,
        0.0,
        0.0,
        0.0,
        0.0,
        0.0,
    ]
)
IMAGE_SIZE = (1920, 1080)
CENTRE = np.array([0.0, 0.0, 10.0])


def rot_y(theta: float) -> np.ndarray:
    c, s = np.cos(theta), np.sin(theta)
    return np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])


def look_at_rig(thetas, centre=CENTRE, d: float = 10.0):
    """Cameras on a circle of radius d around ``centre``, all looking at it. -> R (V,3,3), t (V,3)."""
    Rs, ts = [], []
    for th in thetas:
        R = rot_y(float(th))
        C = np.asarray(centre, float) - d * R.T @ np.array([0.0, 0.0, 1.0])
        Rs.append(R)
        ts.append(-R @ C)
    return np.stack(Rs), np.stack(ts)


def rig(name: str):
    """'2a' = the reference's FIXED pose (cam1 yaw 180 deg at z=20 m, two_view.py:209-221; near
    degenerate, triangulation parity only); '2b' = front/side (cam1 yaw +90 deg); '8' = 8-view ring."""
    if name == "2a":
        return look_at_rig([0.0, np.pi])
    if name == "2b":
        return look_at_rig([0.0, np.pi / 2])
    if name == "8":
        return look_at_rig([2 * np.pi * v / 8 for v in range(8)])
    if name.isdigit():
        n = int(name)
        return look_at_rig([2 * np.pi * v / n for v in range(n)])
    raise ValueError(f"unknown rig {name!r}")


@dataclass
class Clip:
    X: np.ndarray  # (T,J,3) f64 ground truth
    R: np.ndarray  # (V,3,3)
    t: np.ndarray  # (V,3)
    K: np.ndarray  # (V,3,3)
    x_vm: np.ndarray  # (V,T,J,2) f32 observations, view-major
    conf_vm: np.ndarray  # (V,T,J) f32 confidences in U(0.2,1)

    @property
    def x_fm(self) -> np.ndarray:  # (T,V,J,2) frame-major (loss.py layout)
        return np.ascontiguousarray(self.x_vm.transpose(1, 0, 2, 3))

    @property
    def conf_fm(self) -> np.ndarray:
        return np.ascontiguousarray(self.conf_vm.transpose(1, 0, 2))


def skeleton_clip(T: int, J: int, rng) -> np.ndarray:
    """template ~ N(0,0.4^2) fixed over time, Lissajous root motion, 2 cm per-joint jitter."""
    template = rng.normal(0.0, 0.4, (J, 3))
    tt = np.arange(T, dtype=float)
    root = CENTRE + np.stack(
        [1.5 * np.sin(2 * np.pi * tt / 300), 0.3 * np.sin(2 * np.pi * tt / 90), 1.0 * np.cos(2 * np.pi * tt / 240)], -1
    )
    return root[:, None, :] + template[None] + rng.normal(0.0, 0.02, (T, J, 3))


def pinhole(X, R, t, K):
    Xc = X @ R.T + t
    xy = Xc[..., :2] / Xc[..., 2:3]
    return np.stack([K[0, 0] * xy[..., 0] + K[0, 1] * xy[..., 1] + K[0, 2], K[1, 1] * xy[..., 1] + K[1, 2]], -1)


def make_clip(rig_name: str, T: int, J: int, seed: int = 0, noise_px: float = 1.0, K=None) -> Clip:
    rng = np.random.default_rng(seed)
    R, t = rig(rig_name)
    V = len(R)
    K = np.broadcast_to(K_CALIB if K is None else np.asarray(K, float), (V, 3, 3)).copy()
    X = skeleton_clip(T, J, rng)
    x = np.stack([pinhole(X, R[v], t[v], K[v]) for v in range(V)])
    x = (x + rng.normal(0.0, noise_px, x.shape)).astype(np.float32)
    conf = rng.uniform(0.2, 1.0, (V, T, J)).astype(np.float32)
    return Clip(X=X, R=R, t=t, K=K, x_vm=x, conf_vm=conf)


def inject_outliers(x2d: np.ndarray, J: int, frac: float, seed: int = 0) -> np.ndarray:
    """Corrupt a fraction `frac` of the observations of x2d (..., J, 2) IN PLACE, the way monocular 2D detectors fail
    (swapped limbs, invented positions of occluded joints), and return the (..., J) bool mask of corrupted ones.
    Half of them take another joint's observation of the same frame and view (a limb swap); the other half move by a
    uniform 50-300 px in a uniform direction.  Confidences are not touched: they do not flag the outliers."""
    if x2d.shape[-2:] != (J, 2):
        raise ValueError(f"x2d must end in ({J}, 2), got {x2d.shape}")
    rng = np.random.default_rng(seed)
    flat = x2d.reshape(-1, J, 2)
    n = flat.shape[0] * J
    k = int(round(frac * n))
    pick = rng.choice(n, size=k, replace=False)
    row, j = pick // J, pick % J
    orig = flat.copy()
    half = k // 2
    if J > 1:
        other = (j[:half] + rng.integers(1, J, half)) % J
        flat[row[:half], j[:half]] = orig[row[:half], other]
    r = rng.uniform(50.0, 300.0, k - half)
    phi = rng.uniform(0.0, 2 * np.pi, k - half)
    flat[row[half:], j[half:]] = orig[row[half:], j[half:]] + np.stack([r * np.cos(phi), r * np.sin(phi)], -1).astype(flat.dtype)
    mask = np.zeros(n, bool)
    mask[pick] = True
    return mask.reshape(x2d.shape[:-1])


def so3_exp(w):
    w = np.asarray(w, float)
    th = np.linalg.norm(w)
    W = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-8:
        return np.eye(3) + W
    return np.eye(3) + np.sin(th) / th * W + (1 - np.cos(th)) / th**2 * (W @ W)


def perturb_cameras(R, t, seed: int = 1, rot_sigma: float = 0.01, trans_sigma: float = 0.05):
    """BA initialisation: left-multiply exp(N(0,rot_sigma^2)) and add N(0,trans_sigma^2) to every
    camera except camera 0 (the gauge, SURVEY.md section 8c)."""
    rng = np.random.default_rng(seed)
    R2, t2 = R.copy(), t.copy()
    for c in range(1, len(R)):
        R2[c] = so3_exp(rng.normal(0.0, rot_sigma, 3)) @ R[c]
        t2[c] = t[c] + rng.normal(0.0, trans_sigma, 3)
    return R2, t2


CALIB_THETA_PERTURB = np.array([1.01, 0.99, 4.0, -3.0, 0.05, -0.02, 1e-3, -1e-3, 0.01])
CALIB_PRIOR_RHO = np.array([1e-4, 1e-4, 1e-4, 1e-4, 1.0, 1.0, 1.0, 1.0, 1.0])


def theta_from_K(K, dist=None):
    """K (C,3,3) zero skew (+ optional [k1 k2 p1 p2 k3]) -> (C,9) intrinsic vectors [fx fy cx cy k1 k2 p1 p2 k3]."""
    K = np.asarray(K, float)
    th = np.zeros((K.shape[0], 9))
    th[:, 0], th[:, 1], th[:, 2], th[:, 3] = K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]
    if dist is not None:
        th[:, 4:] = np.broadcast_to(np.asarray(dist, float), (K.shape[0], 5))
    return th


def perturb_intrinsics(K):
    """Initial intrinsics of the calibrating-BA test / bench problems: (C,9) [fx fy cx cy k1 k2 p1 p2 k3] with
    fx * 1.01, fy * 0.99, (cx, cy) + (4, -3) px and a small non-zero distortion vector, sign alternating per camera.
    The synthetic observations are pinhole under K, so the optimiser has ~1 % focal error, a few px of principal-point
    error and the distortion to remove.  CALIB_PRIOR_RHO is the matching prior precision (100 px / unit-coefficient sigma)."""
    th = theta_from_K(K)
    for c in range(len(th)):
        sg = 1.0 if c % 2 == 0 else -1.0
        th[c, 0] *= 1.0 + sg * (CALIB_THETA_PERTURB[0] - 1.0)
        th[c, 1] *= 1.0 + sg * (CALIB_THETA_PERTURB[1] - 1.0)
        th[c, 2:4] += sg * CALIB_THETA_PERTURB[2:4]
        th[c, 4:] = sg * CALIB_THETA_PERTURB[4:]
    return th


def theta_to_K_dist(th):
    """(C,9) intrinsic vectors -> K (C,3,3), dist (C,5)."""
    th = np.asarray(th, float)
    K = np.zeros((len(th), 3, 3))
    K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2], K[:, 2, 2] = th[:, 0], th[:, 1], th[:, 2], th[:, 3], 1.0
    return K, th[:, 4:].copy()


def make_clip_device(rig_name: str, T: int, J: int, device, seed: int = 0, noise_px: float = 1.0, layout: str = "TCJ2",
                     chunk_frames: int = 65536, frame_offset: int = 0, shardable: bool = False):
    """Same statistical model as make_clip but generated on the GPU with torch (synthetic-data
    plumbing for the full-size benchmark shapes: 1M frames x 70 joints x 8 views is 560M observations,
    minutes of numpy on the host).  Returns dict(x2d, conf, X, R, t, K) with x2d (T,C,J,2) / conf (T,C,J)
    for layout "TCJ2" or (C,T,J,2) / (C,T,J) for "CTJ2"; R, t, K are host fp64 arrays.
    shardable=True: every block of 500 frames draws from its own generator seeded by (seed, block index), so frames
    [frame_offset, frame_offset + T) are the SAME numbers whichever rank generates them - a clip split over N GPUs is the
    clip one GPU would hold (frame_offset and T multiples of 500)."""
    import torch

    R, t = rig(rig_name)
    V = len(R)
    K = np.broadcast_to(K_CALIB, (V, 3, 3)).copy()
    g = torch.Generator(device=device).manual_seed(seed)
    f64 = dict(dtype=torch.float64, device=device)
    template = torch.randn(J, 3, generator=g, **f64) * 0.4
    Rt = torch.tensor(R, **f64)
    tt = torch.tensor(t, **f64)
    Kt = torch.tensor(K, **f64)
    fm = layout == "TCJ2"
    x2d = torch.empty((T, V, J, 2) if fm else (V, T, J, 2), dtype=torch.float32, device=device)
    conf = torch.empty((T, V, J) if fm else (V, T, J), dtype=torch.float32, device=device)
    X = torch.empty((T, J, 3), **f64)
    if shardable:
        chunk_frames = 500
        if frame_offset % chunk_frames or T % chunk_frames:
            raise ValueError("shardable clips are generated in blocks of 500 frames")
    elif frame_offset:
        raise ValueError("frame_offset needs shardable=True")
    for a in range(0, T, chunk_frames):
        b = min(T, a + chunk_frames)
        if shardable:
            g = torch.Generator(device=device).manual_seed(seed * 1_000_003 + (frame_offset + a) // chunk_frames + 1)
        tt_ = torch.arange(frame_offset + a, frame_offset + b, **f64)
        root = torch.stack([1.5 * torch.sin(2 * np.pi * tt_ / 300), 0.3 * torch.sin(2 * np.pi * tt_ / 90),
                            10.0 + 1.0 * torch.cos(2 * np.pi * tt_ / 240)], -1)
        Xc = root[:, None, :] + template[None] + torch.randn(b - a, J, 3, generator=g, **f64) * 0.02
        X[a:b] = Xc
        cam = torch.einsum("vab,tjb->tvja", Rt, Xc) + tt[None, :, None, :]
        xy = cam[..., :2] / cam[..., 2:3]
        u = Kt[None, :, None, 0, 0] * xy[..., 0] + Kt[None, :, None, 0, 1] * xy[..., 1] + Kt[None, :, None, 0, 2]
        v = Kt[None, :, None, 1, 1] * xy[..., 1] + Kt[None, :, None, 1, 2]
        obs = (torch.stack([u, v], -1) + torch.randn(b - a, V, J, 2, generator=g, **f64) * noise_px).float()
        cf = (torch.rand(b - a, V, J, generator=g, device=device) * 0.8 + 0.2).float()
        if fm:
            x2d[a:b] = obs
            conf[a:b] = cf
        else:
            x2d[:, a:b] = obs.permute(1, 0, 2, 3)
            conf[:, a:b] = cf.permute(1, 0, 2)
    return dict(x2d=x2d, conf=conf, X=X, R=R, t=t, K=K)


def make_fusion_clip(T: int, J: int = 70, seed: int = 0, nan_frac: float = 0.03, outlier_frac: float = 0.05, dtype=np.float64):
    """Two monocular 3D estimates of the same skeleton (what SAM-3D-Body gives per view: `pred_keypoints_3d` in each
    camera's own frame + `pred_keypoints_2d`; fuse/main_raw.py:192-197) for the fusion path (SURVEY row N3).
    Xl / Xr (T,J,3): the ground truth in the left / right camera frame of rig '2b' + N(0, 2 cm) + a few 30 cm outliers;
    Ul / Ur (T,J,2): pinhole pixels + N(0, 2 px); a fraction of joints is missing (NaN rows) in either view - except the
    five key joints of the canonical frame, which only go missing in whole frames (1 %).  Returns dict of arrays."""
    rng = np.random.default_rng(seed)
    R, t = rig("2b")
    X = skeleton_clip(T, J, rng)
    out = {}
    for name, v in (("l", 0), ("r", 1)):
        Xc = X @ R[v].T + t[v]
        U = pinhole(X, R[v], t[v], K_CALIB) + rng.normal(0.0, 2.0, (T, J, 2))
        Xn = Xc + rng.normal(0.0, 0.02, Xc.shape)
        o = rng.random((T, J)) < outlier_frac
        Xn[o] += rng.normal(0.0, 0.3, (int(o.sum()), 3))
        m3 = rng.random((T, J)) < nan_frac
        m2 = rng.random((T, J)) < nan_frac
        key = [k for k in (14, 11, 12, 5, 6) if k < J]
        m3[:, key] = False
        whole = rng.random(T) < 0.01
        m3[np.ix_(whole, key)] = True
        Xn[m3] = np.nan
        U[m2] = np.nan
        out["X" + name], out["U" + name] = Xn.astype(dtype), U.astype(dtype)
    return out
