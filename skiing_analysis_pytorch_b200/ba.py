"""Levenberg-Marquardt bundle adjustment driver (host side).

All arithmetic runs in libska.so (ska_ba_* entry points, include/ska.h): linearise + Schur
accumulation, reduced-system Cholesky, back-substitution + trial cost, and the accept/reject
controller are CUDA kernels; this module owns the device buffers, enqueues the four launches of a
trial on the current stream and - when the clip is sharded over ranks - all-reduces the two tiny
fp64 payloads with torch.distributed (NCCL on GPUs).  Nothing here synchronises with the host until
the caller reads the results, so a whole solve can be captured in a CUDA graph (``graph=True``).

Fills the slot of the reference's undefined ``run_local_ba`` (vggt/multi_view_process.py:553-564)
on the cost the reference defines in bundle_adjustment/loss.py:17-94.  Algorithm spec: oracle/lm.py.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi, _lib

MODES = ("pose_only", "pose_cam_t", "full")  # vggt/multi_view_process.py:338, configs/vggt.yaml:52


def free_mask(n_cams: int, mode: str = "full") -> int:
    """Bit (6*c + r) set = parameter r of camera c is optimised (r 0..2 rotation, 3..5 translation).
    Camera 0 is the gauge and never moves.  pose_only: points only; pose_cam_t: points + camera
    translations; full: points + rotations + translations."""
    if mode not in MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {MODES}")
    per_cam = {"pose_only": 0, "pose_cam_t": 0b111000, "full": 0b111111}[mode]
    m = 0
    for c in range(1, n_cams):
        m |= per_cam << (6 * c)
    return m


def _stream_ptr(dev) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def frame_shard(total_frames: int, world: int, rank: int):
    """Contiguous frame range [t0, t1) of `rank` when a clip is sharded over `world` ranks (points
    are private to a frame, so BA and triangulation shard by frame range; SURVEY.md section 8e)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, rem = divmod(int(total_frames), int(world))
    t0 = rank * base + min(rank, rem)
    return t0, t0 + base + (1 if rank < rem else 0)


class LMSequencer:
    """Engine-agnostic sequencing of LM trials over a frame-sharded clip.

    A trial is  linearize -> all-reduce(red) -> solve -> backsub -> all-reduce(red2) -> control;
    every rank holds its own frame range, runs the identical reduced solve and controller on the
    reduced sums, and therefore takes the identical accept/reject decision without any further
    communication.  Subclasses provide the four steps and the two payload tensors `red` / `red2`
    (the CUDA engine below; an fp64 numpy engine in tests/ exercises this class over gloo)."""

    group = None
    local_only = False  # True: never all-reduce even inside an initialised process group (unsharded solve)
    max_iters = 0
    iters_done = 0
    _graph = None

    def _distributed(self) -> bool:
        return (not self.local_only and torch.distributed.is_available() and torch.distributed.is_initialized()
                and torch.distributed.get_world_size(self.group) > 1)

    peer = None  # peer.PeerExchange: the exchange over NVLink peer memory instead of NCCL (CUDA engines)

    def _allreduce(self, t: torch.Tensor):
        if self._distributed():
            if self.peer is not None and self.peer.fits(t):
                self.peer.all_reduce(t)
            else:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=self.group)

    fused_exchange = False  # CUDA engines with a peer exchange: solve / control all-reduce their payloads in their own prologue

    def trial(self):
        """Enqueue one LM trial (accepted or rejected by the controller)."""
        self.linearize()
        if not self.fused_exchange:
            self._allreduce(self.red)
        self.solve()
        self.backsub()
        if not self.fused_exchange:
            self._allreduce(self.red2)
        self.control()

    def run(self, num_iters: int, graph: bool = False):
        """Enqueue `num_iters` trials.  graph=True captures one trial - its launches AND, on a sharded clip, its NCCL
        all-reduces - in a CUDA graph and replays it: the trial of a 100k-frame clip on 8 GPUs is ~20 us of kernels
        behind ~8 launches and 2 collectives, i.e. launch-latency bound when enqueued one by one."""
        num_iters = int(num_iters)
        if num_iters <= 0:
            return self
        if self.iters_done + num_iters > self.max_iters:
            raise ValueError(f"history buffer holds {self.max_iters} trials; raise max_iters")
        if graph:
            if self._graph is None:
                self.trial()  # warm-up outside capture (module load, attribute setting, NCCL communicator set-up)
                num_iters -= 1
                self.iters_done += 1
                g = torch.cuda.CUDAGraph()
                s = torch.cuda.Stream(self.dev)
                s.wait_stream(torch.cuda.current_stream(self.dev))
                with torch.cuda.stream(s):
                    with torch.cuda.graph(g, stream=s):
                        self.trial()
                torch.cuda.current_stream(self.dev).wait_stream(s)
                self._graph = g
                # capture does not execute: the captured trial still has to run num_iters times
            for _ in range(num_iters):
                self._graph.replay()
        else:
            for _ in range(num_iters):
                self.trial()
        self.iters_done += num_iters
        return self


class BundleAdjuster(LMSequencer):
    """One BA problem resident on one GPU (this rank's frame shard).

    x2d   (T,C,J,2) float32 CUDA [layout "TCJ2", the reference's] or (C,T,J,2) ["CTJ2"]
    conf  (T,C,J) / (C,T,J) float32 CUDA
    K     (C,3,3) | (3,3); R0 (C,3,3); t0 (C,3): host arrays, world->camera, shared over the clip
    X0    (T,J,3) CUDA tensor (any float dtype) - e.g. the output of triangulate_reproject
    group torch.distributed process group when the clip is sharded by frame range over ranks
          (None = the default group when torch.distributed is initialised with world size > 1);
          local_only=True solves this rank's data alone, without any collective
    loss  "l2" (default: loss.py's squared pixel error), "huber" or "cauchy": a robust M-estimator against gross 2D
          detector failures, solved by iteratively reweighted Gauss-Newton (include/ska.h, DESIGN.md section 5);
    loss_scale  its scale in pixels (required, > 0, for "huber" / "cauchy").  `history` and `cost` report the robust cost
    """

    def __init__(self, x2d, conf, K, R0, t0, X0, *, layout: str = "TCJ2", mode: str = "full", lam0: float = 1e-3,
                 max_iters: int = 64, group=None, force_wide: bool = False, local_only: bool = False, tensor_core: bool = False,
                 peer_exchange: bool = True, fuse_exchange: bool = True, loss: str = "l2", loss_scale=None):
        self.local_only = bool(local_only)
        loss_id, loss_scale = _cabi.check_loss(loss, loss_scale)
        if loss != "l2" and tensor_core:
            raise ValueError("tensor_core=True implements the L2 loss only")
        if not (x2d.is_cuda and conf.is_cuda and X0.is_cuda):
            raise RuntimeError("x2d, conf and X0 must be CUDA tensors: this package has no CPU path")
        if x2d.dtype != torch.float32 or conf.dtype != torch.float32:
            raise TypeError("x2d and conf must be float32")
        if x2d.dim() != 4 or x2d.shape[-1] != 2:
            raise ValueError(f"x2d must be 4-D with last dim 2, got {tuple(x2d.shape)}")
        if layout == "TCJ2":
            T, Cn, J, _ = x2d.shape
            self.layout = _cabi.LAYOUT_FRAME_MAJOR
            cshape = (T, Cn, J)
        elif layout == "CTJ2":
            Cn, T, J, _ = x2d.shape
            self.layout = _cabi.LAYOUT_VIEW_MAJOR
            cshape = (Cn, T, J)
        else:
            raise ValueError("layout must be 'TCJ2' or 'CTJ2'")
        if tuple(conf.shape) != cshape:
            raise ValueError(f"conf shape {tuple(conf.shape)} does not match {cshape}")
        if tuple(X0.shape) != (T, J, 3):
            raise ValueError(f"X0 must be ({T},{J},3), got {tuple(X0.shape)}")
        if not 2 <= Cn <= _cabi.MAX_BA_VIEWS:
            raise ValueError(f"need 2..{_cabi.MAX_BA_VIEWS} cameras, got {Cn}")
        R0 = np.asarray(R0, np.float64)
        t0 = np.asarray(t0, np.float64).reshape(Cn, 3)
        K = np.asarray(K, np.float64)
        K = np.broadcast_to(K, (Cn, 3, 3)) if K.ndim == 2 else K.reshape(Cn, 3, 3)
        if R0.shape != (Cn, 3, 3):
            raise ValueError(f"R0 must be ({Cn},3,3), got {R0.shape}")
        self.T, self.C, self.J = T, Cn, J
        self.N = T * J
        self.dev = x2d.device
        self.group = group
        if peer_exchange and self._distributed():
            from . import peer as _peer

            self.peer = _peer.shared(group, self.dev)  # None where peer memory cannot be mapped: NCCL then
        self.mask = free_mask(Cn, mode)
        self.mode = mode
        self.max_iters = int(max_iters)
        self.x2d = x2d.contiguous()
        self.conf = conf.contiguous()
        self.lib = _lib.load()
        dev = self.dev
        f64 = dict(dtype=torch.float64, device=dev)
        cams = np.zeros((2, Cn, _cabi.BA_CAM_DOUBLES))
        for s in range(2):
            cams[s, :, 0:9] = R0.reshape(Cn, 9)
            cams[s, :, 9:12] = t0
            cams[s, :, 12:21] = K.reshape(Cn, 9)
        self.cams = torch.from_numpy(cams).to(dev)
        self.Xpp = torch.empty((2, max(self.N, 1), 3), dtype=torch.float32, device=dev)
        if self.N:
            self.Xpp[0, : self.N].copy_(X0.reshape(-1, 3))
        ctrl = np.zeros(_cabi.BA_CTRL_DOUBLES)
        ctrl[_cabi.BA_CTRL_LAMBDA] = lam0
        ctrl[_cabi.BA_CTRL_NU] = 2.0
        self.ctrl = torch.from_numpy(ctrl).to(dev)
        self.red = torch.zeros(int(self.lib.ska_ba_red_doubles(Cn)), **f64)
        self.red2 = torch.zeros(_cabi.BA_RED2_DOUBLES, **f64)
        self.delta = torch.zeros(Cn * 6, **f64)
        self.hist = torch.zeros((self.max_iters, _cabi.BA_HIST_DOUBLES), **f64)
        with torch.cuda.device(dev):
            ws = int(self.lib.ska_ba_workspace_bytes(Cn))
        self.ws = torch.empty(ws, dtype=torch.uint8, device=dev)
        self.prob = _cabi.SkaBaProblem(
            C=Cn, J=J, T=T, layout=self.layout, flags=(_cabi.BA_FORCE_WIDE if force_wide else 0) | (_cabi.BA_TENSOR_CORE if tensor_core else 0),
            d_x2d=self.x2d.data_ptr(), d_conf=self.conf.data_ptr(), d_Xpp=self.Xpp.data_ptr(),
            d_cams=self.cams.data_ptr(), d_ctrl=self.ctrl.data_ptr(), d_red=self.red.data_ptr(),
            d_red2=self.red2.data_ptr(), d_delta=self.delta.data_ptr(), d_hist=self.hist.data_ptr(),
            d_workspace=self.ws.data_ptr(), ws_bytes=ws, hist_rows=self.max_iters,
            peer=(C.addressof(self.peer.comm) if fuse_exchange and self.peer is not None and self.peer.slot >= 1024 else None),
            loss=loss_id, loss_scale=loss_scale,
        )
        self.loss = loss
        self.fused_exchange = bool(self.prob.peer)
        self._graph = None
        self.iters_done = 0
        # global sum of confidences (loss.py:94 denominator), computed on the device
        sum_out = C.c_void_p(self.ctrl.data_ptr() + 8 * _cabi.BA_CTRL_SUMCONF)
        with torch.cuda.device(dev):
            _lib.check(self.lib.ska_ba_sum_f32(C.c_void_p(self.conf.data_ptr()), self.conf.numel(), sum_out,
                                               C.c_void_p(self.ws.data_ptr()), ws, _stream_ptr(dev)))
        self._allreduce(self.ctrl[_cabi.BA_CTRL_SUMCONF: _cabi.BA_CTRL_SUMCONF + 1])

    # ------------------------------------------------------------------ pieces of one trial
    def linearize(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_linearize_f32(C.byref(self.prob), _stream_ptr(self.dev)))

    def solve(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_solve_f64(C.byref(self.prob), C.c_uint64(self.mask), _stream_ptr(self.dev)))

    def backsub(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_backsub_f32(C.byref(self.prob), _stream_ptr(self.dev)))

    def control(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_control_f64(C.byref(self.prob), _stream_ptr(self.dev)))

    # ------------------------------------------------------------------ results (synchronise)
    @property
    def history(self):
        if self.peer is not None:
            self.peer.check()  # an exchange that gave up waiting for a peer invalidates the trajectory: raise, never return it
        h = self.hist[: self.iters_done].cpu().numpy()
        keys = ("iter", "cost", "trial_cost", "lam", "rho", "accepted", "n_clamped", "pred")
        out = []
        for row in h:
            d = dict(zip(keys, (float(x) for x in row)))
            d["iter"] = int(d["iter"])
            d["accepted"] = bool(d["accepted"])
            d["n_clamped"] = int(d["n_clamped"])
            out.append(d)
        return out

    @property
    def X(self) -> torch.Tensor:
        cur = int(self.ctrl[_cabi.BA_CTRL_CUR].item())
        return self.Xpp[cur, : self.N].view(self.T, self.J, 3)

    @property
    def R(self) -> np.ndarray:
        return self.cams[0, :, 0:9].cpu().numpy().reshape(self.C, 3, 3)

    @property
    def t(self) -> np.ndarray:
        return self.cams[0, :, 9:12].cpu().numpy()

    @property
    def cost(self) -> float:
        return float(self.ctrl[_cabi.BA_CTRL_COST].item())


CALIB_MODES = ("full", "extr_focal", "intr_only")
CALIB_PARAM_NAMES = ("wx", "wy", "wz", "tx", "ty", "tz", "fx", "fy", "cx", "cy", "k1", "k2", "p1", "p2", "k3")


def calib_free_mask(n_cams: int, mode: str = "full") -> int:
    """Bit (15*c + r) set = parameter r of camera c is optimised; r indexes CALIB_PARAM_NAMES.  Camera 0's extrinsics
    are the gauge.  full: all extrinsics (c >= 1) + every camera's 9 intrinsics; extr_focal: extrinsics + fx fy cx cy;
    intr_only: the 9 intrinsics of every camera with all extrinsics fixed."""
    if mode not in CALIB_MODES:
        raise ValueError(f"unknown calibration mode {mode!r}; expected one of {CALIB_MODES}")
    intr = {"full": 0x7FC0, "extr_focal": 0x03C0, "intr_only": 0x7FC0}[mode]
    extr = 0 if mode == "intr_only" else 0x3F
    m = 0
    for c in range(n_cams):
        m |= (intr | (extr if c >= 1 else 0)) << (_cabi.BA_CALIB_PARAMS * c)
    return m


class CalibratingBundleAdjuster(BundleAdjuster):
    """LM over the points, the extrinsics AND every camera's intrinsics + distortion (15 parameters per camera) -
    BASELINE config 3's "Rodrigues extrinsics + intrinsics/distortion".  Specification: oracle/lm_calib.py.

    Arguments as BundleAdjuster, plus
      K            (C,3,3) | (3,3) zero-skew intrinsics (fx, fy, cx, cy are read from it)
      dist         None | (5,) | (C,5): initial [k1, k2, p1, p2, k3] (cv2 order, the model of triangulation/reproject.py:77-78)
      calib        one of CALIB_MODES, or an explicit integer free mask (calib_free_mask)
      prior_rho    None | (9,) | (C,9): precision of a Gaussian prior on [fx fy cx cy k1 k2 p1 p2 k3]
                   (cost += sum rho (theta - prior_theta)^2); prior_theta defaults to the initial intrinsics
    Built for 2 cameras (config 3); libska returns SKA_EUNSUPPORTED otherwise."""

    def __init__(self, x2d, conf, K, R0, t0, X0, *, dist=None, calib="full", prior_rho=None, prior_theta=None, **kw):
        kw.pop("mode", None)
        kw.pop("force_wide", None)
        super().__init__(x2d, conf, K, R0, t0, X0, **kw)
        Cn, dev = self.C, self.dev
        if Cn != 2:
            raise ValueError("the calibrating BA is built for 2 cameras (BASELINE config 3)")
        K = np.asarray(K, np.float64)
        K = np.broadcast_to(K, (Cn, 3, 3)) if K.ndim == 2 else K.reshape(Cn, 3, 3)
        if np.abs(K[:, 0, 1]).max() > 0 or np.abs(K[:, 1, 0]).max() > 0:
            raise ValueError("the calibrating BA uses cv2's zero-skew camera matrix")
        theta = np.zeros((Cn, _cabi.BA_CALIB_INTRINSICS))
        theta[:, 0], theta[:, 1], theta[:, 2], theta[:, 3] = K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]
        if dist is not None:
            theta[:, 4:] = np.broadcast_to(np.asarray(dist, np.float64), (Cn, 5))
        cams = self.cams.cpu().numpy()
        cams[:, :, 12:24] = 0.0
        cams[:, :, 12:21] = theta[None]
        self.cams = torch.from_numpy(cams).to(dev)
        self.mask = calib_free_mask(Cn, calib) if isinstance(calib, str) else int(calib)
        self.mode = calib
        f64 = dict(dtype=torch.float64, device=dev)
        self.prior = None
        if prior_rho is not None:
            pr = np.zeros((Cn, 2, _cabi.BA_CALIB_INTRINSICS))
            pr[:, 0] = theta if prior_theta is None else np.broadcast_to(np.asarray(prior_theta, np.float64), theta.shape)
            pr[:, 1] = np.broadcast_to(np.asarray(prior_rho, np.float64), theta.shape)
            self.prior = torch.from_numpy(pr).to(dev)
        self.red = torch.zeros(int(self.lib.ska_ba_calib_red_doubles(Cn)), **f64)
        self.delta = torch.zeros(Cn * _cabi.BA_CALIB_PARAMS, **f64)
        with torch.cuda.device(dev):
            ws = max(int(self.lib.ska_ba_calib_workspace_bytes(Cn)), self.ws.numel())
        self.ws = torch.empty(ws, dtype=torch.uint8, device=dev)
        self.prob.d_cams = self.cams.data_ptr()
        self.prob.d_red = self.red.data_ptr()
        self.prob.d_delta = self.delta.data_ptr()
        self.prob.d_workspace = self.ws.data_ptr()
        self.prob.ws_bytes = ws
        self.prob.flags = 0

    def linearize(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_calib_linearize_f32(C.byref(self.prob), _stream_ptr(self.dev)))

    def solve(self):
        pr = C.c_void_p(self.prior.data_ptr()) if self.prior is not None else None
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_calib_solve_f64(C.byref(self.prob), C.c_uint64(self.mask), pr, _stream_ptr(self.dev)))

    def backsub(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_calib_backsub_f32(C.byref(self.prob), _stream_ptr(self.dev)))

    def control(self):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ska_ba_calib_control_f64(C.byref(self.prob), _stream_ptr(self.dev)))

    @property
    def theta(self) -> np.ndarray:
        """(C,9) current [fx fy cx cy k1 k2 p1 p2 k3]."""
        return self.cams[0, :, 12:21].cpu().numpy()

    @property
    def K(self) -> np.ndarray:
        th = self.theta
        K = np.zeros((self.C, 3, 3))
        K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2], K[:, 2, 2] = th[:, 0], th[:, 1], th[:, 2], th[:, 3], 1.0
        return K

    @property
    def dist(self) -> np.ndarray:
        return self.theta[:, 4:].copy()


def ba_calibrate(x2d, conf, K, R0, t0, X0, num_iters: int = 20, **kw):
    """Convenience wrapper: build a CalibratingBundleAdjuster, run `num_iters` trials, return it."""
    graph = kw.pop("graph", False)
    kw.setdefault("max_iters", num_iters)
    return CalibratingBundleAdjuster(x2d, conf, K, R0, t0, X0, **kw).run(num_iters, graph=graph)


def ba_solve(x2d, conf, K, R0, t0, X0, num_iters: int = 20, **kw):
    """Convenience wrapper: build a BundleAdjuster, run `num_iters` trials, return it."""
    graph = kw.pop("graph", False)
    kw.setdefault("max_iters", num_iters)
    return BundleAdjuster(x2d, conf, K, R0, t0, X0, **kw).run(num_iters, graph=graph)


def _mean_rotation(R: np.ndarray) -> np.ndarray:
    """Chordal mean of rotations (T,3,3) -> (3,3): SVD projection of the arithmetic mean."""
    U, _, Vt = np.linalg.svd(R.mean(0))
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(U @ Vt))])
    return U @ D @ Vt


FIRST_ORDER_WEIGHTS = dict(reproj=1.0, smooth=0.1, baseline=0.01, bone_length=0.1, pose_temporal=0.1)  # configs/vggt.yaml:46-50
FIRST_ORDER_TERMS = ("reproj", "smooth", "baseline", "bone_length", "pose_temporal")


class _DeviceAdam:
    """torch.optim.Adam's update applied by libska (ska_adam_step_*): state and parameters stay on the device.  The
    per-iteration scalars lr / (1 - b1^k) and 1 / sqrt(1 - b2^k) live in device memory (`scal`, refreshed by `begin`
    from the device-side iteration counter `k`), so one captured CUDA graph of an iteration replays for every k."""

    def __init__(self, lr, dev, betas=(0.9, 0.999), eps=1e-8):
        self.lr, self.b1, self.b2, self.eps, self.state = float(lr), betas[0], betas[1], float(eps), {}
        self.lib = _lib.load()
        self.k = torch.zeros(1, dtype=torch.float64, device=dev)
        self.scal = torch.zeros(2, dtype=torch.float64, device=dev)

    def begin(self):
        self.k += 1.0
        self.scal[0:1] = self.lr / (1.0 - torch.pow(self.b1, self.k))
        self.scal[1:2] = torch.rsqrt(1.0 - torch.pow(self.b2, self.k))

    def apply(self, name, p, g, step_out=None):
        """p <- p - step (p may be None: only step_out is written)."""
        ref = p if p is not None else step_out
        m, v = self.state.setdefault(name, (torch.zeros_like(ref), torch.zeros_like(ref)))
        g = g.contiguous()
        sfx = "f32" if ref.dtype == torch.float32 else "f64"
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        with torch.cuda.device(ref.device):
            _lib.check(getattr(self.lib, f"ska_adam_step_{sfx}")(ptr(p), ptr(g), ptr(m), ptr(v), ref.numel(), 0.0, self.b1, self.b2, self.eps,
                                                                 1.0, ptr(step_out), ptr(self.scal), _stream_ptr(ref.device)))


def run_local_ba_first_order(K_torch, R_init_torch, t_init_torch, X3d_init_torch, x2d_torch, conf2d_torch, num_iters=200, lr=1e-3,
                             device="cuda", mode="pose_only", weights=None, graph=True, fused=True, group=None):
    """First-order (Adam) minimisation of the reference's full configured objective (SURVEY row N1, first-order form;
    specification oracle/first_order.py):
        w_reproj reprojection_loss + w_smooth camera_smooth_loss + w_baseline baseline_reg_loss
        + w_bone_length bone_length_loss + w_pose_temporal pose_temporal_loss        (bundle_adjustment/loss.py:90-155)
    with the weights / lr / num_iters of configs/vggt.yaml:43-52 and PER-FRAME cameras R (T,C,3,3), t (T,C,3) exactly as
    the call site passes them (vggt/multi_view_process.py:546-564).  mode: "pose_only" (X), "pose_cam_t" (X, t), "full"
    (X, t and R; rotations move on SO(3) through the left tangent).  Every loss value and analytic gradient comes from the
    loss kernels (losses.py -> libska), the updates from ska_adam_step_* / ska_so3_*; computed in X3d_init's dtype
    (float32 / float64) like loss.py:27-32.  graph=True captures one iteration in a CUDA graph and replays it; nothing
    synchronises with the host until the history is read back.  fused=True (default) calls the loss entry points
    directly and folds every weight / count into the multi-term Adam kernel (ska_adam_step_terms_*): ~35 launches per
    iteration and no element-wise torch arithmetic; fused=False goes through the autograd wrappers of losses.py (the
    same kernels plus ~100 small torch kernels of gradient scaling / accumulation) - kept as the cross-check.
    group: a torch.distributed process group = the clip is sharded by contiguous frame ranges in rank order and the
    arguments are THIS rank's frames (SURVEY row e3).  The temporal / smoothness terms then read a one-frame halo of the
    neighbouring shards (exchanged after every step), the bone / baseline means and every loss sum are all-reduced, the counts
    are the clip's; every rank records the same history and returns its own frames.
    Returns (R_opt, t_opt, X_opt, history) with one history row per iteration:
    {iter, loss, reproj, smooth, baseline, bone_length, pose_temporal} (values before that iteration's step)."""
    from . import losses

    if mode not in MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {MODES}")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("run_local_ba runs on a CUDA device: this package has no CPU path")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    w = dict(FIRST_ORDER_WEIGHTS, **(weights or {}))
    dt = X3d_init_torch.dtype if X3d_init_torch.dtype in (torch.float32, torch.float64) else torch.float32
    to = lambda a: a.detach().to(dev, dt).contiguous().clone()
    X, R, t = to(X3d_init_torch), to(R_init_torch), to(t_init_torch)
    if R.dim() != 4 or t.dim() != 3:
        raise ValueError(f"per-frame cameras expected: R (T,C,3,3), t (T,C,3); got {tuple(R.shape)}, {tuple(t.shape)}")
    K, x2d, conf = to(K_torch), to(x2d_torch), to(conf2d_torch)
    lib = _lib.load()
    sfx = "f32" if dt == torch.float32 else "f64"
    num_iters = int(num_iters)
    # ---- frame sharding: this rank's frames live in rows 1..Tl of buffers with one halo frame on each side
    tdist = torch.distributed
    world, rank = (tdist.get_world_size(group), tdist.get_rank(group)) if group is not None else (1, 0)
    sharded = world > 1
    Tl = X.shape[0]
    T_glob = Tl
    if sharded:
        if not fused:
            raise ValueError("the sharded first-order solve runs the fused form (fused=True)")
        if Tl < 1:
            raise ValueError("every rank needs at least one frame")
        tot = torch.tensor([float(Tl)], dtype=torch.float64, device=dev)
        tdist.all_reduce(tot, group=group)
        T_glob = int(round(float(tot.item())))
        Xe = torch.zeros((Tl + 2,) + tuple(X.shape[1:]), dtype=dt, device=dev)
        Re = torch.eye(3, dtype=dt, device=dev).expand(Tl + 2, R.shape[1], 3, 3).contiguous()
        te = torch.zeros((Tl + 2,) + tuple(t.shape[1:]), dtype=dt, device=dev)
        Xe[1:-1], Re[1:-1], te[1:-1] = X, R, t
        X, R, t = Xe[1:-1], Re[1:-1], te[1:-1]  # contiguous views: the kernels update the halo buffers' interior in place
        has_prev, has_next = rank > 0, rank < world - 1
        lo, hi = (0 if has_prev else 1), (Tl + 2 if has_next else Tl + 1)  # rows whose gradient needs both neighbours: [lo, hi)
        n_edge = X.shape[1] * 3 + R.shape[1] * 12

        def exchange_halo():
            mine = torch.empty((2, n_edge), dtype=dt, device=dev)
            for e, row_ in enumerate((1, Tl)):
                mine[e] = torch.cat([Xe[row_].reshape(-1), Re[row_].reshape(-1), te[row_].reshape(-1)])
            flat = torch.empty(world * mine.numel(), dtype=dt, device=dev)
            tdist.all_gather_into_tensor(flat, mine.reshape(-1), group=group)
            everyone = flat.view(world, 2, n_edge)
            j3, c9 = X.shape[1] * 3, R.shape[1] * 9
            for row_, src in ((0, everyone[rank - 1, 1] if has_prev else None), (Tl + 1, everyone[rank + 1, 0] if has_next else None)):
                if src is not None:
                    Xe[row_] = src[:j3].view_as(Xe[row_])
                    Re[row_] = src[j3:j3 + c9].view_as(Re[row_])
                    te[row_] = src[j3 + c9:].view_as(te[row_])

        exchange_halo()
    opt = _DeviceAdam(lr, dev)
    n_rot = R.shape[0] * R.shape[1]
    gw = torch.empty((n_rot, 3), dtype=dt, device=dev)
    sw = torch.empty((n_rot, 3), dtype=dt, device=dev)
    hist = torch.zeros((max(num_iters, 1), 1 + len(FIRST_ORDER_TERMS)), dtype=torch.float64, device=dev)
    row = torch.zeros((1, 1 + len(FIRST_ORDER_TERMS)), dtype=torch.float64, device=dev)
    ptr = lambda a: C.c_void_p(a.data_ptr())

    # ---------------------------------------------------------------- fused form: raw kernels, weights folded into Adam
    Tn, Jn, Cn = X.shape[0], X.shape[1], R.shape[1]
    keep = [k for k, (i, j) in enumerate(losses.BONES) if i < Jn and j < Jn]
    nb = len(keep)
    use = dict(reproj=bool(w["reproj"]), smooth=bool(w["smooth"]) and T_glob > 1, baseline=bool(w["baseline"]) and Cn >= 2,
               bone_length=bool(w["bone_length"]) and nb > 0, pose_temporal=bool(w["pose_temporal"]) and T_glob > 1)
    cam_free, rot_free = mode != "pose_only", mode == "full"
    f64d = dict(dtype=torch.float64, device=dev)
    if fused:
        bi = (C.c_int32 * max(nb, 1))(*[losses.BONES[k][0] for k in keep])
        bj = (C.c_int32 * max(nb, 1))(*[losses.BONES[k][1] for k in keep])
        with torch.cuda.device(dev):
            ws_bytes = max(int(lib.ska_loss_workspace_bytes(Cn)), int(lib.ska_reg_workspace_bytes()), 1 << 20)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        like = lambda a, on: torch.zeros_like(a) if on else None
        gX_r, gX_b, gX_t = like(X, use["reproj"]), like(X, use["bone_length"]), like(X, use["pose_temporal"])
        gR_r, gR_s, gR_b = like(R, use["reproj"] and rot_free), like(R, use["smooth"] and cam_free), like(R, use["baseline"] and cam_free)
        gt_r, gt_s, gt_b = like(t, use["reproj"] and cam_free), like(t, use["smooth"] and cam_free), like(t, use["baseline"] and cam_free)
        # the loss sums in ONE buffer (one all-reduce per iteration when sharded), the two means in another (needed in between)
        fin, mid = torch.zeros(7 + _cabi.MAX_BONES, **f64d), torch.zeros(_cabi.MAX_BONES + 1, **f64d)
        s_r, s_t, s_s, s_bl, s_b1 = fin[0:4], fin[4:5], fin[5:6], fin[6:7], fin[7:]
        s_b0, s_m = mid[:_cabi.MAX_BONES], mid[_cabi.MAX_BONES:]
        if sharded:  # gradients of the coupled terms over [halo | own | halo]; the Adam step reads the interior
            scratch1 = torch.zeros(1, **f64d)
            gX_t_e = torch.zeros_like(Xe) if use["pose_temporal"] else None
            gR_s_e = torch.zeros_like(Re) if use["smooth"] and cam_free else None
            gt_s_e = torch.zeros_like(te) if use["smooth"] and cam_free else None
            gX_t = gX_t_e[1:-1] if gX_t_e is not None else None
            gR_s = gR_s_e[1:-1] if gR_s_e is not None else None
            gt_s = gt_s_e[1:-1] if gt_s_e is not None else None
        gw3 = [torch.empty((n_rot, 3), dtype=dt, device=dev) for _ in range(3)] if rot_free else None
        P = lambda a: None if a is None else C.c_void_p(a.data_ptr())
        fn = lambda name: getattr(lib, f"{name}_{sfx}")
        strm = lambda: _stream_ptr(dev)

        def eval_terms_sharded():
            PO = lambda a, r0: None if a is None else C.c_void_p(a[r0:].data_ptr())
            with torch.cuda.device(dev):
                if use["reproj"]:
                    _lib.check(fn("ska_reprojection_loss")(P(X), Tn, Jn, Cn, P(R), Cn * 9, P(t), Cn * 3, P(K), 0, P(x2d), P(conf), P(s_r), P(gX_r),
                                                          P(gR_r), P(gt_r), None, P(ws), ws_bytes, strm()))
                if use["pose_temporal"]:  # gradient over every row that has both neighbours here; value over the pairs (t, t+1) this rank owns
                    _lib.check(fn("ska_pose_temporal")(PO(Xe, lo), hi - lo, Jn, P(scratch1), PO(gX_t_e, lo), P(ws), ws_bytes, strm()))
                    _lib.check(fn("ska_pose_temporal")(PO(Xe, 1), hi - 1, Jn, P(s_t), None, P(ws), ws_bytes, strm()))
                if use["smooth"]:
                    _lib.check(fn("ska_camera_smooth")(PO(Re, lo), PO(te, lo), hi - lo, Cn, P(scratch1), PO(gR_s_e, lo), PO(gt_s_e, lo), P(ws), ws_bytes, strm()))
                    _lib.check(fn("ska_camera_smooth")(PO(Re, 1), PO(te, 1), hi - 1, Cn, P(s_s), None, None, P(ws), ws_bytes, strm()))
                if use["bone_length"]:
                    _lib.check(fn("ska_bone_length")(P(X), Tn, Jn, bi, bj, nb, None, P(s_b0), None, P(ws), ws_bytes, strm()))
                if use["baseline"]:
                    _lib.check(fn("ska_baseline_reg")(P(R), P(t), Tn, Cn, None, P(s_m), None, None, P(ws), ws_bytes, strm()))
            if use["bone_length"] or use["baseline"]:
                tdist.all_reduce(mid, group=group)  # the clip's bone lengths / baselines
                mid.div_(T_glob)
            with torch.cuda.device(dev):
                if use["bone_length"]:
                    _lib.check(fn("ska_bone_length")(P(X), Tn, Jn, bi, bj, nb, P(s_b0), P(s_b1), P(gX_b), P(ws), ws_bytes, strm()))
                if use["baseline"]:
                    _lib.check(fn("ska_baseline_reg")(P(R), P(t), Tn, Cn, P(s_m), P(s_bl), P(gR_b), P(gt_b), P(ws), ws_bytes, strm()))
            tdist.all_reduce(fin, group=group)

        def eval_terms():
            if sharded:
                return eval_terms_sharded()
            with torch.cuda.device(dev):
                if use["reproj"]:
                    _lib.check(fn("ska_reprojection_loss")(P(X), Tn, Jn, Cn, P(R), Cn * 9, P(t), Cn * 3, P(K), 0, P(x2d), P(conf), P(s_r), P(gX_r),
                                                          P(gR_r), P(gt_r), None, P(ws), ws_bytes, strm()))
                if use["pose_temporal"]:
                    _lib.check(fn("ska_pose_temporal")(P(X), Tn, Jn, P(s_t), P(gX_t), P(ws), ws_bytes, strm()))
                if use["bone_length"]:
                    _lib.check(fn("ska_bone_length")(P(X), Tn, Jn, bi, bj, nb, None, P(s_b0), None, P(ws), ws_bytes, strm()))
                    s_b0.div_(Tn)  # per-bone mean length over the clip: the (detached) reference of loss.py:141-146
                    _lib.check(fn("ska_bone_length")(P(X), Tn, Jn, bi, bj, nb, P(s_b0), P(s_b1), P(gX_b), P(ws), ws_bytes, strm()))
                if use["smooth"]:
                    _lib.check(fn("ska_camera_smooth")(P(R), P(t), Tn, Cn, P(s_s), P(gR_s), P(gt_s), P(ws), ws_bytes, strm()))
                if use["baseline"]:
                    _lib.check(fn("ska_baseline_reg")(P(R), P(t), Tn, Cn, None, P(s_m), None, None, P(ws), ws_bytes, strm()))
                    s_m.div_(Tn)
                    _lib.check(fn("ska_baseline_reg")(P(R), P(t), Tn, Cn, P(s_m), P(s_bl), P(gR_b), P(gt_b), P(ws), ws_bytes, strm()))

        eval_terms()  # set-up evaluation: the sum of confidences (constant over the solve) fixes the reprojection scale
        sum_conf = float(s_r[1].item()) if use["reproj"] else 1.0
        c_r = w["reproj"] / (sum_conf + 1e-6)
        c_t = w["pose_temporal"] / max((T_glob - 1) * Jn * 3, 1)
        c_b = w["bone_length"] / max(T_glob * nb, 1)
        c_s = w["smooth"] / max((T_glob - 1) * Cn * 3, 1)
        c_bl = w["baseline"] / max(T_glob, 1)

        def terms3(cands):
            live = [(g, sc) for g, sc in cands if g is not None]
            while len(live) < 3:
                live.append((None, 0.0))
            return live

        def adam_terms(name, p, cands, step_out=None):
            (g0, a0), (g1, a1), (g2, a2) = terms3(cands)
            ref = p if p is not None else step_out
            if g0 is None:
                return
            m, v = opt.state.setdefault(name, (torch.zeros_like(ref), torch.zeros_like(ref)))
            with torch.cuda.device(dev):
                _lib.check(fn("ska_adam_step_terms")(P(p), P(g0), a0, P(g1), a1, P(g2), a2, P(m), P(v), ref.numel(), opt.b1, opt.b2, opt.eps,
                                                    P(step_out), P(opt.scal), strm()))

        order = ("reproj", "smooth", "baseline", "bone_length", "pose_temporal")   # FIRST_ORDER_TERMS
        sums5 = (C.c_void_p * 5)(*[(src.data_ptr() if use[name] else None) for name, src in zip(order, (s_r, s_s, s_bl, s_b1, s_t))])
        coef5 = (C.c_double * 5)(w["reproj"], c_s, c_bl, c_b, c_t)

        def fused_iteration():
            eval_terms()
            with torch.cuda.device(dev):   # history row k, k <- k + 1, Adam scalars of step k: one single-thread launch
                _lib.check(lib.ska_first_order_record_f64(P(opt.k), P(opt.scal), P(hist), hist.shape[0], sums5, P(s_r[1:2]) if use["reproj"] else None,
                                                          coef5, opt.lr, opt.b1, opt.b2, strm()))
            adam_terms("X", X, [(gX_r, 2.0 * c_r), (gX_b, c_b), (gX_t, c_t)])
            if cam_free:
                adam_terms("t", t, [(gt_r, 2.0 * c_r), (gt_s, c_s), (gt_b, c_bl)])
            if rot_free:
                cands = []
                with torch.cuda.device(dev):
                    for buf, (gRk, sc) in zip(gw3, ((gR_r, 2.0 * c_r), (gR_s, c_s), (gR_b, c_bl))):
                        if gRk is not None:
                            _lib.check(fn("ska_so3_tangent_grad")(P(R), P(gRk), n_rot, P(buf), strm()))  # linear in dL/dR
                            cands.append((buf, sc))
                adam_terms("w", None, cands, step_out=sw)
                if cands:
                    with torch.cuda.device(dev):
                        _lib.check(fn("ska_so3_retract")(P(R), P(sw), n_rot, strm()))
            if sharded:
                exchange_halo()

    def iteration():
        if fused:
            return fused_iteration()
        Xv = X.detach().requires_grad_(True)                    # views of the static buffers: the updates below are in place
        tv = t.detach().requires_grad_(mode != "pose_only")
        Rv = R.detach().requires_grad_(mode == "full")
        terms = {}
        if w["reproj"]:
            terms["reproj"] = losses.reprojection_loss(Xv, Rv, tv, K, x2d, conf, w=w["reproj"])
        if w["smooth"]:
            terms["smooth"] = losses.camera_smooth_loss(Rv, tv, w=w["smooth"])
        if w["baseline"]:
            terms["baseline"] = losses.baseline_reg_loss(Rv, tv, w=w["baseline"])
        if w["bone_length"]:
            terms["bone_length"] = losses.bone_length_loss(Xv, None, w=w["bone_length"])
        if w["pose_temporal"]:
            terms["pose_temporal"] = losses.pose_temporal_loss(Xv, w=w["pose_temporal"])
        total = sum(terms.values())
        total.backward()
        row.zero_()
        row[0, 0:1] = total.detach().to(torch.float64)
        for k, name in enumerate(FIRST_ORDER_TERMS):
            if name in terms:
                row[0, 1 + k: 2 + k] = terms[name].detach().to(torch.float64)
        hist.index_copy_(0, opt.k.to(torch.int64), row)       # row k (the counter is incremented by begin() below)
        opt.begin()
        opt.apply("X", X, Xv.grad)
        if mode != "pose_only":
            opt.apply("t", t, tv.grad if tv.grad is not None else torch.zeros_like(t))
        if mode == "full":
            gRc = (Rv.grad if Rv.grad is not None else torch.zeros_like(R)).contiguous()
            with torch.cuda.device(dev):
                _lib.check(getattr(lib, f"ska_so3_tangent_grad_{sfx}")(ptr(R), ptr(gRc), n_rot, ptr(gw), _stream_ptr(dev)))
            opt.apply("w", None, gw, step_out=sw)
            with torch.cuda.device(dev):
                _lib.check(getattr(lib, f"ska_so3_retract_{sfx}")(ptr(R), ptr(sw), n_rot, _stream_ptr(dev)))

    done = 0
    if graph and num_iters >= 4:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            iteration()                                          # warm-up outside capture: a real iteration (k = 1)
            done = 1
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                iteration()                                      # capture does not execute
        torch.cuda.current_stream(dev).wait_stream(side)
        for _ in range(num_iters - done):
            g.replay()
    else:
        for _ in range(num_iters):
            iteration()
    h = hist[:num_iters].cpu().numpy()
    history = [dict(iter=i, loss=float(r[0]), **{n: float(r[1 + k]) for k, n in enumerate(FIRST_ORDER_TERMS)}) for i, r in enumerate(h)]
    od = R_init_torch.dtype
    return R.to(od).clone(), t.to(t_init_torch.dtype).clone(), X.to(X3d_init_torch.dtype).clone(), history


def run_local_ba(K_torch, R_init_torch, t_init_torch, X3d_init_torch, x2d_torch, conf2d_torch, num_iters=200, lr=1e-3,
                 device="cuda", mode="pose_only", optimizer="adam", weights=None, graph=True, fused=True, static_rig_tol=1e-6,
                 loss="l2", loss_scale=None):
    """The optimiser the reference calls but never defines (vggt/multi_view_process.py:553-564;
    argument shapes :546-551).  Returns (R_opt (T,C,3,3), t_opt (T,C,3), X_opt (T,J,3), history).

    optimizer="adam" (default - what the call site's `lr` / `num_iters` and configs/vggt.yaml:43-52 describe): the
    reference's full configured objective - reprojection + the four regularisers of loss.py with the yaml weights - over
    the PER-FRAME cameras exactly as they are passed, minimised by `run_local_ba_first_order`.

    optimizer="lm": the SAME configured objective with the same per-frame cameras, minimised by Levenberg-Marquardt
    (ba_reg.run_local_ba_lm; specification oracle/lm_reg.py): converges in ~10 trials where Adam is configured for 10 000
    steps.  `lr` is the initial damping lambda0.  Computed in fp64, returned in X3d_init's dtype.

    optimizer="lm_rig": the Schur-complement Levenberg-Marquardt of this package on the reprojection term alone with ONE
    camera set shared over the clip (the static-rig problem of BASELINE configs 3 / 5).  Per-frame cameras are accepted
    only if they ARE one rig: they may differ from their mean (chordal mean rotation, mean translation) by at most
    `static_rig_tol` (radians / translation units), otherwise ValueError - averaging a moving rig silently would pull the
    points towards cameras they were not seen by.  mode="pose_only" returns the input cameras untouched (only the
    points move); `lr` is used as the initial damping lambda0; `num_iters` is capped at 64 trials (LM converges in ~10).

    loss="huber" | "cauchy" with loss_scale (pixels): a robust loss on the reprojection term against gross 2D detector
    failures, for optimizer="lm" and "lm_rig" (include/ska.h); the default "l2" is loss.py's squared error."""
    _cabi.check_loss(loss, loss_scale)
    if optimizer == "adam" and loss != "l2":
        raise ValueError(f"loss={loss!r} is implemented by optimizer='lm' and 'lm_rig'; optimizer='adam' minimises the L2 loss only")
    if optimizer == "adam":
        return run_local_ba_first_order(K_torch, R_init_torch, t_init_torch, X3d_init_torch, x2d_torch, conf2d_torch, num_iters, lr,
                                        device, mode, weights, graph, fused)
    if optimizer == "lm":
        from . import ba_reg

        if mode not in MODES:
            raise ValueError(f"unknown mode {mode!r}; expected one of {MODES}")
        return ba_reg.run_local_ba_lm(K_torch, R_init_torch, t_init_torch, X3d_init_torch, x2d_torch, conf2d_torch, num_iters, lr, device,
                                      mode, weights, loss=loss, loss_scale=loss_scale)
    if optimizer != "lm_rig":
        raise ValueError(f"optimizer must be 'adam', 'lm' or 'lm_rig', got {optimizer!r}")
    if mode not in MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {MODES}")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("run_local_ba runs on a CUDA device: this package has no CPU path")
    R = R_init_torch.detach().cpu().numpy().astype(np.float64)
    t = t_init_torch.detach().cpu().numpy().astype(np.float64)
    if R.ndim == 4:
        Tn, Cn = R.shape[:2]
        R0 = np.stack([_mean_rotation(R[:, c]) for c in range(Cn)])
        t0 = t.mean(0)
        # angle of R R0^T per frame and camera, translation spread
        cosang = (np.einsum("tcij,cij->tc", R, R0) - 1.0) / 2.0
        ang = float(np.arccos(np.clip(cosang, -1.0, 1.0)).max())
        dt = float(np.abs(t - t0[None]).max())
        if max(ang, dt) > static_rig_tol:
            raise ValueError(f"optimizer='lm_rig' solves a static rig, but the per-frame cameras differ from their mean by {ang:.3g} rad / "
                             f"{dt:.3g} (tolerance {static_rig_tol:g}); use optimizer='adam' / 'lm' (per-frame cameras) or pass one camera set")
    elif R.ndim == 3:
        Cn = R.shape[0]
        R0, t0 = R, t
        Tn = x2d_torch.shape[0]
    else:
        raise ValueError(f"Unsupported R shape: {R.shape}")
    K = K_torch.detach().cpu().numpy().astype(np.float64)
    x2d = x2d_torch.detach().to(dev, torch.float32)
    conf = conf2d_torch.detach().to(dev, torch.float32)
    X0 = X3d_init_torch.detach().to(dev, torch.float32)
    iters = int(max(1, min(int(num_iters), 64)))
    ba = ba_solve(x2d, conf, K, R0, t0, X0, num_iters=iters, mode=mode, lam0=float(lr), loss=loss, loss_scale=loss_scale)
    out_dtype = R_init_torch.dtype
    if mode == "pose_only":   # the cameras are not parameters: hand the caller's back bit for bit
        Rb = R_init_torch.detach() if R.ndim == 4 else R_init_torch.detach()[None].expand(Tn, Cn, 3, 3)
        tb = t_init_torch.detach().reshape(Tn, Cn, 3) if R.ndim == 4 else t_init_torch.detach().reshape(1, Cn, 3).expand(Tn, Cn, 3)
        R_opt, t_opt = Rb.to(dev, out_dtype).clone(), tb.to(dev, out_dtype).clone()
    else:
        R_opt = torch.from_numpy(np.broadcast_to(ba.R[None], (Tn, Cn, 3, 3)).copy()).to(dev, out_dtype)
        t_opt = torch.from_numpy(np.broadcast_to(ba.t[None], (Tn, Cn, 3)).copy()).to(dev, out_dtype)
    X_opt = ba.X.to(X3d_init_torch.dtype).clone()
    return R_opt, t_opt, X_opt, ba.history
