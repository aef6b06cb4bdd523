"""Levenberg-Marquardt over the reference's full configured objective with per-frame cameras (SURVEY rows N1 / e3): the
second-order form of `run_local_ba` (vggt/multi_view_process.py:553-564; undefined in the reference).

    total = w_reproj reprojection_loss + w_smooth camera_smooth_loss + w_baseline baseline_reg_loss
          + w_bone_length bone_length_loss + w_pose_temporal pose_temporal_loss           (bundle_adjustment/loss.py:90-155)

Specification: oracle/lm_reg.py.  The arithmetic is libska's (csrc/ska_ba_reg.cu through the C ABI of include/ska.h); this
module allocates, sequences the launches and - when the clip is sharded by frame range over ranks - moves the three things
that cross a shard edge: the all-reduced sums (cost terms, CG dot products), and the one-frame halo of the CG direction and
of the trial point (the temporal / smoothness terms couple frame t with t +- 1; the bone / baseline means are global).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi, _lib

MODES = ("pose_only", "pose_cam_t", "full")
DEFAULT_WEIGHTS = dict(reproj=1.0, smooth=0.1, baseline=0.01, bone_length=0.1, pose_temporal=0.1)  # configs/vggt.yaml:46-50
BONES = [(11, 13), (13, 15), (12, 14), (14, 16), (5, 7), (7, 9), (6, 8), (8, 10), (5, 6), (11, 12), (5, 11), (6, 12)]  # loss.py:118-131
HIST_KEYS = ("iter", "cost", "trial_cost", "lam", "rho", "accepted", "n_clamped", "pred", "cg_iters", "reproj", "smooth", "baseline",
             "bone_length", "pose_temporal", "cg_residual")


def coefficients(T: int, J: int, C_: int, conf_sum: float, n_bones: int, weights=None) -> list:
    """[c_r, c_l, c_t, c_s, c_b]: each term's weight over its `mean` denominator (loss.py:94,106,114,150,155)."""
    w = dict(DEFAULT_WEIGHTS, **(weights or {}))
    return [w["reproj"] / (conf_sum + 1e-6),
            w["bone_length"] / (T * n_bones) if n_bones else 0.0,
            w["pose_temporal"] / ((T - 1) * J * 3) if T > 1 else 0.0,
            w["smooth"] / ((T - 1) * C_ * 3) if T > 1 else 0.0,
            w["baseline"] / T if C_ >= 2 else 0.0]


class RegLMSequencer:
    """Engine-agnostic sequencing of one regularised LM trial over a frame-sharded clip.  Subclasses provide the steps
    (linearize, cg(op), apply, cost(which), finish_cost(which), control), the all-reduce payloads `dot` (1 element) and
    `sums` (2, n), and `edges(kind)` -> (first_row, last_row, halo_prev, halo_next) 1-D tensors for kind "p" / "trial".
    The CUDA engine is below; an fp64 numpy engine in tests/ drives this class over gloo."""

    group = None
    local_only = False
    cg_iters = 64
    check_every = 0  # > 0: outside graph capture, read the convergence flag every this many CG iterations and stop early
    max_iters = 0
    iters_done = 0
    _graph = None
    _capturing = False
    _gather_bufs = None

    def _world(self):
        d = torch.distributed
        if self.local_only or not (d.is_available() and d.is_initialized()):
            return 1, 0
        return d.get_world_size(self.group), d.get_rank(self.group)

    peer = None  # peer.PeerExchange: exchanges over NVLink peer memory instead of NCCL (CUDA engine)

    fused_exchange = False  # CUDA engine with a peer exchange: finish_cost / the CG scalar kernels all-reduce in their own prologue
    cg_done = None  # engines: one-element fp64 device tensor, non-zero once CG has converged (identical on every rank)

    def _allreduce(self, t, in_cg: bool = False):
        if self._world()[0] > 1:
            if self.peer is not None and self.peer.fits(t):
                self.peer.all_reduce(t, skip=self.cg_done if in_cg else None)
            else:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=self.group)

    def _allgather(self, mine, in_cg: bool = False):
        """(world,) + mine.shape <- every rank's `mine`."""
        world = self._world()[0]
        if self._gather_bufs is None:
            self._gather_bufs = {}
        bufs = self._gather_bufs
        key = (world * mine.numel(), mine.dtype, mine.device)
        flat = bufs.get(key)
        if flat is None:  # persistent: a skipped exchange (CG converged) leaves the previous, valid contents in place
            flat = bufs[key] = torch.zeros(key[0], dtype=mine.dtype, device=mine.device)
        if self.peer is not None and self.peer.fits(mine):
            self.peer.all_gather(flat, mine.reshape(-1), skip=self.cg_done if in_cg else None)
        else:
            torch.distributed.all_gather_into_tensor(flat, mine.reshape(-1), group=self.group)
        return flat.view((world,) + tuple(mine.shape))

    def exchange_halo(self, kind: str):
        """One all-gather of every rank's first / last row; rank r takes rank r-1's last row and rank r+1's first."""
        world, rank = self._world()
        if world == 1:
            return
        first, last, halo_prev, halo_next = self.edges(kind)
        mine = torch.stack([first, last]).contiguous()
        everyone = self._allgather(mine, in_cg=(kind == "p"))
        if rank > 0:
            halo_prev.copy_(everyone[rank - 1, 1])
        if rank < world - 1:
            halo_next.copy_(everyone[rank + 1, 0])

    def converged(self) -> bool:  # engines that can answer without a device round trip override this
        return False

    def trial(self):
        k = _cabi
        self.linearize()
        fused = self.fused_exchange
        self.cg(k.BA_REG_CG_BEGIN)
        if not fused:
            self._allreduce(self.dot)
        self.cg(k.BA_REG_CG_INIT)
        self.cg(k.BA_REG_CG_DIR)
        for it in range(self.cg_iters):
            if self.check_every and not self._capturing and it and it % self.check_every == 0 and self.converged():
                break
            # inside the loop the convergence flag is current (set by INIT / BETA from all-reduced scalars, identical on every
            # rank): once it is up the kernels return at once and the peer exchanges are skipped on every rank alike
            self.exchange_halo("p")
            self.cg(k.BA_REG_CG_MATVEC)
            if not fused:
                self._allreduce(self.dot, in_cg=True)
            self.cg(k.BA_REG_CG_ALPHA)
            self.cg(k.BA_REG_CG_UPDATE)
            if not fused:
                self._allreduce(self.dot, in_cg=True)
            self.cg(k.BA_REG_CG_BETA)
            self.cg(k.BA_REG_CG_DIR)
        self.apply()
        self.exchange_halo("trial")
        self.cost(1)
        if not fused:
            self._allreduce(self.sums[1])
        self.finish_cost(1)
        self.control()

    def setup_cost(self):
        self.exchange_halo("current")
        self.cost(0)
        if not self.fused_exchange:
            self._allreduce(self.sums[0])
        self.finish_cost(0)

    def run(self, num_iters: int, graph: bool = False):
        num_iters = int(num_iters)
        if num_iters <= 0:
            return self
        if self.iters_done + num_iters > self.max_iters:
            raise ValueError(f"history buffer holds {self.max_iters} trials; raise max_iters")
        if graph:
            if self._graph is None:
                self.trial()  # warm-up outside capture
                num_iters -= 1
                self.iters_done += 1
                g = torch.cuda.CUDAGraph()
                s = torch.cuda.Stream(self.dev)
                s.wait_stream(torch.cuda.current_stream(self.dev))
                self._capturing = True
                try:
                    with torch.cuda.stream(s):
                        with torch.cuda.graph(g, stream=s):
                            self.trial()
                finally:
                    self._capturing = False
                torch.cuda.current_stream(self.dev).wait_stream(s)
                self._graph = g
            for _ in range(num_iters):
                self._graph.replay()
        else:
            for _ in range(num_iters):
                self.trial()
        self.iters_done += num_iters
        return self


def _stream_ptr(dev) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


class RegularisedBundleAdjuster(RegLMSequencer):
    """This rank's frame shard of one regularised BA problem, resident on one GPU.

    x2d (T,C,J,2), conf (T,C,J): float32 CUDA (the call site casts them with .float(), multi_view_process.py:548-549)
    K (C,3,3) | (3,3); R (T,C,3,3) | (C,3,3); t (T,C,3) | (C,3); X0 (T,J,3): tensors or arrays, any float dtype
    mode: "pose_only" (points), "pose_cam_t" (points + every frame's camera translations), "full" (+ rotations)
    group: process group when the clip is sharded by contiguous frame ranges in rank order (None = the default group if
    torch.distributed is initialised); local_only=True solves this rank's frames alone.
    loss: "l2" (default: loss.py's squared pixel error), "huber" or "cauchy" on the reprojection term - a robust M-estimator
    against gross 2D detector failures (swapped limbs, invented occluded joints), solved by iteratively reweighted
    Gauss-Newton (include/ska.h); the four regularisers stay squared.  loss_scale: its scale in pixels (required, > 0, for
    "huber" / "cauchy").  `history` and `cost_value` report the robust cost."""

    def __init__(self, x2d, conf, K, R, t, X0, *, mode: str = "pose_only", weights=None, lam0: float = 1e-3, max_iters: int = 64,
                 cg_iters: int = 64, cg_tol: float = 1e-8, check_every: int = 0, group=None, local_only: bool = False,
                 peer_exchange: bool = True, fuse_exchange: bool = True, loss: str = "l2", loss_scale=None):
        if mode not in MODES:
            raise ValueError(f"unknown mode {mode!r}; expected one of {MODES}")
        self.loss = loss
        self.loss_id, self.loss_scale = _cabi.check_loss(loss, loss_scale)
        if not (x2d.is_cuda and conf.is_cuda):
            raise RuntimeError("x2d and conf must be CUDA tensors: this package has no CPU path")
        if x2d.dim() != 4 or x2d.shape[-1] != 2:
            raise ValueError(f"x2d must be (T,C,J,2), got {tuple(x2d.shape)}")
        Tl, Cn, J, _ = x2d.shape
        if tuple(conf.shape) != (Tl, Cn, J):
            raise ValueError(f"conf must be ({Tl},{Cn},{J}), got {tuple(conf.shape)}")
        if Tl < 1:
            raise ValueError("every rank needs at least one frame")
        if not 1 <= Cn <= _cabi.MAX_VIEWS or J > 96:
            raise ValueError("1..8 cameras and at most 96 joints")
        dev = x2d.device
        self.dev, self.group, self.local_only = dev, group, bool(local_only)
        if peer_exchange and self._world()[0] > 1:
            from . import peer as _peer

            self.peer = _peer.shared(group, dev)  # None where peer memory cannot be mapped: NCCL then
        self.mode, self.Tl, self.C, self.J = mode, Tl, Cn, J
        self.cg_iters, self.check_every, self.max_iters = int(cg_iters), int(check_every), int(max_iters)
        self.lib = _lib.load()
        f64 = dict(dtype=torch.float64, device=dev)
        as64 = lambda a: torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).to(**f64)
        self.x2d = x2d.to(torch.float32).contiguous()
        self.conf = conf.to(torch.float32).contiguous()
        Kt = as64(K)
        self.K = (Kt[None].expand(Cn, 3, 3) if Kt.dim() == 2 else Kt).reshape(Cn, 9).contiguous()
        Rt, tt = as64(R), as64(t)
        if Rt.dim() == 3:
            Rt, tt = Rt[None].expand(Tl, Cn, 3, 3), tt.reshape(1, Cn, 3).expand(Tl, Cn, 3)
        if tuple(Rt.shape) != (Tl, Cn, 3, 3) or tuple(tt.shape) != (Tl, Cn, 3):
            raise ValueError(f"cameras must be ({Tl},{Cn},3,3) / ({Tl},{Cn},3)")
        Xt = as64(X0)
        if tuple(Xt.shape) != (Tl, J, 3):
            raise ValueError(f"X0 must be ({Tl},{J},3), got {tuple(Xt.shape)}")
        self.nf = nf = 3 * J + 6 * Cn
        self.Xh = torch.zeros((2, Tl + 2, J, 3), **f64)
        self.Ch = torch.zeros((2, Tl + 2, Cn, 12), **f64)
        self.Ch[:, :, :, 0] = self.Ch[:, :, :, 4] = self.Ch[:, :, :, 8] = 1.0  # halo rows nobody reads stay valid rotations
        self.Xh[0, 1:-1] = Xt
        self.Ch[0, 1:-1, :, :9] = Rt.reshape(Tl, Cn, 9)
        self.Ch[0, 1:-1, :, 9:] = tt
        self.Xh[1], self.Ch[1] = self.Xh[0], self.Ch[0]
        self.vec = torch.zeros((_cabi.BA_REG_NVEC, Tl + 2, nf), **f64)
        self.pinv = torch.zeros((Tl, J, 6), **f64)
        n6 = 6 * Cn
        self.free = _cabi.BA_REG_FREE[mode]
        self.lfac = torch.zeros((Tl, n6 * (n6 + 1) // 2), **f64) if self.free else None
        self.sc = torch.zeros(_cabi.BA_REG_SC_DOUBLES, **f64)
        self.sums = torch.zeros((2, _cabi.BA_REG_SUMS), **f64)
        self.dot = self.sc[_cabi.BA_REG_SC_DOT: _cabi.BA_REG_SC_DOT + 1]
        self.cg_done = self.sc[13:14]
        self.hist = torch.zeros((self.max_iters, _cabi.BA_REG_HIST_DOUBLES), **f64)
        with torch.cuda.device(dev):
            ws = int(self.lib.ska_ba_reg_workspace_bytes(Tl))
        self.ws = torch.empty(ws, dtype=torch.uint8, device=dev)
        bones = [(i, j) for i, j in BONES if i < J and j < J]
        # global frame count, confidence sum and this rank's position in the clip
        world, rank = self._world()
        tot = torch.tensor([float(Tl), 0.0], **f64)
        tot[1] = self.conf.sum(dtype=torch.float64)
        self._allreduce(tot)
        T_global, conf_sum = int(round(float(tot[0]))), float(tot[1])
        self.T_global = T_global
        coef = coefficients(T_global, J, Cn, conf_sum, len(bones), weights)
        sc = np.zeros(_cabi.BA_REG_SC_DOUBLES)
        sc[_cabi.BA_REG_SC_LAMBDA], sc[_cabi.BA_REG_SC_NU], sc[_cabi.BA_REG_SC_TOL2] = lam0, 2.0, float(cg_tol) ** 2
        sc[_cabi.BA_REG_SC_COEF: _cabi.BA_REG_SC_COEF + 5] = coef
        sc[_cabi.BA_REG_SC_T_GLOBAL] = T_global
        self.sc.copy_(torch.from_numpy(sc))
        P = lambda a: None if a is None else a.data_ptr()
        self.prob = _cabi.SkaBaRegProblem(
            C=Cn, J=J, n_bones=len(bones), free_mask=self.free, T_local=Tl, has_prev=int(rank > 0), has_next=int(rank < world - 1),
            bone_i=(C.c_int32 * 16)(*[b[0] for b in bones]), bone_j=(C.c_int32 * 16)(*[b[1] for b in bones]),
            d_x2d=P(self.x2d), d_conf=P(self.conf), d_K=P(self.K), d_X=P(self.Xh), d_cams=P(self.Ch), d_vec=P(self.vec),
            d_pinv=P(self.pinv), d_lfac=P(self.lfac), d_sc=P(self.sc), d_sums=P(self.sums), d_hist=P(self.hist),
            hist_rows=self.max_iters, d_workspace=P(self.ws), ws_bytes=ws,
            peer=(C.addressof(self.peer.comm) if fuse_exchange and self.peer is not None else None))
        self.fused_exchange = bool(self.prob.peer)
        self._edge_stage = {"x": torch.empty((2, 2, 3 * J + 12 * Cn), **f64)}
        self.iters_done = 0
        self._graph = None
        self.setup_cost()

    # ------------------------------------------------------------------ halo rows
    def edges(self, kind: str):
        if kind == "p":
            p = self.vec[5]
            return p[1], p[self.Tl], p[0], p[self.Tl + 1]
        raise KeyError(kind)

    def exchange_halo(self, kind: str):
        world, rank = self._world()
        if world == 1:
            return
        if kind == "p":
            return super().exchange_halo(kind)
        # points and cameras, BOTH halves (current and trial: which is which is a device-side flag), in one gather
        J3 = 3 * self.J
        mine = self._edge_stage["x"]  # (half, first / last, 3 J + 12 C)
        for e, row in enumerate((1, self.Tl)):
            mine[:, e, :J3] = self.Xh[:, row].reshape(2, -1)
            mine[:, e, J3:] = self.Ch[:, row].reshape(2, -1)
        everyone = self._allgather(mine)
        if rank > 0:
            src = everyone[rank - 1, :, 1]
            self.Xh[:, 0] = src[:, :J3].view(2, self.J, 3)
            self.Ch[:, 0] = src[:, J3:].view(2, self.C, 12)
        if rank < world - 1:
            src = everyone[rank + 1, :, 0]
            self.Xh[:, self.Tl + 1] = src[:, :J3].view(2, self.J, 3)
            self.Ch[:, self.Tl + 1] = src[:, J3:].view(2, self.C, 12)

    def _cur_index(self) -> int:
        return int(self.sc[_cabi.BA_REG_SC_CUR].item())

    # ------------------------------------------------------------------ steps
    def _call(self, fn, *args):
        with torch.cuda.device(self.dev):
            _lib.check(fn(C.byref(self.prob), *args, _stream_ptr(self.dev)))

    def cost(self, which: int):
        self._call(self.lib.ska_ba_reg_cost_robust_f64, which, self.loss_id, self.loss_scale)

    def finish_cost(self, which: int):
        self._call(self.lib.ska_ba_reg_finish_cost_f64, which)

    def linearize(self):
        self._call(self.lib.ska_ba_reg_linearize_robust_f64, self.loss_id, self.loss_scale)

    def cg(self, op: int):
        self._call(self.lib.ska_ba_reg_cg_robust_f64, op, self.loss_id, self.loss_scale)

    def apply(self):
        self._call(self.lib.ska_ba_reg_apply_f64)

    def control(self):
        self._call(self.lib.ska_ba_reg_control_f64)

    def converged(self) -> bool:
        return bool(self.sc[13].item() != 0.0)

    # ------------------------------------------------------------------ results (synchronise)
    @property
    def history(self):
        if self.peer is not None:
            self.peer.check()  # an exchange that gave up waiting for a peer invalidates the trajectory: raise, never return it
        out = []
        for row in self.hist[: self.iters_done].cpu().numpy():
            d = dict(zip(HIST_KEYS, (float(v) for v in row)))
            for k in ("iter", "n_clamped", "cg_iters"):
                d[k] = int(d[k])
            d["accepted"] = bool(d["accepted"])
            out.append(d)
        return out

    @property
    def X(self) -> torch.Tensor:
        return self.Xh[self._cur_index(), 1:-1]

    @property
    def R(self) -> torch.Tensor:
        return self.Ch[self._cur_index(), 1:-1, :, :9].reshape(self.Tl, self.C, 3, 3)

    @property
    def t(self) -> torch.Tensor:
        return self.Ch[self._cur_index(), 1:-1, :, 9:]

    @property
    def cost_value(self) -> float:
        return float(self.sc[_cabi.BA_REG_SC_COST].item())


def run_local_ba_lm(K_torch, R_init_torch, t_init_torch, X3d_init_torch, x2d_torch, conf2d_torch, num_iters=20, lr=1e-3, device="cuda",
                    mode="pose_only", weights=None, cg_iters=64, cg_tol=1e-8, graph=False, group=None, loss="l2", loss_scale=None):
    """The reference's call (vggt/multi_view_process.py:553-564) answered by LM on the configured objective.  `lr` is the
    initial damping lambda0 (the one scalar the call site passes to its optimiser).  `loss` / `loss_scale`: the reprojection
    term's loss, as RegularisedBundleAdjuster takes them.  Returns (R_opt, t_opt, X_opt, history) in X3d_init's dtype;
    history rows: HIST_KEYS."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("run_local_ba runs on a CUDA device: this package has no CPU path")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    dt = X3d_init_torch.dtype if torch.is_tensor(X3d_init_torch) and X3d_init_torch.dtype in (torch.float32, torch.float64) else torch.float32
    to32 = lambda a: torch.as_tensor(a).detach().to(dev, torch.float32).contiguous()
    s = RegularisedBundleAdjuster(to32(x2d_torch), to32(conf2d_torch), torch.as_tensor(K_torch).detach(), torch.as_tensor(R_init_torch).detach(),
                                  torch.as_tensor(t_init_torch).detach(), torch.as_tensor(X3d_init_torch).detach(), mode=mode, weights=weights,
                                  lam0=float(lr), max_iters=max(int(num_iters), 1), cg_iters=cg_iters, cg_tol=cg_tol,
                                  check_every=0 if graph else 8, group=group, local_only=group is None, loss=loss, loss_scale=loss_scale)
    s.run(int(num_iters), graph=graph)
    return s.R.to(dt).clone(), s.t.to(dt).clone(), s.X.to(dt).clone(), s.history

