"""The regularised LM kernels (csrc/ska_ba_reg.cu) piece by piece against a float64 reference, at clip sizes where every
grid-stride loop wraps, and across shard edges on one GPU.  tests/test_ba_reg_gpu.py compares the pieces with the numpy
oracle only at T <= 60, where no warp takes a second frame and the point kernels launch a handful of blocks.

One trial is driven a launch at a time through RegularisedBundleAdjuster's steps and the device state is read in
between:
  cost(0)     the five weighted terms, the clamp count, the bone means and the baseline mean in `sc`;
  linearize   every row of g and D, every point's damped inverse, L L^T of every frame's Schur factor;
  CG          z and r.z after BEGIN; y and p.y for a seeded p; x, r, z after UPDATE with a given alpha; p after DIR
              with a given beta;
  apply       the trial points and cameras after a real CG solve; cost(1) and the predicted decrease; the history row.
The reference is oracle/lm_reg.py restated matrix-free in float64 torch (pinned to the oracle below at the G12 sizes)
and run on the GPU.  A frame-sharded solve is emulated on one GPU: three RegularisedBundleAdjuster(local_only=True)
shards, the middle one a single frame, with the all-reduces done as host-side sums and the halo exchanges as row copies.
Every row a shard writes must equal the unsharded solver's row bit for bit, and four lockstep trials must follow the
unsharded trajectory.

Each large case asserts, from the kernel constants mirrored here (and checked against the source), the grid-stride
passes it needs."""
import re
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

from oracle import lm_reg
from skiing_analysis_pytorch_b200 import _cabi, api, ba_reg, synth
from tests.test_ba_reg_gpu import _check, _expand, _oracle_to_rows, _rows_to_oracle

CSRC = Path(__file__).resolve().parent.parent / "skiing_analysis_pytorch_b200" / "csrc"

# ------------------------------------------------------------------------------------- kernel constants (mirrored)
K_WARPS_PER_BLOCK = 4          # kWarpsPerBlock: the warp-per-frame kernels' blocks
K_MAX_GRID_BLOCKS = 148 * 8    # kMaxGridBlocks: grid cap of the warp-per-frame kernels
K_PT_BLOCK = 256               # kPtBlock: reg_pt_* (pose_only), one thread per point
K_PT_MAX_GRID = 148 * 8        # kPtMaxGrid
DIR_BLOCK, DIR_MAX_GRID = 256, 148 * 8  # reg_dir_kernel launch in ba_reg_cg
SMEM_BLOCK_MAX = 227 * 1024    # ba_reg_linearize halves the warps per block while a block would need more
W_MAX = K_MAX_GRID_BLOCKS * K_WARPS_PER_BLOCK  # 4736 warps: frames one pass covers

# d_sc slots and sums columns (enums of ska_ba_reg.cu)
SC_FT, SC_PRED, SC_ALPHA, SC_BETA, SC_DONE, SC_CGIT = 5, 6, 11, 12, 13, 14
SC_REF, SC_BMEAN, SC_NCL, SC_TERM = 22, 38, 39, 40
SUM_REPROJ, SUM_CLAMP, SUM_TEMP, SUM_SMOOTH, SUM_B, SUM_B2, SUM_PRED, SUM_L, SUM_L2 = 0, 1, 2, 3, 4, 5, 6, 8, 24
N_BONE_SLOTS = 16


def _cdiv(a, b):
    return -(-a // b)


def _warps(T):
    """W: warps of every warp-per-frame launch (grid_blocks x kWarpsPerBlock)."""
    return max(1, min(_cdiv(T, K_WARPS_PER_BLOCK), K_MAX_GRID_BLOCKS)) * K_WARPS_PER_BLOCK


def _warp_passes(T):
    return _cdiv(T, _warps(T))


def _pt_passes(T, J):
    g = max(1, min(_cdiv(T * J, K_PT_BLOCK), K_PT_MAX_GRID, _warps(T)))
    return _cdiv(T * J, g * K_PT_BLOCK)


def _dir_passes(T, J, C):
    n = T * (3 * J + 6 * C)
    return _cdiv(n, min(_cdiv(n, DIR_BLOCK), DIR_MAX_GRID) * DIR_BLOCK)


def _linearize_warps_per_block(J, C):
    n6 = 6 * C
    per_warp = (J * 12 + C * 28 + 3 * J + n6 + n6 * (n6 + 1) // 2 + 96 * n6) * 8
    wpb = K_WARPS_PER_BLOCK
    while wpb > 1 and per_warp * wpb > SMEM_BLOCK_MAX:
        wpb //= 2
    return wpb


def test_mirrored_kernel_constants_match_the_source():
    src = (CSRC / "ska_ba_reg.cu").read_text()
    want = [(r"constexpr int kWarpsPerBlock = (\d+);", K_WARPS_PER_BLOCK),
            (r"constexpr int kMaxGridBlocks = (\d+ \* \d+);", K_MAX_GRID_BLOCKS),
            (r"constexpr int kPtBlock = (\d+);", K_PT_BLOCK),
            (r"constexpr int kPtMaxGrid = (\d+ \* \d+);", K_PT_MAX_GRID),
            (r"if \(g > (\d+ \* \d+)\) g = \d+ \* \d+;\s*reg_dir_kernel", DIR_MAX_GRID),
            (r"while \(wpb > 1 && per_warp \* wpb > \(size_t\)(\d+ \* \d+)\) wpb /= 2;", SMEM_BLOCK_MAX),
            (r"SC_FT = (\d+)", SC_FT), (r"SC_PRED = (\d+)", SC_PRED), (r"SC_ALPHA = (\d+)", SC_ALPHA), (r"SC_BETA = (\d+)", SC_BETA),
            (r"SC_DONE = (\d+)", SC_DONE), (r"SC_CGIT = (\d+)", SC_CGIT), (r"SC_REF = (\d+)", SC_REF), (r"SC_BMEAN = (\d+)", SC_BMEAN),
            (r"SC_NCL = (\d+)", SC_NCL), (r"SC_TERM = (\d+)", SC_TERM), (r"SUM_REPROJ = (\d+)", SUM_REPROJ),
            (r"SUM_CLAMP = (\d+)", SUM_CLAMP), (r"SUM_TEMP = (\d+)", SUM_TEMP), (r"SUM_SMOOTH = (\d+)", SUM_SMOOTH),
            (r"SUM_B = (\d+)", SUM_B), (r"SUM_B2 = (\d+)", SUM_B2), (r"SUM_PRED = (\d+)", SUM_PRED), (r"SUM_L = (\d+)", SUM_L),
            (r"SUM_L2 = (\d+)", SUM_L2)]
    for pat, val in want:
        m = re.search(pat, src)
        assert m is not None, pat
        assert int(np.prod([int(f) for f in m.group(1).split("*")])) == val, (pat, m.group(1), val)  # "148 * 8" style products
    m = re.search(r"int g = \(int\)\(\(n \+ (\d+)\) / (\d+)\);\s*if \(g > (\d+ \* \d+)\) g = \3;\s*reg_dir_kernel<<<g, (\d+), 0, s>>>", src)
    assert m is not None and (int(m.group(1)), int(m.group(2)), int(m.group(4))) == (DIR_BLOCK - 1, DIR_BLOCK, DIR_BLOCK)
    # the launch rules the pass counts below mirror
    assert "if (b > kMaxGridBlocks) b = kMaxGridBlocks;" in src
    assert "a.W = grid_blocks(p.T_local) * kWarpsPerBlock;" in src
    assert "if (g > kPtMaxGrid) g = kPtMaxGrid;" in src and "if (g > a.W) g = a.W;" in src
    assert ("const size_t per_warp = ((size_t)a.J * 12 + (size_t)a.C * 28 + a.nf + a.nS + (size_t)96 * a.n6) * sizeof(double);"
            in src)
    assert "reg_linearize_kernel<<<a.W / wpb, 32 * wpb, bytes, s>>>(a);" in src
    for kern in ("reg_cost_kernel", "reg_apply_kernel"):
        assert re.search(kern + r"<<<a\.W / kWarpsPerBlock, 32 \* kWarpsPerBlock", src), kern
    assert src.count("for (int64_t f = wid; f < a.Tl; f += a.W)") == 5  # cost, linearize, matvec, precond, apply
    assert src.count("i += (int64_t)gridDim.x * kPtBlock)") == 3  # reg_pt_linearize / matvec / precond
    assert _linearize_warps_per_block(96, 8) == 2 and _linearize_warps_per_block(80, 8) == 4


# ---------------------------------------------------------------------------------- float64 reference (torch port)
ZMIN = lm_reg.ZMIN
_FREE = {m: [bool((_cabi.BA_REG_FREE[m] >> k) & 1) for k in range(6)] for m in lm_reg.MODES}


def _hat(v):
    z = torch.zeros_like(v[..., 0])
    return torch.stack([torch.stack([z, -v[..., 2], v[..., 1]], -1), torch.stack([v[..., 2], z, -v[..., 0]], -1),
                        torch.stack([-v[..., 1], v[..., 0], z], -1)], -2)


def _safe_inv3(H):
    """Inverse of each 3x3 block, ZERO where the block is not positive definite (inv_sym3's rule)."""
    d1 = H[..., 0, 0] * H[..., 1, 1] - H[..., 0, 1] * H[..., 1, 0]
    ok = (H[..., 0, 0] > 0) & (d1 > 0) & (torch.linalg.det(H) > 0)
    Hs = torch.where(ok[..., None, None], H, torch.eye(3, dtype=H.dtype, device=H.device))
    return torch.where(ok[..., None, None], torch.linalg.inv(Hs), 0.0)


def _pack3(M):
    return torch.stack([M[..., 0, 0], M[..., 0, 1], M[..., 0, 2], M[..., 1, 1], M[..., 1, 2], M[..., 2, 2]], -1)


def _damped(H, lam):
    return H + lam * torch.diag_embed(H.diagonal(dim1=-2, dim2=-1))


def _so3_exp_left(w, R):
    """exp([w]x) R for batches (series below th^2 = 1e-8, as so3_exp_left)."""
    th2 = (w * w).sum(-1)
    small = th2 < 1e-8
    th = th2.clamp_min(1e-8).sqrt()
    A_ = torch.where(small, 1.0 - th2 / 6.0, torch.sin(th) / th)
    B_ = torch.where(small, 0.5 - th2 / 24.0, (1.0 - torch.cos(th)) / th2.clamp_min(1e-8))
    W = _hat(w)
    E = torch.eye(3, dtype=w.dtype, device=w.device) + A_[..., None, None] * W + B_[..., None, None] * (W @ W)
    return E @ R


def _apply_step(X, R, t, x, mode):
    """Trial point of a (T, 3J + 6C) step row block: X + dX, exp([d_omega]x) R, t + d_t over the free parameters."""
    T, J, _ = X.shape
    C = R.shape[1]
    f = torch.tensor(_FREE[mode], device=X.device)
    dq = torch.where(f, x[:, 3 * J:].reshape(T, C, 6), 0.0)
    Rn = _so3_exp_left(dq[..., :3], R) if mode == "full" else R
    tn = t + dq[..., 3:] if mode != "pose_only" else t
    return X + x[:, : 3 * J].reshape(T, J, 3), Rn, tn


def _cost(X, R, t, K, x2d, conf, coef):
    """(the five weighted terms as oracle/lm_reg.py cost_terms computes them, the kernels' raw sums row, the clamp count)."""
    T, J, _ = X.shape
    C = R.shape[1]
    Xc = torch.einsum("tcab,tjb->tcja", R, X) + t[:, :, None]
    z = Xc[..., 2]
    clamped = z < ZMIN
    iz = 1.0 / z.clamp_min(ZMIN)
    xn, yn = Xc[..., 0] * iz, Xc[..., 1] * iz
    k = K[None, :, None]
    du = k[..., 0, 0] * xn + k[..., 0, 1] * yn + k[..., 0, 2] - x2d[..., 0]
    dv = k[..., 1, 0] * xn + k[..., 1, 1] * yn + k[..., 1, 2] - x2d[..., 1]
    raw = torch.zeros(_cabi.BA_REG_SUMS, dtype=X.dtype, device=X.device)
    raw[SUM_REPROJ] = (conf * (du * du + dv * dv)).sum()
    raw[SUM_CLAMP] = clamped.sum()
    terms = dict(reproj=coef["reproj"] * float(raw[SUM_REPROJ]))
    bl = lm_reg.bones_for(J)
    L = torch.stack([(X[:, i] - X[:, j]).norm(dim=-1) for i, j in bl], -1) if bl else X.new_zeros((T, 0))
    raw[SUM_L: SUM_L + len(bl)] = L.sum(0)
    raw[SUM_L2: SUM_L2 + len(bl)] = (L * L).sum(0)
    terms["bone_length"] = coef["bone_length"] * float(((L - L.mean(0)) ** 2).sum()) if bl and coef["bone_length"] else 0.0
    raw[SUM_TEMP] = ((X[1:] - X[:-1]) ** 2).sum()
    terms["pose_temporal"] = coef["pose_temporal"] * float(raw[SUM_TEMP])
    Cc = -torch.einsum("tcba,tcb->tca", R, t)
    raw[SUM_SMOOTH] = ((Cc[1:] - Cc[:-1]) ** 2).sum()
    terms["smooth"] = coef["smooth"] * float(raw[SUM_SMOOTH])
    if C >= 2:
        b = (Cc[:, 0] - Cc[:, 1]).norm(dim=-1)
        raw[SUM_B], raw[SUM_B2] = b.sum(), (b * b).sum()
    terms["baseline"] = coef["baseline"] * float(((b - b.mean()) ** 2).sum()) if C >= 2 and coef["baseline"] else 0.0
    return terms, raw, int(clamped.sum())


class RegRef:
    """oracle/lm_reg.py matrix-free at one point (X (T,J,3), R (T,C,3,3), t (T,C,3), K (C,3,3), x2d (T,C,J,2), conf
    (T,C,J), float64 tensors on one device).  Vectors over the unknowns are (T, 3J + 6C) frame rows [J x (x,y,z) |
    C x (d_omega, d_t)] as the kernels hold them; camera columns a mode leaves fixed are zero in every Jacobian block.
    The bone / baseline references are the means at this point (constants of the linearisation)."""

    def __init__(self, X, R, t, K, x2d, conf, coef, mode):
        T, J, _ = X.shape
        C = R.shape[1]
        self.T, self.J, self.C, self.coef, self.mode = T, J, C, coef, mode
        self.fm = torch.tensor(_FREE[mode], device=X.device)
        fm = self.fm.to(X.dtype)
        # ---- reprojection rows sqrt(c_r conf) (pi(R X + t) - x): A = d/dX (T,C,J,2,3), B = d/d(d_omega, d_t) (T,C,J,2,6)
        p = torch.einsum("tcab,tjb->tcja", R, X)
        Xc = p + t[:, :, None]
        z = Xc[..., 2]
        live = (z >= ZMIN).to(X.dtype)
        iz = 1.0 / z.clamp_min(ZMIN)
        xn, yn = Xc[..., 0] * iz, Xc[..., 1] * iz
        k = K[None, :, None]
        fu, fv = k[..., 0, 0] * xn + k[..., 0, 1] * yn, k[..., 1, 0] * xn + k[..., 1, 1] * yn
        s = (coef["reproj"] * conf).sqrt()
        self.e = torch.stack([fu + k[..., 0, 2] - x2d[..., 0], fv + k[..., 1, 2] - x2d[..., 1]], -1) * s[..., None]
        ju = torch.stack([k[..., 0, 0] * iz, k[..., 0, 1] * iz, -fu * iz * live], -1)
        jv = torch.stack([k[..., 1, 0] * iz, k[..., 1, 1] * iz, -fv * iz * live], -1)
        Jx = torch.stack([ju, jv], -2) * s[..., None, None]
        self.A = torch.einsum("tcjik,tckl->tcjil", Jx, R)
        self.B = torch.cat([torch.linalg.cross(p[..., None, :].expand_as(Jx), Jx, dim=-1), Jx], -1) * fm
        # ---- bones: unit vectors and lengths; temporal pairs per frame
        self.bones = lm_reg.bones_for(J)
        if self.bones:
            d = torch.stack([X[:, i] - X[:, j] for i, j in self.bones], 1)  # (T,B,3)
            self.L = d.norm(dim=-1)
            self.U = d / self.L[..., None]
        self.npair = torch.zeros(T, dtype=X.dtype, device=X.device)
        self.npair[1:] += 1.0
        self.npair[:-1] += 1.0
        self.X = X
        # ---- camera centres Cc = -R^T t and J_Cc = [-R^T [t]x | -R^T] (T,C,3,6); baseline gradients g0, g1 (T,6)
        self.Cc = -torch.einsum("tcba,tcb->tca", R, t)
        Jt = -R.transpose(-1, -2)
        self.JC = torch.cat([Jt @ _hat(t), Jt], -1) * fm
        if C >= 2:
            dc = self.Cc[:, 0] - self.Cc[:, 1]
            self.b = dc.norm(dim=-1)
            nh = dc / self.b[:, None]
            self.g0 = torch.einsum("ta,tak->tk", nh, self.JC[:, 0])
            self.g1 = -torch.einsum("ta,tak->tk", nh, self.JC[:, 1])

    def _rows(self, vX, vQ):
        return torch.cat([vX.reshape(self.T, -1), vQ.reshape(self.T, -1)], 1)

    def _split(self, v):
        T, J, C = self.T, self.J, self.C
        return v[:, : 3 * J].reshape(T, J, 3), torch.where(self.fm, v[:, 3 * J:].reshape(T, C, 6), 0.0)

    def gradient(self):
        c = self.coef
        gX = torch.einsum("tcjik,tcji->tjk", self.A, self.e)
        gQ = torch.einsum("tcjik,tcji->tck", self.B, self.e)
        if self.bones and c["bone_length"]:
            res = c["bone_length"] * (self.L - self.L.mean(0))
            for b, (i, j) in enumerate(self.bones):
                gX[:, i] += res[:, b, None] * self.U[:, b]
                gX[:, j] -= res[:, b, None] * self.U[:, b]
        if self.T > 1:
            dX = c["pose_temporal"] * (self.X[1:] - self.X[:-1])
            gX[1:] += dX
            gX[:-1] -= dX
            dC = c["smooth"] * (self.Cc[1:] - self.Cc[:-1])
            gQ[1:] += torch.einsum("tcak,tca->tck", self.JC[1:], dC)
            gQ[:-1] -= torch.einsum("tcak,tca->tck", self.JC[:-1], dC)
        if self.C >= 2 and c["baseline"]:
            res = c["baseline"] * (self.b - self.b.mean())
            gQ[:, 0] += res[:, None] * self.g0
            gQ[:, 1] += res[:, None] * self.g1
        return self._rows(gX, gQ)

    def blocks(self):
        """Diagonal blocks of J^T J: points (T,J,3,3), cameras (T,C,6,6); the frame's coupling W (T,J,3,6C)."""
        c = self.coef
        Hpp = torch.einsum("tcjik,tcjil->tjkl", self.A, self.A)
        if self.bones and c["bone_length"]:
            uu = c["bone_length"] * self.U[..., :, None] * self.U[..., None, :]
            for b, (i, j) in enumerate(self.bones):
                Hpp[:, i] += uu[:, b]
                Hpp[:, j] += uu[:, b]
        Hpp += (c["pose_temporal"] * self.npair)[:, None, None, None] * torch.eye(3, dtype=Hpp.dtype, device=Hpp.device)
        Hcc = torch.einsum("tcjik,tcjil->tckl", self.B, self.B)
        Hcc += (c["smooth"] * self.npair)[:, None, None, None] * (self.JC.transpose(-1, -2) @ self.JC)
        if self.C >= 2 and c["baseline"]:
            Hcc[:, 0] += c["baseline"] * self.g0[:, :, None] * self.g0[:, None, :]
            Hcc[:, 1] += c["baseline"] * self.g1[:, :, None] * self.g1[:, None, :]
        W = torch.einsum("tcjik,tcjil->tjkcl", self.A, self.B).reshape(self.T, self.J, 3, 6 * self.C)
        return Hpp, Hcc, W

    def diag(self):
        Hpp, Hcc, _ = self.blocks()
        return self._rows(Hpp.diagonal(dim1=-2, dim2=-1), Hcc.diagonal(dim1=-2, dim2=-1))

    def matvec(self, v, lam):
        """(J^T J + lam diag(J^T J)) v over the free unknowns, one residual group at a time."""
        c = self.coef
        pX, pQ = self._split(v)
        Jp = torch.einsum("tcjik,tjk->tcji", self.A, pX) + torch.einsum("tcjik,tck->tcji", self.B, pQ)
        yX = torch.einsum("tcjik,tcji->tjk", self.A, Jp)
        yQ = torch.einsum("tcjik,tcji->tck", self.B, Jp)
        if self.bones and c["bone_length"]:
            for b, (i, j) in enumerate(self.bones):
                sb = c["bone_length"] * (self.U[:, b] * (pX[:, i] - pX[:, j])).sum(-1, keepdim=True)
                yX[:, i] += sb * self.U[:, b]
                yX[:, j] -= sb * self.U[:, b]
        if self.T > 1:
            dp = c["pose_temporal"] * (pX[1:] - pX[:-1])
            yX[1:] += dp
            yX[:-1] -= dp
            q = torch.einsum("tcak,tck->tca", self.JC, pQ)
            dq = c["smooth"] * (q[1:] - q[:-1])
            yQ[1:] += torch.einsum("tcak,tca->tck", self.JC[1:], dq)
            yQ[:-1] -= torch.einsum("tcak,tca->tck", self.JC[:-1], dq)
        if self.C >= 2 and c["baseline"]:
            db = c["baseline"] * ((self.g0 * pQ[:, 0]).sum(-1) + (self.g1 * pQ[:, 1]).sum(-1))
            yQ[:, 0] += db[:, None] * self.g0
            yQ[:, 1] += db[:, None] * self.g1
        return self._rows(yX, yQ) + lam * self.diag() * self._rows(pX, pQ)

    def point_inverses(self, lam):
        """(T,J,6) packed [00 01 02 11 12 22] damped point-block inverses."""
        return _pack3(_safe_inv3(_damped(self.blocks()[0], lam)))

    def _frame_blocks(self, lam):
        """Damped point blocks (T,J,3,3), the damped camera blocks of each frame with identity on fixed parameters
        (T,6C,6C; no camera-camera coupling: the preconditioner drops it), W (T,J,3,6C)."""
        Hpp, Hcc, W = self.blocks()
        T, C = self.T, self.C
        Dc = torch.zeros((T, 6 * C, 6 * C), dtype=Hcc.dtype, device=Hcc.device)
        for c in range(C):
            Dc[:, 6 * c: 6 * c + 6, 6 * c: 6 * c + 6] = _damped(Hcc[:, c], lam)
        fixed = ~self.fm.repeat(C)
        Dc[:, fixed, :] = 0.0
        Dc[:, :, fixed] = 0.0
        Dc[:, fixed, fixed] = 1.0
        return _damped(Hpp, lam), Dc, W

    def schur(self, lam):
        """S_f = Dc - sum_j W_j^T Dp_j^-1 W_j (T,6C,6C), as reg_linearize_kernel factors it."""
        Dp, Dc, W = self._frame_blocks(lam)
        return Dc - torch.einsum("tjkm,tjkn->tmn", W, _safe_inv3(Dp) @ W)

    def precond(self, r, lam, chunk=None):
        """z = M_f^-1 r: each frame's dense [Dp W; W^T Dc] system (test_linearisation_pieces_match_oracle's M),
        solved by batched dense LU in frame chunks."""
        Dp, Dc, W = self._frame_blocks(lam)
        T, J, C = self.T, self.J, self.C
        n = 3 * J + 6 * C
        z = torch.empty_like(r)
        chunk = chunk or max(1, (1 << 25) // (n * n))  # 256 MB of systems at a time
        for a in range(0, T, chunk):
            b = min(T, a + chunk)
            F = b - a
            M = torch.zeros((F, n, n), dtype=r.dtype, device=r.device)
            M[:, : 3 * J, : 3 * J] = torch.diag_embed(Dp[a:b].permute(0, 2, 3, 1)).permute(0, 3, 1, 4, 2).reshape(F, 3 * J, 3 * J)
            M[:, : 3 * J, 3 * J:] = W[a:b].reshape(F, 3 * J, 6 * C)
            M[:, 3 * J:, : 3 * J] = W[a:b].reshape(F, 3 * J, 6 * C).transpose(1, 2)
            M[:, 3 * J:, 3 * J:] = Dc[a:b]
            z[a:b] = torch.linalg.solve(M, r[a:b])
        return z


# -------------------------------------------------------------------------------------- the port against the oracle
def _rel(got, want):
    got, want = np.asarray(got, float), np.asarray(want, float)
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-300))


@pytest.mark.parametrize("name", sorted(lm_reg.G12_CASES))
def test_reference_port_matches_numpy_oracle(name):
    """The matrix-free float64 torch port equals oracle/lm_reg.py to 1e-12 relative at the G12 sizes: g, diag(J^T J),
    the damped product, the cost terms, the trial step, the point-block inverses, the frame Schur complements and the
    frame preconditioner (the oracle's sparse M solved by LU)."""
    rig, T, J, mode = lm_reg.G12_CASES[name]
    clip, R, t, X = lm_reg.make_problem(rig, T, J, cam_jitter=0.01)
    C = R.shape[1]
    x2d, conf = clip.x_fm.astype(float), clip.conf_fm.astype(float)
    coef = lm_reg.coefficients(T, J, C, conf.sum(), None)
    H, g, free, _ = lm_reg.normal_system(X, R, t, clip.K, x2d, conf, coef, mode)
    lam = 1e-3
    th = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))  # noqa: E731
    ref = RegRef(th(X), th(R), th(t), th(clip.K), th(x2d), th(conf), coef, mode)
    to_o = lambda v: _rows_to_oracle(v.numpy(), T, J, C)  # noqa: E731
    assert _rel(to_o(ref.gradient()), _expand(g, free)) <= 1e-12
    assert _rel(to_o(ref.diag()), _expand(H.diagonal(), free)) <= 1e-12
    A = (H + lam * sp.diags(H.diagonal())).tocsr()
    rng = np.random.default_rng(5)
    v = rng.normal(size=g.shape[0])
    y = ref.matvec(th(_oracle_to_rows(_expand(v, free), T, J, C)), lam)
    assert _rel(to_o(y), _expand(A @ v, free)) <= 1e-12
    # a step whose fixed camera columns hold garbage: the port must ignore them as the kernels do
    step = rng.normal(0.0, 1e-2, (T, 3 * J + 6 * C))
    terms, raw, ncl = _cost(th(X), th(R), th(t), th(clip.K), th(x2d), th(conf), coef)
    o_terms, o_ncl = lm_reg.cost_terms(X, R, t, clip.K, x2d, conf, coef)
    assert ncl == o_ncl
    for k in lm_reg.TERMS:
        assert abs(terms[k] - o_terms[k]) <= 1e-12 * abs(o_terms[k]), k
    Xn, Rn, tn = _apply_step(th(X), th(R), th(t), th(step), mode)
    delta = _rows_to_oracle(step, T, J, C) * free
    for got, want in zip((Xn, Rn, tn), lm_reg.apply_step(X, R, t, delta, mode)):
        assert _rel(got.numpy(), want) <= 1e-12
    # the preconditioner's pieces from the oracle's sparse matrix: per frame [Dp W; W^T Dc] (M of
    # test_linearisation_pieces_match_oracle), its 3x3 point blocks and its Schur complement onto the frame's cameras
    nX = T * J * 3
    k = {"pose_only": 0, "pose_cam_t": 3, "full": 6}[mode]
    fr = np.concatenate([np.repeat(np.arange(T), J * 3), np.repeat(np.arange(T), C * k)])
    blk = np.concatenate([np.repeat(np.arange(T * J), 3), T * J + np.repeat(np.arange(T * C), k)])
    ispt = np.concatenate([np.ones(nX, bool), np.zeros(T * C * k, bool)])
    Ac = A.tocoo()
    keep = (blk[Ac.row] == blk[Ac.col]) | ((fr[Ac.row] == fr[Ac.col]) & (ispt[Ac.row] != ispt[Ac.col]))
    M = sp.coo_matrix((Ac.data[keep], (Ac.row[keep], Ac.col[keep])), shape=Ac.shape).tocsc()
    r = rng.normal(size=g.shape[0])
    z = ref.precond(th(_oracle_to_rows(_expand(r, free), T, J, C)), lam, chunk=7)  # several chunks, a ragged last one
    assert _rel(to_o(z), _expand(spla.splu(M).solve(r), free)) <= 1e-12
    Md = M.toarray()
    pinv = ref.point_inverses(lam).numpy()
    pinv_o = np.stack([np.linalg.inv(Md[3 * i: 3 * i + 3, 3 * i: 3 * i + 3]) for i in range(T * J)])
    assert _rel(pinv.reshape(-1, 6), pinv_o[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]) <= 1e-12
    S = ref.schur(lam).numpy()
    cols = np.array([6 * c + q for c in range(C) for q in range(6) if _FREE[mode][q]], int)
    fixed = np.setdiff1d(np.arange(6 * C), cols)
    assert np.array_equal(S[:, fixed][:, :, fixed], np.broadcast_to(np.eye(len(fixed)), (T, len(fixed), len(fixed))))
    assert np.all(S[:, fixed][:, :, cols] == 0.0)
    for f in range(T) if k else ():
        pi = np.arange(f * J * 3, (f + 1) * J * 3)
        ci = nX + np.arange(f * C * k, (f + 1) * C * k)
        So = Md[np.ix_(ci, ci)] - Md[np.ix_(ci, pi)] @ np.linalg.solve(Md[np.ix_(pi, pi)], Md[np.ix_(pi, ci)])
        assert _rel(S[f][np.ix_(cols, cols)], So) <= 1e-12, f


# ------------------------------------------------------------------------------------------------------ tolerances
# Measured on one NVIDIA B200 (1000 W power limit) with about a 3x margin; each comment gives the largest error measured
# over the four cases below.  The starting point was the small-size bounds of tests/test_ba_reg_gpu.py (1e-11 of the
# vector's largest entry for g / D / y, 1e-8 for z, 1e-12 for the cost): every piece stays far inside them.
TOL = dict(
    coef=1e-15,      # c_r .. c_b in sc (the confidence sum in another order), relative (0)
    cost=1e-14,      # F and the reprojection, smoothness and temporal terms, relative (3.6e-15: smoothness)
    # bone and baseline terms: the kernel's one-pass variance c (sum b^2 - (sum b)^2 / T), the form whose two sums the
    # shards all-reduce, cancels - relative to the term it is off by up to 2e-12 at T = 9509 - so the error is measured
    # against c sum b^2, the size of what cancels (4.3e-16)
    cost_var=1.5e-15,
    sums=1e-14,      # every raw sums entry, relative to the entry (3.7e-15)
    means=1e-15,     # the 16 bone means and the baseline mean in sc, relative (2.3e-16)
    g=1e-14,         # of max |g| (3.4e-15)
    D=5e-15,         # of max |D| (1.4e-15)
    pinv=5e-15,      # per point, of the block's largest entry (1.6e-15)
    lfac=1e-14,      # L L^T against S_f, per frame, of the frame's largest |S_f| entry (3.4e-15)
    # z = M_f^-1 r: the frame Schur complements lose ~1/lambda of their digits; largest at 96 joints x 8 cameras for the
    # r left by a seeded update (1.5e-10; 2.4e-11 for r = -g)
    z=5e-10,
    y=1.5e-15,       # of max |y| (4.9e-16)
    dot=1e-15,       # r.z / p.y against the reference vectors, relative (2.3e-16)
    axpy=4e-16,      # x + alpha p, r - alpha y, z + beta p: one rounding here, up to two in torch; of max |v| (1.7e-16)
    R=6e-16,         # trial rotations, absolute (2.2e-16)
    pred=4e-16,      # SUM_PRED against x.(lam D x - g) from the GPU's own x, D, g; of sum |terms| (1.2e-16)
)
SHARD_SUM_TOL = 1e-14  # the shards' raw sums rows and dot partials against the unsharded, relative (3.3e-16)
TRAJ_COST_TOL, TRAJ_X_TOL = 1e-12, 1e-10  # lockstep trials: trial cost relative (1.9e-15), X absolute (3.4e-14)


def _err(got, ref, scale):
    return float((got - ref).abs().max() / scale) if got.numel() else 0.0


def _within(name, err, tol):
    print(f"    {name:<30s} {err:.3e}  (tol {tol:.1e})")
    assert err <= tol, (name, err, tol)


def _rel_t(got, ref):
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


# ------------------------------------------------------------------------------------------------------ large cases
# name -> (rig, T, J, mode): the frame counts come from W_MAX (frames of one warp pass) and are checked below
CASES = {
    "A_full_3_warp_passes": ("2b", 2 * W_MAX + 37, 17, "full"),
    "B_pose_cam_t": ("2b", 2 * W_MAX + 37, 17, "pose_cam_t"),
    "C_pose_only_3_point_passes": ("2b", 40_000, 17, "pose_only"),
    "D_96_joints_8_cams": ("8", W_MAX + 64, 96, "full"),
}
CG_ITERS = 48


@pytest.fixture(scope="module")
def clips(cuda):
    """Device clips as tools/ba_reg_multi_gpu_check.py builds them: perturbed cameras, triangulated X0, and a random
    walk on every frame's t so the smoothness and baseline terms are active."""
    cache = {}

    def get(rig, T, J):
        if (rig, T, J) not in cache:
            d = synth.make_clip_device(rig, T, J, cuda, seed=7)
            R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
            X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), d["K"], R0, t0, want=("X",)).X
            C = len(R0)
            g = torch.Generator(device=cuda).manual_seed(11)
            R = torch.tensor(R0, device=cuda)[None].expand(T, C, 3, 3).contiguous()
            walk = torch.cumsum(0.002 * torch.randn(T, C, 3, generator=g, device=cuda, dtype=torch.float64), 0)
            t = (torch.tensor(t0, device=cuda)[None] + walk).contiguous()
            cache[(rig, T, J)] = dict(x2d=d["x2d"], conf=d["conf"], K=d["K"], R=R, t=t, X0=X0.double().contiguous())
        return cache[(rig, T, J)]

    yield get
    cache.clear()
    torch.cuda.empty_cache()


def _solver(clip, mode, a=0, b=None, **kw):
    b = clip["X0"].shape[0] if b is None else b
    return ba_reg.RegularisedBundleAdjuster(clip["x2d"][a:b].contiguous(), clip["conf"][a:b].contiguous(), clip["K"],
                                            clip["R"][a:b], clip["t"][a:b], clip["X0"][a:b], mode=mode, max_iters=8,
                                            cg_iters=CG_ITERS, **kw)


def _point(s, which=0):
    """(X, R, t) of the current (which = 0) or trial (1) buffer, interior rows."""
    cur = int(s.sc[_cabi.BA_REG_SC_CUR].item())
    buf = cur if which == 0 else 1 - cur
    return s.Xh[buf, 1:-1], s.Ch[buf, 1:-1, :, :9].reshape(s.Tl, s.C, 3, 3), s.Ch[buf, 1:-1, :, 9:]


def _reference(s, mode, which=0):
    X, R, t = _point(s, which)
    conf = s.conf.double()
    coef = lm_reg.coefficients(s.Tl, s.J, s.C, float(conf.sum()), None)
    return RegRef(X, R, t, s.K.view(s.C, 3, 3), s.x2d.double(), conf, coef, mode), coef


def _interior(s, k):
    return s.vec[k, 1:-1]


def _term_tol(term):
    return "cost_var" if term in ("bone_length", "baseline") else "cost"


def _term_err(got, term, terms, raw, coef):
    """Error of one weighted term.  The bone and baseline terms are one-pass variances, c (sum b^2 - (sum b)^2 / T) -
    the form whose two sums the shards all-reduce - so their rounding is relative to c sum b^2, not to the term."""
    if term == "bone_length":
        scale = coef[term] * float(raw[SUM_L2: SUM_L2 + N_BONE_SLOTS].sum())
    elif term == "baseline":
        scale = coef[term] * float(raw[SUM_B2])
    else:
        scale = abs(terms[term])
    return abs(got - terms[term]) / max(scale, 1e-300)


def _check_cost(s, ref_args, which):
    X, R, t, K, x2d, conf, coef = ref_args
    terms, raw, ncl = _cost(X, R, t, K, x2d, conf, coef)
    cols = [c for c in range(_cabi.BA_REG_SUMS) if c not in (SUM_PRED, 7)]
    got, want = s.sums[which, cols], raw[cols]
    assert torch.all(got[want == 0.0] == 0.0)  # clamp count, unused bone slots
    _within(f"cost({which}) raw sums", float(((got - want).abs() / want.abs().clamp_min(1e-300)).max()), TOL["sums"])
    F = sum(terms.values())
    if which == 0:
        for k, term in enumerate(lm_reg.TERMS):
            _within(f"cost(0) {term}", _term_err(float(s.sc[SC_TERM + k]), term, terms, raw, coef), TOL[_term_tol(term)])
        _within("cost(0) F", abs(s.cost_value - F) / F, TOL["cost"])
        assert int(s.sc[SC_NCL].item()) == ncl
        T = s.Tl
        nb = len(lm_reg.bones_for(s.J))
        means = torch.zeros(N_BONE_SLOTS, dtype=torch.float64, device=X.device)
        means[:nb] = raw[SUM_L: SUM_L + nb] / T
        _within("cost(0) bone means", _rel_t(s.sc[SC_REF: SC_REF + N_BONE_SLOTS], means), TOL["means"])
        assert torch.all(s.sc[SC_REF + nb: SC_REF + N_BONE_SLOTS] == 0.0)
        _within("cost(0) baseline mean", abs(float(s.sc[SC_BMEAN]) - float(raw[SUM_B]) / T) / (float(raw[SUM_B]) / T), TOL["means"])
    else:
        _within("cost(1) F_trial", abs(float(s.sc[SC_FT]) - F) / F, TOL["cost"])
    return terms, F, ncl


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_lm_trial_pieces_at_scale(cuda, clips, name):
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    C = clip["R"].shape[1]
    s = _solver(clip, mode)
    k = _cabi
    wp, pp, dp, wpb = _warp_passes(T), _pt_passes(T, J), _dir_passes(T, J, C), _linearize_warps_per_block(J, C)
    print(f"\n[{name}] T = {T}, J = {J}, C = {C}, {mode}: warp passes {wp} (last {T - (wp - 1) * _warps(T)} frames), "
          f"point passes {pp}, DIR passes {dp}, linearize {wpb} warps per block")
    if mode == "pose_only":
        assert pp >= 2 and wp >= 2  # reg_pt_*; cost / apply warp kernels
    else:
        assert wp >= 2 and dp >= 2
    if (J, C) == (96, 8):  # the largest frame: two warps per linearize block
        assert wpb == 2 and wp >= 2
    lam = float(s.sc[k.BA_REG_SC_LAMBDA])
    ref, coef = _reference(s, mode)
    _within("coefficients", _rel_t(s.sc[k.BA_REG_SC_COEF: k.BA_REG_SC_COEF + 5],
                                   torch.tensor([coef[c] for c in ("reproj", "bone_length", "pose_temporal", "smooth", "baseline")],
                                                dtype=torch.float64, device=cuda)), TOL["coef"])
    X, R, t = _point(s)
    cost_args = (X, R, t, s.K.view(C, 3, 3), s.x2d.double(), s.conf.double(), coef)
    # ---- cost(0) / finish_cost(0)
    s.cost(0)
    s.finish_cost(0)
    terms0, F0, _ = _check_cost(s, cost_args, 0)
    raw0 = s.sums[0].clone()
    # ---- linearize
    s.linearize()
    g_ref, D_ref = ref.gradient(), ref.diag()
    g, D = _interior(s, 0), _interior(s, 1)
    _within("linearize g", _err(g, g_ref, g_ref.abs().max()), TOL["g"])
    _within("linearize D", _err(D, D_ref, D_ref.abs().max()), TOL["D"])
    assert torch.equal(_interior(s, 3), -g)  # r = -g
    pinv_ref = ref.point_inverses(lam)
    scale = pinv_ref.abs().amax(-1, keepdim=True)
    _within("linearize pinv", float(((s.pinv - pinv_ref).abs() / scale).max()), TOL["pinv"])
    if s.lfac is not None:
        n6 = 6 * C
        Lm = torch.zeros((T, n6, n6), dtype=torch.float64, device=cuda)
        ii = torch.tril_indices(n6, n6, device=cuda)
        Lm[:, ii[0], ii[1]] = s.lfac
        S_ref = ref.schur(lam)
        err = ((Lm @ Lm.transpose(1, 2) - S_ref).abs().amax((1, 2)) / S_ref.abs().amax((1, 2))).max()
        _within("linearize L L^T vs S_f", float(err), TOL["lfac"])
    # ---- CG_BEGIN: x = 0, z = M^-1 r, r.z
    s.cg(k.BA_REG_CG_BEGIN)
    r = _interior(s, 3)
    z_ref = ref.precond(r, lam)
    assert torch.all(s.vec[2] == 0.0) and torch.all(s.vec[5] == 0.0) and torch.all(s.vec[6] == 0.0)
    _within("BEGIN z", _err(_interior(s, 4), z_ref, z_ref.abs().max()), TOL["z"])
    rz = float((r * z_ref).sum())
    _within("BEGIN r.z", abs(float(s.dot) - rz) / abs(rz), TOL["dot"])
    # ---- CG_MATVEC with a seeded p
    gen = torch.Generator(device=cuda).manual_seed(5)
    fmask = torch.cat([torch.ones(3 * J, dtype=torch.bool, device=cuda), torch.tensor(_FREE[mode], device=cuda).repeat(C)])
    p = torch.randn(T, 3 * J + 6 * C, generator=gen, device=cuda, dtype=torch.float64) * fmask
    s.vec[5, 1:-1] = p
    s.sc[SC_DONE] = 0.0
    s.cg(k.BA_REG_CG_MATVEC)
    y_ref = ref.matvec(p, lam)
    _within("MATVEC y", _err(_interior(s, 6), y_ref, y_ref.abs().max()), TOL["y"])
    py = float((p * y_ref).sum())
    _within("MATVEC p.y", abs(float(s.dot) - py) / abs(py), TOL["dot"])
    # ---- CG_UPDATE with alpha
    alpha = 0.37
    x0, r0, y = _interior(s, 2).clone(), r.clone(), _interior(s, 6).clone()
    s.sc[SC_ALPHA] = alpha
    s.cg(k.BA_REG_CG_UPDATE)
    xa, ra = x0 + alpha * p, r0 - alpha * y
    _within("UPDATE x", _err(_interior(s, 2), xa, xa.abs().max()), TOL["axpy"])
    _within("UPDATE r", _err(_interior(s, 3), ra, ra.abs().max()), TOL["axpy"])
    z_ref = ref.precond(_interior(s, 3), lam)
    _within("UPDATE z", _err(_interior(s, 4), z_ref, z_ref.abs().max()), TOL["z"])
    rz = float((_interior(s, 3) * z_ref).sum())
    _within("UPDATE r.z", abs(float(s.dot) - rz) / abs(rz), TOL["dot"])
    # ---- CG_DIR with beta
    beta = 0.61
    z = _interior(s, 4).clone()
    s.sc[SC_BETA] = beta
    s.cg(k.BA_REG_CG_DIR)
    pb = z + beta * p
    _within("DIR p", _err(_interior(s, 5), pb, pb.abs().max()), TOL["axpy"])
    # ---- a real CG solve (RegLMSequencer.trial's launches) from r = -g again, then the trial point
    s.linearize()
    s.cg(k.BA_REG_CG_BEGIN)
    s.cg(k.BA_REG_CG_INIT)
    s.cg(k.BA_REG_CG_DIR)
    for _ in range(CG_ITERS):
        for op in (k.BA_REG_CG_MATVEC, k.BA_REG_CG_ALPHA, k.BA_REG_CG_UPDATE, k.BA_REG_CG_BETA, k.BA_REG_CG_DIR):
            s.cg(op)
    s.apply()
    x = _interior(s, 2)
    Xn, Rn, tn = _point(s, 1)
    Xr, Rr, tr = _apply_step(X, R, t, x, mode)
    assert torch.equal(Xn, Xr) and torch.equal(tn, tr)
    if mode == "full":
        _within("apply R", _err(Rn, Rr, 1.0), TOL["R"])
    else:
        assert torch.equal(Rn, R)  # rotations untouched bit for bit
    # ---- cost(1): trial terms and the predicted decrease from the GPU's own x, D, g
    s.cost(1)
    s.finish_cost(1)
    _, Ft, _ = _check_cost(s, (Xn, Rn, tn) + cost_args[3:], 1)
    terms = x * (lam * D * x - g)
    _within("cost(1) SUM_PRED", abs(float(s.sums[1, SUM_PRED]) - float(terms.sum())) / float(terms.abs().sum()), TOL["pred"])
    assert float(s.sc[SC_PRED]) == float(s.sums[1, SUM_PRED])
    # ---- control: the history row against the reference costs
    s.control()
    h = s.hist[0].cpu().numpy()
    pred = float(s.sums[1, SUM_PRED])
    _within("control F", abs(h[1] - F0) / F0, TOL["cost"])
    _within("control F_trial", abs(h[2] - Ft) / Ft, TOL["cost"])
    assert h[0] == 0 and h[3] == lam and h[5] == float(Ft < F0) and h[7] == pred and h[8] == float(s.sc[SC_CGIT])
    assert h[4] == ((h[1] - h[2]) / pred if pred > 0 else 0.0)
    for i, term in enumerate(lm_reg.TERMS):
        assert _term_err(h[9 + i], term, terms0, raw0, coef) <= TOL[_term_tol(term)], term
    assert h[5] == 1.0 and int(s.sc[k.BA_REG_SC_CUR].item()) == 1  # the first trial from a perturbed start is accepted


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A_full_3_warp_passes", "C_pose_only_3_point_passes", "D_96_joints_8_cams"])
def test_whole_trials_bitwise_repeatable(cuda, clips, name):
    """Two solves of two trials each are bit-identical in every device buffer: a warp that reuses its shared-memory
    slice for a second frame without the synchronisation it needs would break this."""
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    runs = []
    for _ in range(2):
        s = _solver(clip, mode)
        s.run(2)
        runs.append([v.clone() for v in (s.Xh, s.Ch, s.vec, s.pinv, s.sc, s.sums, s.hist) + ((s.lfac,) if s.lfac is not None else ())])
        del s
    for u, v in zip(*runs):
        assert torch.equal(u, v)


# ------------------------------------------------------------------------------------------ shard edges, one GPU
def _bounds(T):
    """[0, W+1), [W+1, W+2), [W+2, T): the middle shard is one frame with a halo on both sides; both outer shards wrap
    (their warps take a second frame)."""
    return [(0, W_MAX + 1), (W_MAX + 1, W_MAX + 2), (W_MAX + 2, T)]


def _sharded(clip, mode, full):
    """Shards over frame ranges with the unsharded solver's scalars (coefficients, T_global, lambda, nu, the bone and
    baseline means) and state (both halves of X and the cameras, every vector) including the halo rows."""
    T = clip["X0"].shape[0]
    shards = []
    for a, b in _bounds(T):
        s = _solver(clip, mode, a, b, local_only=True)
        s.prob.has_prev, s.prob.has_next = int(a > 0), int(b < T)
        s.sc.copy_(full.sc)
        s.Xh.copy_(full.Xh[:, a: b + 2])
        s.Ch.copy_(full.Ch[:, a: b + 2])
        s.vec.copy_(full.vec[:, a: b + 2])
        s.span = (a, b)
        shards.append(s)
    assert [s.Tl for s in shards][1] == 1 and all(_warp_passes(s.Tl) >= 2 for s in (shards[0], shards[2]))
    return shards


def _allreduce(ts):
    tot = ts[0].clone()
    for v in ts[1:]:
        tot += v
    for v in ts:
        v.copy_(tot)


def _halo(shards, kind):
    """The one-frame halo: rank r's row 0 <- rank r-1's last row, its row Tl+1 <- rank r+1's first row."""
    for i, s in enumerate(shards):
        for nb, dst, src in ((i - 1, 0, None), (i + 1, s.Tl + 1, 1)):
            if not 0 <= nb < len(shards):
                continue
            o = shards[nb]
            srow = o.Tl if src is None else src
            if kind == "p":
                s.vec[5, dst] = o.vec[5, srow]
            else:
                s.Xh[:, dst] = o.Xh[:, srow]
                s.Ch[:, dst] = o.Ch[:, srow]


def _same_rows(full, shards, what):
    for s in shards:
        a, b = s.span
        for name, u, v in what(s, a, b):
            assert torch.equal(u, v), (name, s.span, float((u - v).abs().max()))


def _sum_check(full_t, shard_ts, what):
    tot = shard_ts[0].clone()
    for v in shard_ts[1:]:
        tot += v
    assert torch.all(tot[full_t == 0.0] == 0.0), what
    _within("shards: " + what, float(((tot - full_t).abs() / full_t.abs().clamp_min(1e-300)).max()), SHARD_SUM_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A_full_3_warp_passes", "C_pose_only_3_point_passes"])
def test_shard_rows_equal_unsharded_rows(cuda, clips, name):
    """Every per-frame row a shard writes equals the unsharded row bit for bit (the per-frame arithmetic does not depend
    on which warp or shard runs it), after each launch; the shards' raw sums and dot partials add up to the unsharded."""
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    k = _cabi
    full = _solver(clip, mode)
    shards = _sharded(clip, mode, full)
    vec_rows = lambda ids: lambda s, a, b: [(f"vec[{i}]", s.vec[i, 1:-1], full.vec[i, a + 1: b + 1]) for i in ids]  # noqa: E731
    for s in shards:
        s.cost(0)
    _sum_check(full.sums[0], [s.sums[0] for s in shards], "cost(0) sums")
    full.linearize()
    for s in shards:
        s.linearize()
    _same_rows(full, shards, lambda s, a, b: vec_rows((0, 1, 3))(s, a, b) + [("pinv", s.pinv, full.pinv[a:b])]
               + ([("lfac", s.lfac, full.lfac[a:b])] if s.lfac is not None else []))

    def cg(op):
        full.cg(op)
        for s in shards:
            s.cg(op)
        return full.dot.clone(), [s.dot.clone() for s in shards]

    _sum_check(*cg(k.BA_REG_CG_BEGIN), "BEGIN r.z")
    _same_rows(full, shards, vec_rows((2, 3, 4, 5, 6)))
    gen = torch.Generator(device=cuda).manual_seed(9)
    fmask = torch.cat([torch.ones(3 * J, dtype=torch.bool, device=cuda), torch.tensor(_FREE[mode], device=cuda).repeat(full.C)])
    full.vec[5, 1:-1] = torch.randn(T, full.nf, generator=gen, device=cuda, dtype=torch.float64) * fmask
    for s in shards:
        a, b = s.span
        s.vec[5].copy_(full.vec[5, a: b + 2])  # interior and both halo rows
    for e in [full] + shards:
        e.sc[SC_DONE], e.sc[SC_ALPHA], e.sc[SC_BETA] = 0.0, 0.37, 0.61
    _sum_check(*cg(k.BA_REG_CG_MATVEC), "MATVEC p.y")
    _same_rows(full, shards, vec_rows((6,)))
    _sum_check(*cg(k.BA_REG_CG_UPDATE), "UPDATE r.z")
    _same_rows(full, shards, vec_rows((2, 3, 4)))
    cg(k.BA_REG_CG_DIR)
    _same_rows(full, shards, vec_rows((5,)))
    full.apply()
    for s in shards:
        s.apply()
    _same_rows(full, shards, lambda s, a, b: [("X", s.Xh[:, 1:-1], full.Xh[:, a + 1: b + 1]), ("cams", s.Ch[:, 1:-1], full.Ch[:, a + 1: b + 1])])
    _halo(shards, "trial")
    full.cost(1)
    for s in shards:
        s.cost(1)
    _sum_check(full.sums[1], [s.sums[1] for s in shards], "cost(1) sums")


def _lockstep_trial(shards):
    """RegLMSequencer.trial over the shards: all-reduces as host-side sums, halo exchanges as row copies."""
    k = _cabi

    def each(fn, *args):
        for s in shards:
            getattr(s, fn)(*args)

    each("linearize")
    each("cg", k.BA_REG_CG_BEGIN)
    _allreduce([s.dot for s in shards])
    each("cg", k.BA_REG_CG_INIT)
    each("cg", k.BA_REG_CG_DIR)
    for _ in range(CG_ITERS):
        _halo(shards, "p")
        each("cg", k.BA_REG_CG_MATVEC)
        _allreduce([s.dot for s in shards])
        each("cg", k.BA_REG_CG_ALPHA)
        each("cg", k.BA_REG_CG_UPDATE)
        _allreduce([s.dot for s in shards])
        each("cg", k.BA_REG_CG_BETA)
        each("cg", k.BA_REG_CG_DIR)
    each("apply")
    _halo(shards, "trial")
    each("cost", 1)
    _allreduce([s.sums[1] for s in shards])
    each("finish_cost", 1)
    each("control")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A_full_3_warp_passes", "C_pose_only_3_point_passes"])
def test_lockstep_shards_follow_the_unsharded_trajectory(cuda, clips, name):
    """Four trials over the three shards in RegLMSequencer.trial's order: trial costs within 1e-12 relative of the
    unsharded CUDA solve, the same decisions and CG iteration counts, X within 1e-10."""
    rig, T, J, mode = CASES[name]
    clip = clips(rig, T, J)
    n = 4
    full = _solver(clip, mode)
    shards = _sharded(clip, mode, full)
    for s in shards:  # RegLMSequencer.setup_cost: the halos are already in place
        s.cost(0)
    _allreduce([s.sums[0] for s in shards])
    for s in shards:
        s.finish_cost(0)
    full.run(n)
    for _ in range(n):
        _lockstep_trial(shards)
    for s in shards:
        s.iters_done = n
    hf, hs = full.history, shards[0].history
    for s in shards[1:]:
        assert s.history == hs  # every shard writes the same row
    n_cmp = _check(hs, hf, n)
    for i in range(n):
        dev = abs(hs[i]["trial_cost"] - hf[i]["trial_cost"]) / hf[i]["trial_cost"]
        print(f"    trial {i}: trial cost {hf[i]['trial_cost']:.9f}  dev {dev:.2e}  cg {hs[i]['cg_iters']} / {hf[i]['cg_iters']}  "
              f"accepted {hs[i]['accepted']} / {hf[i]['accepted']}")
        assert dev <= TRAJ_COST_TOL and abs(hs[i]["cost"] - hf[i]["cost"]) <= TRAJ_COST_TOL * hf[i]["cost"]
        if i < n_cmp:
            assert hs[i]["accepted"] == hf[i]["accepted"] and hs[i]["cg_iters"] == hf[i]["cg_iters"], i
    Xs = torch.cat([s.X for s in shards])
    dx = float((Xs - full.X).abs().max())
    print(f"    max |X_sharded - X| {dx:.2e}")
    assert dx <= TRAJ_X_TOL
