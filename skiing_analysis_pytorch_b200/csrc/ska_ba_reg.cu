// ska_ba_reg.cu - Levenberg-Marquardt over the reference's FULL configured objective (SURVEY rows N1 / e3):
//     F = w_r reprojection_loss + w_s camera_smooth_loss + w_b baseline_reg_loss + w_l bone_length_loss + w_t pose_temporal_loss
//                loss.py:90-94        loss.py:103-106          loss.py:109-114         loss.py:134-150         loss.py:153-155
// with PER-FRAME cameras R (T,C,3,3), t (T,C,3) as the call site passes them (vggt/multi_view_process.py:546-564) and the
// weights of configs/vggt.yaml:46-50.  Specification: oracle/lm_reg.py (the optimiser itself is an undefined symbol in the
// reference).  The coupling terms make J^T J block-tridiagonal in time, so the damped normal equations
//     (J^T J + lam diag(J^T J)) delta = -J^T r
// are solved matrix-free by preconditioned conjugate gradients.  The preconditioner is the exact inverse of each FRAME's
// reprojection system [Dp W; W^T Dc] (3x3 point blocks, the frame's cameras, their coupling) through the frame's Schur
// complement onto its cameras - the inter-frame terms it leaves out are weak, and CG converges in 2 (points only) to ~30
// (free cameras, small lambda) iterations where point-block Jacobi needs hundreds (measured in oracle/lm_reg.py).
//
// Layout: a frame is a row.  Vectors over the unknowns are (T_local + 2, 3 J + 6 C) fp64 rows [J x (x,y,z) | C x (d_omega, d_t)]
// with one halo row on each side - the neighbouring shard's edge frame when the clip is sharded by frame range over GPUs
// (the temporal / smoothness terms couple frame t with t +- 1); X and the cameras carry the same halo.  One WARP owns one
// frame: lanes are joints (J <= 96: up to three per lane), camera sums are warp-reduced, everything a frame needs sits in
// the warp's slice of shared memory.  All arithmetic is fp64 (the reference's loss.py computes in the dtype of X; the
// frame Schur complements lose ~1/lambda of their digits).  Every sum is a fixed-order reduction: per-warp partial rows,
// then ba_reduce_columns.  Nothing synchronises with the host: the CG scalars, the convergence flag, the gain ratio and
// the accept / reject decision live in d_sc, so a whole LM iteration (with its NCCL all-reduces when sharded) replays
// as one CUDA graph.
//
// Robust loss (Huber / Cauchy, include/ska.h; spec tests/oracle_robust_reg.py run_lm_reg): the kernels that read observations
// take it as a template argument.  The reprojection weight becomes c_r conf omega(s) in every sum of the step (observe<Loss>)
// and the cost sums conf rho(s); the regularisers and every other kernel are the L2 solver's.
#include <cuda_runtime.h>
#include <math.h>

#include "ska_ba.cuh"
#include "ska_internal.h"
#include "ska_peer.cuh"

namespace ska {
namespace {

constexpr int kWarpsPerBlock = 4;
constexpr int kMaxGridBlocks = 148 * 8;
constexpr int NS = SKA_BA_REG_SUMS;  // 40
constexpr double kZMin = 1e-6;

// d_sc slots (include/ska.h documents the ones a caller reads)
enum : int {
  SC_CUR = SKA_BA_REG_SC_CUR, SC_LAM = SKA_BA_REG_SC_LAMBDA, SC_NU = SKA_BA_REG_SC_NU, SC_ITER = SKA_BA_REG_SC_ITER,
  SC_F = SKA_BA_REG_SC_COST, SC_FT = 5, SC_PRED = 6, SC_ACC = SKA_BA_REG_SC_ACCEPTED, SC_RZ0 = 8, SC_RZ = 9, SC_PAP = 10, SC_ALPHA = 11,
  SC_BETA = 12, SC_DONE = 13, SC_CGIT = 14, SC_TOL2 = SKA_BA_REG_SC_TOL2, SC_CR = SKA_BA_REG_SC_COEF, SC_CL = SC_CR + 1, SC_CT = SC_CR + 2,
  SC_CS = SC_CR + 3, SC_CB = SC_CR + 4, SC_TG = SKA_BA_REG_SC_T_GLOBAL, SC_REF = 22 /* 16 bone means */, SC_BMEAN = 38, SC_NCL = 39,
  SC_TERM = 40 /* 5 weighted terms of the current cost */, SC_DOT = SKA_BA_REG_SC_DOT
};
enum : int { SUM_REPROJ = 0, SUM_CLAMP = 1, SUM_TEMP = 2, SUM_SMOOTH = 3, SUM_B = 4, SUM_B2 = 5, SUM_PRED = 6, SUM_L = 8, SUM_L2 = 24 };

struct RegArgs {
  int64_t Tl;
  int J, C, nb, has_prev, has_next, nf, n6, nS;
  uint32_t free6;
  int32_t bi[SKA_MAX_BONES], bj[SKA_MAX_BONES];
  const float* x2d;
  const float* conf;
  const double* K;
  double* Xh;
  double* Ch;
  double *g, *D, *x, *r, *z, *p, *y;
  double* pinv;
  double* lfac;
  double* sc;
  double* sums;
  double* part;   // [W][NS]
  double* dpart;  // [W]
  double* ppart;  // [W]  predicted-decrease partials (apply -> cost(trial))
  int W;
};
// The robust scale goes after everything the L2 solver passes a kernel, so that the L2 instantiations read every parameter
// at its old offset: appended to the argument block of the kernels that take nothing else (linearisation, matrix-vector
// product), a trailing parameter of reg_cost_kernel and reg_precond_kernel.
struct RegArgsRs : RegArgs {
  RobustScale rs;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void cross(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ void matvec3(const double* R, const double v[3], double o[3]) {  // o = R v
  o[0] = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
  o[1] = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
  o[2] = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
}
__device__ __forceinline__ void matTvec3(const double* R, const double v[3], double o[3]) {  // o = R^T v
  o[0] = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
  o[1] = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
  o[2] = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
}
// symmetric 3x3 packed [00 01 02 11 12 22] times a vector
__device__ __forceinline__ void sym3vec(const double N[6], const double v[3], double o[3]) {
  o[0] = N[0] * v[0] + N[1] * v[1] + N[2] * v[2];
  o[1] = N[1] * v[0] + N[3] * v[1] + N[4] * v[2];
  o[2] = N[2] * v[0] + N[4] * v[1] + N[5] * v[2];
}

// One observation: camera-frame point, residual, N = w' (ju ju^T + jv jv^T), q = w' (ju eu + jv ev).  loss.py:17-87.
// w' = w under L2; under a robust loss w' = w omega(|e|^2), omega at the current state and not differentiated (iteratively
// reweighted Gauss-Newton).  Every kernel that needs N recomputes omega from the same d2 expression, so the linearisation,
// the matrix-vector product and the preconditioner of a trial weight each observation with the same bits.
struct Obs {
  double p[3];  // R X
  double N[6];
  double q[3];
  double d2;    // |e|^2
  bool clamped;
};
template <int Loss>
__device__ __forceinline__ void observe(const double* cam /*R(9) t(3)*/, const double* K, const double X[3], double u_obs, double v_obs,
                                        double w, const RobustScale& rs, Obs& o) {
  matvec3(cam, X, o.p);
  const double xc = o.p[0] + cam[9], yc = o.p[1] + cam[10], zc = o.p[2] + cam[11];
  o.clamped = zc < kZMin;
  const double iz = 1.0 / fmax(zc, kZMin);
  const double x = xc * iz, y = yc * iz;
  const double eu = K[0] * x + K[1] * y + K[2] - u_obs, ev = K[3] * x + K[4] * y + K[5] - v_obs;
  const double live = o.clamped ? 0.0 : 1.0;  // the clamp has zero derivative (what autograd of loss.py:67 gives)
  const double ju[3] = {K[0] * iz, K[1] * iz, -(K[0] * x + K[1] * y) * iz * live};
  const double jv[3] = {K[3] * iz, K[4] * iz, -(K[3] * x + K[4] * y) * iz * live};
  o.d2 = eu * eu + ev * ev;
  if constexpr (Loss != kLossL2) w *= robust_omega<Loss>(o.d2, rs);
  o.N[0] = w * (ju[0] * ju[0] + jv[0] * jv[0]);
  o.N[1] = w * (ju[0] * ju[1] + jv[0] * jv[1]);
  o.N[2] = w * (ju[0] * ju[2] + jv[0] * jv[2]);
  o.N[3] = w * (ju[1] * ju[1] + jv[1] * jv[1]);
  o.N[4] = w * (ju[1] * ju[2] + jv[1] * jv[2]);
  o.N[5] = w * (ju[2] * ju[2] + jv[2] * jv[2]);
#pragma unroll
  for (int k = 0; k < 3; ++k) o.q[k] = w * (ju[k] * eu + jv[k] * ev);
}

// camera centre Cc = -R^T t and, for a parameter direction (d_omega, d_t), its first-order change -R^T (d_t + t x d_omega)
__device__ __forceinline__ void centre(const double* cam, double o[3]) {
  matTvec3(cam, cam + 9, o);
  o[0] = -o[0], o[1] = -o[1], o[2] = -o[2];
}
__device__ __forceinline__ void centre_dir(const double* cam, const double* pc /*6*/, uint32_t free6, double o[3]) {
  double w[3], tt[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    w[k] = (free6 >> k) & 1u ? pc[k] : 0.0;
    tt[k] = (free6 >> (3 + k)) & 1u ? pc[3 + k] : 0.0;
  }
  double c[3];
  cross(cam + 9, w, c);
  const double s[3] = {tt[0] + c[0], tt[1] + c[1], tt[2] + c[2]};
  matTvec3(cam, s, o);
  o[0] = -o[0], o[1] = -o[1], o[2] = -o[2];
}
// J_Cc^T v for v in world coordinates: d_t part -R v, d_omega part t x (R v)
__device__ __forceinline__ void centre_adj(const double* cam, const double v[3], double o6[6]) {
  double m[3];
  matvec3(cam, v, m);
  cross(cam + 9, m, o6);
  o6[3] = -m[0], o6[4] = -m[1], o6[5] = -m[2];
}

__device__ __forceinline__ int tri(int r, int c) { return r * (r + 1) / 2 + c; }  // packed lower triangle, c <= r

// inverse of a symmetric 3x3 [00 01 02 11 12 22]; not positive definite -> the zero matrix (no step for that point: the
// rule of oracle/lm.py _safe_inverse)
__device__ __forceinline__ void inv_sym3(const double H[6], double o[6]) {
  const double c00 = H[3] * H[5] - H[4] * H[4], c01 = H[2] * H[4] - H[1] * H[5], c02 = H[1] * H[4] - H[2] * H[3];
  const double det = H[0] * c00 + H[1] * c01 + H[2] * c02;
  const bool ok = H[0] > 0.0 && (H[0] * H[3] - H[1] * H[1]) > 0.0 && det > 0.0 && isfinite(det);
  const double id = ok ? 1.0 / det : 0.0;
  o[0] = c00 * id;
  o[1] = c01 * id;
  o[2] = c02 * id;
  o[3] = (H[0] * H[5] - H[2] * H[2]) * id;
  o[4] = (H[1] * H[2] - H[0] * H[4]) * id;
  o[5] = (H[0] * H[3] - H[1] * H[1]) * id;
}

__device__ __forceinline__ const double* frame_X(const RegArgs& a, int buf, int64_t row) {
  return a.Xh + ((int64_t)buf * (a.Tl + 2) + row) * a.J * 3;
}
__device__ __forceinline__ const double* frame_C(const RegArgs& a, int buf, int64_t row) {
  return a.Ch + ((int64_t)buf * (a.Tl + 2) + row) * a.C * 12;
}

// ------------------------------------------------------------------------------------------------ cost
// sums of one point (buffer `buf`): raw reprojection sum, clamp count, temporal / smoothness pairs (t, t+1) owned by t,
// per-bone sum L and sum L^2, baseline sum b and sum b^2.  The weights and the means enter in reg_finish_cost.
template <int Loss>
__global__ void __launch_bounds__(32 * kWarpsPerBlock) reg_cost_kernel(const RegArgs a, int which, const RobustScale rs) {
  const int lane = threadIdx.x & 31, wid = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int buf = which == 0 ? (int)a.sc[SC_CUR] : 1 - (int)a.sc[SC_CUR];
  double s_rep = 0.0, s_cl = 0.0, s_tmp = 0.0, s_sm = 0.0, s_b = 0.0, s_b2 = 0.0, s_L = 0.0, s_L2 = 0.0;
  for (int64_t f = wid; f < a.Tl; f += a.W) {
    const int64_t row = f + 1;
    const double* X = frame_X(a, buf, row);
    const double* Cm = frame_C(a, buf, row);
    const bool next = f + 1 < a.Tl || a.has_next;
    for (int j = lane; j < a.J; j += 32) {
      const double Xj[3] = {X[3 * j], X[3 * j + 1], X[3 * j + 2]};
      for (int c = 0; c < a.C; ++c) {
        const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
        const double w = (double)a.conf[(f * a.C + c) * a.J + j];
        Obs o;
        observe<kLossL2>(Cm + 12 * c, a.K + 9 * c, Xj, (double)uv.x, (double)uv.y, 1.0, rs, o);
        s_rep += w * robust_rho<Loss>(o.d2, rs);
        s_cl += o.clamped ? 1.0 : 0.0;
      }
      if (next) {
        const double* Xn = X + a.J * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double d = Xn[3 * j + k] - Xj[k];
          s_tmp += d * d;
        }
      }
    }
    if (lane < a.nb) {
      const int i = a.bi[lane], j = a.bj[lane];
      const double d0 = X[3 * i] - X[3 * j], d1 = X[3 * i + 1] - X[3 * j + 1], d2 = X[3 * i + 2] - X[3 * j + 2];
      const double L2 = d0 * d0 + d1 * d1 + d2 * d2;
      s_L += sqrt(L2);
      s_L2 += L2;
    }
    if (lane < a.C) {
      double c0[3];
      centre(Cm + 12 * lane, c0);
      if (next) {
        double c1[3];
        centre(Cm + 12 * (a.C + lane), c1);
#pragma unroll
        for (int k = 0; k < 3; ++k) s_sm += (c1[k] - c0[k]) * (c1[k] - c0[k]);
      }
      if (lane == 0 && a.C >= 2) {
        double c1[3];
        centre(Cm + 12, c1);
        const double b2 = (c0[0] - c1[0]) * (c0[0] - c1[0]) + (c0[1] - c1[1]) * (c0[1] - c1[1]) + (c0[2] - c1[2]) * (c0[2] - c1[2]);
        s_b += sqrt(b2);
        s_b2 += b2;
      }
    }
  }
  s_rep = warp_sum(s_rep), s_cl = warp_sum(s_cl), s_tmp = warp_sum(s_tmp), s_sm = warp_sum(s_sm);
  double* out = a.part + (int64_t)wid * NS;
  if (lane == 0) {
    out[SUM_REPROJ] = s_rep, out[SUM_CLAMP] = s_cl, out[SUM_TEMP] = s_tmp, out[SUM_SMOOTH] = s_sm, out[SUM_B] = s_b, out[SUM_B2] = s_b2;
    out[SUM_PRED] = 0.0, out[7] = 0.0;
  }
  if (lane < SKA_MAX_BONES) out[SUM_L + lane] = s_L, out[SUM_L2 + lane] = s_L2;
}

// after the all-reduce of the sums: the weighted terms, F, and (for the current point) the detached means
__global__ void reg_finish_cost_kernel(const RegArgs a, int which, const PeerDev peer) {
  if (peer.world > 1) peer_exchange_block(peer, a.sums + which * NS, NS, a.sums + which * NS, 0);  // the sums' all-reduce, fused
  if (threadIdx.x != 0) return;
  double* sc = a.sc;
  const double* s = a.sums + which * NS;
  const double Tg = sc[SC_TG];
  double bone = 0.0;
  for (int b = 0; b < a.nb; ++b) bone += s[SUM_L2 + b] - s[SUM_L + b] * s[SUM_L + b] / Tg;
  const double base = a.C >= 2 ? s[SUM_B2] - s[SUM_B] * s[SUM_B] / Tg : 0.0;
  const double terms[5] = {sc[SC_CR] * s[SUM_REPROJ], sc[SC_CS] * s[SUM_SMOOTH], sc[SC_CB] * base, sc[SC_CL] * bone, sc[SC_CT] * s[SUM_TEMP]};
  const double F = terms[0] + terms[1] + terms[2] + terms[3] + terms[4];
  if (which == 0) {
    sc[SC_F] = F;
    sc[SC_NCL] = s[SUM_CLAMP];
    for (int k = 0; k < 5; ++k) sc[SC_TERM + k] = terms[k];
    for (int b = 0; b < SKA_MAX_BONES; ++b) sc[SC_REF + b] = s[SUM_L + b] / Tg;
    sc[SC_BMEAN] = s[SUM_B] / Tg;
  } else {
    sc[SC_FT] = F;
    sc[SC_PRED] = s[SUM_PRED];
  }
}

// ------------------------------------------------------------------------------------------------ per-warp shared memory
struct Smem {
  double *X, *P, *Cam, *Y, *S, *V;
  __device__ Smem(double* base, const RegArgs& a) {
    X = base;                  // J*3   the frame's points
    P = X + a.J * 3;           // J*9   per point: block (6) + 3 scratch
    Cam = P + a.J * 9;         // C*28  per camera: block (21) + vector (6) + pad
    V = Cam + a.C * 28;        // nf    a vector row
    S = V + a.nf;              // nS    frame Schur complement / its Cholesky factor
    Y = S + a.nS;              // 96 * n6  staged rows
  }
};
static size_t smem_doubles_per_warp(int J, int C) {
  const int n6 = 6 * C, nS = n6 * (n6 + 1) / 2, nf = 3 * J + 6 * C;
  return (size_t)J * 3 + (size_t)J * 9 + (size_t)C * 28 + nf + nS + (size_t)96 * n6;
}

// Hcc block of one observation: G^T N G with G = [-[p]x | I] (21 upper-triangle entries, row-major) and G^T q (6)
__device__ __forceinline__ void camera_block(const Obs& o, double H[21], double gq[6], bool with_q) {
  // G columns: k < 3: e_k x p; k >= 3: e_{k-3}
  double G[6][3];
  G[0][0] = 0.0, G[0][1] = -o.p[2], G[0][2] = o.p[1];
  G[1][0] = o.p[2], G[1][1] = 0.0, G[1][2] = -o.p[0];
  G[2][0] = -o.p[1], G[2][1] = o.p[0], G[2][2] = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int i = 0; i < 3; ++i) G[3 + k][i] = i == k ? 1.0 : 0.0;
  int e = 0;
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    double NG[3];
    sym3vec(o.N, G[r], NG);
#pragma unroll
    for (int c = r; c < 6; ++c, ++e) H[e] += G[c][0] * NG[0] + G[c][1] * NG[1] + G[c][2] * NG[2];
    if (with_q) gq[r] += G[r][0] * o.q[0] + G[r][1] * o.q[1] + G[r][2] * o.q[2];
  }
}
__device__ __forceinline__ int up6(int r, int c) { return r * 6 - r * (r - 1) / 2 + (c - r); }  // 6x6 upper triangle, c >= r

// ------------------------------------------------------------------------------------------------ linearisation
// per frame: gradient g = J^T r, D = diag(J^T J), r_cg = -g, the damped point blocks' inverses, and the Cholesky factor of
// the frame's Schur complement S = Dc - sum_j W_j^T Dp_j^-1 W_j  (Dp, Dc: damped diagonal blocks of J^T J).
template <int Loss>
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 4) reg_linearize_kernel(const RegArgsRs a) {
  extern __shared__ double smem_d[];
  // launched with 4, 2 or 1 warps per block (the largest frames - 96 joints x 8 cameras - need 60 KB of shared memory per warp)
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, wid = blockIdx.x * (int)(blockDim.x >> 5) + wl;
  const size_t per_warp = (size_t)a.J * 12 + (size_t)a.C * 28 + a.nf + a.nS + (size_t)96 * a.n6;
  Smem sm(smem_d + wl * per_warp, a);
  const double* sc = a.sc;
  const int buf = (int)sc[SC_CUR];
  const double lam = sc[SC_LAM], cr = sc[SC_CR], cl = sc[SC_CL], ct = sc[SC_CT], cs = sc[SC_CS], cb = sc[SC_CB];
  const bool cams_free = a.free6 != 0;
  for (int64_t f = wid; f < a.Tl; f += a.W) {
    const int64_t row = f + 1;
    const double* X = frame_X(a, buf, row);
    const double* Cm = frame_C(a, buf, row);
    const bool prev = f > 0 || a.has_prev, next = f + 1 < a.Tl || a.has_next;
    __syncwarp();
    for (int i = lane; i < a.J * 3; i += 32) sm.X[i] = X[i];
    for (int i = lane; i < a.J * 9; i += 32) sm.P[i] = 0.0;
    for (int i = lane; i < a.nS; i += 32) sm.S[i] = 0.0;
    __syncwarp();
    // ---- reprojection: point blocks (lane-private rows of sm.P), camera blocks (warp-reduced)
    for (int c = 0; c < a.C; ++c) {
      const double* cam = Cm + 12 * c;
      const double* K = a.K + 9 * c;
      double H[21], gq[6];
#pragma unroll
      for (int k = 0; k < 21; ++k) H[k] = 0.0;
#pragma unroll
      for (int k = 0; k < 6; ++k) gq[k] = 0.0;
      for (int j = lane; j < a.J; j += 32) {
        const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
        const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
        Obs o;
        observe<Loss>(cam, K, sm.X + 3 * j, (double)uv.x, (double)uv.y, w, a.rs, o);
        // Hpp += R^T N R, gX += R^T q
        double RtN[3][3];  // rows of R^T N: (R^T N)[i][k] = sum_a R[a][i] N[a][k]
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const double col[3] = {cam[i], cam[3 + i], cam[6 + i]};
          sym3vec(o.N, col, RtN[i]);  // N symmetric: N col = (col^T N)^T
        }
        double* P = sm.P + 9 * j;
        int e = 0;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int k = i; k < 3; ++k, ++e) P[e] += RtN[i][0] * cam[k] + RtN[i][1] * cam[3 + k] + RtN[i][2] * cam[6 + k];
        double gx[3];
        matTvec3(cam, o.q, gx);
        P[6] += gx[0], P[7] += gx[1], P[8] += gx[2];
        if (cams_free) camera_block(o, H, gq, true);
      }
      if (cams_free) {
#pragma unroll
        for (int k = 0; k < 21; ++k) H[k] = warp_sum(H[k]);
#pragma unroll
        for (int k = 0; k < 6; ++k) gq[k] = warp_sum(gq[k]);
        if (lane == 0) {
#pragma unroll
          for (int k = 0; k < 21; ++k) sm.Cam[28 * c + k] = H[k];
#pragma unroll
          for (int k = 0; k < 6; ++k) sm.Cam[28 * c + 21 + k] = gq[k];
        }
      }
    }
    __syncwarp();
    // ---- point regularisers, D, damped inverse, g
    double* gr = a.g + row * a.nf;
    double* Dr = a.D + row * a.nf;
    double* rr = a.r + row * a.nf;
    for (int j = lane; j < a.J; j += 32) {
      double* P = sm.P + 9 * j;
      const double Xj[3] = {sm.X[3 * j], sm.X[3 * j + 1], sm.X[3 * j + 2]};
      for (int b = 0; b < a.nb; ++b) {
        const int bi = a.bi[b], bj = a.bj[b];
        if (bi != j && bj != j) continue;
        const int o = bi == j ? bj : bi;
        const double sgn = bi == j ? 1.0 : -1.0;
        double u[3] = {sgn * (Xj[0] - sm.X[3 * o]), sgn * (Xj[1] - sm.X[3 * o + 1]), sgn * (Xj[2] - sm.X[3 * o + 2])};  // X_bi - X_bj
        const double L = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        const double iL = 1.0 / L;
        u[0] *= iL, u[1] *= iL, u[2] *= iL;
        const double res = cl * (L - sc[SC_REF + b]) * sgn;
        P[0] += cl * u[0] * u[0], P[1] += cl * u[0] * u[1], P[2] += cl * u[0] * u[2];
        P[3] += cl * u[1] * u[1], P[4] += cl * u[1] * u[2], P[5] += cl * u[2] * u[2];
        P[6] += res * u[0], P[7] += res * u[1], P[8] += res * u[2];
      }
      const double nn = ct * ((prev ? 1.0 : 0.0) + (next ? 1.0 : 0.0));
      P[0] += nn, P[3] += nn, P[5] += nn;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        double gk = 0.0;
        if (prev) gk += Xj[k] - X[3 * j + k - a.J * 3];
        if (next) gk -= X[3 * j + k + a.J * 3] - Xj[k];
        P[6 + k] += ct * gk;
      }
      const double d[3] = {P[0], P[3], P[5]};
      const double Hd[6] = {P[0] + lam * d[0], P[1], P[2], P[3] + lam * d[1], P[4], P[5] + lam * d[2]};
      double inv[6];
      inv_sym3(Hd, inv);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        gr[3 * j + k] = P[6 + k];
        rr[3 * j + k] = -P[6 + k];
        Dr[3 * j + k] = d[k];
      }
      double* pg = a.pinv + (f * a.J + j) * 6;
#pragma unroll
      for (int k = 0; k < 6; ++k) pg[k] = inv[k], P[k] = inv[k];
    }
    if (!cams_free) {
      for (int i = lane; i < 6 * a.C; i += 32) gr[3 * a.J + i] = 0.0, rr[3 * a.J + i] = 0.0, Dr[3 * a.J + i] = 0.0;
      continue;
    }
    // ---- camera regularisers (lane c owns camera c), D, g, damped diagonal blocks into S
    if (lane < a.C) {
      const int c = lane;
      const double* cam = Cm + 12 * c;
      double* B = sm.Cam + 28 * c;
      double c0[3];
      centre(cam, c0);
      const double nn = cs * ((prev ? 1.0 : 0.0) + (next ? 1.0 : 0.0));
      double v[3] = {0.0, 0.0, 0.0};
      if (prev) {
        double cp[3];
        centre(cam - 12 * a.C, cp);
#pragma unroll
        for (int k = 0; k < 3; ++k) v[k] += cs * (c0[k] - cp[k]);
      }
      if (next) {
        double cn[3];
        centre(cam + 12 * a.C, cn);
#pragma unroll
        for (int k = 0; k < 3; ++k) v[k] -= cs * (cn[k] - c0[k]);
      }
      double adj[6];
      centre_adj(cam, v, adj);
#pragma unroll
      for (int k = 0; k < 6; ++k) B[21 + k] += adj[k];
      // J_Cc^T J_Cc = [[t]x^T [t]x, [t]x^T; [t]x, I]  (R cancels)
      const double* t = cam + 9;
      const double tx[3][3] = {{0.0, -t[2], t[1]}, {t[2], 0.0, -t[0]}, {-t[1], t[0], 0.0}};
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int q = r; q < 3; ++q) B[up6(r, q)] += nn * (tx[0][r] * tx[0][q] + tx[1][r] * tx[1][q] + tx[2][r] * tx[2][q]);
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int q = 0; q < 3; ++q) B[up6(r, 3 + q)] += nn * tx[q][r];  // ([t]x^T)[r][q] = [t]x[q][r]
      B[up6(3, 3)] += nn, B[up6(4, 4)] += nn, B[up6(5, 5)] += nn;
      if (a.C >= 2 && c < 2 && cb != 0.0) {
        double co[3];
        centre(Cm + 12 * (1 - c), co);
        const double sgn = c == 0 ? 1.0 : -1.0;
        double nh[3] = {sgn * (c0[0] - co[0]), sgn * (c0[1] - co[1]), sgn * (c0[2] - co[2])};  // Cc_0 - Cc_1
        const double b = sqrt(nh[0] * nh[0] + nh[1] * nh[1] + nh[2] * nh[2]);
        nh[0] /= b, nh[1] /= b, nh[2] /= b;
        const double nv[3] = {sgn * nh[0], sgn * nh[1], sgn * nh[2]};
        double jn[6];
        centre_adj(cam, nv, jn);  // gradient of the baseline w.r.t. this camera's parameters
        const double res = cb * (b - sc[SC_BMEAN]);
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          B[21 + r] += res * jn[r];
#pragma unroll
          for (int q = r; q < 6; ++q) B[up6(r, q)] += cb * jn[r] * jn[q];
        }
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        const bool fr = (a.free6 >> r) & 1u;
        const double d = fr ? B[up6(r, r)] : 0.0;
        const double gk = fr ? B[21 + r] : 0.0;
        gr[3 * a.J + 6 * c + r] = gk;
        rr[3 * a.J + 6 * c + r] = -gk;
        Dr[3 * a.J + 6 * c + r] = d;
#pragma unroll
        for (int q = 0; q <= r; ++q) {
          const bool fq = (a.free6 >> q) & 1u;
          double val = (fr && fq) ? B[up6(q, r)] : 0.0;
          if (q == r) val = fr ? val + lam * d : 1.0;
          sm.S[tri(6 * c + r, 6 * c + q)] = val;
        }
      }
    }
    __syncwarp();
    // ---- S -= sum_j Y_j^T Y_j,  Y_j = Li_j^T W_j  (Li Li^T = Dp_j^-1),  W_jc = R_c^T N_jc G_jc   (3 x 6 per camera)
    for (int j0 = 0; j0 < a.J; j0 += 32) {
      const int j = j0 + lane;
      double* Yr = sm.Y + (size_t)lane * 3 * a.n6;
      if (j < a.J) {
        const double* inv = sm.P + 9 * j;
        // Cholesky Dp^-1 = Li Li^T (lower); a zero matrix (unobserved point) stays zero
        double l00 = inv[0] > 0.0 ? sqrt(inv[0]) : 0.0;
        const double il00 = l00 > 0.0 ? 1.0 / l00 : 0.0;
        const double l10 = inv[1] * il00, l20 = inv[2] * il00;
        const double d11 = inv[3] - l10 * l10;
        const double l11 = d11 > 0.0 ? sqrt(d11) : 0.0;
        const double il11 = l11 > 0.0 ? 1.0 / l11 : 0.0;
        const double l21 = (inv[4] - l20 * l10) * il11;
        const double d22 = inv[5] - l20 * l20 - l21 * l21;
        const double l22 = d22 > 0.0 ? sqrt(d22) : 0.0;
        for (int c = 0; c < a.C; ++c) {
          const double* cam = Cm + 12 * c;
          const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
          const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
          Obs o;
          observe<Loss>(cam, a.K + 9 * c, sm.X + 3 * j, (double)uv.x, (double)uv.y, w, a.rs, o);
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            double col[3] = {0.0, 0.0, 0.0};
            if ((a.free6 >> k) & 1u) {
              double gk[3];
              if (k < 3) {
                const double ek[3] = {k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0};
                cross(ek, o.p, gk);
              } else {
                gk[0] = k == 3 ? 1.0 : 0.0, gk[1] = k == 4 ? 1.0 : 0.0, gk[2] = k == 5 ? 1.0 : 0.0;
              }
              double ng[3];
              sym3vec(o.N, gk, ng);
              matTvec3(cam, ng, col);  // column k of W_jc
            }
            // Y = Li^T W: row 0 = l00 w0 + l10 w1 + l20 w2, row 1 = l11 w1 + l21 w2, row 2 = l22 w2
            Yr[0 * a.n6 + 6 * c + k] = l00 * col[0] + l10 * col[1] + l20 * col[2];
            Yr[1 * a.n6 + 6 * c + k] = l11 * col[1] + l21 * col[2];
            Yr[2 * a.n6 + 6 * c + k] = l22 * col[2];
          }
        }
      } else {
        for (int k = 0; k < 3 * a.n6; ++k) Yr[k] = 0.0;
      }
      __syncwarp();
      for (int e = lane; e < a.nS; e += 32) {
        int r = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
        while (tri(r + 1, 0) <= e) ++r;
        while (tri(r, 0) > e) --r;
        const int c = e - tri(r, 0);
        double s = 0.0;
        for (int q = 0; q < 96; ++q) s += sm.Y[(size_t)q * a.n6 + r] * sm.Y[(size_t)q * a.n6 + c];
        sm.S[e] -= s;
      }
      __syncwarp();
    }
    // ---- in-place Cholesky S = L L^T (packed lower); a non-positive pivot decouples that parameter
    for (int k = 0; k < a.n6; ++k) {
      const double d = sm.S[tri(k, k)];
      const bool ok = d > 0.0 && isfinite(d);
      const double l = ok ? sqrt(d) : 1.0;
      __syncwarp();
      if (lane == 0) sm.S[tri(k, k)] = l;
      for (int r = k + 1 + lane; r < a.n6; r += 32) sm.S[tri(r, k)] = ok ? sm.S[tri(r, k)] / l : 0.0;
      __syncwarp();
      for (int r = k + 1 + lane; r < a.n6; r += 32) {
        const double lrk = sm.S[tri(r, k)];
        for (int c = k + 1; c <= r; ++c) sm.S[tri(r, c)] -= lrk * sm.S[tri(c, k)];
      }
      __syncwarp();
    }
    double* Lg = a.lfac + f * a.nS;
    for (int e = lane; e < a.nS; e += 32) Lg[e] = sm.S[e];
  }
}

// ------------------------------------------------------------------------------------------------ matrix-vector product
// y = (J^T J + lam D) p for the frame's row; partial dot p . y
template <int Loss>
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 4) reg_matvec_kernel(const RegArgsRs a) {
  extern __shared__ double smem_d[];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, wid = blockIdx.x * kWarpsPerBlock + wl;
  const double* sc = a.sc;
  double dot = 0.0;
  if (sc[SC_DONE] == 0.0) {
    double* V = smem_d + (size_t)wl * (a.nf + 3 * a.J);
    double* sX = V + a.nf;
    const int buf = (int)sc[SC_CUR];
    const double lam = sc[SC_LAM], cr = sc[SC_CR], cl = sc[SC_CL], ct = sc[SC_CT], cs = sc[SC_CS], cb = sc[SC_CB];
    const bool cams_free = a.free6 != 0;
    for (int64_t f = wid; f < a.Tl; f += a.W) {
      const int64_t row = f + 1;
      const double* X = frame_X(a, buf, row);
      const double* Cm = frame_C(a, buf, row);
      const double* pr = a.p + row * a.nf;
      double* yr = a.y + row * a.nf;
      const double* Dr = a.D + row * a.nf;
      const bool prev = f > 0 || a.has_prev, next = f + 1 < a.Tl || a.has_next;
      __syncwarp();
      for (int i = lane; i < a.nf; i += 32) V[i] = pr[i];
      for (int i = lane; i < 3 * a.J; i += 32) sX[i] = X[i];
      __syncwarp();
      double yx[3][3];  // up to three joints per lane
#pragma unroll
      for (int q = 0; q < 3; ++q) yx[q][0] = yx[q][1] = yx[q][2] = 0.0;
      for (int c = 0; c < a.C; ++c) {
        const double* cam = Cm + 12 * c;
        const double* pc = V + 3 * a.J + 6 * c;
        double yc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const int j = lane + 32 * q;
          if (j >= a.J) break;
          const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
          const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
          Obs o;
          observe<Loss>(cam, a.K + 9 * c, sX + 3 * j, (double)uv.x, (double)uv.y, w, a.rs, o);
          double dxc[3];
          matvec3(cam, V + 3 * j, dxc);  // R pX
          if (cams_free) {
            double wv[3], cx[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) wv[k] = pc[k];
            cross(wv, o.p, cx);
#pragma unroll
            for (int k = 0; k < 3; ++k) dxc[k] += cx[k] + pc[3 + k];
          }
          double nq[3];
          sym3vec(o.N, dxc, nq);
          double back[3];
          matTvec3(cam, nq, back);
          yx[q][0] += back[0], yx[q][1] += back[1], yx[q][2] += back[2];
          if (cams_free) {
            double pw[3];
            cross(o.p, nq, pw);
            yc[0] += pw[0], yc[1] += pw[1], yc[2] += pw[2], yc[3] += nq[0], yc[4] += nq[1], yc[5] += nq[2];
          }
        }
        if (cams_free) {
#pragma unroll
          for (int k = 0; k < 6; ++k) yc[k] = warp_sum(yc[k]);
          if (lane == c) {  // lane c keeps camera c's sums for the regularisers below
#pragma unroll
            for (int k = 0; k < 6; ++k) yr[3 * a.J + 6 * c + k] = yc[k];
          }
        }
      }
      // ---- points: bones, temporal, damping
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int j = lane + 32 * q;
        if (j >= a.J) break;
        for (int b = 0; b < a.nb; ++b) {
          const int bi = a.bi[b], bj = a.bj[b];
          if (bi != j && bj != j) continue;
          double u[3] = {sX[3 * bi] - sX[3 * bj], sX[3 * bi + 1] - sX[3 * bj + 1], sX[3 * bi + 2] - sX[3 * bj + 2]};
          const double iL = rsqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
          u[0] *= iL, u[1] *= iL, u[2] *= iL;
          const double s = cl * (u[0] * (V[3 * bi] - V[3 * bj]) + u[1] * (V[3 * bi + 1] - V[3 * bj + 1]) + u[2] * (V[3 * bi + 2] - V[3 * bj + 2]));
          const double sg = bi == j ? s : -s;
          yx[q][0] += sg * u[0], yx[q][1] += sg * u[1], yx[q][2] += sg * u[2];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double pv = V[3 * j + k];
          double tv = 0.0;
          if (prev) tv += pv - pr[3 * j + k - a.nf];
          if (next) tv += pv - pr[3 * j + k + a.nf];
          const double yv = yx[q][k] + ct * tv + lam * Dr[3 * j + k] * pv;
          yr[3 * j + k] = yv;
          dot += pv * yv;
        }
      }
      // ---- cameras: smoothness, baseline, damping, mask
      if (lane < a.C) {
        const int c = lane;
        double* yc = yr + 3 * a.J + 6 * c;
        if (!cams_free) {
#pragma unroll
          for (int k = 0; k < 6; ++k) yc[k] = 0.0;
        } else {
          const double* cam = Cm + 12 * c;
          const double* pc = V + 3 * a.J + 6 * c;
          double q0[3], v[3] = {0.0, 0.0, 0.0};
          centre_dir(cam, pc, a.free6, q0);
          if (prev) {
            double qp[3];
            centre_dir(cam - 12 * a.C, pr - a.nf + 3 * a.J + 6 * c, a.free6, qp);
#pragma unroll
            for (int k = 0; k < 3; ++k) v[k] += cs * (q0[k] - qp[k]);
          }
          if (next) {
            double qn[3];
            centre_dir(cam + 12 * a.C, pr + a.nf + 3 * a.J + 6 * c, a.free6, qn);
#pragma unroll
            for (int k = 0; k < 3; ++k) v[k] += cs * (q0[k] - qn[k]);
          }
          if (a.C >= 2 && c < 2 && cb != 0.0) {
            double c0[3], co[3], qo[3];
            centre(cam, c0);
            centre(Cm + 12 * (1 - c), co);
            centre_dir(Cm + 12 * (1 - c), V + 3 * a.J + 6 * (1 - c), a.free6, qo);
            const double sgn = c == 0 ? 1.0 : -1.0;
            double nh[3] = {sgn * (c0[0] - co[0]), sgn * (c0[1] - co[1]), sgn * (c0[2] - co[2])};
            const double ib = rsqrt(nh[0] * nh[0] + nh[1] * nh[1] + nh[2] * nh[2]);
            nh[0] *= ib, nh[1] *= ib, nh[2] *= ib;
            const double db = sgn * (nh[0] * (q0[0] - qo[0]) + nh[1] * (q0[1] - qo[1]) + nh[2] * (q0[2] - qo[2]));  // n . (q_0 - q_1)
            const double s = cb * db * sgn;
#pragma unroll
            for (int k = 0; k < 3; ++k) v[k] += s * nh[k];
          }
          double adj[6];
          centre_adj(cam, v, adj);
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            const bool fr = (a.free6 >> k) & 1u;
            const double pv = fr ? pc[k] : 0.0;
            const double yv = fr ? yc[k] + adj[k] + lam * Dr[3 * a.J + 6 * c + k] * pv : 0.0;
            yc[k] = yv;
            dot += pv * yv;
          }
        }
      }
    }
  }
  dot = warp_sum(dot);
  if (lane == 0) a.dpart[wid] = dot;
}

// ------------------------------------------------------------------------------------------------ CG update + preconditioner
// x += alpha p, r -= alpha y, z = M^-1 r (the frame's system through its Schur complement); partial dot r . z
template <int Loss>
__global__ void __launch_bounds__(32 * kWarpsPerBlock, 4) reg_precond_kernel(const RegArgs a, int first, const RobustScale rs) {
  extern __shared__ double smem_d[];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, wid = blockIdx.x * kWarpsPerBlock + wl;
  const double* sc = a.sc;
  double dot = 0.0;
  if (first || sc[SC_DONE] == 0.0) {
    const size_t per_warp = (size_t)a.nf + 3 * a.J + 3 * a.J + a.nS + a.n6;
    double* V = smem_d + wl * per_warp;  // r row, then z
    double* sX = V + a.nf;
    double* U = sX + 3 * a.J;            // Dp^-1 r_p
    double* L = U + 3 * a.J;
    double* B = L + a.nS;                // camera right-hand side / solution
    const int buf = (int)sc[SC_CUR];
    const double alpha = first ? 0.0 : sc[SC_ALPHA], cr = sc[SC_CR];
    const bool cams_free = a.free6 != 0;
    for (int64_t f = wid; f < a.Tl; f += a.W) {
      const int64_t row = f + 1;
      double* xr = a.x + row * a.nf;
      double* rr = a.r + row * a.nf;
      double* zr = a.z + row * a.nf;
      const double* pr = a.p + row * a.nf;
      const double* yr = a.y + row * a.nf;
      const double* X = frame_X(a, buf, row);
      const double* Cm = frame_C(a, buf, row);
      __syncwarp();
      for (int i = lane; i < a.nf; i += 32) {
        double rv = rr[i];
        if (!first) {
          xr[i] += alpha * pr[i];
          rv -= alpha * yr[i];
          rr[i] = rv;
        } else {
          xr[i] = 0.0;
        }
        V[i] = rv;
      }
      for (int i = lane; i < 3 * a.J; i += 32) sX[i] = X[i];
      if (cams_free)
        for (int i = lane; i < a.nS; i += 32) L[i] = a.lfac[f * a.nS + i];
      __syncwarp();
      for (int j = lane; j < a.J; j += 32) {
        const double* inv = a.pinv + (f * a.J + j) * 6;
        const double iv[6] = {inv[0], inv[1], inv[2], inv[3], inv[4], inv[5]};
        sym3vec(iv, V + 3 * j, U + 3 * j);
      }
      if (!cams_free) {
        for (int j = lane; j < a.J; j += 32)
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            zr[3 * j + k] = U[3 * j + k];
            dot += V[3 * j + k] * U[3 * j + k];
          }
        for (int i = lane; i < 6 * a.C; i += 32) zr[3 * a.J + i] = 0.0;
        continue;
      }
      // ---- b_c = r_c - sum_j W_jc^T u_j
      for (int c = 0; c < a.C; ++c) {
        const double* cam = Cm + 12 * c;
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int j = lane; j < a.J; j += 32) {
          const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
          const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
          Obs o;
          observe<Loss>(cam, a.K + 9 * c, sX + 3 * j, (double)uv.x, (double)uv.y, w, rs, o);
          double ru[3], nb[3], pw[3];
          matvec3(cam, U + 3 * j, ru);
          sym3vec(o.N, ru, nb);
          cross(o.p, nb, pw);
          acc[0] += pw[0], acc[1] += pw[1], acc[2] += pw[2], acc[3] += nb[0], acc[4] += nb[1], acc[5] += nb[2];
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
        if (lane == 0) {
#pragma unroll
          for (int k = 0; k < 6; ++k) B[6 * c + k] = ((a.free6 >> k) & 1u) ? V[3 * a.J + 6 * c + k] - acc[k] : 0.0;
        }
      }
      __syncwarp();
      // ---- L L^T z_c = b  (column sweeps: lanes over rows)
      for (int k = 0; k < a.n6; ++k) {
        const double zk = B[k] / L[tri(k, k)];
        __syncwarp();
        if (lane == 0) B[k] = zk;
        for (int r = k + 1 + lane; r < a.n6; r += 32) B[r] -= L[tri(r, k)] * zk;
        __syncwarp();
      }
      for (int k = a.n6 - 1; k >= 0; --k) {
        const double zk = B[k] / L[tri(k, k)];
        __syncwarp();
        if (lane == 0) B[k] = zk;
        for (int r = lane; r < k; r += 32) B[r] -= L[tri(k, r)] * zk;
        __syncwarp();
      }
      // ---- z_p = u - Dp^-1 sum_c W_jc z_c
      for (int j = lane; j < a.J; j += 32) {
        double acc[3] = {0.0, 0.0, 0.0};
        for (int c = 0; c < a.C; ++c) {
          const double* cam = Cm + 12 * c;
          const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
          const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
          Obs o;
          observe<Loss>(cam, a.K + 9 * c, sX + 3 * j, (double)uv.x, (double)uv.y, w, rs, o);
          const double* zc = B + 6 * c;
          double cx[3];
          cross(zc, o.p, cx);
          const double v[3] = {cx[0] + zc[3], cx[1] + zc[4], cx[2] + zc[5]};
          double nv[3], back[3];
          sym3vec(o.N, v, nv);
          matTvec3(cam, nv, back);
          acc[0] += back[0], acc[1] += back[1], acc[2] += back[2];
        }
        const double* inv = a.pinv + (f * a.J + j) * 6;
        const double iv[6] = {inv[0], inv[1], inv[2], inv[3], inv[4], inv[5]};
        double corr[3];
        sym3vec(iv, acc, corr);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double zv = U[3 * j + k] - corr[k];
          zr[3 * j + k] = zv;
          dot += V[3 * j + k] * zv;
        }
      }
      for (int i = lane; i < a.n6; i += 32) {
        zr[3 * a.J + i] = B[i];
        dot += V[3 * a.J + i] * B[i];
      }
    }
  }
  dot = warp_sum(dot);
  if (lane == 0) a.dpart[wid] = dot;
}

// p = z + beta p
__global__ void reg_dir_kernel(const RegArgs a) {
  const double* sc = a.sc;
  if (sc[SC_DONE] != 0.0 && sc[SC_CGIT] > 0.0) return;
  const double beta = sc[SC_BETA];
  const int64_t n = a.Tl * a.nf;
  double* p = a.p + a.nf;
  const double* z = a.z + a.nf;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = z[i] + beta * p[i];
}

// the scalar recurrences of CG, after the all-reduce of the dot in SC_DOT
__global__ void reg_scalar_kernel(const RegArgs a, int stage, const PeerDev peer) {
  if (peer.world > 1) peer_exchange_block(peer, a.sc + SC_DOT, 1, a.sc + SC_DOT, 0);  // the dot product's all-reduce, fused
  if (threadIdx.x != 0) return;
  double* sc = a.sc;
  const double v = sc[SC_DOT];
  if (stage == SKA_BA_REG_CG_INIT) {
    sc[SC_RZ0] = sc[SC_RZ] = v;
    sc[SC_BETA] = 0.0;
    sc[SC_ALPHA] = 0.0;
    sc[SC_CGIT] = 0.0;
    sc[SC_DONE] = (v > 0.0 && isfinite(v)) ? 0.0 : 1.0;
  } else if (stage == SKA_BA_REG_CG_ALPHA) {
    if (sc[SC_DONE] != 0.0) return;
    sc[SC_PAP] = v;
    if (v > 0.0 && isfinite(v)) {
      sc[SC_ALPHA] = sc[SC_RZ] / v;
    } else {
      sc[SC_ALPHA] = 0.0;
      sc[SC_DONE] = 1.0;
    }
  } else {
    if (sc[SC_DONE] != 0.0) return;
    sc[SC_BETA] = v / sc[SC_RZ];
    sc[SC_RZ] = v;
    sc[SC_CGIT] += 1.0;
    if (!(v > sc[SC_TOL2] * sc[SC_RZ0])) sc[SC_DONE] = 1.0;
  }
}

// ------------------------------------------------------------------------------------------------ trial point
// trial = current (+) x; partial of the predicted decrease  x . (lam D x - g)
__global__ void __launch_bounds__(32 * kWarpsPerBlock) reg_apply_kernel(const RegArgs a) {
  const int lane = threadIdx.x & 31, wid = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const double* sc = a.sc;
  const int buf = (int)sc[SC_CUR];
  const double lam = sc[SC_LAM];
  double pred = 0.0;
  for (int64_t f = wid; f < a.Tl; f += a.W) {
    const int64_t row = f + 1;
    const double* xr = a.x + row * a.nf;
    const double* gr = a.g + row * a.nf;
    const double* Dr = a.D + row * a.nf;
    const double* X = frame_X(a, buf, row);
    double* Xt = const_cast<double*>(frame_X(a, 1 - buf, row));
    for (int i = lane; i < a.nf; i += 32) pred += xr[i] * (lam * Dr[i] * xr[i] - gr[i]);
    for (int i = lane; i < 3 * a.J; i += 32) Xt[i] = X[i] + xr[i];
    if (lane < a.C) {
      const double* cam = frame_C(a, buf, row) + 12 * lane;
      double* camt = const_cast<double*>(frame_C(a, 1 - buf, row)) + 12 * lane;
      const double* dc = xr + 3 * a.J + 6 * lane;
      double w[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) w[k] = ((a.free6 >> k) & 1u) ? dc[k] : 0.0;
      if (a.free6 & 7u) {
        so3_exp_left(w, cam, camt);
      } else {
#pragma unroll
        for (int k = 0; k < 9; ++k) camt[k] = cam[k];
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) camt[9 + k] = cam[9 + k] + (((a.free6 >> (3 + k)) & 1u) ? dc[3 + k] : 0.0);
    }
  }
  pred = warp_sum(pred);
  if (lane == 0) a.ppart[wid] = pred;
}

// gain ratio, accept / reject, Nielsen's damping update, history row (oracle/lm_reg.py run_lm)
__global__ void reg_control_kernel(const RegArgs a, double* hist, int64_t hist_rows) {
  if (threadIdx.x != 0) return;
  double* sc = a.sc;
  const double F = sc[SC_F], Ft = sc[SC_FT], pred = sc[SC_PRED], lam = sc[SC_LAM], nu = sc[SC_NU];
  const double rho = pred > 0.0 ? (F - Ft) / pred : 0.0;
  const bool acc = isfinite(Ft) && Ft < F;
  const int64_t it = (int64_t)sc[SC_ITER];
  if (hist != nullptr && it < hist_rows) {
    double* h = hist + it * SKA_BA_REG_HIST_DOUBLES;
    h[0] = (double)it, h[1] = F, h[2] = Ft, h[3] = lam, h[4] = rho, h[5] = acc ? 1.0 : 0.0, h[6] = sc[SC_NCL], h[7] = pred, h[8] = sc[SC_CGIT];
    for (int k = 0; k < 5; ++k) h[9 + k] = sc[SC_TERM + k];
    h[14] = sc[SC_RZ0] > 0.0 ? sqrt(sc[SC_RZ] / sc[SC_RZ0]) : 0.0;
    h[15] = 0.0;
  }
  sc[SC_ITER] = (double)(it + 1);
  sc[SC_ACC] = acc ? 1.0 : 0.0;
  if (acc) {
    const double q = 2.0 * rho - 1.0;
    sc[SC_LAM] = lam * fmax(1.0 / 3.0, 1.0 - q * q * q);
    sc[SC_NU] = 2.0;
    sc[SC_CUR] = 1.0 - sc[SC_CUR];
    // the trial point's sums become the current point's: cost, terms and the detached means
    const double* s = a.sums + NS;
    double* s0 = a.sums;
    for (int k = 0; k < NS; ++k) s0[k] = s[k];
    const double Tg = sc[SC_TG];
    double bone = 0.0;
    for (int b = 0; b < a.nb; ++b) bone += s[SUM_L2 + b] - s[SUM_L + b] * s[SUM_L + b] / Tg;
    const double base = a.C >= 2 ? s[SUM_B2] - s[SUM_B] * s[SUM_B] / Tg : 0.0;
    sc[SC_TERM + 0] = sc[SC_CR] * s[SUM_REPROJ];
    sc[SC_TERM + 1] = sc[SC_CS] * s[SUM_SMOOTH];
    sc[SC_TERM + 2] = sc[SC_CB] * base;
    sc[SC_TERM + 3] = sc[SC_CL] * bone;
    sc[SC_TERM + 4] = sc[SC_CT] * s[SUM_TEMP];
    sc[SC_F] = Ft;
    sc[SC_NCL] = s[SUM_CLAMP];
    for (int b = 0; b < SKA_MAX_BONES; ++b) sc[SC_REF + b] = s[SUM_L + b] / Tg;
    sc[SC_BMEAN] = s[SUM_B] / Tg;
  } else {
    sc[SC_LAM] = lam * nu;
    sc[SC_NU] = 2.0 * nu;
  }
}


// ------------------------------------------------------------------------------------------------ points only ("pose_only")
// With the cameras fixed (the reference's configured default, configs/vggt.yaml:52) nothing is reduced over a frame: the
// normal matrix is the 3x3 point blocks plus the bone / temporal couplings, and its block-Jacobi preconditioner is exact up
// to those weak couplings (CG converges in 2 iterations).  ONE THREAD PER POINT then: every lane busy (a warp per frame
// leaves 15 of 32 lanes idle at J = 17), no shuffles, no shared memory; the frame's cameras are read through L1.
constexpr int kPtBlock = 256;
constexpr int kPtMaxGrid = 148 * 8;

__device__ __forceinline__ double block_sum_to(double v, double* sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kPtBlock / 32; ++w) t += sh[w];
  return t;
}

template <int Loss>
__global__ void __launch_bounds__(kPtBlock) reg_pt_linearize_kernel(const RegArgsRs a) {
  const double* sc = a.sc;
  const int buf = (int)sc[SC_CUR];
  const double lam = sc[SC_LAM], cr = sc[SC_CR], cl = sc[SC_CL], ct = sc[SC_CT];
  const int64_t N = a.Tl * a.J;
  for (int64_t i = blockIdx.x * (int64_t)kPtBlock + threadIdx.x; i < N; i += (int64_t)gridDim.x * kPtBlock) {
    const int64_t f = i / a.J;
    const int j = (int)(i - f * a.J);
    const int64_t row = f + 1;
    const double* Xf = frame_X(a, buf, row);
    const double* Cm = frame_C(a, buf, row);
    const bool prev = f > 0 || a.has_prev, next = f + 1 < a.Tl || a.has_next;
    const double Xj[3] = {Xf[3 * j], Xf[3 * j + 1], Xf[3 * j + 2]};
    double P[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int c = 0; c < a.C; ++c) {
      const double* cam = Cm + 12 * c;
      const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
      const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
      Obs o;
      observe<Loss>(cam, a.K + 9 * c, Xj, (double)uv.x, (double)uv.y, w, a.rs, o);
      double RtN[3][3];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const double col[3] = {cam[r], cam[3 + r], cam[6 + r]};
        sym3vec(o.N, col, RtN[r]);
      }
      int e = 0;
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = r; k < 3; ++k, ++e) P[e] += RtN[r][0] * cam[k] + RtN[r][1] * cam[3 + k] + RtN[r][2] * cam[6 + k];
      double gx[3];
      matTvec3(cam, o.q, gx);
      P[6] += gx[0], P[7] += gx[1], P[8] += gx[2];
    }
    for (int b = 0; b < a.nb; ++b) {
      const int bi = a.bi[b], bj = a.bj[b];
      if (bi != j && bj != j) continue;
      const int o = bi == j ? bj : bi;
      const double sgn = bi == j ? 1.0 : -1.0;
      double u[3] = {sgn * (Xj[0] - Xf[3 * o]), sgn * (Xj[1] - Xf[3 * o + 1]), sgn * (Xj[2] - Xf[3 * o + 2])};
      const double L = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
      const double iL = 1.0 / L;
      u[0] *= iL, u[1] *= iL, u[2] *= iL;
      const double res = cl * (L - sc[SC_REF + b]) * sgn;
      P[0] += cl * u[0] * u[0], P[1] += cl * u[0] * u[1], P[2] += cl * u[0] * u[2];
      P[3] += cl * u[1] * u[1], P[4] += cl * u[1] * u[2], P[5] += cl * u[2] * u[2];
      P[6] += res * u[0], P[7] += res * u[1], P[8] += res * u[2];
    }
    const double nn = ct * ((prev ? 1.0 : 0.0) + (next ? 1.0 : 0.0));
    P[0] += nn, P[3] += nn, P[5] += nn;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double gk = 0.0;
      if (prev) gk += Xj[k] - Xf[3 * j + k - a.J * 3];
      if (next) gk -= Xf[3 * j + k + a.J * 3] - Xj[k];
      P[6 + k] += ct * gk;
    }
    const double d[3] = {P[0], P[3], P[5]};
    const double Hd[6] = {P[0] + lam * d[0], P[1], P[2], P[3] + lam * d[1], P[4], P[5] + lam * d[2]};
    double inv[6];
    inv_sym3(Hd, inv);
    double* gr = a.g + row * a.nf;
    double* Dr = a.D + row * a.nf;
    double* rr = a.r + row * a.nf;
#pragma unroll
    for (int k = 0; k < 3; ++k) gr[3 * j + k] = P[6 + k], rr[3 * j + k] = -P[6 + k], Dr[3 * j + k] = d[k];
    double* pg = a.pinv + i * 6;
#pragma unroll
    for (int k = 0; k < 6; ++k) pg[k] = inv[k];
    if (j == 0)
      for (int k = 0; k < 6 * a.C; ++k) gr[3 * a.J + k] = 0.0, rr[3 * a.J + k] = 0.0, Dr[3 * a.J + k] = 0.0;
  }
}

template <int Loss>
__global__ void __launch_bounds__(kPtBlock) reg_pt_matvec_kernel(const RegArgsRs a) {
  __shared__ double sh[kPtBlock / 32];
  const double* sc = a.sc;
  double dot = 0.0;
  if (sc[SC_DONE] == 0.0) {
    const int buf = (int)sc[SC_CUR];
    const double lam = sc[SC_LAM], cr = sc[SC_CR], cl = sc[SC_CL], ct = sc[SC_CT];
    const int64_t N = a.Tl * a.J;
    for (int64_t i = blockIdx.x * (int64_t)kPtBlock + threadIdx.x; i < N; i += (int64_t)gridDim.x * kPtBlock) {
      const int64_t f = i / a.J;
      const int j = (int)(i - f * a.J);
      const int64_t row = f + 1;
      const double* Xf = frame_X(a, buf, row);
      const double* Cm = frame_C(a, buf, row);
      const double* pr = a.p + row * a.nf;
      const bool prev = f > 0 || a.has_prev, next = f + 1 < a.Tl || a.has_next;
      const double Xj[3] = {Xf[3 * j], Xf[3 * j + 1], Xf[3 * j + 2]};
      const double pj[3] = {pr[3 * j], pr[3 * j + 1], pr[3 * j + 2]};
      double y[3] = {0.0, 0.0, 0.0};
      for (int c = 0; c < a.C; ++c) {
        const double* cam = Cm + 12 * c;
        const float2 uv = *reinterpret_cast<const float2*>(a.x2d + ((f * a.C + c) * a.J + j) * 2);
        const double w = cr * (double)a.conf[(f * a.C + c) * a.J + j];
        Obs o;
        observe<Loss>(cam, a.K + 9 * c, Xj, (double)uv.x, (double)uv.y, w, a.rs, o);
        double dxc[3], nq[3], back[3];
        matvec3(cam, pj, dxc);
        sym3vec(o.N, dxc, nq);
        matTvec3(cam, nq, back);
        y[0] += back[0], y[1] += back[1], y[2] += back[2];
      }
      for (int b = 0; b < a.nb; ++b) {
        const int bi = a.bi[b], bj = a.bj[b];
        if (bi != j && bj != j) continue;
        double u[3] = {Xf[3 * bi] - Xf[3 * bj], Xf[3 * bi + 1] - Xf[3 * bj + 1], Xf[3 * bi + 2] - Xf[3 * bj + 2]};
        const double iL = rsqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        u[0] *= iL, u[1] *= iL, u[2] *= iL;
        const double s = cl * (u[0] * (pr[3 * bi] - pr[3 * bj]) + u[1] * (pr[3 * bi + 1] - pr[3 * bj + 1]) + u[2] * (pr[3 * bi + 2] - pr[3 * bj + 2]));
        const double sg = bi == j ? s : -s;
        y[0] += sg * u[0], y[1] += sg * u[1], y[2] += sg * u[2];
      }
      double* yr = a.y + row * a.nf;
      const double* Dr = a.D + row * a.nf;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        double tv = 0.0;
        if (prev) tv += pj[k] - pr[3 * j + k - a.nf];
        if (next) tv += pj[k] - pr[3 * j + k + a.nf];
        const double yv = y[k] + ct * tv + lam * Dr[3 * j + k] * pj[k];
        yr[3 * j + k] = yv;
        dot += pj[k] * yv;
      }
      if (j == 0)
        for (int k = 0; k < 6 * a.C; ++k) yr[3 * a.J + k] = 0.0;
    }
  }
  const double t = block_sum_to(dot, sh);
  if (threadIdx.x == 0) a.dpart[blockIdx.x] = t;
}

// x += alpha p, r -= alpha y, z = Dp^-1 r; partial dot r . z
__global__ void __launch_bounds__(kPtBlock) reg_pt_precond_kernel(const RegArgs a, int first) {
  __shared__ double sh[kPtBlock / 32];
  const double* sc = a.sc;
  double dot = 0.0;
  if (first || sc[SC_DONE] == 0.0) {
    const double alpha = first ? 0.0 : sc[SC_ALPHA];
    const int64_t N = a.Tl * a.J;
    for (int64_t i = blockIdx.x * (int64_t)kPtBlock + threadIdx.x; i < N; i += (int64_t)gridDim.x * kPtBlock) {
      const int64_t f = i / a.J;
      const int j = (int)(i - f * a.J);
      const int64_t o = (f + 1) * a.nf + 3 * j;
      double rv[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        rv[k] = a.r[o + k];
        if (!first) {
          a.x[o + k] += alpha * a.p[o + k];
          rv[k] -= alpha * a.y[o + k];
          a.r[o + k] = rv[k];
        } else {
          a.x[o + k] = 0.0;
        }
      }
      const double* inv = a.pinv + i * 6;
      const double iv[6] = {inv[0], inv[1], inv[2], inv[3], inv[4], inv[5]};
      double zv[3];
      sym3vec(iv, rv, zv);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        a.z[o + k] = zv[k];
        dot += rv[k] * zv[k];
      }
      if (j == 0)
        for (int k = 0; k < 6 * a.C; ++k) a.z[(f + 1) * a.nf + 3 * a.J + k] = 0.0, a.x[(f + 1) * a.nf + 3 * a.J + k] = 0.0;
    }
  }
  const double t = block_sum_to(dot, sh);
  if (threadIdx.x == 0) a.dpart[blockIdx.x] = t;
}

static int pt_grid(const RegArgs& a) {
  int64_t g = (a.Tl * a.J + kPtBlock - 1) / kPtBlock;
  if (g > kPtMaxGrid) g = kPtMaxGrid;
  if (g > a.W) g = a.W;  // dpart holds W rows
  return g < 1 ? 1 : (int)g;
}

// ------------------------------------------------------------------------------------------------ host side
static int grid_blocks(int64_t Tl) {
  int64_t b = (Tl + kWarpsPerBlock - 1) / kWarpsPerBlock;
  if (b > kMaxGridBlocks) b = kMaxGridBlocks;
  return b < 1 ? 1 : (int)b;
}

static int fill(const SkaBaRegProblem& p, RegArgs& a) {
  if (p.C < 1 || p.C > SKA_MAX_VIEWS) return set_error(SKA_EINVAL, "C must be in 1..8");
  if (p.J < 1 || p.J > 96) return set_error(SKA_EINVAL, "J must be in 1..96");
  if (p.n_bones < 0 || p.n_bones > SKA_MAX_BONES) return set_error(SKA_EINVAL, "n_bones must be in 0..SKA_MAX_BONES");
  if (p.T_local < 1) return set_error(SKA_EINVAL, "every rank needs at least one frame");
  for (int b = 0; b < p.n_bones; ++b)
    if (p.bone_i[b] < 0 || p.bone_i[b] >= p.J || p.bone_j[b] < 0 || p.bone_j[b] >= p.J) return set_error(SKA_EINVAL, "bone joint index out of range");
  if (!p.d_x2d || !p.d_conf || !p.d_K || !p.d_X || !p.d_cams || !p.d_vec || !p.d_pinv || !p.d_sc || !p.d_sums || !p.d_workspace ||
      (p.free_mask && !p.d_lfac))
    return set_error(SKA_EINVAL, "null device pointer");
  a.Tl = p.T_local;
  a.J = p.J, a.C = p.C, a.nb = p.n_bones, a.has_prev = p.has_prev, a.has_next = p.has_next;
  a.nf = 3 * p.J + 6 * p.C;
  a.n6 = 6 * p.C;
  a.nS = a.n6 * (a.n6 + 1) / 2;
  a.free6 = p.free_mask & 63u;
  for (int b = 0; b < SKA_MAX_BONES; ++b) a.bi[b] = b < p.n_bones ? p.bone_i[b] : 0, a.bj[b] = b < p.n_bones ? p.bone_j[b] : 0;
  a.x2d = p.d_x2d, a.conf = p.d_conf, a.K = p.d_K, a.Xh = p.d_X, a.Ch = p.d_cams;
  const int64_t stride = (p.T_local + 2) * a.nf;
  a.g = p.d_vec, a.D = p.d_vec + stride, a.x = p.d_vec + 2 * stride, a.r = p.d_vec + 3 * stride, a.z = p.d_vec + 4 * stride;
  a.p = p.d_vec + 5 * stride, a.y = p.d_vec + 6 * stride;
  a.pinv = p.d_pinv, a.lfac = p.d_lfac, a.sc = p.d_sc, a.sums = p.d_sums;
  a.W = grid_blocks(p.T_local) * kWarpsPerBlock;
  if (p.ws_bytes < (size_t)a.W * (NS + 2) * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_reg_workspace_bytes)");
  a.part = (double*)p.d_workspace;
  a.dpart = a.part + (size_t)a.W * NS;
  a.ppart = a.dpart + a.W;
  return SKA_OK;
}

static int check_launch() {
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

template <typename Kern>
static int set_smem(Kern kern, size_t bytes) {
  if (bytes > 227 * 1024) return set_error(SKA_EUNSUPPORTED, "frame too large for one warp's shared memory (J, C)");
  if (bytes > 48 * 1024) {
    const cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  }
  return SKA_OK;
}

// The instantiation of a loss-templated kernel for `loss` (SKA_BA_LOSS_*, validated by the C ABI).  The launch sites bind
// it to a local pointer of the kernel's own name, so that every loss runs through the same launch code.
template <typename Kern>
static Kern by_loss(int loss, Kern l2, Kern huber, Kern cauchy) {
  return loss == SKA_BA_LOSS_HUBER ? huber : loss == SKA_BA_LOSS_CAUCHY ? cauchy : l2;
}
#define SKA_REG_BY_LOSS(kern) by_loss(loss, ska::kern<kLossL2>, ska::kern<kLossHuber>, ska::kern<kLossCauchy>)

static RobustScale robust_scale(double d) { return RobustScale{d, d * d, d > 0.0 ? 1.0 / (d * d) : 0.0}; }

}  // namespace

size_t ba_reg_workspace_bytes(int64_t T_local) { return (size_t)grid_blocks(T_local) * kWarpsPerBlock * (NS + 2) * sizeof(double); }

int ba_reg_cost(const SkaBaRegProblem& p, int which, int loss, double loss_scale, cudaStream_t s) {
  RegArgs a;
  int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  const RobustScale rs = robust_scale(loss_scale);
  const auto reg_cost_kernel = SKA_REG_BY_LOSS(reg_cost_kernel);
  reg_cost_kernel<<<a.W / kWarpsPerBlock, 32 * kWarpsPerBlock, 0, s>>>(a, which, rs);
  if ((rc = check_launch()) != SKA_OK) return rc;
  if ((rc = launch_reduce(a.part, a.W, NS, a.sums + (which ? NS : 0), s)) != SKA_OK) return rc;
  if (which) rc = launch_reduce(a.ppart, a.W, 1, a.sums + NS + SUM_PRED, s);
  return rc;
}

int ba_reg_finish_cost(const SkaBaRegProblem& p, int which, cudaStream_t s) {
  RegArgs a;
  const int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  PeerDev pd;
  pd.world = 0;
  if (p.peer != nullptr) {
    const int rp = peer_fill(*p.peer, pd);
    if (rp != SKA_OK) return rp;
    if (p.peer->slot_doubles < NS) return set_error(SKA_EINVAL, "peer slot smaller than the sums row");
    pd.skip = nullptr;
  }
  reg_finish_cost_kernel<<<1, 32, 0, s>>>(a, which ? 1 : 0, pd);
  return check_launch();
}

int ba_reg_linearize(const SkaBaRegProblem& p, int loss, double loss_scale, cudaStream_t s) {
  RegArgsRs a;
  int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  a.rs = robust_scale(loss_scale);
  if (a.free6 == 0) {  // points only: one thread per point
    const auto reg_pt_linearize_kernel = SKA_REG_BY_LOSS(reg_pt_linearize_kernel);
    reg_pt_linearize_kernel<<<pt_grid(a), kPtBlock, 0, s>>>(a);
    return check_launch();
  }
  const size_t per_warp = ((size_t)a.J * 12 + (size_t)a.C * 28 + a.nf + a.nS + (size_t)96 * a.n6) * sizeof(double);
  int wpb = kWarpsPerBlock;
  while (wpb > 1 && per_warp * wpb > (size_t)227 * 1024) wpb /= 2;
  const size_t bytes = per_warp * wpb;
  const auto reg_linearize_kernel = SKA_REG_BY_LOSS(reg_linearize_kernel);
  if ((rc = set_smem(reg_linearize_kernel, bytes)) != SKA_OK) return rc;
  reg_linearize_kernel<<<a.W / wpb, 32 * wpb, bytes, s>>>(a);
  return check_launch();
}

int ba_reg_cg(const SkaBaRegProblem& p, int op, int loss, double loss_scale, cudaStream_t s) {
  RegArgsRs a;
  int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  a.rs = robust_scale(loss_scale);  // read by MATVEC, and by BEGIN / UPDATE with free cameras: the ops that read observations
  const auto reg_precond_kernel = SKA_REG_BY_LOSS(reg_precond_kernel);
  const auto reg_matvec_kernel = SKA_REG_BY_LOSS(reg_matvec_kernel);
  const auto reg_pt_matvec_kernel = SKA_REG_BY_LOSS(reg_pt_matvec_kernel);
  const int blocks = a.W / kWarpsPerBlock;
  switch (op) {
    case SKA_BA_REG_CG_BEGIN:
    case SKA_BA_REG_CG_UPDATE: {
      if (a.free6 == 0) {
        if (op == SKA_BA_REG_CG_BEGIN) {
          const size_t n = (size_t)(a.Tl + 2) * a.nf * sizeof(double);
          cudaError_t ce = cudaMemsetAsync(a.p, 0, n, s);
          if (ce == cudaSuccess) ce = cudaMemsetAsync(a.y, 0, n, s);
          if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
        }
        const int g = pt_grid(a);
        reg_pt_precond_kernel<<<g, kPtBlock, 0, s>>>(a, op == SKA_BA_REG_CG_BEGIN ? 1 : 0);
        if ((rc = check_launch()) != SKA_OK) return rc;
        return launch_reduce(a.dpart, g, 1, a.sc + SC_DOT, s);
      }
      const size_t bytes = ((size_t)a.nf + 6 * a.J + a.nS + a.n6) * sizeof(double) * kWarpsPerBlock;
      if ((rc = set_smem(reg_precond_kernel, bytes)) != SKA_OK) return rc;
      if (op == SKA_BA_REG_CG_BEGIN) {
        const size_t n = (size_t)(a.Tl + 2) * a.nf * sizeof(double);
        cudaError_t ce = cudaMemsetAsync(a.p, 0, n, s);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(a.y, 0, n, s);
        if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
      }
      reg_precond_kernel<<<blocks, 32 * kWarpsPerBlock, bytes, s>>>(a, op == SKA_BA_REG_CG_BEGIN ? 1 : 0, a.rs);
      if ((rc = check_launch()) != SKA_OK) return rc;
      return launch_reduce(a.dpart, a.W, 1, a.sc + SC_DOT, s);
    }
    case SKA_BA_REG_CG_MATVEC: {
      if (a.free6 == 0) {
        const int g = pt_grid(a);
        reg_pt_matvec_kernel<<<g, kPtBlock, 0, s>>>(a);
        if ((rc = check_launch()) != SKA_OK) return rc;
        return launch_reduce(a.dpart, g, 1, a.sc + SC_DOT, s);
      }
      const size_t bytes = ((size_t)a.nf + 3 * a.J) * sizeof(double) * kWarpsPerBlock;
      if ((rc = set_smem(reg_matvec_kernel, bytes)) != SKA_OK) return rc;
      reg_matvec_kernel<<<blocks, 32 * kWarpsPerBlock, bytes, s>>>(a);
      if ((rc = check_launch()) != SKA_OK) return rc;
      return launch_reduce(a.dpart, a.W, 1, a.sc + SC_DOT, s);
    }
    case SKA_BA_REG_CG_DIR: {
      const int64_t n = a.Tl * a.nf;
      int g = (int)((n + 255) / 256);
      if (g > 148 * 8) g = 148 * 8;
      reg_dir_kernel<<<g, 256, 0, s>>>(a);
      return check_launch();
    }
    case SKA_BA_REG_CG_INIT:
    case SKA_BA_REG_CG_ALPHA:
    case SKA_BA_REG_CG_BETA: {
      PeerDev pd;
      pd.world = 0;
      if (p.peer != nullptr) {
        if ((rc = peer_fill(*p.peer, pd)) != SKA_OK) return rc;
        // inside the CG loop the convergence flag is current and identical on every rank: converged = every rank skips
        pd.skip = op == SKA_BA_REG_CG_INIT ? nullptr : a.sc + SC_DONE;
      }
      reg_scalar_kernel<<<1, 32, 0, s>>>(a, op, pd);
      return check_launch();
    }
    default:
      return set_error(SKA_EINVAL, "unknown CG operation");
  }
}

int ba_reg_apply(const SkaBaRegProblem& p, cudaStream_t s) {
  RegArgs a;
  const int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  reg_apply_kernel<<<a.W / kWarpsPerBlock, 32 * kWarpsPerBlock, 0, s>>>(a);
  return check_launch();
}

int ba_reg_control(const SkaBaRegProblem& p, cudaStream_t s) {
  RegArgs a;
  const int rc = fill(p, a);
  if (rc != SKA_OK) return rc;
  reg_control_kernel<<<1, 32, 0, s>>>(a, p.d_hist, p.hist_rows);
  return check_launch();
}

#undef SKA_REG_BY_LOSS

}  // namespace ska
