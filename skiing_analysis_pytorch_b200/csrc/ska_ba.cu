// ska_ba.cu - Levenberg-Marquardt bundle adjustment, Schur-complement form, sm_100a.
//
// One LM trial = four launches, no host synchronisation, no atomics:
//   ba_linearize   one thread per point (frame, joint): residuals, analytic Jacobians (left SO(3)
//                  perturbation + pinhole, loss.py projection), damped 3x3 point block, its Cholesky,
//                  Y = L^-1 W, and the point's contribution to the reduced camera system
//                  (Sw += Y^T Y, bw += Y^T L^-1 gp, Hcc, gc, cost).  fp32 per point, fp64 reductions:
//                  warp shuffles -> fixed-order shared-memory sum -> one fp64 partial row per CTA ->
//                  fixed-order column sum (ba_reduce_columns).
//   [NCCL all-reduce of the packed fp64 reduced system when the clip is sharded over GPUs]
//   ba_solve       one CTA: S = Hcc + lam diag(Hcc) - Sw (fp64), gauge/free mask, Cholesky, delta_c,
//                  trial cameras R <- exp([d_omega]x) R, t <- t + d_t.
//   ba_backsub     one thread per point: recompute the point block from the observations (12 B/obs
//                  re-read instead of >= 100 B/point stored), delta_p = -Hd^-1 (gp + W delta_c),
//                  write the trial point and evaluate the trial cost with the trial cameras from the
//                  observations still in registers.
//   [all-reduce of (trial cost, predicted decrease, clamp count)]
//   ba_control     one thread: gain ratio, accept/reject, Nielsen damping update, history row, flips
//                  the point ping-pong index / commits the trial cameras on accept.
//
// Reference anchors: cost = bundle_adjustment/loss.py:17-94 (project_points + reprojection_loss);
// the optimiser slot = run_local_ba, vggt/multi_view_process.py:553-564 (undefined in the
// reference); algorithm spec = oracle/lm.py.
#include <cuda_runtime.h>
#include <math.h>

#include "ska_ba.cuh"
#include "ska_internal.h"
#include "ska_peer.cuh"

namespace ska {

// packed layout of the reduced system (fp64), the multi-GPU all-reduce payload
struct RedLayout {
  int NC, n, nS, oSw, oBw, oGc, oHcc, oCost, oClamp, size;
  __host__ __device__ explicit RedLayout(int C) {
    NC = C - 1;
    n = 6 * NC;
    nS = n * (n + 1) / 2;
    oSw = 0;
    oBw = nS;
    oGc = nS + n;
    oHcc = nS + 2 * n;
    oCost = oHcc + 21 * NC;
    oClamp = oCost + 1;
    size = oClamp + 1;
  }
  __host__ __device__ int sw(int a, int b) const { return a * n - (a * (a - 1)) / 2 + (b - a); }  // a <= b
};

template <int C>
struct RedConst {
  static constexpr int NC = C - 1, n = 6 * NC, nS = n * (n + 1) / 2;
  static constexpr int oBw = nS, oGc = nS + n, oHcc = nS + 2 * n, oCost = oHcc + 21 * NC, oClamp = oCost + 1, size = oClamp + 1;
};

struct BaKernelArgs {
  ObsLayout lay;
  int64_t N;
  const float* x2d;
  const float* conf;
  const double* cams;   // [2][C][kCamStride]: slot 0 current, slot 1 trial
  const double* ctrl;
  const double* delta;  // [C][6] (backsub)
  float* Xpp;           // [2][N][3] ping-pong
  double* partials;     // [grid][row]
  int32_t loss;         // SKA_BA_LOSS_* (the kernel's Loss template argument selects the code)
  float loss_scale;     // robust scale d in pixels (unused by L2)
};

template <int C>
__device__ __forceinline__ void load_cams_shared(const double* __restrict__ cams, CamF* s_cam) {
  if (threadIdx.x < C) load_cam(cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
  __syncthreads();
}

template <int C>
struct PointObs {
  float u[C], v[C], cw[C];
  float X[3];
};

template <int C>
__device__ __forceinline__ void load_point(const BaKernelArgs& a, const float* __restrict__ X, int64_t i, PointObs<C>& o) {
  int64_t koff, coff;
  obs_offsets(a.lay, i, koff, coff);
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float2 q = __ldg(reinterpret_cast<const float2*>(a.x2d + koff + c * a.lay.k_sV));
    o.u[c] = q.x;
    o.v[c] = q.y;
    o.cw[c] = __ldg(a.conf + coff + c * a.lay.c_sV);
  }
  o.X[0] = __ldg(X + 3 * i);
  o.X[1] = __ldg(X + 3 * i + 1);
  o.X[2] = __ldg(X + 3 * i + 2);
}

// ------------------------------------------------------------------------------------------------
// linearise, register path (C == 2: one free camera, 56 fp32 accumulators per thread)
template <int C, int Loss>
__global__ void __launch_bounds__(kBaBlock, 2) ba_linearize_reg(const BaKernelArgs a) {
  using L = RedConst<C>;
  static_assert(C == 2, "register path holds the whole reduced system per thread: C == 2 only");
  __shared__ CamF s_cam[C];
  __shared__ double scratch[(kBaBlock / 32) * L::size];
  load_cams_shared<C>(a.cams, s_cam);
  const float lam = (float)a.ctrl[kCtrlLambda];
  const int cur = (int)a.ctrl[kCtrlCur];
  const float* X = a.Xpp + (int64_t)cur * 3 * a.N;

  float acc[L::size];
#pragma unroll
  for (int k = 0; k < L::size; ++k) acc[k] = 0.f;

  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.N; i += stride) {
    PointObs<C> o;
    load_point<C>(a, X, i, o);
    PointBlock pb;
    pb_zero(pb);
    float W[3][6], cost = 0.f;
    int ncl = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsLin ol;
      project_lin(s_cam[c], o.X, o.u[c], o.v[c], ol);
      float au[3], av[3];
      point_rows(s_cam[c], ol, au, av);
      float cw = o.cw[c];
      if constexpr (Loss == kLossL2) {  // written out: the robust form below moves this kernel's register allocation
        pb_add(pb, cw, au, av, ol.eu, ol.ev);
        cost = fmaf(cw, fmaf(ol.eu, ol.eu, ol.ev * ol.ev), cost);
      } else {
        float rho, om;
        robust_loss<Loss>(fmaf(ol.eu, ol.eu, ol.ev * ol.ev), a.loss_scale, rho, om);
        cost = fmaf(cw, rho, cost);
        cw *= om;
        pb_add(pb, cw, au, av, ol.eu, ol.ev);
      }
      ncl += ol.clamped ? 1 : 0;
      if (c >= 1) {
        float bu[6], bv[6];
        camera_rows(ol, bu, bv);
        float* hcc = acc + L::oHcc + 21 * (c - 1);
        float* gc = acc + L::oGc + 6 * (c - 1);
        int q = 0;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          const float su = cw * bu[r], sv = cw * bv[r];
#pragma unroll
          for (int s = r; s < 6; ++s, ++q) hcc[q] = fmaf(su, bu[s], fmaf(sv, bv[s], hcc[q]));
          gc[r] = fmaf(su, ol.eu, fmaf(sv, ol.ev, gc[r]));
#pragma unroll
          for (int k = 0; k < 3; ++k) W[k][r] = fmaf(su, au[k], sv * av[k]);
        }
      }
    }
    acc[L::oCost] += cost;
    acc[L::oClamp] += (float)ncl;
    const Chol3 f = chol3_damped(pb, lam);
    {  // no branch on f.ok: a point without a factor has a zeroed one (chol3), so Y = 0 and it adds exact zeros
      float yg0, yg1, yg2;
      chol3_fwd(f, pb.g0, pb.g1, pb.g2, yg0, yg1, yg2);
      float Y[3][6];
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        chol3_fwd(f, W[0][r], W[1][r], W[2][r], Y[0][r], Y[1][r], Y[2][r]);
        acc[L::oBw + r] = fmaf(Y[0][r], yg0, fmaf(Y[1][r], yg1, fmaf(Y[2][r], yg2, acc[L::oBw + r])));
      }
      int q = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int s = r; s < 6; ++s, ++q)
          acc[q] = fmaf(Y[0][r], Y[0][s], fmaf(Y[1][r], Y[1][s], fmaf(Y[2][r], Y[2][s], acc[q])));
    }
  }
  block_reduce_store<L::size>(acc, scratch, a.partials + (int64_t)blockIdx.x * L::size);
}

// ------------------------------------------------------------------------------------------------
// back-substitution + trial point + trial cost
constexpr int kBackAcc = 3;  // trial cost, predicted decrease (points), clamped count

template <int C, int Loss>
__global__ void __launch_bounds__(kBaBlock, 2) ba_backsub_kernel(const BaKernelArgs a) {
  __shared__ CamF s_cam[C], s_trial[C];
  __shared__ float s_delta[C][6];
  __shared__ double scratch[(kBaBlock / 32) * kBackAcc];
  if (threadIdx.x < C) {
    load_cam(a.cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
    load_cam(a.cams + (C + threadIdx.x) * kCamStride, s_trial[threadIdx.x]);
  }
  if (threadIdx.x < 6 * C) s_delta[threadIdx.x / 6][threadIdx.x % 6] = (float)a.delta[threadIdx.x];
  __syncthreads();
  const float lam = (float)a.ctrl[kCtrlLambda];
  const int cur = (int)a.ctrl[kCtrlCur];
  const float* X = a.Xpp + (int64_t)cur * 3 * a.N;
  float* Xn = a.Xpp + (int64_t)(1 - cur) * 3 * a.N;

  float acc[kBackAcc] = {0.f, 0.f, 0.f};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.N; i += stride) {
    PointObs<C> o;
    load_point<C>(a, X, i, o);
    PointBlock pb;
    pb_zero(pb);
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;  // gp + W delta_c
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsLin ol;
      project_lin(s_cam[c], o.X, o.u[c], o.v[c], ol);
      float au[3], av[3];
      point_rows(s_cam[c], ol, au, av);
      float rho, om;  // the linearisation's weight: the same fp32 expression at the same state
      robust_loss<Loss>(fmaf(ol.eu, ol.eu, ol.ev * ol.ev), a.loss_scale, rho, om);
      const float cw = o.cw[c] * om;
      pb_add(pb, cw, au, av, ol.eu, ol.ev);
      float lu = ol.eu, lv = ol.ev;
      if (c >= 1) {
        float bu[6], bv[6];
        camera_rows(ol, bu, bv);
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          lu = fmaf(bu[r], s_delta[c][r], lu);
          lv = fmaf(bv[r], s_delta[c][r], lv);
        }
      }
      r0 = fmaf(cw * au[0], lu, fmaf(cw * av[0], lv, r0));
      r1 = fmaf(cw * au[1], lu, fmaf(cw * av[1], lv, r1));
      r2 = fmaf(cw * au[2], lu, fmaf(cw * av[2], lv, r2));
    }
    const Chol3 f = chol3_damped(pb, lam);
    float d0, d1, d2;
    {  // branch-free: zeroed factor -> zero step for a point without a factor
      float y0, y1, y2;
      chol3_fwd(f, -r0, -r1, -r2, y0, y1, y2);
      chol3_bwd(f, y0, y1, y2, d0, d1, d2);
      d0 = f.ok ? d0 : 0.f;  // selects, not a branch (a non-finite residual times the zeroed factor would be NaN)
      d1 = f.ok ? d1 : 0.f;
      d2 = f.ok ? d2 : 0.f;
      // predicted decrease of the quadratic model, point part: dp . (lam diag(Hpp) dp - gp)
      acc[1] += d0 * fmaf(lam * pb.h00, d0, -pb.g0) + d1 * fmaf(lam * pb.h11, d1, -pb.g1) + d2 * fmaf(lam * pb.h22, d2, -pb.g2);
    }
    float Xt[3] = {o.X[0] + d0, o.X[1] + d1, o.X[2] + d2};
    Xn[3 * i] = Xt[0];
    Xn[3 * i + 1] = Xt[1];
    Xn[3 * i + 2] = Xt[2];
    float tc = 0.f;
    int ncl = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      bool cl;
      float rho, om;
      robust_loss<Loss>(project_err2(s_trial[c], Xt, o.u[c], o.v[c], cl), a.loss_scale, rho, om);
      tc = fmaf(o.cw[c], rho, tc);
      ncl += cl ? 1 : 0;
    }
    acc[0] += tc;
    acc[2] += (float)ncl;
  }
  block_reduce_store<kBackAcc>(acc, scratch, a.partials + (int64_t)blockIdx.x * kBackAcc);
}

// ------------------------------------------------------------------------------------------------
// fixed-order column sums of the per-CTA partial rows: out[col] = sum_r partials[r][col].
// One warp per column: lane l sums rows l, l+32, ... (independent loads, a handful per lane - a serial
// walk over ~300 rows is a 20-microsecond chain of dependent L2 round trips), then a fixed shuffle tree.
constexpr int kRedCols = 8;  // columns (= warps) per CTA
__global__ void __launch_bounds__(32 * kRedCols) ba_reduce_columns(const double* __restrict__ partials, int rows, int ncol,
                                                                   double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * kRedCols + (threadIdx.x >> 5);
  if (col >= ncol) return;
  double s0 = 0.0, s1 = 0.0;
  int r = lane;
  for (; r + 32 < rows; r += 64) {
    s0 += partials[(int64_t)r * ncol + col];
    s1 += partials[(int64_t)(r + 32) * ncol + col];
  }
  if (r < rows) s0 += partials[(int64_t)r * ncol + col];
  double s = s0 + s1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) out[col] = s;
}

// plain sum of a float array (sum of confidences), same deterministic scheme
__global__ void __launch_bounds__(kBaBlock) ba_sum_kernel(const float* __restrict__ x, int64_t n, double* __restrict__ partials) {
  __shared__ double scratch[kBaBlock / 32];
  float acc[1] = {0.f};
  double d = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int k = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    acc[0] += __ldg(x + i);
    if (++k == 64) {  // bound the fp32 run length
      d += (double)acc[0];
      acc[0] = 0.f;
      k = 0;
    }
  }
  d += (double)acc[0];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_down_sync(0xffffffffu, d, o);
  if (lane == 0) scratch[warp] = d;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kBaBlock / 32; ++w) s += scratch[w];
    partials[blockIdx.x] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// reduced camera system: one CTA, fp64
constexpr int kMaxN = 6 * (SKA_MAX_VIEWS - 1);

// `peer.world > 1`: the all-reduce of the packed reduced system over NVLink peer memory is this kernel's prologue (push /
// release flag / poll / rank-ordered sum, ska_peer.cuh) - exchange and solve are one launch.
__global__ void __launch_bounds__(256) ba_solve_kernel(int C, uint64_t free_mask, double* red, double* cams, double* ctrl, double* delta,
                                                      const PeerDev peer) {
  __shared__ double S[kMaxN][kMaxN + 1];
  __shared__ double b[kMaxN], hd[kMaxN], gc[kMaxN], d[kMaxN];
  __shared__ int s_ok;
  const RedLayout L(C);
  const int n = L.n, tid = threadIdx.x, nt = blockDim.x;
  if (peer.world > 1) peer_exchange_block(peer, red, L.size, red, 0);
  const double lam = ctrl[kCtrlLambda];
  const double s = 1.0 / (ctrl[kCtrlSumConf] + 1e-6);
  if (tid == 0) s_ok = 1;
  // parameter k = 6*(c-1) + r of camera c >= 1 is free iff bit (6*c + r) of free_mask is set
  for (int idx = tid; idx < n * n; idx += nt) {
    const int i = idx / n, j = idx % n;
    const int a = i < j ? i : j, bb = i < j ? j : i;
    double v = -red[L.oSw + L.sw(a, bb)];
    if (a / 6 == bb / 6) {
      const int c = a / 6, r = a % 6, q = bb % 6;
      const double h = red[L.oHcc + 21 * c + (r * 6 - (r * (r - 1)) / 2 + (q - r))];
      v += (a == bb) ? h * (1.0 + lam) : h;
    }
    const bool fi = (free_mask >> (6 + i)) & 1ull, fj = (free_mask >> (6 + j)) & 1ull;
    S[i][j] = (fi && fj) ? v * s : (i == j ? 1.0 : 0.0);
  }
  for (int i = tid; i < n; i += nt) {
    const bool fi = (free_mask >> (6 + i)) & 1ull;
    const int c = i / 6, r = i % 6;
    hd[i] = s * red[L.oHcc + 21 * c + (r * 6 - (r * (r - 1)) / 2)];
    gc[i] = s * red[L.oGc + i];
    b[i] = fi ? s * (red[L.oBw + i] - red[L.oGc + i]) : 0.0;
  }
  __syncthreads();
  // right-looking Cholesky, lower triangle
  for (int k = 0; k < n; ++k) {
    if (tid == 0) {
      const double p = S[k][k];
      if (!(p > 0.0) || !isfinite(p)) {
        s_ok = 0;
        S[k][k] = 1.0;
      } else {
        S[k][k] = sqrt(p);
      }
    }
    __syncthreads();
    const double inv = 1.0 / S[k][k];
    for (int i = k + 1 + tid; i < n; i += nt) S[i][k] *= inv;
    __syncthreads();
    const int m = n - k - 1;
    for (int idx = tid; idx < m * m; idx += nt) {
      const int i = k + 1 + idx / m, j = k + 1 + idx % m;
      if (j <= i) S[i][j] -= S[i][k] * S[j][k];
    }
    __syncthreads();
  }
  // forward / backward substitution, column oriented: thread 0 finishes one unknown, every thread
  // eliminates it from its rows (a single-thread triangular solve is ~n^2 dependent shared-memory
  // round trips: 27 us at n = 42)
  for (int i = tid; i < n; i += nt) d[i] = b[i];
  __syncthreads();
  for (int k = 0; k < n; ++k) {
    if (tid == 0) d[k] = d[k] / S[k][k];
    __syncthreads();
    const double dk = d[k];
    for (int i = k + 1 + tid; i < n; i += nt) d[i] -= S[i][k] * dk;
    __syncthreads();
  }
  for (int k = n - 1; k >= 0; --k) {
    if (tid == 0) d[k] = d[k] / S[k][k];
    __syncthreads();
    const double dk = d[k];
    for (int i = tid; i < k; i += nt) d[i] -= S[k][i] * dk;
    __syncthreads();
  }
  if (tid == 0) {
    double pred = 0.0;
    bool fin = true;
    for (int i = 0; i < n; ++i) fin = fin && isfinite(d[i]);
    for (int i = 0; i < n; ++i) {
      const bool fi = (free_mask >> (6 + i)) & 1ull;
      if (!s_ok || !isfinite(d[i])) d[i] = 0.0;
      if (fi) pred += d[i] * (lam * hd[i] * d[i] - gc[i]);
    }
    ctrl[kCtrlOk] = (s_ok && fin) ? 1.0 : 0.0;
    ctrl[kCtrlPredCam] = pred;
  }
  __syncthreads();
  // delta (C,6) with the gauge camera's zeros, and the trial cameras in slot 1
  for (int i = tid; i < 6 * C; i += nt) delta[i] = (i < 6) ? 0.0 : d[i - 6];
  // trial cameras: K (and camera 0 entirely) copied by all threads, then R / t of the free cameras
  for (int k = tid; k < C * kCamStride; k += nt)
    if (k < kCamStride || (k % kCamStride) >= 12) cams[C * kCamStride + k] = cams[k];
  for (int c = 1 + tid; c < C; c += nt) {
    const double* src = cams + c * kCamStride;
    double* dst = cams + (C + c) * kCamStride;
    const double* dc = d + 6 * (c - 1);
    so3_exp_left(dc, src, dst);
    for (int k = 0; k < 3; ++k) dst[9 + k] = src[9 + k] + dc[3 + k];
  }
}

// LM controller: gain ratio, accept / reject, Nielsen update (oracle/lm.py run_lm / nielsen_update).
// One warp: lane 0 decides, all lanes commit the trial cameras (a serial copy by one thread is a
// chain of dependent global round trips - microseconds in a 100-microsecond trial).
__global__ void __launch_bounds__(32) ba_control_kernel(int C, const double* red, double* red2, double* cams, double* ctrl, double* hist,
                                                        int64_t hist_rows, const PeerDev peer) {
  if (blockIdx.x != 0) return;
  if (peer.world > 1) peer_exchange_block(peer, red2, SKA_BA_RED2_DOUBLES, red2, 0);  // the trial scalars' all-reduce, fused
  const RedLayout L(C);
  int accepted_i = 0;
  if (threadIdx.x == 0) {
    const double s = 1.0 / (ctrl[kCtrlSumConf] + 1e-6);
    const double F = s * red[L.oCost], Ft = s * red2[0];
    const double pred = ctrl[kCtrlPredCam] + s * red2[1];
    const double lam = ctrl[kCtrlLambda], nu = ctrl[kCtrlNu];
    const bool ok = ctrl[kCtrlOk] > 0.5;
    const double rho = pred > 0.0 ? (F - Ft) / pred : 0.0;
    const bool accepted = ok && isfinite(Ft) && (Ft < F);
    const int it = (int)ctrl[kCtrlIter];
    if (hist != nullptr && it < hist_rows) {
      double* h = hist + (int64_t)it * kHistRow;
      h[0] = (double)it;
      h[1] = F;
      h[2] = Ft;
      h[3] = lam;
      h[4] = rho;
      h[5] = accepted ? 1.0 : 0.0;
      h[6] = red[L.oClamp];
      h[7] = pred;
    }
    if (accepted) {
      const double q = 2.0 * rho - 1.0;
      const double f = 1.0 - q * q * q;
      ctrl[kCtrlLambda] = lam * (f > 1.0 / 3.0 ? f : 1.0 / 3.0);
      ctrl[kCtrlNu] = 2.0;
      ctrl[kCtrlCur] = 1.0 - ctrl[kCtrlCur];
      ctrl[kCtrlCost] = Ft;
    } else {
      ctrl[kCtrlLambda] = lam * nu;
      ctrl[kCtrlNu] = 2.0 * nu;
      ctrl[kCtrlCost] = F;
    }
    ctrl[kCtrlAccepted] = accepted ? 1.0 : 0.0;
    ctrl[kCtrlIter] = (double)(it + 1);
    accepted_i = accepted ? 1 : 0;
  }
  accepted_i = __shfl_sync(0xffffffffu, accepted_i, 0);
  if (accepted_i)
    for (int k = threadIdx.x; k < C * kCamStride; k += 32) cams[k] = cams[C * kCamStride + k];
}

// ------------------------------------------------------------------------------------------------
// host side
static int grid_for(const void* kern, int64_t N, int& grid) {
  int dev = 0, sms = 0, per_sm = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce == cudaSuccess) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBaBlock, 0);
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  if (per_sm < 1) per_sm = 1;
  int64_t g = (int64_t)sms * per_sm;
  const int64_t need = (N + kBaBlock - 1) / kBaBlock;
  if (g > need) g = need;
  if (g < 1) g = 1;
  grid = (int)g;
  return SKA_OK;
}

int ba_max_grid() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  return sms * 8;  // kBaBlock = 256 threads: at most 8 resident CTAs per SM
}

int ba_red_size(int C) { return RedLayout(C).size; }

static int fill_layout(const SkaBaProblem& in, BaKernelArgs& a) {
  a.N = in.T * (int64_t)in.J;
  a.lay.J = in.J;
  if (in.layout == SKA_LAYOUT_FRAME_MAJOR) {
    a.lay.k_sV = 2 * (int64_t)in.J;
    a.lay.k_sT = 2 * (int64_t)in.J * in.C;
    a.lay.c_sV = in.J;
    a.lay.c_sT = (int64_t)in.J * in.C;
  } else {
    a.lay.k_sV = 2 * a.N;
    a.lay.k_sT = 2 * (int64_t)in.J;
    a.lay.c_sV = a.N;
    a.lay.c_sT = in.J;
  }
  a.x2d = in.d_x2d;
  a.conf = in.d_conf;
  a.cams = in.d_cams;
  a.ctrl = in.d_ctrl;
  a.delta = in.d_delta;
  a.Xpp = in.d_Xpp;
  a.partials = (double*)in.d_workspace;
  a.loss = in.loss;
  a.loss_scale = (float)in.loss_scale;
  return SKA_OK;
}

int launch_reduce(const double* partials, int rows, int ncol, double* out, cudaStream_t s) {
  ba_reduce_columns<<<(ncol + kRedCols - 1) / kRedCols, 32 * kRedCols, 0, s>>>(partials, rows, ncol, out);
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

template <int Loss>
static int linearize_reg(const SkaBaProblem& in, const BaKernelArgs& a, cudaStream_t s) {
  int grid = 1;
  const int rc = grid_for((const void*)ba_linearize_reg<2, Loss>, a.N, grid);
  if (rc != SKA_OK) return rc;
  const size_t need = (size_t)grid * RedConst<2>::size * sizeof(double);
  if (in.ws_bytes < need) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_workspace_bytes)");
  ba_linearize_reg<2, Loss><<<grid, kBaBlock, 0, s>>>(a);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, grid, RedConst<2>::size, in.d_red, s);
}

int ba_linearize(const SkaBaProblem& in, cudaStream_t s) {
  if (in.C != 2 || (in.flags & SKA_BA_FORCE_WIDE)) return ba_linearize_wide(in, s);
  BaKernelArgs a;
  fill_layout(in, a);
  switch (in.loss) {
    case SKA_BA_LOSS_HUBER: return linearize_reg<kLossHuber>(in, a, s);
    case SKA_BA_LOSS_CAUCHY: return linearize_reg<kLossCauchy>(in, a, s);
    default: return linearize_reg<kLossL2>(in, a, s);
  }
}

template <int C, int Loss>
static int backsub_cl(const SkaBaProblem& in, const BaKernelArgs& a, cudaStream_t s) {
  int grid = 1;
  const int rc = grid_for((const void*)ba_backsub_kernel<C, Loss>, a.N, grid);
  if (rc != SKA_OK) return rc;
  if (in.ws_bytes < (size_t)grid * kBackAcc * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_workspace_bytes)");
  ba_backsub_kernel<C, Loss><<<grid, kBaBlock, 0, s>>>(a);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, grid, kBackAcc, in.d_red2, s);
}

template <int C>
static int backsub_c(const SkaBaProblem& in, const BaKernelArgs& a, cudaStream_t s) {
  switch (in.loss) {
    case SKA_BA_LOSS_HUBER: return backsub_cl<C, kLossHuber>(in, a, s);
    case SKA_BA_LOSS_CAUCHY: return backsub_cl<C, kLossCauchy>(in, a, s);
    default: return backsub_cl<C, kLossL2>(in, a, s);
  }
}

int ba_backsub(const SkaBaProblem& in, cudaStream_t s) {
  BaKernelArgs a;
  fill_layout(in, a);
  switch (in.C) {
    case 2: return backsub_c<2>(in, a, s);
    case 3: return backsub_c<3>(in, a, s);
    case 4: return backsub_c<4>(in, a, s);
    case 5: return backsub_c<5>(in, a, s);
    case 6: return backsub_c<6>(in, a, s);
    case 7: return backsub_c<7>(in, a, s);
    case 8: return backsub_c<8>(in, a, s);
    default: return set_error(SKA_EINVAL, "C must be in 2..8");
  }
}

static int peer_of(const SkaPeerComm* c, int payload, PeerDev& pd) {
  pd.world = 0;
  if (c == nullptr) return SKA_OK;
  const int rc = peer_fill(*c, pd);
  if (rc != SKA_OK) return rc;
  if (payload > c->slot_doubles) return set_error(SKA_EINVAL, "reduced system larger than the peer slot");
  return SKA_OK;
}

int ba_solve(int C, uint64_t free_mask, double* red, double* cams, double* ctrl, double* delta, const SkaPeerComm* peer, void* stream) {
  PeerDev pd;
  const int rc = peer_of(peer, ba_red_size(C), pd);
  if (rc != SKA_OK) return rc;
  ba_solve_kernel<<<1, C <= 3 ? 64 : 256, 0, (cudaStream_t)stream>>>(C, free_mask, red, cams, ctrl, delta, pd);
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

int ba_control(int C, const double* red, double* red2, double* cams, double* ctrl, double* hist, int64_t hist_rows, const SkaPeerComm* peer,
               void* stream) {
  PeerDev pd;
  const int rc = peer_of(peer, SKA_BA_RED2_DOUBLES, pd);
  if (rc != SKA_OK) return rc;
  ba_control_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(C, red, red2, cams, ctrl, hist, hist_rows, pd);
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

int ba_sum(const float* x, int64_t n, double* out, void* workspace, size_t ws_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  int grid = ba_max_grid() / 4;
  const int64_t need = (n + kBaBlock - 1) / kBaBlock;
  if (grid > need) grid = (int)(need < 1 ? 1 : need);
  if (ws_bytes < (size_t)grid * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_workspace_bytes)");
  ba_sum_kernel<<<grid, kBaBlock, 0, s>>>(x, n, (double*)workspace);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce((const double*)workspace, grid, 1, out, s);
}

}  // namespace ska
