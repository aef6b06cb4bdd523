// ska_ba_calib.cu - CALIBRATING bundle adjustment: Levenberg-Marquardt over the points, the camera extrinsics
// AND every camera's intrinsics + distortion (15 parameters per camera), Schur-complement form, sm_100a.
//
// BASELINE config 3 names "2 cameras, Rodrigues extrinsics + intrinsics/distortion"; SURVEY.md section 8d calls this
// the p = 15 block.  The projection is cv2.projectPoints' 5-coefficient model the reference reprojects with
// (triangulation/reproject.py:77-78); the optimiser slot is the reference's undefined run_local_ba
// (vggt/multi_view_process.py:553-564); the algorithm specification is oracle/lm_calib.py.
//
// Same trial structure as ska_ba.cu: linearise -> [all-reduce red] -> solve -> back-substitute + trial cost ->
// [all-reduce red2] -> control; no host synchronisation, no atomics, fixed summation orders.
//
// Reduced system: n = 15 C - 6 free-able parameters (camera 0 keeps only its 9 intrinsics: its extrinsics are the
// gauge).  Packed fp64 payload `red`:
//   [0, n(n+1)/2)        upper triangle of Sw = sum_points Y^T Y,  Y = L^-1 W   (L L^T = damped 3x3 point block)
//   then per camera c    160 doubles: the upper triangle (153) of  sum_obs w row^T row  with the 17-entry row
//                        [B (15) | e | a.dp0]: entries (r,s<=14) = Hcc, (r,15) = gc, (r,16) = bw, (15,15) = cost;
//                        slot 153 = number of depth-clamped observations; slot 154 = the robust cost correction
//                        sum w (rho(s) - omega s), so that (15,15) + slot 154 = sum w rho(s) (0 under L2)
// all sums with the raw confidences; the fp64 solve / control kernels scale by 1/(sum conf + 1e-6) once.
//
// ba_calib_linearize_kernel<C>: a warp owns 32 points per tile.
//   phase 1  thread = point: pass A builds the damped point block, its Cholesky and dp0 = -Hd^-1 gp; pass B
//            re-linearises each camera, writes Y_c (3 x 15) into the warp's staging buffer and reduces the camera's
//            153 row products over the 32 points with five TRANSPOSING butterflies (lane i ends with the warp total of
//            product 32 b + i; the product list is resolved at compile time).
//   phase 2  lane = one 6x6 block of Sw and a third of the 96 staged rows: 36 fp32 accumulators, 128-bit shared loads.
//   every kFlush tiles the fp32 accumulators are folded into the CTA's fp64 copy in a fixed warp order.
#include <cuda_runtime.h>
#include <math.h>

#include <utility>

#include "ska_ba.cuh"
#include "ska_ba_calib.cuh"
#include "ska_internal.h"
#include "ska_peer.cuh"

namespace ska {

#ifndef SKA_BA_CALIB_WARPS
#define SKA_BA_CALIB_WARPS 12
#endif

struct CalibLayout {
  int C, n, nS, oCam, size;
  __host__ __device__ explicit CalibLayout(int C_) : C(C_), n(kCalibP * C_ - 6), nS(n * (n + 1) / 2), oCam(nS), size(nS + kCalibCamBlock * C_) {}
  __host__ __device__ int sw(int a, int b) const { return a * n - (a * (a - 1)) / 2 + (b - a); }  // a <= b
  __host__ __device__ void param(int i, int& c, int& r) const {
    if (i < kCalibNI) {
      c = 0;
      r = i + 6;
    } else {
      c = 1 + (i - kCalibNI) / kCalibP;
      r = (i - kCalibNI) % kCalibP;
    }
  }
};

template <int C>
struct Calib {
  static constexpr int n = kCalibP * C - 6, nS = n * (n + 1) / 2, oCam = nS, size = nS + kCalibCamBlock * C;
  static constexpr int NB = n / 6;                   // 6-column blocks of Sw
  static constexpr int NPAIR = NB * (NB + 1) / 2;    // block pairs a <= b
  static constexpr int SL = largest_div(24, 32 / NPAIR);
  static constexpr int CH = 24 / SL;                 // chunks of 4 staged rows per lane
  static constexpr int W = SKA_BA_CALIB_WARPS;
  static constexpr int warp_floats = n * kYStride;
  static constexpr size_t smem = (size_t)W * warp_floats * sizeof(float) + (size_t)size * sizeof(double) + C * sizeof(CamC);
  static_assert(n % 6 == 0 && NPAIR <= 32, "Sw block decomposition: one lane per 6x6 block pair");
  __host__ __device__ static constexpr int col(int c, int r) { return c == 0 ? r - 6 : kCalibNI + kCalibP * (c - 1) + r; }
};

struct CalibArgs {
  ObsLayout lay;
  int64_t N;
  int64_t n_tiles;
  const float* x2d;
  const float* conf;
  const double* cams;   // [2][C][24]: R(9) t(3) theta(9) pad(3); slot 0 current, slot 1 trial
  const double* ctrl;
  const double* delta;  // [C][15]
  float* Xpp;
  double* partials;
  int32_t loss;       // SKA_BA_LOSS_* (the kernel's Loss template argument selects the code)
  float loss_scale;   // robust scale d in pixels (unused by L2)
};

__device__ __forceinline__ void load_cam_calib(const double* __restrict__ s, CamC& c) {
#pragma unroll
  for (int i = 0; i < 9; ++i) c.R[i] = (float)s[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) c.t[i] = (float)s[9 + i];
  c.fx = (float)s[12]; c.fy = (float)s[13]; c.cx = (float)s[14]; c.cy = (float)s[15];
  c.k1 = (float)s[16]; c.k2 = (float)s[17]; c.p1 = (float)s[18]; c.p2 = (float)s[19]; c.k3 = (float)s[20];
}

// product Q of the per-camera block, resolved at compile time
template <int Q>
__device__ __forceinline__ float calib_prod(const float (&su)[kCalibRow], const float (&sv)[kCalibRow], const ObsCalib& o, float clampv,
                                            float robustv) {
  if constexpr (Q < kCalibTri) {
    constexpr int r = calib_tri_row(Q), s = calib_tri_col(Q);
    return fmaf(su[r], o.bu[s], sv[r] * o.bv[s]);
  } else if constexpr (Q == kCalibClampSlot) {
    return clampv;
  } else if constexpr (Q == kCalibRobustSlot) {
    return robustv;
  } else {
    return 0.0f;
  }
}
template <int B, int... I>
__device__ __forceinline__ void calib_fill(float (&v)[32], const float (&su)[kCalibRow], const float (&sv)[kCalibRow], const ObsCalib& o,
                                           float clampv, float robustv, std::integer_sequence<int, I...>) {
  ((v[I] = calib_prod<32 * B + I>(su, sv, o, clampv, robustv)), ...);
}
template <int B>
__device__ __forceinline__ float calib_batch(const float (&su)[kCalibRow], const float (&sv)[kCalibRow], const ObsCalib& o, float clampv,
                                             float robustv, int lane) {
  float v[32];
  calib_fill<B>(v, su, sv, o, clampv, robustv, std::make_integer_sequence<int, 32>{});
  return transpose_reduce32(v, lane);
}

template <int C, int Loss>
__global__ void __launch_bounds__(32 * Calib<C>::W, 1) ba_calib_linearize_kernel(const CalibArgs a) {
  using L = Calib<C>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_warp = reinterpret_cast<float*>(smem_raw);
  double* s_red = reinterpret_cast<double*>(s_warp + (size_t)L::W * L::warp_floats);
  CamC* s_cam = reinterpret_cast<CamC*>(s_red + L::size);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* Yt = s_warp + (size_t)warp * L::warp_floats;

  if (threadIdx.x < C) load_cam_calib(a.cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) s_red[k] = 0.0;
  __syncthreads();
  const float lam = (float)a.ctrl[kCtrlLambda];
  const int cur = (int)a.ctrl[kCtrlCur];
  const float* X = a.Xpp + (int64_t)cur * 3 * a.N;

  // phase-2 role: 6x6 block pair (pa <= pb_) and row slice
  int pa = 0, pb_ = 0;
  const int pair = lane % L::NPAIR, slice = lane / L::NPAIR;
  {
    int q = pair;
    for (int r = 0; r < L::NB; ++r) {
      const int len = L::NB - r;
      if (q < len) {
        pa = r;
        pb_ = r + q;
        break;
      }
      q -= len;
    }
  }
  const bool act = slice < L::SL;

  float accS[6][6], accH[C][5];
#pragma unroll
  for (int k = 0; k < 6; ++k)
#pragma unroll
    for (int l = 0; l < 6; ++l) accS[k][l] = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c)
#pragma unroll
    for (int b = 0; b < 5; ++b) accH[c][b] = 0.f;
  int since = 0;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t i = (tile * L::W + warp) * 32 + lane;
    const bool valid = i < a.N;
    const int64_t il = valid ? i : a.N - 1;  // a padding lane re-reads the last point with zero weights
    // ---------------------------------------------------------------- phase 1
    float u[C], v[C], cw[C], Xp[3];
    {
      int64_t koff, coff;
      obs_offsets(a.lay, il, koff, coff);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float2 q = __ldg(reinterpret_cast<const float2*>(a.x2d + koff + c * a.lay.k_sV));
        u[c] = q.x;
        v[c] = q.y;
        cw[c] = valid ? __ldg(a.conf + coff + c * a.lay.c_sV) : 0.f;
      }
      Xp[0] = __ldg(X + 3 * il);
      Xp[1] = __ldg(X + 3 * il + 1);
      Xp[2] = __ldg(X + 3 * il + 2);
    }
    PointBlock pb;
    pb_zero(pb);
    float rcorr[C];  // cw (rho - omega s): slot 154
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsCalib o;
      calib_obs(s_cam[c], Xp, u[c], v[c], o);
      cw[c] = o.clamped ? 0.f : cw[c];  // a depth-clamped observation is excluded (ska_ba_calib.cuh)
      rcorr[c] = 0.f;
      if constexpr (Loss != kLossL2) {
        const float s2 = fmaf(o.bu[15], o.bu[15], o.bv[15] * o.bv[15]);
        float rho, om;
        robust_loss<Loss>(s2, a.loss_scale, rho, om);
        rcorr[c] = cw[c] * fmaf(-om, s2, rho);
        cw[c] *= om;  // pass B re-linearises the same state: it uses this weight
      }
      pb_add(pb, cw[c], o.au, o.av, o.bu[15], o.bv[15]);
    }
    const Chol3 f = chol3_damped(pb, lam);
    float d0, d1, d2;  // dp0 = -Hd^-1 gp (zero for a point without a factor: chol3 zeroes it)
    {
      float y0, y1, y2;
      chol3_fwd(f, -pb.g0, -pb.g1, -pb.g2, y0, y1, y2);
      chol3_bwd(f, y0, y1, y2, d0, d1, d2);
      d0 = f.ok ? d0 : 0.f;
      d1 = f.ok ? d1 : 0.f;
      d2 = f.ok ? d2 : 0.f;
    }
    __syncwarp();  // previous tile's phase 2 is done with the staging buffer
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsCalib o;
      calib_obs(s_cam[c], Xp, u[c], v[c], o);
      // slot 16 of the row: a . dp0, so that sum w B^T (a . dp0) = -W^T Hd^-1 gp ... sign folded below
      o.bu[16] = -fmaf(o.au[0], d0, fmaf(o.au[1], d1, o.au[2] * d2));
      o.bv[16] = -fmaf(o.av[0], d0, fmaf(o.av[1], d1, o.av[2] * d2));
      const float w = cw[c];
      float su[kCalibRow], sv[kCalibRow];
#pragma unroll
      for (int r = 0; r < kCalibRow; ++r) {
        su[r] = w * o.bu[r];
        sv[r] = w * o.bv[r];
      }
#pragma unroll
      for (int r = (c == 0 ? 6 : 0); r < kCalibP; ++r) {
        float y0, y1, y2;  // a point without a factor has a zeroed one: Y = 0 without a branch
        chol3_fwd(f, fmaf(su[r], o.au[0], sv[r] * o.av[0]), fmaf(su[r], o.au[1], sv[r] * o.av[1]),
                  fmaf(su[r], o.au[2], sv[r] * o.av[2]), y0, y1, y2);
        float* yt = Yt + L::col(c, r) * kYStride + 3 * lane;
        yt[0] = y0;
        yt[1] = y1;
        yt[2] = y2;
      }
      const float clampv = (valid && o.clamped) ? 1.f : 0.f;
      accH[c][0] += calib_batch<0>(su, sv, o, clampv, rcorr[c], lane);
      accH[c][1] += calib_batch<1>(su, sv, o, clampv, rcorr[c], lane);
      accH[c][2] += calib_batch<2>(su, sv, o, clampv, rcorr[c], lane);
      accH[c][3] += calib_batch<3>(su, sv, o, clampv, rcorr[c], lane);
      accH[c][4] += calib_batch<4>(su, sv, o, clampv, rcorr[c], lane);
    }
    __syncwarp();
    // ---------------------------------------------------------------- phase 2: Sw block (pa, pb_)
    if (act) {
      const float* ya = Yt + (6 * pa) * kYStride + 4 * slice * L::CH;
      const float* yb = Yt + (6 * pb_) * kYStride + 4 * slice * L::CH;
#pragma unroll 2
      for (int ch = 0; ch < L::CH; ++ch) {
        float4 A4[6], B4[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          A4[k] = *reinterpret_cast<const float4*>(ya + k * kYStride + 4 * ch);
          B4[k] = *reinterpret_cast<const float4*>(yb + k * kYStride + 4 * ch);
        }
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
          for (int l = 0; l < 6; ++l)
            accS[k][l] = fmaf(A4[k].x, B4[l].x, fmaf(A4[k].y, B4[l].y, fmaf(A4[k].z, B4[l].z, fmaf(A4[k].w, B4[l].w, accS[k][l]))));
      }
    }
    // ---------------------------------------------------------------- periodic fp64 fold
    const bool last = tile + gridDim.x >= a.n_tiles;
    if (++since == kFlush || last) {
      since = 0;
      for (int w = 0; w < L::W; ++w) {
        __syncthreads();
        if (warp == w) {
          for (int sl = 0; sl < L::SL; ++sl) {
            if (act && slice == sl) {
#pragma unroll
              for (int k = 0; k < 6; ++k)
#pragma unroll
                for (int l = 0; l < 6; ++l) {
                  const int ra = 6 * pa + k, rb = 6 * pb_ + l;
                  if (rb >= ra) s_red[ra * L::n - (ra * (ra - 1)) / 2 + (rb - ra)] += (double)accS[k][l];
                }
            }
            __syncwarp();
          }
#pragma unroll
          for (int c = 0; c < C; ++c)
#pragma unroll
            for (int b = 0; b < 5; ++b) s_red[L::oCam + kCalibCamBlock * c + 32 * b + lane] += (double)accH[c][b];
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int l = 0; l < 6; ++l) accS[k][l] = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c)
#pragma unroll
        for (int b = 0; b < 5; ++b) accH[c][b] = 0.f;
    }
  }
  __syncthreads();
  double* out = a.partials + (int64_t)blockIdx.x * L::size;
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) out[k] = s_red[k];
}

// ------------------------------------------------------------------------------------------------
// back-substitution + trial point + trial cost (thread per point)
constexpr int kCalibBackAcc = 3;  // trial cost, predicted decrease (points), clamped count

template <int C, int Loss>
__global__ void __launch_bounds__(kBaBlock, 2) ba_calib_backsub_kernel(const CalibArgs a) {
  __shared__ CamC s_cam[C], s_trial[C];
  __shared__ float s_delta[C][kCalibP];
  __shared__ double scratch[(kBaBlock / 32) * kCalibBackAcc];
  if (threadIdx.x < C) {
    load_cam_calib(a.cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
    load_cam_calib(a.cams + (C + threadIdx.x) * kCamStride, s_trial[threadIdx.x]);
  }
  if (threadIdx.x < kCalibP * C) s_delta[threadIdx.x / kCalibP][threadIdx.x % kCalibP] = (float)a.delta[threadIdx.x];
  __syncthreads();
  const float lam = (float)a.ctrl[kCtrlLambda];
  const int cur = (int)a.ctrl[kCtrlCur];
  const float* X = a.Xpp + (int64_t)cur * 3 * a.N;
  float* Xn = a.Xpp + (int64_t)(1 - cur) * 3 * a.N;

  float acc[kCalibBackAcc] = {0.f, 0.f, 0.f};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.N; i += stride) {
    int64_t koff, coff;
    obs_offsets(a.lay, i, koff, coff);
    float u[C], v[C], cw[C], Xp[3];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float2 q = __ldg(reinterpret_cast<const float2*>(a.x2d + koff + c * a.lay.k_sV));
      u[c] = q.x;
      v[c] = q.y;
      cw[c] = __ldg(a.conf + coff + c * a.lay.c_sV);
    }
    Xp[0] = __ldg(X + 3 * i);
    Xp[1] = __ldg(X + 3 * i + 1);
    Xp[2] = __ldg(X + 3 * i + 2);
    PointBlock pb;
    pb_zero(pb);
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;  // gp + W delta_c
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsCalib o;
      calib_obs(s_cam[c], Xp, u[c], v[c], o);
      float w = o.clamped ? 0.f : cw[c];  // excluded observation
      if constexpr (Loss != kLossL2) {  // the linearisation's weight: the same fp32 expression at the same state
        float rho, om;
        robust_loss<Loss>(fmaf(o.bu[15], o.bu[15], o.bv[15] * o.bv[15]), a.loss_scale, rho, om);
        w *= om;
      }
      pb_add(pb, w, o.au, o.av, o.bu[15], o.bv[15]);
      float lu = o.bu[15], lv = o.bv[15];
#pragma unroll
      for (int r = (c == 0 ? 6 : 0); r < kCalibP; ++r) {
        lu = fmaf(o.bu[r], s_delta[c][r], lu);
        lv = fmaf(o.bv[r], s_delta[c][r], lv);
      }
      r0 = fmaf(w * o.au[0], lu, fmaf(w * o.av[0], lv, r0));
      r1 = fmaf(w * o.au[1], lu, fmaf(w * o.av[1], lv, r1));
      r2 = fmaf(w * o.au[2], lu, fmaf(w * o.av[2], lv, r2));
    }
    const Chol3 f = chol3_damped(pb, lam);
    float d0, d1, d2;
    {
      float y0, y1, y2;
      chol3_fwd(f, -r0, -r1, -r2, y0, y1, y2);
      chol3_bwd(f, y0, y1, y2, d0, d1, d2);
      d0 = f.ok ? d0 : 0.f;
      d1 = f.ok ? d1 : 0.f;
      d2 = f.ok ? d2 : 0.f;
      acc[1] += d0 * fmaf(lam * pb.h00, d0, -pb.g0) + d1 * fmaf(lam * pb.h11, d1, -pb.g1) + d2 * fmaf(lam * pb.h22, d2, -pb.g2);
    }
    const float Xt[3] = {Xp[0] + d0, Xp[1] + d1, Xp[2] + d2};
    Xn[3 * i] = Xt[0];
    Xn[3 * i + 1] = Xt[1];
    Xn[3 * i + 2] = Xt[2];
    float tc = 0.f;
    int ncl = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      bool cl;
      float rho, om;
      robust_loss<Loss>(calib_err2(s_trial[c], Xt, u[c], v[c], cl), a.loss_scale, rho, om);
      tc = fmaf(cw[c], rho, tc);
      ncl += cl ? 1 : 0;
    }
    acc[0] += tc;
    acc[2] += (float)ncl;
  }
  block_reduce_store<kCalibBackAcc>(acc, scratch, a.partials + (int64_t)blockIdx.x * kCalibBackAcc);
}

// ------------------------------------------------------------------------------------------------
// reduced camera system with the intrinsics prior: one CTA, fp64
constexpr int kCalibMaxN = kCalibP * 2 - 6;  // C == 2

__global__ void __launch_bounds__(256) ba_calib_solve_kernel(int C, uint64_t free_mask, double* red, const double* __restrict__ prior,
                                                            double* cams, double* ctrl, double* delta, const PeerDev peer) {
  __shared__ double S[kCalibMaxN][kCalibMaxN + 1];
  __shared__ double b[kCalibMaxN], hd[kCalibMaxN], g[kCalibMaxN], d[kCalibMaxN];
  __shared__ int s_ok;
  const CalibLayout L(C);
  const int n = L.n, tid = threadIdx.x, nt = blockDim.x;
  if (peer.world > 1) peer_exchange_block(peer, red, L.size, red, 0);  // the reduced system's all-reduce, fused (ska_peer.cuh)
  const double lam = ctrl[kCtrlLambda];
  const double s = 1.0 / (ctrl[kCtrlSumConf] + 1e-6);
  if (tid == 0) s_ok = 1;
  // parameter r of camera c is free iff bit (15 c + r) of free_mask is set (camera 0: r >= 6 only)
  for (int i = tid; i < n; i += nt) {
    int c, r;
    L.param(i, c, r);
    const double* cb = red + L.oCam + kCalibCamBlock * c;
    double pr = 0.0, pg = 0.0;
    if (prior != nullptr && r >= 6) {
      pr = prior[c * 2 * kCalibNI + kCalibNI + (r - 6)];
      pg = pr * (cams[c * kCamStride + 12 + (r - 6)] - prior[c * 2 * kCalibNI + (r - 6)]);
    }
    const bool fi = (free_mask >> (kCalibP * c + r)) & 1ull;
    hd[i] = s * cb[calib_tri(r, r)] + pr;
    g[i] = s * cb[calib_tri(r, 15)] + pg;
    b[i] = fi ? s * cb[calib_tri(r, 16)] - g[i] : 0.0;
  }
  __syncthreads();
  for (int idx = tid; idx < n * n; idx += nt) {
    const int i = idx / n, j = idx % n;
    const int a = i < j ? i : j, bb = i < j ? j : i;
    int ci, ri, cj, rj;
    L.param(a, ci, ri);
    L.param(bb, cj, rj);
    double v = -s * red[L.sw(a, bb)];
    if (ci == cj) v += s * red[L.oCam + kCalibCamBlock * ci + calib_tri(ri, rj)];  // ri <= rj because a <= bb
    if (i == j) v = hd[i] * (1.0 + lam) - s * red[L.sw(a, a)];
    const bool fi = (free_mask >> (kCalibP * ci + ri)) & 1ull, fj = (free_mask >> (kCalibP * cj + rj)) & 1ull;
    S[i][j] = (fi && fj) ? v : (i == j ? 1.0 : 0.0);
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
      int c, r;
      L.param(i, c, r);
      const bool fi = (free_mask >> (kCalibP * c + r)) & 1ull;
      if (!s_ok || !isfinite(d[i])) d[i] = 0.0;
      if (fi) pred += d[i] * (lam * hd[i] * d[i] - g[i]);
    }
    ctrl[kCtrlOk] = (s_ok && fin) ? 1.0 : 0.0;
    ctrl[kCtrlPredCam] = pred;
  }
  __syncthreads();
  // delta (C,15) with the gauge zeros; trial cameras in slot 1
  for (int k = tid; k < kCalibP * C; k += nt) {
    const int c = k / kCalibP, r = k % kCalibP;
    delta[k] = (c == 0 && r < 6) ? 0.0 : d[Calib<2>::col(c, r)];
  }
  for (int c = tid; c < C; c += nt) {
    const double* src = cams + c * kCamStride;
    double* dst = cams + (C + c) * kCamStride;
    double dc[kCalibP];
    for (int r = 0; r < kCalibP; ++r) dc[r] = (c == 0 && r < 6) ? 0.0 : d[Calib<2>::col(c, r)];
    so3_exp_left(dc, src, dst);
    for (int k = 0; k < 3; ++k) dst[9 + k] = src[9 + k] + dc[3 + k];
    for (int k = 0; k < kCalibNI; ++k) dst[12 + k] = src[12 + k] + dc[6 + k];
    for (int k = 21; k < kCamStride; ++k) dst[k] = src[k];
  }
  __syncthreads();
  if (tid == 0) {  // prior part of the cost at the current and at the trial intrinsics
    double pc = 0.0, pt = 0.0;
    if (prior != nullptr)
      for (int c = 0; c < C; ++c)
        for (int k = 0; k < kCalibNI; ++k) {
          const double rho = prior[c * 2 * kCalibNI + kCalibNI + k], th0 = prior[c * 2 * kCalibNI + k];
          const double e0 = cams[c * kCamStride + 12 + k] - th0, e1 = cams[(C + c) * kCamStride + 12 + k] - th0;
          pc += rho * e0 * e0;
          pt += rho * e1 * e1;
        }
    ctrl[kCtrlPriorCur] = pc;
    ctrl[kCtrlPriorTrial] = pt;
  }
}

// LM controller (oracle/lm_calib.py run_lm): as ba_control_kernel with the prior inside the cost.
__global__ void __launch_bounds__(32) ba_calib_control_kernel(int C, const double* red, double* red2, double* cams, double* ctrl,
                                                              double* hist, int64_t hist_rows, const PeerDev peer) {
  if (blockIdx.x != 0) return;
  if (peer.world > 1) peer_exchange_block(peer, red2, SKA_BA_RED2_DOUBLES, red2, 0);
  const CalibLayout L(C);
  int accepted_i = 0;
  if (threadIdx.x == 0) {
    const double s = 1.0 / (ctrl[kCtrlSumConf] + 1e-6);
    double data = 0.0, ncl = 0.0;
    for (int c = 0; c < C; ++c) {
      data += red[L.oCam + kCalibCamBlock * c + calib_tri(15, 15)];
      data += red[L.oCam + kCalibCamBlock * c + kCalibRobustSlot];  // robust cost correction; +0.0 under L2
      ncl += red[L.oCam + kCalibCamBlock * c + kCalibClampSlot];
    }
    const double F = s * data + ctrl[kCtrlPriorCur], Ft = s * red2[0] + ctrl[kCtrlPriorTrial];
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
      h[6] = ncl;
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
static void fill_args(const SkaBaProblem& in, CalibArgs& a) {
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
  a.n_tiles = 0;
  a.x2d = in.d_x2d;
  a.conf = in.d_conf;
  a.cams = in.d_cams;
  a.ctrl = in.d_ctrl;
  a.delta = in.d_delta;
  a.Xpp = in.d_Xpp;
  a.partials = (double*)in.d_workspace;
  a.loss = in.loss;
  a.loss_scale = (float)in.loss_scale;
}

int ba_calib_red_size(int C) { return CalibLayout(C).size; }

static int unsupported_c() {
  return set_error(SKA_EUNSUPPORTED, "calibrating BA (free intrinsics / distortion) is built for C == 2 cameras (BASELINE config 3)");
}

template <int Loss>
static int calib_linearize(const SkaBaProblem& in, cudaStream_t s) {
  using L = Calib<2>;
  CalibArgs a;
  fill_args(in, a);
  auto kern = ba_calib_linearize_kernel<2, Loss>;
  static bool attr_set[64] = {};
  int dev = 0, sms = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  if (dev < 64 && !attr_set[dev]) {  // idempotent; a benign race sets it twice
    ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::smem);
    if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
    attr_set[dev] = true;
  }
  int per_sm = 1;
  ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * L::W, L::smem);
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  if (per_sm < 1) per_sm = 1;
  const int64_t per_tile = 32 * L::W;
  a.n_tiles = (a.N + per_tile - 1) / per_tile;
  int64_t grid = (int64_t)sms * per_sm;
  if (grid > a.n_tiles) grid = a.n_tiles;
  if (grid < 1) grid = 1;
  if (in.ws_bytes < (size_t)grid * L::size * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_calib_workspace_bytes)");
  kern<<<(unsigned)grid, 32 * L::W, L::smem, s>>>(a);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, (int)grid, L::size, in.d_red, s);
}

int ba_calib_linearize(const SkaBaProblem& in, cudaStream_t s) {
  if (in.C != 2) return unsupported_c();
  switch (in.loss) {
    case SKA_BA_LOSS_HUBER: return calib_linearize<kLossHuber>(in, s);
    case SKA_BA_LOSS_CAUCHY: return calib_linearize<kLossCauchy>(in, s);
    default: return calib_linearize<kLossL2>(in, s);
  }
}

template <int Loss>
static int calib_backsub(const SkaBaProblem& in, cudaStream_t s) {
  CalibArgs a;
  fill_args(in, a);
  int dev = 0, sms = 0, per_sm = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce == cudaSuccess) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_calib_backsub_kernel<2, Loss>, kBaBlock, 0);
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)sms * per_sm;
  const int64_t need = (a.N + kBaBlock - 1) / kBaBlock;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  if (in.ws_bytes < (size_t)grid * kCalibBackAcc * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_calib_workspace_bytes)");
  ba_calib_backsub_kernel<2, Loss><<<(unsigned)grid, kBaBlock, 0, s>>>(a);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, (int)grid, kCalibBackAcc, in.d_red2, s);
}

int ba_calib_backsub(const SkaBaProblem& in, cudaStream_t s) {
  if (in.C != 2) return unsupported_c();
  switch (in.loss) {
    case SKA_BA_LOSS_HUBER: return calib_backsub<kLossHuber>(in, s);
    case SKA_BA_LOSS_CAUCHY: return calib_backsub<kLossCauchy>(in, s);
    default: return calib_backsub<kLossL2>(in, s);
  }
}

static int calib_peer_of(const SkaPeerComm* c, int payload, PeerDev& pd) {
  pd.world = 0;
  if (c == nullptr) return SKA_OK;
  const int rc = peer_fill(*c, pd);
  if (rc != SKA_OK) return rc;
  if (payload > c->slot_doubles) return set_error(SKA_EINVAL, "reduced system larger than the peer slot");
  return SKA_OK;
}

int ba_calib_solve(int C, uint64_t free_mask, double* red, const double* prior, double* cams, double* ctrl, double* delta,
                   const SkaPeerComm* peer, void* stream) {
  if (C != 2) return unsupported_c();
  PeerDev pd;
  const int rc = calib_peer_of(peer, ba_calib_red_size(C), pd);
  if (rc != SKA_OK) return rc;
  ba_calib_solve_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(C, free_mask, red, prior, cams, ctrl, delta, pd);
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

int ba_calib_control(int C, const double* red, double* red2, double* cams, double* ctrl, double* hist, int64_t hist_rows,
                     const SkaPeerComm* peer, void* stream) {
  if (C != 2) return unsupported_c();
  PeerDev pd;
  const int rc = calib_peer_of(peer, SKA_BA_RED2_DOUBLES, pd);
  if (rc != SKA_OK) return rc;
  ba_calib_control_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(C, red, red2, cams, ctrl, hist, hist_rows, pd);
  const cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SKA_OK : set_error((int)ce, cudaGetErrorString(ce));
}

}  // namespace ska
