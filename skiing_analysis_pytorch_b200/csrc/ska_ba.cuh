// ska_ba.cuh - device-side pieces shared by the bundle-adjustment kernels.
//
// Cost and projection are the reference's (bundle_adjustment/loss.py:17-94):
//   X_c = R X + t;  Z = max(z, 1e-6);  (x, y) = X_c.xy / Z;  (u, v) = (K [x, y, 1])[:2]  (full K)
//   F = sum_tcj conf/(sum conf + 1e-6) |(u, v) - x2d|^2
// The LM algorithm on top of it is specified in oracle/lm.py / DESIGN.md section 5 (the reference's
// run_local_ba is an undefined symbol, vggt/multi_view_process.py:553).
//
// Scaling: every accumulated quantity (Hpp, gp, W, Hcc, gc, Sw, bw, cost) is linear in the
// observation weight w = conf * s, s = 1/(sum conf + 1e-6).  The kernels accumulate with the raw
// conf and the fp64 solve / control kernels apply s once, so fp32 never sees the ~1e-9 weights of
// a 1e8-observation clip.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ska {

constexpr int kBaBlock = 256;
constexpr float kZMin = 1e-6f;

// fp64 camera state as it lives in device memory: R(9) t(3) K(9) pad(3)
constexpr int kCamStride = 24;

// device control block (doubles); one per solve, owned by the caller
enum : int {
  kCtrlLambda = 0,   // damping used by the NEXT linearise / solve / backsub
  kCtrlNu = 1,       // Nielsen growth factor
  kCtrlSumConf = 2,  // global sum of conf (all ranks)
  kCtrlCur = 3,      // which half of the X ping-pong buffer is current (0/1)
  kCtrlIter = 4,     // trial counter = history row to write
  kCtrlPredCam = 5,  // camera part of the predicted decrease (written by solve)
  kCtrlOk = 6,       // 1 if the reduced system was positive definite (written by solve)
  kCtrlCost = 7,     // cost at the current point (written by control)
  kCtrlAccepted = 8, // last decision
  kCtrlPriorCur = 9,    // calibrating BA: intrinsics-prior part of the cost at the current cameras (written by solve)
  kCtrlPriorTrial = 10, // ... and at the trial cameras
  kCtrlSize = 16
};
constexpr int kHistRow = 8;  // iter, cost, trial_cost, lambda, rho, accepted, n_clamped, pred

struct CamF {
  float R[9], t[3];
  float k00, k01, k02, k10, k11, k12;
};

__device__ __forceinline__ void load_cam(const double* __restrict__ s, CamF& c) {
#pragma unroll
  for (int i = 0; i < 9; ++i) c.R[i] = (float)s[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) c.t[i] = (float)s[9 + i];
  const double k22 = s[12 + 8];
  c.k00 = (float)(s[12 + 0] / k22); c.k01 = (float)(s[12 + 1] / k22); c.k02 = (float)(s[12 + 2] / k22);
  c.k10 = (float)(s[12 + 3] / k22); c.k11 = (float)(s[12 + 4] / k22); c.k12 = (float)(s[12 + 5] / k22);
}

// 1/z: one MUFU.RCP plus one Newton step (full fp32 accuracy, a third of the IEEE-division sequence)
__device__ __forceinline__ float ba_rcp(float z) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(z));
  return fmaf(r, fmaf(-z, r, 1.0f), r);
}

// Robust loss of one observation's squared pixel error s = e_u^2 + e_v^2 (tests/oracle_robust.py, DESIGN.md section 5):
//   l2      rho = s                                  omega = 1
//   huber   rho = s (s <= d^2), 2 d sqrt(s) - d^2    omega = 1 (s <= d^2), d / sqrt(s)
//   cauchy  rho = d^2 ln(1 + s / d^2)                omega = 1 / (1 + s / d^2)
// The kernels weight the observation by conf * omega in every sum of the step (iteratively reweighted Gauss-Newton,
// omega not differentiated) and add conf * rho to the cost.  Huber's inlier branch is the L2 expression itself, so a
// solve whose every residual lies inside d is bit-identical to L2.  `d` is the scale in pixels (> 0).
enum : int { kLossL2 = 0, kLossHuber = 1, kLossCauchy = 2 };  // SKA_BA_LOSS_* (include/ska.h)

template <int Loss>
__device__ __forceinline__ void robust_loss(float s, float d, float& rho, float& omega) {
  if constexpr (Loss == kLossHuber) {
    const bool in = s <= d * d;
    omega = in ? 1.0f : d * rsqrtf(s);
    rho = in ? s : fmaf(2.0f * s, omega, -(d * d));  // 2 s d / sqrt(s) = 2 d sqrt(s)
  } else if constexpr (Loss == kLossCauchy) {
    const float q = s * ba_rcp(d * d);
    omega = ba_rcp(1.0f + q);
    rho = (d * d) * log1pf(q);
  } else {
    rho = s;
    omega = 1.0f;
  }
}

// fp64 twin for the regularised LM (ska_ba_reg.cu), split because only its cost kernel needs rho: the scale arrives as
// d, d^2 and 1/d^2 (computed once on the host), so omega costs Huber one rsqrt and a select and Cauchy one reciprocal.
// The same s gives the same bits in every kernel that recomputes omega.
struct RobustScale {
  double d, d2, id2;
};
template <int Loss>
__device__ __forceinline__ double robust_omega(double s, const RobustScale& r) {
  if constexpr (Loss == kLossHuber) {
    return s <= r.d2 ? 1.0 : r.d * rsqrt(s);
  } else if constexpr (Loss == kLossCauchy) {
    return 1.0 / (1.0 + s * r.id2);
  } else {
    return 1.0;
  }
}
template <int Loss>
__device__ __forceinline__ double robust_rho(double s, const RobustScale& r) {
  if constexpr (Loss == kLossHuber) {
    return s <= r.d2 ? s : 2.0 * r.d * sqrt(s) - r.d2;
  } else if constexpr (Loss == kLossCauchy) {
    return r.d2 * log1p(s * r.id2);
  } else {
    return s;
  }
}

// One observation: residual e, Jacobian rows of (u,v) w.r.t. X_c (ju, jv) and p = R X.
struct ObsLin {
  float eu, ev;
  float ju[3], jv[3];
  float p[3];
  bool clamped;
};

__device__ __forceinline__ void project_lin(const CamF& c, const float X[3], float uo, float vo, ObsLin& o) {
  o.p[0] = fmaf(c.R[0], X[0], fmaf(c.R[1], X[1], c.R[2] * X[2]));
  o.p[1] = fmaf(c.R[3], X[0], fmaf(c.R[4], X[1], c.R[5] * X[2]));
  o.p[2] = fmaf(c.R[6], X[0], fmaf(c.R[7], X[1], c.R[8] * X[2]));
  const float xc = o.p[0] + c.t[0], yc = o.p[1] + c.t[1], zc = o.p[2] + c.t[2];
  o.clamped = zc < kZMin;
  const float iz = ba_rcp(fmaxf(zc, kZMin));
  const float x = xc * iz, y = yc * iz;
  const float fu = fmaf(c.k00, x, c.k01 * y), fv = fmaf(c.k10, x, c.k11 * y);
  o.eu = (fu + c.k02) - uo;
  o.ev = (fv + c.k12) - vo;
  const float live = o.clamped ? 0.0f : 1.0f;  // d/dz vanishes while the clamp is active (autograd of loss.py:67)
  o.ju[0] = c.k00 * iz; o.ju[1] = c.k01 * iz; o.ju[2] = -fu * iz * live;
  o.jv[0] = c.k10 * iz; o.jv[1] = c.k11 * iz; o.jv[2] = -fv * iz * live;
}

// residual only (trial cost)
__device__ __forceinline__ float project_err2(const CamF& c, const float X[3], float uo, float vo, bool& clamped) {
  const float xc = fmaf(c.R[0], X[0], fmaf(c.R[1], X[1], fmaf(c.R[2], X[2], c.t[0])));
  const float yc = fmaf(c.R[3], X[0], fmaf(c.R[4], X[1], fmaf(c.R[5], X[2], c.t[1])));
  const float zc = fmaf(c.R[6], X[0], fmaf(c.R[7], X[1], fmaf(c.R[8], X[2], c.t[2])));
  clamped = zc < kZMin;
  const float iz = ba_rcp(fmaxf(zc, kZMin));
  const float x = xc * iz, y = yc * iz;
  const float eu = fmaf(c.k00, x, fmaf(c.k01, y, c.k02)) - uo;
  const float ev = fmaf(c.k10, x, fmaf(c.k11, y, c.k12)) - vo;
  return fmaf(eu, eu, ev * ev);
}

// point Jacobian rows A_u = ju R, A_v = jv R
__device__ __forceinline__ void point_rows(const CamF& c, const ObsLin& o, float au[3], float av[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    au[k] = fmaf(o.ju[0], c.R[k], fmaf(o.ju[1], c.R[3 + k], o.ju[2] * c.R[6 + k]));
    av[k] = fmaf(o.jv[0], c.R[k], fmaf(o.jv[1], c.R[3 + k], o.jv[2] * c.R[6 + k]));
  }
}

// camera Jacobian rows B_u = [p x ju | ju], B_v = [p x jv | jv]  (left-multiplicative d_omega, additive d_t)
__device__ __forceinline__ void camera_rows(const ObsLin& o, float bu[6], float bv[6]) {
  bu[0] = o.p[1] * o.ju[2] - o.p[2] * o.ju[1];
  bu[1] = o.p[2] * o.ju[0] - o.p[0] * o.ju[2];
  bu[2] = o.p[0] * o.ju[1] - o.p[1] * o.ju[0];
  bv[0] = o.p[1] * o.jv[2] - o.p[2] * o.jv[1];
  bv[1] = o.p[2] * o.jv[0] - o.p[0] * o.jv[2];
  bv[2] = o.p[0] * o.jv[1] - o.p[1] * o.jv[0];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    bu[3 + k] = o.ju[k];
    bv[3 + k] = o.jv[k];
  }
}

// Symmetric 3x3 point block accumulator + gradient
struct PointBlock {
  float h00, h01, h02, h11, h12, h22, g0, g1, g2;
};
__device__ __forceinline__ void pb_zero(PointBlock& b) { b.h00 = b.h01 = b.h02 = b.h11 = b.h12 = b.h22 = b.g0 = b.g1 = b.g2 = 0.f; }
__device__ __forceinline__ void pb_add(PointBlock& b, float cw, const float au[3], const float av[3], float eu, float ev) {
  const float u0 = cw * au[0], u1 = cw * au[1], u2 = cw * au[2];
  const float v0 = cw * av[0], v1 = cw * av[1], v2 = cw * av[2];
  b.h00 = fmaf(u0, au[0], fmaf(v0, av[0], b.h00));
  b.h01 = fmaf(u0, au[1], fmaf(v0, av[1], b.h01));
  b.h02 = fmaf(u0, au[2], fmaf(v0, av[2], b.h02));
  b.h11 = fmaf(u1, au[1], fmaf(v1, av[1], b.h11));
  b.h12 = fmaf(u1, au[2], fmaf(v1, av[2], b.h12));
  b.h22 = fmaf(u2, au[2], fmaf(v2, av[2], b.h22));
  b.g0 = fmaf(u0, eu, fmaf(v0, ev, b.g0));
  b.g1 = fmaf(u1, eu, fmaf(v1, ev, b.g1));
  b.g2 = fmaf(u2, eu, fmaf(v2, ev, b.g2));
}

// Cholesky of the damped 3x3 point block, lower factor with inverted diagonal.
struct Chol3 {
  float i0, l10, l20, i1, l21, i2;
  bool ok;
};
__device__ __forceinline__ Chol3 chol3(float h00, float h01, float h02, float h11, float h12, float h22) {
  Chol3 f;
  f.i0 = rsqrtf(h00);
  f.l10 = h01 * f.i0;
  f.l20 = h02 * f.i0;
  const float d1 = fmaf(-f.l10, f.l10, h11);
  f.i1 = rsqrtf(d1);
  f.l21 = fmaf(-f.l20, f.l10, h12) * f.i1;
  const float d2 = fmaf(-f.l21, f.l21, fmaf(-f.l20, f.l20, h22));
  f.i2 = rsqrtf(d2);
  // a point nobody observes (all conf 0) or a rank-deficient block has no step and no Schur term:
  // its factor is zeroed so that chol3_fwd / chol3_bwd return exact zeros without a branch
  f.ok = (h00 > 0.f) && (d1 > 0.f) && (d2 > 0.f) && (d2 <= 3.0e38f);
  if (!f.ok) f.i0 = f.l10 = f.l20 = f.i1 = f.l21 = f.i2 = 0.f;
  return f;
}
__device__ __forceinline__ Chol3 chol3_damped(const PointBlock& b, float lam) {
  const float s = 1.0f + lam;
  return chol3(b.h00 * s, b.h01, b.h02, b.h11 * s, b.h12, b.h22 * s);
}
// y = L^-1 b
__device__ __forceinline__ void chol3_fwd(const Chol3& f, float b0, float b1, float b2, float& y0, float& y1, float& y2) {
  y0 = b0 * f.i0;
  y1 = fmaf(-f.l10, y0, b1) * f.i1;
  y2 = fmaf(-f.l21, y1, fmaf(-f.l20, y0, b2)) * f.i2;
}
// x = L^-T y
__device__ __forceinline__ void chol3_bwd(const Chol3& f, float y0, float y1, float y2, float& x0, float& x1, float& x2) {
  x2 = y2 * f.i2;
  x1 = fmaf(-f.l21, x2, y1) * f.i1;
  x0 = fmaf(-f.l20, x2, fmaf(-f.l10, x1, y0)) * f.i0;
}

// Deterministic block reduction of NV values per thread: fp64 warp shuffles, then a fixed-order sum
// of the per-warp values in shared memory; thread k < NV writes column k of `out`.  No atomics.
// `scratch` holds (blockDim/32)*NV doubles.
template <int NV>
__device__ __forceinline__ void block_reduce_store(const float (&v)[NV], double* scratch, double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = (double)v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) scratch[warp * NV + i] = x;
  }
  __syncthreads();
  const int nw = (int)(blockDim.x >> 5);
  for (int i = threadIdx.x; i < NV; i += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += scratch[w * NV + i];
    out[i] = s;
  }
  __syncthreads();
}

// R_new = exp([w]x) R (fp64; the camera update of the reduced-system solve kernels)
__device__ inline void so3_exp_left(const double w[3], const double* R, double* Rn) {
  const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  double A, B;
  if (th2 < 1e-8) {
    A = 1.0 - th2 / 6.0;
    B = 0.5 - th2 / 24.0;
  } else {
    const double th = sqrt(th2);
    A = sin(th) / th;
    B = (1.0 - cos(th)) / th2;
  }
  // E = I + A [w]x + B [w]x^2
  const double wx = w[0], wy = w[1], wz = w[2];
  double E[9];
  E[0] = 1.0 - B * (wy * wy + wz * wz);
  E[1] = -A * wz + B * wx * wy;
  E[2] = A * wy + B * wx * wz;
  E[3] = A * wz + B * wx * wy;
  E[4] = 1.0 - B * (wx * wx + wz * wz);
  E[5] = -A * wx + B * wy * wz;
  E[6] = -A * wy + B * wx * wz;
  E[7] = A * wx + B * wy * wz;
  E[8] = 1.0 - B * (wx * wx + wy * wy);
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) Rn[3 * r + c] = E[3 * r] * R[c] + E[3 * r + 1] * R[3 + c] + E[3 * r + 2] * R[6 + c];
}

// ---- shared by the warp-cooperative linearisation kernels (ska_ba_wide.cu, ska_ba_calib.cu)
constexpr int kFlush = 16;
constexpr int kYStride = 100;  // 96 rows + 4: column stride = 4 banks mod 32

constexpr int largest_div(int n, int cap) {
  int best = 1;
  for (int d = 1; d <= n; ++d)
    if (n % d == 0 && d <= cap) best = d;
  return best;
}

// lane i ends up with the sum over the warp of v[i] (i < 32); v is destroyed
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = up ? v[i] : v[i + o];
      const float keep = up ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0];
}

// Observation addressing for both layouts: frame-major (T,C,J,.) is the reference's
// (bundle_adjustment/loss.py x2d / conf2d), view-major (C,T,J,.) is the triangulation layout.
struct ObsLayout {
  int64_t k_sT, k_sV;  // strides in floats for x2d
  int64_t c_sT, c_sV;  // strides in floats for conf
  int32_t J;
};
__device__ __forceinline__ void obs_offsets(const ObsLayout& L, int64_t i, int64_t& koff, int64_t& coff) {
  const uint32_t t = (uint32_t)i / (uint32_t)L.J;
  const uint32_t j = (uint32_t)i - t * (uint32_t)L.J;
  koff = (int64_t)t * L.k_sT + 2 * (int64_t)j;
  coff = (int64_t)t * L.c_sT + (int64_t)j;
}

}  // namespace ska
