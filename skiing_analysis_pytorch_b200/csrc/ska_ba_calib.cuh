// ska_ba_calib.cuh - per-observation arithmetic of the CALIBRATING bundle adjustment (free intrinsics +
// distortion; BASELINE config 3 "Rodrigues extrinsics + intrinsics/distortion", SURVEY.md section 8d "p = 15").
// __host__ __device__ so tests/hostemu can run the exact fp32 sequence against the fp64 oracle
// (oracle/lm_calib.py) on the CPU-only authoring box; the product only calls it from device code.
//
// Projection = cv2.projectPoints' 5-coefficient model, the one the reference reprojects with
// (triangulation/reproject.py:77-78, bundle_adjustment/reproject.py:147-148), with loss.py's depth clamp
// (bundle_adjustment/loss.py:67):
//   X_c = R X + t;  x = X_c.x / z, y = X_c.y / z;  r2 = x^2 + y^2   (observations with z < 1e-6 - loss.py:67's clamp
//   threshold - are excluded and counted: a polynomial distortion of a clamped projection is meaningless)
//   rad = 1 + k1 r2 + k2 r2^2 + k3 r2^3
//   x" = x rad + 2 p1 x y + p2 (r2 + 2 x^2);   y" = y rad + p1 (r2 + 2 y^2) + 2 p2 x y
//   u = fx x" + cx;  v = fy y" + cy
// Camera parameter block (15): [d_omega(3) (R <- exp([d_omega]x) R), d_t(3), fx, fy, cx, cy, k1, k2, p1, p2, k3].
#pragma once
#include <math.h>
#include <stdint.h>

#include "ska_vec.cuh"

#if defined(__CUDACC__)
#define SKA_CX __host__ __device__ constexpr
#else
#define SKA_CX constexpr
#endif

namespace ska {

constexpr int kCalibP = 15;          // parameters per camera
constexpr int kCalibNI = 9;          // intrinsic parameters theta = fx fy cx cy k1 k2 p1 p2 k3
constexpr int kCalibRow = 17;        // per-observation row [B (15) | e | a.dp0]
constexpr int kCalibTri = 153;       // upper triangle of the 17 x 17 per-camera matrix sum w row^T row
constexpr int kCalibClampSlot = 153; // per-camera count of depth-clamped observations
constexpr int kCalibRobustSlot = 154; // per-camera robust cost correction sum w (rho(s) - omega s); 0 under L2
constexpr int kCalibCamBlock = 160;  // padded per-camera block of the packed reduced system (5 x 32)
constexpr float kCalibZMin = 1e-6f;

// index of entry (r, s), r <= s, in the row-major upper triangle of the 17 x 17 per-camera matrix
SKA_CX int calib_tri(int r, int s) { return r * kCalibRow - (r * (r - 1)) / 2 + (s - r); }
// (r, s) of triangle entry q
SKA_CX int calib_tri_row(int q) {
  int r = 0;
  while (q >= kCalibRow - r) {
    q -= kCalibRow - r;
    ++r;
  }
  return r;
}
SKA_CX int calib_tri_col(int q) {
  const int r = calib_tri_row(q);
  return r + (q - calib_tri(r, r));
}

// fp32 camera as the kernels hold it in shared memory
struct CamC {
  float R[9], t[3];
  float fx, fy, cx, cy, k1, k2, p1, p2, k3;
};

SKA_HD float calib_rcp(float z) {
#if defined(__CUDA_ARCH__)
  float r;  // MUFU.RCP + one Newton step: full fp32 accuracy at a third of the IEEE-division sequence
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(z));
  return fmaf(r, fmaf(-z, r, 1.0f), r);
#else
  return 1.0f / z;
#endif
}

// Everything one observation contributes to the linearisation.
struct ObsCalib {
  float au[3], av[3];                    // point Jacobian rows d(u, v) / dX
  float bu[kCalibRow], bv[kCalibRow];    // [camera Jacobian rows (15) | residual | slot 16 filled by the caller]
  bool clamped;
};

SKA_HD void calib_obs(const CamC& c, const float X[3], float uo, float vo, ObsCalib& o) {
  const float p0 = fmaf(c.R[0], X[0], fmaf(c.R[1], X[1], c.R[2] * X[2]));
  const float p1 = fmaf(c.R[3], X[0], fmaf(c.R[4], X[1], c.R[5] * X[2]));
  const float p2 = fmaf(c.R[6], X[0], fmaf(c.R[7], X[1], c.R[8] * X[2]));
  float xc = p0 + c.t[0], yc = p1 + c.t[1], zc = p2 + c.t[2];
  o.clamped = zc < kCalibZMin;
  // A depth-clamped observation (the point is at / behind the camera plane) is EXCLUDED from the calibrating problem:
  // the caller gives it zero weight (oracle/lm_calib.py does the same).  loss.py's clamp would put it at |x| ~ 1e6,
  // where the r^6 distortion term overflows fp32 and 0 * inf would poison every sum; evaluating the row at the optical
  // axis instead keeps all of its entries finite.
  xc = o.clamped ? 0.0f : xc;
  yc = o.clamped ? 0.0f : yc;
  zc = o.clamped ? 1.0f : zc;
  const float iz = calib_rcp(zc);
  const float live = 1.0f;
  const float x = xc * iz, y = yc * iz;
  const float xx = x * x, yy = y * y, xy = x * y;
  const float r2 = xx + yy, r4 = r2 * r2, r6 = r4 * r2;
  const float rad = fmaf(r2, fmaf(r2, fmaf(r2, c.k3, c.k2), c.k1), 1.0f);
  const float drad = fmaf(r2, fmaf(3.0f * c.k3, r2, 2.0f * c.k2), c.k1);
  const float tx = fmaf(2.0f, xx, r2), ty = fmaf(2.0f, yy, r2);  // r2 + 2x^2, r2 + 2y^2
  const float xd = fmaf(x, rad, fmaf(2.0f * c.p1, xy, c.p2 * tx));
  const float yd = fmaf(y, rad, fmaf(c.p1, ty, 2.0f * c.p2 * xy));
  const float eu = fmaf(c.fx, xd, c.cx) - uo;
  const float ev = fmaf(c.fy, yd, c.cy) - vo;
  // 2 x 2 Jacobian of (x", y") w.r.t. (x, y): symmetric off-diagonal
  const float a11 = fmaf(2.0f * xx, drad, rad) + fmaf(2.0f * c.p1, y, 6.0f * c.p2 * x);
  const float a12 = fmaf(2.0f * xy, drad, fmaf(2.0f * c.p1, x, 2.0f * c.p2 * y));
  const float a22 = fmaf(2.0f * yy, drad, rad) + fmaf(6.0f * c.p1, y, 2.0f * c.p2 * x);
  const float fiz = c.fx * iz, giz = c.fy * iz;
  const float ju0 = fiz * a11, ju1 = fiz * a12, ju2 = -fmaf(ju0, x, ju1 * y) * live;
  const float jv0 = giz * a12, jv1 = giz * a22, jv2 = -fmaf(jv0, x, jv1 * y) * live;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    o.au[k] = fmaf(ju0, c.R[k], fmaf(ju1, c.R[3 + k], ju2 * c.R[6 + k]));
    o.av[k] = fmaf(jv0, c.R[k], fmaf(jv1, c.R[3 + k], jv2 * c.R[6 + k]));
  }
  // rotation (left-multiplicative d_omega): p x j with p = R X;  translation: j
  o.bu[0] = p1 * ju2 - p2 * ju1; o.bu[1] = p2 * ju0 - p0 * ju2; o.bu[2] = p0 * ju1 - p1 * ju0;
  o.bv[0] = p1 * jv2 - p2 * jv1; o.bv[1] = p2 * jv0 - p0 * jv2; o.bv[2] = p0 * jv1 - p1 * jv0;
  o.bu[3] = ju0; o.bu[4] = ju1; o.bu[5] = ju2;
  o.bv[3] = jv0; o.bv[4] = jv1; o.bv[5] = jv2;
  // fx fy cx cy k1 k2 p1 p2 k3
  const float fxx = c.fx * x, fyy = c.fy * y;
  o.bu[6] = xd;   o.bu[7] = 0.0f; o.bu[8] = 1.0f; o.bu[9] = 0.0f;
  o.bv[6] = 0.0f; o.bv[7] = yd;   o.bv[8] = 0.0f; o.bv[9] = 1.0f;
  o.bu[10] = fxx * r2; o.bu[11] = fxx * r4; o.bu[12] = 2.0f * c.fx * xy; o.bu[13] = c.fx * tx; o.bu[14] = fxx * r6;
  o.bv[10] = fyy * r2; o.bv[11] = fyy * r4; o.bv[12] = c.fy * ty; o.bv[13] = 2.0f * c.fy * xy; o.bv[14] = fyy * r6;
  o.bu[15] = eu;
  o.bv[15] = ev;
  o.bu[16] = 0.0f;
  o.bv[16] = 0.0f;
}

// squared pixel error only (trial cost); 0 for a depth-clamped (excluded) observation
SKA_HD float calib_err2(const CamC& c, const float X[3], float uo, float vo, bool& clamped) {
  const float xc = fmaf(c.R[0], X[0], fmaf(c.R[1], X[1], fmaf(c.R[2], X[2], c.t[0])));
  const float yc = fmaf(c.R[3], X[0], fmaf(c.R[4], X[1], fmaf(c.R[5], X[2], c.t[1])));
  const float zc = fmaf(c.R[6], X[0], fmaf(c.R[7], X[1], fmaf(c.R[8], X[2], c.t[2])));
  clamped = zc < kCalibZMin;
  if (clamped) return 0.0f;
  const float iz = calib_rcp(zc);
  const float x = xc * iz, y = yc * iz;
  const float xx = x * x, yy = y * y, xy = x * y, r2 = xx + yy;
  const float rad = fmaf(r2, fmaf(r2, fmaf(r2, c.k3, c.k2), c.k1), 1.0f);
  const float xd = fmaf(x, rad, fmaf(2.0f * c.p1, xy, c.p2 * fmaf(2.0f, xx, r2)));
  const float yd = fmaf(y, rad, fmaf(c.p1, fmaf(2.0f, yy, r2), 2.0f * c.p2 * xy));
  const float eu = fmaf(c.fx, xd, c.cx) - uo;
  const float ev = fmaf(c.fy, yd, c.cy) - vo;
  return fmaf(eu, eu, ev * ev);
}

}  // namespace ska
