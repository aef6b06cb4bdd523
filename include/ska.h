/* ska.h - C ABI of libska.so: B200 (sm_100a) kernels for batched multi-view 3D keypoint
 * reconstruction (weighted DLT triangulation + fused reprojection scoring + Schur LM bundle
 * adjustment).
 *
 * The reference (ChenKaiXuSan/Skiing_Analysis_PyTorch) is pure Python and has no FFI layer; its
 * boundary for this path is a set of Python call signatures (SURVEY.md section 8b).  Each entry
 * point below names the reference interface whose arithmetic it replaces (file:line relative to
 * the reference checkout); INTEGRATION.md shows the ctypes stub a maintainer adds on that side.
 *
 * Conventions
 *  - plain C, no torch / C++ types; every `d_*` pointer is a DEVICE pointer owned by the caller
 *    (e.g. the PyTorch allocator); the library never allocates, frees or retains caller memory.
 *  - `SkaCamera` arrays and `centre` are HOST pointers, read during the call only.
 *  - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation.
 *  - return value: 0 = ok, negative = SKA_E* argument error, positive = cudaError_t.
 *    `ska_last_error()` returns a thread-local message for the last non-zero return.
 *  - re-entrant and thread safe: no mutable globals, per-call constants travel as kernel
 *    parameters (never through a shared __constant__ symbol).
 */
#ifndef SKA_H_
#define SKA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKA_ABI_VERSION 9

#define SKA_OK 0
#define SKA_EINVAL -1       /* null pointer / bad size / bad enum */
#define SKA_EUNSUPPORTED -2 /* valid request outside what the kernels implement (e.g. tilted sensor) */
#define SKA_EALIGN -3       /* pointer not aligned as documented */
#define SKA_EWORKSPACE -4   /* workspace too small */

#define SKA_MAX_VIEWS 8
#define SKA_MAX_BONES 16 /* bundle_adjustment/loss.py:118-131 lists 12 */

/* memory layout of per-observation tensors */
#define SKA_LAYOUT_VIEW_MAJOR 0  /* kpts (V,T,J,2), conf/err (V,T,J): the reference's separate
                                    left_kpts/right_kpts arrays, triangulation/main.py:99-109 */
#define SKA_LAYOUT_FRAME_MAJOR 1 /* kpts (T,V,J,2), conf/err (T,V,J): bundle_adjustment/loss.py x2d/conf2d */

/* flags for ska_triangulate_reproject_f32 */
#define SKA_SOLVER_SECULAR 0u    /* default: fp32 secular/Rayleigh iteration with interlacing certificate,
                                    fp64 Jacobi fallback for points that fail it */
#define SKA_SOLVER_JACOBI64 1u   /* fp64 rows + fp64 register-resident cyclic Jacobi for every point */
#define SKA_SOLVER_JACOBI32 2u   /* fp32 register-resident cyclic Jacobi (north-star design point; measurement) */
#define SKA_SOLVER_MASK 3u
#define SKA_WEIGHT_SQRT 4u       /* DLT row weight = sqrt(conf) (matches loss.py's conf*err^2); default = conf */
#define SKA_PINHOLE_REPROJ 8u    /* ignore dist[] when scoring (quirk Q1 switch: dist=None) */

/* One calibrated camera, world->camera x_c = R x_w + t, fp64, row-major. HOST struct.
 * K is the full 3x3 intrinsic matrix: triangulation uses P = K [R|t] (triangulate.py:65-66,
 * vggt/triangulate.py:13-16); cv2-style reprojection uses fx,fy,cx,cy only (skew ignored, like
 * cv2.projectPoints); loss-style projection uses all of K (loss.py:74-82).
 * dist: OpenCV order k1,k2,p1,p2,k3,k4,k5,k6,s1,s2,s3,s4,taux,tauy; all zero = pinhole.
 * taux/tauy != 0 -> SKA_EUNSUPPORTED. */
typedef struct SkaCamera {
  double K[9];
  double R[9];
  double t[3];
  double dist[14];
} SkaCamera;

int ska_abi_version(void);
const char* ska_last_error(void);
/* compiled-for architecture string, e.g. "sm_100a" */
const char* ska_build_arch(void);

/* Fused weighted V-view DLT triangulation + reprojection scoring.
 * Replaces, for a whole clip in ONE launch:
 *   triangulate_joints         triangulation/triangulate.py:60-68   (cv2.triangulatePoints)
 *   triangulate_point / loop   vggt/triangulate.py:19-34, :64-71    (np.linalg.svd per joint)
 *   reproject_points + errors  triangulation/reproject.py:49-83, :243-244 (cv2.projectPoints, |proj-kpt|)
 *   the per-frame loop         triangulation/triangulate.py:76-116
 * cams[V]   host; static rig shared by every frame (per-frame extrinsics: the _frames_ variant below).
 * centre    host[3] or NULL: numerical conditioning origin only (results do not depend on it
 *           beyond rounding); NULL = least-squares intersection of the optical axes.
 * d_kpts    pixels, layout per `layout`; d_conf nullable (NULL = unit weights = reference behaviour).
 * d_X       (T,J,3) f32 out.  d_err: per-view pixel error |proj-kpt|, same layout as conf, nullable.
 * d_proj    reprojected pixels, same layout as kpts, nullable.
 * d_status  nullable (T,J) uint8 out: 0 = fast path certified, 1 = Jacobi fallback used,
 *           2 = non-finite result.
 * Alignment: d_kpts 8 B, everything else 4 B (16 B on all of them enables the 128-bit path). */
int ska_triangulate_reproject_f32(const SkaCamera* cams, int32_t V, const double* centre, const float* d_kpts,
                                  const float* d_conf, int64_t T, int32_t J, int32_t layout, uint32_t flags,
                                  float* d_X, float* d_err, float* d_proj, uint8_t* d_status, void* stream);

/* Same, with PER-FRAME extrinsics: process_triangulate hands every frame its own R[i], T[i]
 * (triangulation/triangulate.py:76-82; vggt/multi_view_process.py:220-234 likewise).
 * d_Rt_frames  (T,V,12) fp64 device = [R row-major (9), t (3)] world->camera per frame and view;
 *              cams[v].K / dist are shared over the clip, cams[v].R / t are ignored.
 * d_workspace  may be NULL (ws_bytes 0) when the fused kernel takes the call: view-major layout, V <= 4, >= 8 joints, no skew /
 *              thin prism, d_kpts / d_X / d_proj (and d_conf, with T*J % 4 == 0) 16-byte aligned - it builds every frame's centred
 *              cameras in shared memory (fp64, conditioning origin chosen per frame) and writes nothing per frame to global memory.
 *              Any other call needs >= ska_tri_frames_workspace_bytes(V, T) bytes, 16-byte aligned (a prep kernel stores the
 *              per-frame kernel-side cameras there) and returns SKA_EWORKSPACE without it.
 * Solver flags are ignored (fp32 secular path with fp64 fallback). */
size_t ska_tri_frames_workspace_bytes(int32_t V, int64_t T);
int ska_triangulate_reproject_frames_f32(const SkaCamera* cams, int32_t V, const double* d_Rt_frames,
                                         const float* d_kpts, const float* d_conf, int64_t T, int32_t J,
                                         int32_t layout, uint32_t flags, float* d_X, float* d_err, float* d_proj,
                                         uint8_t* d_status, void* d_workspace, size_t ws_bytes, void* stream);

/* cv2-style reprojection of GIVEN 3D points (no triangulation) into V cameras, with the rational /
 * tangential / thin-prism distortion model, computed in fp64 like cv2.projectPoints and stored as
 * float32 pixels.  Replaces
 *   reproject_points   triangulation/reproject.py:49-83; bundle_adjustment/reproject.py:74-153
 *                      (== vggt/reproject.py, front_side/side/reproject.py, fuse/side/reproject.py)
 * d_X (T,J,3) f32 in the coordinates cams[v] maps from; d_proj like kpts in `layout`, nullable;
 * d_err (needs d_kpts) = |proj_f32 - kpt| per view as reproject.py:243-244, nullable. */
int ska_reproject_points_f32(const SkaCamera* cams, int32_t V, const float* d_X, const float* d_kpts, int64_t T,
                             int32_t J, int32_t layout, float* d_proj, float* d_err, void* stream);

/* nan-aware per-(frame, view) statistics of the pixel errors: d_stats (T,V,4) f32 =
 * [rmse, mean, median, max] (np.nanmean / nanmedian / nanmax of triangulation/reproject.py:254-261);
 * all-NaN rows give NaN.  d_err in `layout` ((V,T,J) or (T,V,J)); J <= 1024. */
int ska_frame_stats_f32(const float* d_err, int64_t T, int32_t J, int32_t V, int32_t layout, float* d_stats,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * bundle_adjustment/loss.py as kernels.  All pointers are device pointers in the caller's dtype
 * (f32 / f64 variants).  Cameras: d_R (.,C,3,3), d_t (.,C,3), d_K (.,C,3,3) with a FRAME STRIDE in
 * elements: 0 = one camera set shared over the clip (loss.py's (C,3,3) inputs), 9*C / 3*C / 9*C =
 * per-frame cameras ((T,C,3,3) inputs); the three strides are independent (loss.py:40-50, :74-79).
 *
 * project_points     loss.py:17-84:  d_out (T,C,J,2); Z clamp at 1e-6 (:67), rows 0-1 of the full K. */
int ska_project_points_f32(const float* d_X, int64_t T, int32_t J, int32_t C, const float* d_R, int64_t R_frame_stride,
                           const float* d_t, int64_t t_frame_stride, const float* d_K, int64_t K_frame_stride,
                           float* d_out, void* stream);
int ska_project_points_f64(const double* d_X, int64_t T, int32_t J, int32_t C, const double* d_R, int64_t R_frame_stride,
                           const double* d_t, int64_t t_frame_stride, const double* d_K, int64_t K_frame_stride,
                           double* d_out, void* stream);
/* reprojection_loss  loss.py:90-94, value and analytic gradient in one pass over the observations.
 * d_sums[4] (fp64): [sum conf |proj - x2d|^2, sum conf, #clamped observations, reserved (not written)];
 *                   loss = w * d_sums[0] / (d_sums[1] + 1e-6).
 * d_gX (T,J,3), d_gR / d_gt / d_gK shaped like d_R / d_t / d_K: nullable; UNSCALED gradients
 * sum conf J^T e - multiply by 2 w / (d_sums[1] + 1e-6) (what torch.autograd derives from loss.py).
 * d_conf == NULL selects vector-Jacobian mode: d_x2d then holds a cotangent g (T,C,J,2) of
 * project_points' output and the gradients are sum J^T g (the backward of project_points). */
size_t ska_loss_workspace_bytes(int32_t C);
int ska_reprojection_loss_f32(const float* d_X, int64_t T, int32_t J, int32_t C, const float* d_R, int64_t R_frame_stride,
                              const float* d_t, int64_t t_frame_stride, const float* d_K, int64_t K_frame_stride,
                              const float* d_x2d, const float* d_conf, double* d_sums, float* d_gX, float* d_gR,
                              float* d_gt, float* d_gK, void* d_workspace, size_t ws_bytes, void* stream);
int ska_reprojection_loss_f64(const double* d_X, int64_t T, int32_t J, int32_t C, const double* d_R, int64_t R_frame_stride,
                              const double* d_t, int64_t t_frame_stride, const double* d_K, int64_t K_frame_stride,
                              const double* d_x2d, const double* d_conf, double* d_sums, double* d_gX, double* d_gR,
                              double* d_gt, double* d_gK, void* d_workspace, size_t ws_bytes, void* stream);
/* Regularisers (loss.py:97-155): raw fp64 sums + UNSCALED gradients (nullable); the caller applies
 * w / count.  d_workspace >= ska_reg_workspace_bytes().
 *   pose_temporal   :153-155  d_sum[0] = sum_{t<T-1} |X[t+1]-X[t]|^2            count = (T-1)*J*3
 *   bone_length     :134-150  d_ref == NULL: d_sums[b] = sum_t len[t][b] (the caller forms the mean);
 *                             else d_sums[0] = sum_{t,b} (len - d_ref[b])^2      count = T*n_bones
 *                             bone_i / bone_j: HOST index arrays (BONES, :118-131), n_bones <= SKA_MAX_BONES;
 *                             d_sums holds SKA_MAX_BONES doubles
 *   camera_centre   :97-100   d_C (n,3) = -R^T t
 *   camera_smooth   :103-106  cameras (D0, M): d_sum[0] = sum_{d<D0-1,m} |C[d+1][m]-C[d][m]|^2   count = (D0-1)*M*3
 *   baseline_reg    :109-114  cameras (T, C>=2): d_mean == NULL: d_sum[0] = sum_t |C0-C1|;
 *                             else d_sum[0] = sum_t (|C0-C1| - d_mean[0])^2      count = T */
size_t ska_reg_workspace_bytes(void);
int ska_pose_temporal_f32(const float* d_X, int64_t T, int32_t J, double* d_sum, float* d_gX, void* d_workspace, size_t ws_bytes, void* stream);
int ska_pose_temporal_f64(const double* d_X, int64_t T, int32_t J, double* d_sum, double* d_gX, void* d_workspace, size_t ws_bytes, void* stream);
int ska_bone_length_f32(const float* d_X, int64_t T, int32_t J, const int32_t* bone_i, const int32_t* bone_j, int32_t n_bones,
                        const double* d_ref, double* d_sums, float* d_gX, void* d_workspace, size_t ws_bytes, void* stream);
int ska_bone_length_f64(const double* d_X, int64_t T, int32_t J, const int32_t* bone_i, const int32_t* bone_j, int32_t n_bones,
                        const double* d_ref, double* d_sums, double* d_gX, void* d_workspace, size_t ws_bytes, void* stream);
int ska_camera_centre_f32(const float* d_R, const float* d_t, int64_t n, float* d_C, void* stream);
int ska_camera_centre_f64(const double* d_R, const double* d_t, int64_t n, double* d_C, void* stream);
int ska_camera_smooth_f32(const float* d_R, const float* d_t, int64_t D0, int64_t M, double* d_sum, float* d_gR, float* d_gt,
                          void* d_workspace, size_t ws_bytes, void* stream);
int ska_camera_smooth_f64(const double* d_R, const double* d_t, int64_t D0, int64_t M, double* d_sum, double* d_gR, double* d_gt,
                          void* d_workspace, size_t ws_bytes, void* stream);
int ska_baseline_reg_f32(const float* d_R, const float* d_t, int64_t T, int32_t C, const double* d_mean, double* d_sum,
                         float* d_gR, float* d_gt, void* d_workspace, size_t ws_bytes, void* stream);
int ska_baseline_reg_f64(const double* d_R, const double* d_t, int64_t T, int32_t C, const double* d_mean, double* d_sum,
                         double* d_gR, double* d_gt, void* d_workspace, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Bundle adjustment: Levenberg-Marquardt with Schur complement over a whole clip.
 * Fills the slot of the reference's undefined optimiser
 *   run_local_ba(K, R_init, t_init, X3d_init, x2d, conf2d, num_iters, lr, device, mode)
 *                                                       vggt/multi_view_process.py:553-564, :546-551
 * on the cost the reference does define:
 *   project_points + reprojection_loss                  bundle_adjustment/loss.py:17-94
 * Algorithm (oracle/lm.py is the fp64 specification): residual r = sqrt(conf/(sum conf + 1e-6)) (pi_c(X) - x2d),
 * pi = loss.py's projection (Z clamp at 1e-6, full 3x3 K); parameters = every point X (T,J,3) and, per
 * camera c >= 1, [d_omega(3), d_t(3)] with R <- exp([d_omega]x) R, t <- t + d_t (camera 0 is the gauge);
 * Marquardt damping lam*diag(H) on both blocks; Schur complement onto the cameras; Cholesky;
 * back-substitution; accept iff the cost decreases; Nielsen gain-ratio damping update.
 *
 * Robust loss (SkaBaProblem.loss / loss_scale; DESIGN.md section 5): with s = |pi_c(X) - x2d|^2 in px^2 and d > 0 the scale
 * in pixels, the cost becomes F = sum conf/(sum conf + 1e-6) rho(s) with
 *   SKA_BA_LOSS_L2      rho = s                                       omega = 1
 *   SKA_BA_LOSS_HUBER   rho = s if s <= d^2, else 2 d sqrt(s) - d^2   omega = 1 if s <= d^2, else d / sqrt(s)
 *   SKA_BA_LOSS_CAUCHY  rho = d^2 ln(1 + s / d^2)                     omega = 1 / (1 + s / d^2)
 * and the step is iteratively reweighted Gauss-Newton: every sum above uses the weight conf * omega(s), with omega
 * evaluated at the current state and not differentiated (the gradient is still exactly half that of F, so the gain
 * ratio and the accept rule keep their meaning).  A depth-clamped observation is weighted by omega of its error.  Huber
 * computes an inlier's rho and omega with the L2 expressions: a solve with every residual inside d is bit-identical to
 * L2.  The reduced-system layout does not change.  SKA_BA_TENSOR_CORE with a robust loss returns SKA_EUNSUPPORTED.
 *
 * One LM trial = ska_ba_linearize_f32 -> [all-reduce d_red over ranks] -> ska_ba_solve_f64 ->
 * ska_ba_backsub_f32 -> [all-reduce d_red2] -> ska_ba_control_f64.  Nothing synchronises with the host;
 * the sequence can be captured in a CUDA graph.  All state lives in caller-owned device buffers:
 */
#define SKA_BA_CAM_DOUBLES 24   /* per camera: R(9) row-major, t(3), K(9), pad(3) */
#define SKA_BA_CTRL_DOUBLES 16
#define SKA_BA_HIST_DOUBLES 8   /* iter, cost, trial_cost, lambda, rho, accepted, n_clamped, pred */
#define SKA_BA_RED2_DOUBLES 4   /* trial cost, predicted decrease of the points, clamped count, pad (unscaled sums) */
/* d_ctrl slots the caller initialises (all others 0): */
#define SKA_BA_CTRL_LAMBDA 0    /* initial damping, oracle default 1e-3 */
#define SKA_BA_CTRL_NU 1        /* 2.0 */
#define SKA_BA_CTRL_SUMCONF 2   /* global sum of conf over ALL ranks (ska_ba_sum_f32 + all-reduce) */
#define SKA_BA_CTRL_CUR 3       /* which half of d_Xpp holds the current points (0) */
#define SKA_BA_CTRL_ITER 4      /* next history row (0) */
#define SKA_BA_CTRL_COST 7      /* out: cost at the current point */
#define SKA_BA_CTRL_ACCEPTED 8  /* out: last decision */

#define SKA_BA_FORCE_WIDE 1u    /* flags: run the shared-memory SYRK linearisation even for C == 2 (testing) */
#define SKA_BA_LOSS_L2 0        /* SkaBaProblem.loss: plain squared pixel error (a zeroed struct) */
#define SKA_BA_LOSS_HUBER 1
#define SKA_BA_LOSS_CAUCHY 2
#define SKA_BA_TENSOR_CORE 2u   /* flags: 5..8 cameras: Schur accumulation on the tensor cores (tcgen05 kind::tf32, three-product split).
                                   Same reduced system to fp32 accuracy; measured SLOWER than the CUDA-core form on B200
                                   (26.3 vs 23.1 ms per 1M x 70 x 8 linearisation, profiles/README.md), hence opt-in */

struct SkaPeerComm;
typedef struct SkaBaProblem {
  int32_t C;            /* cameras, 2..SKA_MAX_VIEWS */
  int32_t J;            /* joints per frame */
  int64_t T;            /* frames of THIS rank's shard */
  int32_t layout;       /* SKA_LAYOUT_FRAME_MAJOR: x2d (T,C,J,2), conf (T,C,J) = loss.py's; or VIEW_MAJOR */
  uint32_t flags;
  const float* d_x2d;
  const float* d_conf;
  float* d_Xpp;         /* [2][T*J*3]: point ping-pong, half d_ctrl[CUR] is current */
  double* d_cams;       /* [2][C][SKA_BA_CAM_DOUBLES]: slot 0 current, slot 1 trial */
  double* d_ctrl;       /* [SKA_BA_CTRL_DOUBLES] */
  double* d_red;        /* [ska_ba_red_doubles(C)]: packed reduced system of this rank (all-reduce payload):
                           Sw upper triangle (n(n+1)/2, n = 6(C-1)), bw (n), gc (n), Hcc upper triangles (21 per
                           free camera), cost, clamped count - all sums with raw conf weights */
  double* d_red2;       /* [SKA_BA_RED2_DOUBLES] */
  double* d_delta;      /* [C*6] camera step of the current trial */
  double* d_hist;       /* nullable [hist_rows][SKA_BA_HIST_DOUBLES] */
  void* d_workspace;    /* >= ska_ba_workspace_bytes(C), 16-byte aligned */
  size_t ws_bytes;
  int64_t hist_rows;    /* rows of d_hist: trials beyond them still run, their history row is dropped */
  const struct SkaPeerComm* peer; /* nullable HOST pointer (see "exchange step" below).  Non-NULL: ska_ba_solve_f64 /
                           ska_ba_calib_solve_f64 all-reduce d_red over NVLink peer memory in their prologue and
                           ska_ba_control_f64 / ska_ba_calib_control_f64 do the same for d_red2 - exchange and consumer are ONE
                           kernel, and the caller runs no collective: linearize -> solve -> backsub -> control */
  int32_t loss;         /* SKA_BA_LOSS_*: read by the linearize and backsub entry points (solve and control ignore it) */
  double loss_scale;    /* robust scale d in pixels: finite and > 0 unless loss == SKA_BA_LOSS_L2 */
} SkaBaProblem;

int32_t ska_ba_red_doubles(int32_t C);
size_t ska_ba_workspace_bytes(int32_t C);
/* d_out[0] = sum of x[0..count) in fp64, fixed summation order (sum of confidences) */
int ska_ba_sum_f32(const float* d_x, int64_t count, double* d_out, void* d_workspace, size_t ws_bytes, void* stream);
int ska_ba_linearize_f32(const SkaBaProblem* p, void* stream);
/* free_mask: bit (6*c + r) set = parameter r of camera c is optimised (r: 0..2 d_omega, 3..5 d_t);
 * bits of camera 0 are ignored (gauge).  Modes of vggt/multi_view_process.py:338. */
int ska_ba_solve_f64(const SkaBaProblem* p, uint64_t free_mask, void* stream);
int ska_ba_backsub_f32(const SkaBaProblem* p, void* stream);
int ska_ba_control_f64(const SkaBaProblem* p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CALIBRATING bundle adjustment: the same LM with every camera's intrinsics and distortion free as well
 * (BASELINE config 3: "2 cameras, Rodrigues extrinsics + intrinsics/distortion"; specification: oracle/lm_calib.py).
 * Projection = cv2.projectPoints' 5-coefficient model the reference reprojects with
 * (triangulation/reproject.py:77-78, bundle_adjustment/reproject.py:147-148) + loss.py's depth clamp (:67):
 *   x = X_c.x/Z, y = X_c.y/Z, r2 = x^2 + y^2, rad = 1 + k1 r2 + k2 r2^2 + k3 r2^3
 *   u = fx (x rad + 2 p1 x y + p2 (r2 + 2 x^2)) + cx,   v = fy (y rad + p1 (r2 + 2 y^2) + 2 p2 x y) + cy
 * Observations with depth < 1e-6 (loss.py:67's clamp threshold) are EXCLUDED (zero weight, counted): the polynomial
 * distortion of a clamped projection overflows fp32.
 * 15 parameters per camera: [d_omega(3), d_t(3), fx, fy, cx, cy, k1, k2, p1, p2, k3]; camera 0's extrinsics are the gauge.
 * Cost = loss.py's confidence-weighted mean squared error under that projection
 *        + sum_c sum_k rho_ck (theta_ck - theta0_ck)^2   (optional Gaussian prior on the 9 intrinsics; d_prior).
 * The SkaBaProblem fields keep their meaning except:
 *   d_cams  [2][C][SKA_BA_CAM_DOUBLES]: R(9), t(3), theta(9) = fx fy cx cy k1 k2 p1 p2 k3, pad(3)
 *   d_delta [C * SKA_BA_CALIB_PARAMS]
 *   d_red   [ska_ba_calib_red_doubles(C)]: upper triangle of Sw (n(n+1)/2, n = 15 C - 6: camera 0 contributes its 9
 *           intrinsics only), then per camera 160 doubles: the row-major upper triangle (153) of sum w row^T row with
 *           row = [B(15) | e | a.dp0] - entries (r,s<=14) Hcc, (r,15) gc, (r,16) bw, (15,15) sum w omega s - in slot 153,
 *           the count of depth-clamped observations, and in slot 154 the robust cost correction sum w (rho(s) - omega s)
 *           (0 under L2; the data cost is (15,15) + slot 154); all sums with raw conf weights
 * The robust loss applies as above; depth-clamped observations stay excluded.
 *   d_workspace >= ska_ba_calib_workspace_bytes(C)
 * free_mask: bit (15*c + r) set = parameter r of camera c is optimised (bits 0..5 of camera 0 are ignored).
 * d_prior: nullable [C][18] = theta0(9), rho(9) per camera.
 * Built for C == 2 (config 3); other camera counts return SKA_EUNSUPPORTED.  One trial = linearize ->
 * [all-reduce d_red] -> solve -> backsub -> [all-reduce d_red2] -> control, as above. */
#define SKA_BA_CALIB_PARAMS 15
#define SKA_BA_CALIB_INTRINSICS 9
#define SKA_BA_CALIB_CAM_BLOCK 160
int32_t ska_ba_calib_red_doubles(int32_t C);
size_t ska_ba_calib_workspace_bytes(int32_t C);
int ska_ba_calib_linearize_f32(const SkaBaProblem* p, void* stream);
int ska_ba_calib_solve_f64(const SkaBaProblem* p, uint64_t free_mask, const double* d_prior, void* stream);
int ska_ba_calib_backsub_f32(const SkaBaProblem* p, void* stream);
int ska_ba_calib_control_f64(const SkaBaProblem* p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Regularised bundle adjustment: Levenberg-Marquardt over the reference's FULL configured objective (SURVEY rows N1, e3)
 *     w_r reprojection_loss + w_s camera_smooth_loss + w_b baseline_reg_loss + w_l bone_length_loss + w_t pose_temporal_loss
 *     (bundle_adjustment/loss.py:90-94, :103-106, :109-114, :134-150, :153-155; weights configs/vggt.yaml:46-50)
 * with PER-FRAME cameras as the call site passes them (vggt/multi_view_process.py:546-564) - the second-order form of the
 * optimiser the reference calls but never defines (run_local_ba).  Specification: oracle/lm_reg.py.  All fp64.
 * The damped normal equations (J^T J + lambda diag(J^T J)) delta = -J^T r are solved matrix-free by conjugate gradients,
 * preconditioned with each frame's exact reprojection system (Schur complement onto the frame's cameras).
 *
 * Frames are rows; every per-frame array carries ONE HALO ROW on each side (row 0 = the frame before this rank's first,
 * row T_local + 1 = the frame after its last), which the CALLER fills from the neighbouring ranks when the clip is sharded
 * by frame range (has_prev / has_next say whether those frames exist).  free_mask: bits 0..5 = [d_omega(3), d_t(3)] of
 * EVERY camera of every frame are optimised ("pose_only" 0, "pose_cam_t" 0x38, "full" 0x3f; multi_view_process.py:338).
 *   d_x2d (T_local,C,J,2) f32, d_conf (T_local,C,J) f32, d_K (C,9) f64
 *   d_X    [2][T_local+2][J][3]   current / trial points (d_sc[SKA_BA_REG_SC_CUR] says which half is current)
 *   d_cams [2][T_local+2][C][12]  R (9, row-major), t (3)
 *   d_vec  [SKA_BA_REG_NVEC][T_local+2][3J+6C]: g, D, x (the step), r, z, p, y   - rows [J x xyz | C x (d_omega, d_t)]
 *   d_pinv [T_local][J][6]; d_lfac [T_local][3C(6C+1)] (nullable when free_mask == 0)
 *   d_sc   [SKA_BA_REG_SC_DOUBLES]: the caller sets CUR = 0, LAMBDA (1e-3), NU = 2, ITER = 0, TOL2 (squared relative CG
 *          tolerance, 1e-16), COEF[5] = c_r c_l c_t c_s c_b (oracle/lm_reg.py coefficients()) and T_GLOBAL
 *   d_sums [2][SKA_BA_REG_SUMS]: raw sums of the current / the trial point (the multi-GPU all-reduce payloads)
 *   d_hist nullable [hist_rows][SKA_BA_REG_HIST_DOUBLES]: iter, cost, trial_cost, lambda, rho, accepted, n_clamped, pred,
 *          cg_iters, reproj, smooth, baseline, bone_length, pose_temporal (terms of `cost`), final CG residual, pad
 * One LM trial:
 *   [set-up only: ska_ba_reg_cost_f64(p, 0) -> all-reduce d_sums[0] -> ska_ba_reg_finish_cost_f64(p, 0)]
 *   ska_ba_reg_linearize_f64
 *   ska_ba_reg_cg_f64(BEGIN) -> [all-reduce d_sc[DOT]] -> cg(INIT) -> cg(DIR)
 *   repeat: [halo exchange of p] cg(MATVEC) -> [all-reduce DOT] -> cg(ALPHA) -> cg(UPDATE) -> [all-reduce DOT] -> cg(BETA) -> cg(DIR)
 *           (a fixed number of times: once converged every kernel returns at once - no host round trip)
 *   ska_ba_reg_apply_f64 -> [halo exchange of the trial X / cameras] -> ska_ba_reg_cost_f64(p, 1) -> [all-reduce d_sums[1]]
 *   -> ska_ba_reg_finish_cost_f64(p, 1) -> ska_ba_reg_control_f64
 *
 * Robust loss (ska_ba_reg_{cost,linearize,cg}_robust_f64; `loss` = SKA_BA_LOSS_*, `loss_scale` = d in pixels): rho and omega
 * as in the Schur-LM section above, on the REPROJECTION group only.  Its term becomes c_r sum conf rho(s), s = e_u^2 + e_v^2
 * (c_r still from the raw sum of conf); bone length, pose temporal, smoothness and baseline stay squared.  The step is
 * iteratively reweighted Gauss-Newton: every reprojection contribution to g, D, the matrix-vector product and the frame
 * preconditioner uses the weight c_r conf omega(s), omega at the current point and not differentiated, so g is still half
 * the gradient of F and the predicted decrease, the gain ratio and the accept rule keep their meaning.  Depth-clamped
 * observations keep their residual and are weighted by omega of it.  d_sums' reprojection column, the history's `reproj`
 * and `cost` are the robust values; the clamp count is unchanged.  Huber computes an inlier with the L2 expressions: a
 * solve with every residual inside d is bit-identical to L2.
 *   - The loss and scale must be the same for every call of a trial (the kernels recompute omega from the observations
 *     instead of storing it, so the linearisation and the CG operators agree bit for bit only then).
 *   - cg ops that read no observations (INIT, ALPHA, BETA, DIR, and BEGIN / UPDATE with free_mask == 0) ignore it.
 *   - An unknown loss, or for a robust loss a scale that is not finite and > 0 with d^2 a normal fp64 number, returns
 *     SKA_EINVAL before any CUDA call.
 * ska_ba_reg_cost_f64 / _linearize_f64 / _cg_f64 are the robust entry points with SKA_BA_LOSS_L2. */
#define SKA_BA_REG_NVEC 7
#define SKA_BA_REG_SUMS 40
#define SKA_BA_REG_SC_DOUBLES 64
#define SKA_BA_REG_HIST_DOUBLES 16
#define SKA_BA_REG_SC_CUR 0
#define SKA_BA_REG_SC_LAMBDA 1
#define SKA_BA_REG_SC_NU 2
#define SKA_BA_REG_SC_ITER 3
#define SKA_BA_REG_SC_COST 4
#define SKA_BA_REG_SC_ACCEPTED 7
#define SKA_BA_REG_SC_TOL2 15
#define SKA_BA_REG_SC_COEF 16
#define SKA_BA_REG_SC_T_GLOBAL 21
#define SKA_BA_REG_SC_DOT 47
#define SKA_BA_REG_CG_BEGIN 0
#define SKA_BA_REG_CG_INIT 1
#define SKA_BA_REG_CG_MATVEC 2
#define SKA_BA_REG_CG_ALPHA 3
#define SKA_BA_REG_CG_UPDATE 4
#define SKA_BA_REG_CG_BETA 5
#define SKA_BA_REG_CG_DIR 6
typedef struct SkaBaRegProblem {
  int32_t C, J, n_bones;
  uint32_t free_mask;
  int64_t T_local;
  int32_t has_prev, has_next;
  int32_t bone_i[SKA_MAX_BONES], bone_j[SKA_MAX_BONES];
  const float* d_x2d;
  const float* d_conf;
  const double* d_K;
  double* d_X;
  double* d_cams;
  double* d_vec;
  double* d_pinv;
  double* d_lfac;
  double* d_sc;
  double* d_sums;
  double* d_hist;
  int64_t hist_rows;
  void* d_workspace;
  size_t ws_bytes;
  const struct SkaPeerComm* peer; /* nullable HOST pointer: non-NULL = ska_ba_reg_finish_cost_f64 all-reduces d_sums[which] and
                                     ska_ba_reg_cg_f64(INIT / ALPHA / BETA) all-reduce d_sc[DOT] over NVLink peer memory in their own
                                     prologue (the caller then runs no collective for them; the halo all-gathers stay the caller's) */
} SkaBaRegProblem;
size_t ska_ba_reg_workspace_bytes(int64_t T_local);
int ska_ba_reg_cost_f64(const SkaBaRegProblem* p, int32_t which, void* stream);
int ska_ba_reg_finish_cost_f64(const SkaBaRegProblem* p, int32_t which, void* stream);
int ska_ba_reg_linearize_f64(const SkaBaRegProblem* p, void* stream);
int ska_ba_reg_cg_f64(const SkaBaRegProblem* p, int32_t op, void* stream);
int ska_ba_reg_apply_f64(const SkaBaRegProblem* p, void* stream);
int ska_ba_reg_control_f64(const SkaBaRegProblem* p, void* stream);
int ska_ba_reg_cost_robust_f64(const SkaBaRegProblem* p, int32_t which, int32_t loss, double loss_scale, void* stream);
int ska_ba_reg_linearize_robust_f64(const SkaBaRegProblem* p, int32_t loss, double loss_scale, void* stream);
int ska_ba_reg_cg_robust_f64(const SkaBaRegProblem* p, int32_t op, int32_t loss, double loss_scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The exchange step of the sharded solvers over NVLink peer memory (SURVEY row e: the NCCL all-reduce of the packed
 * reduced system / the trial scalars / the CG dot products, and the all-gather of the one-frame halos, replaced by one
 * single-CTA kernel per exchange).  Every rank pushes its payload into every peer's receive area with plain 8-byte stores
 * (each word tagged with the exchange number), polls its own words and sums (all-reduce, fixed rank order: bit-identical on every
 * rank) or copies (all-gather) the world's payloads.  One process per GPU on one node; fp64 payloads of at most
 * `slot_doubles`.  Set-up (host, once): ska_peer_alloc a region of ska_peer_region_bytes(world, slot_doubles)
 * (cudaMalloc: IPC-exportable; zero-filled), ska_peer_export its 64-byte handle, exchange the handles (e.g.
 * torch.distributed.all_gather_object), ska_peer_import the peers' regions, fill SkaPeerComm:
 *   recv[r]  = region_r   [2][world][slot_doubles][2] 64-bit words: every double travels as {low half | exchange number} and
 *              {high half | exchange number}, so a word is its own arrival flag (no fence, no separate flag round trip)
 *   flags[r] = unused (reserved)
 *   d_state  = local [2] uint64 (zero): exchange counter, and the number of the first exchange that timed out (0 = none:
 *              a peer that never arrives makes the kernel give up after 2^poll_limit_log2 polls instead of hanging the GPU)
 * Every rank must issue the same sequence of exchanges.  Enqueues on `stream`; capturable in a CUDA graph. */
#define SKA_MAX_PEERS 8
typedef struct SkaPeerComm {
  int32_t world, rank, slot_doubles;
  int32_t poll_limit_log2; /* 0 = default (24) */
  double* recv[SKA_MAX_PEERS];
  uint64_t* flags[SKA_MAX_PEERS];
  uint64_t* d_state;
  const double* d_skip; /* nullable: a device flag that is IDENTICAL on every rank (e.g. the CG convergence flag computed from
                           all-reduced scalars); non-zero = every rank skips this exchange */
} SkaPeerComm;
size_t ska_peer_region_bytes(int32_t world, int32_t slot_doubles);
int ska_peer_alloc(size_t bytes, void** d_ptr);
int ska_peer_free(void* d_ptr);
int ska_peer_export(void* d_ptr, unsigned char* handle64);
int ska_peer_import(const unsigned char* handle64, void** d_ptr);
int ska_peer_close(void* d_ptr);
int ska_peer_allreduce_f64(const SkaPeerComm* comm, double* d_buf, int32_t n, void* stream);
int ska_peer_allgather_f64(const SkaPeerComm* comm, const double* d_in, int32_t n, double* d_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Post-triangulation triage and temporal smoothing (the step right after the path; SURVEY row N2).
 * Replaces post_triage_single / post_triage_sequence and smooth_skeleton of
 * triangulation/postprocess.py:54-170 for a whole clip.
 *
 * ska_post_triage_f32: cams[2] host (cam 0 = K1 [I|0] in the reference, cam 1 = K2 [R|T]; any world->camera
 *   pair is accepted); d_X (T,J,3); d_kpts (2,T,J,2) view-major; d_conf (2,T,J) nullable.
 *   flags: SKA_TRIAGE_UNDISTORT0/1 = undistort that view's pixels with cams[v].dist first
 *   (cv2.undistortPoints(x, K, d, P=K): 5 fixed-point iterations, float32 result, postprocess.py:93-98).
 *   A joint is kept iff depth > 0 in both cameras (:47-52), 0.5 (e1 + e2) is finite and <= err_thresh_px (:112)
 *   and both confidences >= conf_thr (:108-110).  Outputs: d_Xclean (T,J,3) = X or NaN (:115-116);
 *   d_em (T,J) mean pixel error, nullable; d_flags (T,J) nullable: SKA_TRIAGE_POS | _ERR | _CONF | _KEEP.
 * ska_frame_flag_counts_u8: d_counts (T,4) int32, 16-byte aligned = per-frame count of each of the four flag bits
 *   (pos_depth_ratio, kept_ratio, kept_count of :118-124; rmse / median of d_em via ska_frame_stats_f32, V = 1).
 * ska_savgol_f32: Savitzky-Golay (scipy.signal.savgol_filter, mode="interp") along T for each of the S = J*3
 *   series of d_X (T,S), over the series' FINITE samples only (compacted in time, filtered, scattered back;
 *   non-finite entries stay; series with fewer finite samples than `win` pass through) - smooth_skeleton :54-68.
 *   win odd <= 25, poly < win.  d_workspace >= ska_savgol_workspace_bytes(T, S).  d_out may not alias d_X. */
#define SKA_TRIAGE_UNDISTORT0 1u
#define SKA_TRIAGE_UNDISTORT1 2u
#define SKA_TRIAGE_POS 1
#define SKA_TRIAGE_ERR 2
#define SKA_TRIAGE_CONF 4
#define SKA_TRIAGE_KEEP 8
int ska_post_triage_f32(const SkaCamera* cams, const float* d_X, const float* d_kpts, const float* d_conf, int64_t T, int32_t J,
                        uint32_t flags, double conf_thr, double err_thresh_px, float* d_Xclean, float* d_em, uint8_t* d_flags,
                        void* stream);
int ska_frame_flag_counts_u8(const uint8_t* d_flags, int64_t T, int32_t J, int32_t* d_counts, void* stream);
size_t ska_savgol_workspace_bytes(int64_t T, int32_t S);
int ska_savgol_f32(const float* d_X, int64_t T, int32_t S, int32_t win, int32_t poly, float* d_out, void* d_workspace,
                   size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Two-view 3D-3D fusion of monocular pose estimates + adaptive EMA smoothing (SURVEY row N3), whole clip per call.
 * Replaces the per-frame numpy of the reference's `fuse` pipeline (fuse/main_raw.py:199-250):
 *   _align_right_to_left (Kabsch, main_raw.py:48-95) -> weakpersp_reproj_confidence per view (fuse/confidence.py:9-108)
 *   -> crossview_consistency_confidence (confidence.py:118-224) -> q = sqrt(conf1 * conf2) -> fuse_frame_3d
 *   (softmax2 weights, fuse/fuse.py:87-94, 289-326); then temporal_smooth_ema (fuse/fuse.py:329-412).
 * All arrays are fp64 device arrays (the reference computes in numpy float64); a missing joint is a NaN row.
 * ska_fuse_frames_f64: d_Xl, d_Xr (T,J,3) per-view 3D in each view's own frame; d_Ul, d_Ur (T,J,2) pixels; J <= 96.
 *   d_fused (T,J,3); nullable d_ql, d_qr (T,J), d_aligned (T,J,3) = right view in the left frame, d_status (T,) bit set:
 *   SKA_FUSE_NO_ALIGN (fewer than 3 common joints: right view used unaligned, main_raw.py:83-84),
 *   SKA_FUSE_FIT_LEFT_FAILED / _RIGHT_FAILED (weak-perspective fit impossible: the reference raises ValueError,
 *   confidence.py:31-32,52-53; the frame's outputs are NaN).  d_workspace >= ska_fuse_workspace_bytes(T) (56 doubles per
 *   frame: the frame's raw moments, then its alignment / fit / canonical-frame parameters), 8-byte aligned; three launches:
 *   moments (warp per frame) -> parameters (thread per frame) -> fusion (thread per joint).
 * ska_ema_f64: d_X (T,J,3) -> d_Y (T,J,3) (may not alias); d_alpha_joint (J,) per-joint base alpha (fuse.py:362-376);
 *   adaptive != 0: alpha_t = clip(alpha_joint + speed_gain |x_t - y_{t-1}|, alpha_min, alpha_max), else the fixed `alpha`.
 *   Frames are processed in chunks of `chunk` frames, each replaying `halo` finite samples before its start; halo < 0
 *   (or chunk >= T) runs the exact sequential scan.  The recurrence contracts by rho = max(1 - alpha_min,
 *   |1 + alpha_min - 2 alpha_max|) per step, so halo >= log(1e-18) / log(rho) reproduces the sequential result to below
 *   fp64 rounding. */
typedef struct SkaFuseParams {
  double sigma_px;     /* 12.0  (main_raw.py:133) */
  double sigma_3d;     /* 0.08  (main_raw.py:134) */
  int32_t scale_mode;  /* 0 = "hip", 1 = "torso" (confidence.py:170-175) */
  int32_t min_points;  /* 8     (confidence.py:12) */
  int32_t root, lhip, rhip, lsho, rsho; /* 14, 11, 12, 5, 6 (main_raw.py:18-22) */
  int32_t pad_;        /* flags: bit 0 = always take the Jacobi SVD path of the rigid alignment (test hook);
                          bit 1 = skip the rigid alignment (views already in one frame: fuse/main_unity.py:96-132);
                          bit 2 = run the single warp-per-frame kernel (no workspace) instead of the three-stage path (A/B testing) */
} SkaFuseParams;
#define SKA_FUSE_NO_ALIGN 1
#define SKA_FUSE_FIT_LEFT_FAILED 2
#define SKA_FUSE_FIT_RIGHT_FAILED 4
size_t ska_fuse_workspace_bytes(int64_t T);
int ska_fuse_frames_f64(const double* d_Xl, const double* d_Xr, const double* d_Ul, const double* d_Ur, int64_t T, int32_t J,
                        const SkaFuseParams* prm, double* d_fused, double* d_ql, double* d_qr, double* d_aligned,
                        uint8_t* d_status, void* d_workspace, size_t ws_bytes, void* stream);
/* ska_rigid_fuse_f64: rigid_transform_3D of bundle_adjustment/fuse/fuse.py:96-232 (== fuse/side/fuse/fuse.py,
 *   front_side/side/fuse/fuse.py; called at bundle_adjustment/run.py:225) for a whole clip.  d_L (target / left), d_R
 *   (source / right) (T,J,3) fp64, NaN rows = missing.  Per frame: Umeyama alignment s R x + t of the right view onto the
 *   left from the joints torso5 (HOST array of 5 indices; fuse.py:27-31 uses 69, 9, 10, 5, 6) exactly as
 *   estimate_rigid_umeyama does (fuse_check.py:26-78: cross-covariance / N, det-fixed rotation, s = sum(S) / (var + 1e-12)
 *   when allow_scale, else 1), then per joint (fuse.py:55-93): one view missing -> the other; both present and farther
 *   apart than tau (d_tau_j (J,) if not NULL, else the scalar) -> the view with the larger weight (left on ties); else the
 *   weighted mean / (wL + wR + 1e-9).  d_wL / d_wR nullable (weights 1): (T,J) with w_frame_stride = J or (J,) with 0.
 *   Outputs: d_fused (T,J,3); d_Rts (T,13) = R (9, row-major), t (3), s; nullable d_diag (T,4) = LR_before, Fused_vs_L,
 *   Fused_vs_R, gain (plain means over the joints: NaN if one is missing, like the reference); nullable d_status (T,):
 *   1 = fewer than 3 usable torso joints (the reference raises ValueError; that frame's d_Rts is NaN). */
int ska_rigid_fuse_f64(const double* d_L, const double* d_R, int64_t T, int32_t J, const int32_t* torso5, double tau,
                       const double* d_tau_j, int32_t allow_scale, const double* d_wL, const double* d_wR, int64_t w_frame_stride,
                       double* d_fused, double* d_Rts, double* d_diag, uint8_t* d_status, void* stream);
int ska_ema_f64(const double* d_X, int64_t T, int32_t J, const double* d_alpha_joint, int32_t adaptive, double alpha,
                double alpha_min, double alpha_max, double speed_gain, int64_t chunk, int32_t halo, double* d_Y, void* stream);

/* ------------------------------------------------------------------------------------------------
 * First-order (Adam) form of the regularised bundle adjustment (SURVEY row N1): the update kernels.  The objective
 *   w_reproj * reprojection_loss + w_smooth * camera_smooth_loss + w_baseline * baseline_reg_loss
 *   + w_bone_length * bone_length_loss + w_pose_temporal * pose_temporal_loss      (bundle_adjustment/loss.py:90-155)
 * with the weights, `lr` and `num_iters` of configs/vggt.yaml:43-52 and per-frame cameras (vggt/multi_view_process.py:546-564)
 * is evaluated, value and analytic gradient, by the loss entry points above; these three apply the step
 * (specification: oracle/first_order.py).
 *   ska_adam_step_*: torch.optim.Adam's update on n elements: m <- m + (1-beta1)(g-m); v <- beta2 v + (1-beta2) g^2;
 *       step = step_size * m / (sqrt(v) * inv_sqrt_bc2 + eps), step_size = lr / (1 - beta1^k), inv_sqrt_bc2 = 1 / sqrt(1 - beta2^k);
 *       d_p (nullable) <- d_p - step; d_step_out (nullable) <- step.  d_scalars (nullable): device [2] = {step_size,
 *       inv_sqrt_bc2} overriding the by-value arguments, so a captured CUDA graph of one iteration replays for every k.
 *   ska_so3_tangent_grad_*: n rotations (row-major 3x3) and dL/dR -> gradient w.r.t. the left tangent of R = exp([w]x) R.
 *   ska_so3_retract_*: R <- exp([-step]x) R. */
int ska_adam_step_f32(float* d_p, const float* d_g, float* d_m, float* d_v, int64_t n, double step_size, double beta1, double beta2,
                      double eps, double inv_sqrt_bc2, float* d_step_out, const double* d_scalars, void* stream);
int ska_adam_step_f64(double* d_p, const double* d_g, double* d_m, double* d_v, int64_t n, double step_size, double beta1, double beta2,
                      double eps, double inv_sqrt_bc2, double* d_step_out, const double* d_scalars, void* stream);
/* the same update with the gradient given as up to three UNSCALED terms, g = s0 g0 + s1 g1 + s2 g2 (d_g1 / d_g2 nullable):
 * the loss entry points return gradients of their raw sums, the weights / counts are folded in here; step_size and
 * inv_sqrt_bc2 always come from d_scalars. */
int ska_adam_step_terms_f32(float* d_p, const float* d_g0, double s0, const float* d_g1, double s1, const float* d_g2, double s2,
                            float* d_m, float* d_v, int64_t n, double beta1, double beta2, double eps, float* d_step_out,
                            const double* d_scalars, void* stream);
int ska_adam_step_terms_f64(double* d_p, const double* d_g0, double s0, const double* d_g1, double s1, const double* d_g2, double s2,
                            double* d_m, double* d_v, int64_t n, double beta1, double beta2, double eps, double* d_step_out,
                            const double* d_scalars, void* stream);
/* scalar bookkeeping of one first-order iteration in one launch: d_hist[k] (6 doubles per row, nullable, max_rows rows) =
 * [total, coef5[0] * sums5[0][0] / (d_den[0] + 1e-6) (d_den NULL: no division), coef5[q] * sums5[q][0] for q = 1..4] where
 * sums5 / coef5 are HOST arrays of 5 device pointers (NULL = term off) / 5 coefficients in the order reproj, smooth,
 * baseline, bone_length, pose_temporal; then d_k[0] <- k + 1 and d_scal = {lr / (1 - beta1^k), 1 / sqrt(1 - beta2^k)}. */
int ska_first_order_record_f64(double* d_k, double* d_scal, double* d_hist, int64_t max_rows, const double* const* sums5,
                               const double* d_den, const double* coef5, double lr, double beta1, double beta2, void* stream);
int ska_so3_tangent_grad_f32(const float* d_R, const float* d_gR, int64_t n, float* d_gw, void* stream);
int ska_so3_tangent_grad_f64(const double* d_R, const double* d_gR, int64_t n, double* d_gw, void* stream);
int ska_so3_retract_f32(float* d_R, const float* d_step, int64_t n, void* stream);
int ska_so3_retract_f64(double* d_R, const double* d_step, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SKA_H_ */
