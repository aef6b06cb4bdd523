// ska_capi.cu - the extern "C" boundary of libska.so: argument validation and dispatch only.
#include <cuda_runtime.h>
#include <float.h>
#include <stdio.h>
#include <string.h>

#include "ska_internal.h"

namespace ska {

static thread_local char g_err[512] = "";

int set_error(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg ? msg : "");
  return code;
}

}  // namespace ska

using namespace ska;

extern "C" {
#pragma GCC visibility push(default)

int ska_abi_version(void) { return SKA_ABI_VERSION; }
const char* ska_last_error(void) { return g_err; }
const char* ska_build_arch(void) { return "sm_100a"; }

static int check_tri_common(const SkaCamera* cams, int32_t V, const float* d_kpts, const float* d_conf, int64_t T, int32_t J,
                            int32_t layout, uint32_t flags, float* d_X, float* d_err, float* d_proj) {
  if (cams == nullptr || d_kpts == nullptr || d_X == nullptr) return set_error(SKA_EINVAL, "cams, d_kpts and d_X must not be NULL");
  if (V < 2 || V > SKA_MAX_VIEWS) return set_error(SKA_EINVAL, "V must be in 2..SKA_MAX_VIEWS");
  if (T < 0 || J < 1) return set_error(SKA_EINVAL, "T must be >= 0 and J >= 1");
  if (layout != SKA_LAYOUT_VIEW_MAJOR && layout != SKA_LAYOUT_FRAME_MAJOR) return set_error(SKA_EINVAL, "bad layout");
  if ((flags & SKA_SOLVER_MASK) == 3u) return set_error(SKA_EINVAL, "bad solver");
  if (T * (int64_t)J >= (int64_t)1 << 31) return set_error(SKA_EINVAL, "T*J must be < 2^31 per call; shard the clip");
  auto al = [](const void* p, uintptr_t n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; };
  if (!al(d_kpts, 8) || !al(d_proj, 8)) return set_error(SKA_EALIGN, "d_kpts / d_proj must be 8-byte aligned");
  if (!al(d_conf, 4) || !al(d_err, 4) || !al(d_X, 4)) return set_error(SKA_EALIGN, "float pointers must be 4-byte aligned");
  return SKA_OK;
}

int ska_triangulate_reproject_f32(const SkaCamera* cams, int32_t V, const double* centre, const float* d_kpts,
                                  const float* d_conf, int64_t T, int32_t J, int32_t layout, uint32_t flags, float* d_X,
                                  float* d_err, float* d_proj, uint8_t* d_status, void* stream) {
  const int rc = check_tri_common(cams, V, d_kpts, d_conf, T, J, layout, flags, d_X, d_err, d_proj);
  if (rc != SKA_OK) return rc;
  if (T == 0) return SKA_OK;
  TriArgs a;
  a.cams = cams;
  a.V = V;
  if (centre != nullptr) {
    for (int k = 0; k < 3; ++k) {
      if (!isfinite(centre[k])) return set_error(SKA_EINVAL, "centre must be finite");
      a.centre[k] = (double)(float)centre[k];
    }
  } else {
    default_centre(cams, V, a.centre);
  }
  a.Rt_frames = nullptr;
  a.kpts = d_kpts;
  a.conf = d_conf;
  a.T = T;
  a.J = J;
  a.layout = layout;
  a.flags = flags;
  a.X = d_X;
  a.err = d_err;
  a.proj = d_proj;
  a.status = d_status;
  a.stream = stream;
  a.workspace = nullptr;
  a.ws_bytes = 0;
  return triangulate_dispatch(a);
}

size_t ska_tri_frames_workspace_bytes(int32_t V, int64_t T) {
  if (V < 2 || V > SKA_MAX_VIEWS || T < 0) return 0;
  return tri_frames_workspace(V, T);
}

int ska_triangulate_reproject_frames_f32(const SkaCamera* cams, int32_t V, const double* d_Rt_frames, const float* d_kpts,
                                         const float* d_conf, int64_t T, int32_t J, int32_t layout, uint32_t flags,
                                         float* d_X, float* d_err, float* d_proj, uint8_t* d_status, void* d_workspace,
                                         size_t ws_bytes, void* stream) {
  const int rc = check_tri_common(cams, V, d_kpts, d_conf, T, J, layout, flags, d_X, d_err, d_proj);
  if (rc != SKA_OK) return rc;
  if (T == 0) return SKA_OK;
  if (d_Rt_frames == nullptr) return set_error(SKA_EINVAL, "d_Rt_frames must not be NULL");
  if (reinterpret_cast<uintptr_t>(d_Rt_frames) % 8 != 0) return set_error(SKA_EALIGN, "d_Rt_frames must be 8-byte aligned");
  TriArgs a;
  a.cams = cams;
  a.V = V;
  a.centre[0] = a.centre[1] = a.centre[2] = 0.0;
  a.Rt_frames = d_Rt_frames;
  a.kpts = d_kpts;
  a.conf = d_conf;
  a.T = T;
  a.J = J;
  a.layout = layout;
  a.flags = flags;
  a.X = d_X;
  a.err = d_err;
  a.proj = d_proj;
  a.status = d_status;
  a.stream = stream;
  a.workspace = d_workspace;
  a.ws_bytes = ws_bytes;
  return triangulate_dispatch(a);
}

int ska_reproject_points_f32(const SkaCamera* cams, int32_t V, const float* d_X, const float* d_kpts, int64_t T, int32_t J,
                             int32_t layout, float* d_proj, float* d_err, void* stream) {
  if (cams == nullptr || d_X == nullptr) return set_error(SKA_EINVAL, "cams and d_X must not be NULL");
  if (V < 1 || V > SKA_MAX_VIEWS) return set_error(SKA_EINVAL, "V must be in 1..SKA_MAX_VIEWS");
  if (T < 0 || J < 1) return set_error(SKA_EINVAL, "T must be >= 0 and J >= 1");
  if (layout != SKA_LAYOUT_VIEW_MAJOR && layout != SKA_LAYOUT_FRAME_MAJOR) return set_error(SKA_EINVAL, "bad layout");
  if (d_err != nullptr && d_kpts == nullptr) return set_error(SKA_EINVAL, "d_err needs d_kpts");
  if (d_proj == nullptr && d_err == nullptr) return set_error(SKA_EINVAL, "nothing to compute: d_proj and d_err are both NULL");
  auto al = [](const void* p, uintptr_t n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; };
  if (!al(d_kpts, 8) || !al(d_proj, 8)) return set_error(SKA_EALIGN, "d_kpts / d_proj must be 8-byte aligned");
  if (T == 0) return SKA_OK;
  return project_cv(cams, V, d_X, d_kpts, T, J, layout, d_proj, d_err, (cudaStream_t)stream);
}

int ska_frame_stats_f32(const float* d_err, int64_t T, int32_t J, int32_t V, int32_t layout, float* d_stats, void* stream) {
  if (T < 0 || J < 1 || V < 1) return set_error(SKA_EINVAL, "T >= 0, J >= 1, V >= 1");
  if (layout != SKA_LAYOUT_VIEW_MAJOR && layout != SKA_LAYOUT_FRAME_MAJOR) return set_error(SKA_EINVAL, "bad layout");
  if (T == 0) return SKA_OK;
  if (d_err == nullptr || d_stats == nullptr) return set_error(SKA_EINVAL, "d_err and d_stats must not be NULL");
  return frame_stats(d_err, T, J, V, layout, d_stats, (cudaStream_t)stream);
}

// ---- loss.py entry points: thin typed wrappers over the templates
#define SKA_LOSS_CHECK()                                                                                     \
  do {                                                                                                       \
    if (T < 0 || J < 1 || C < 1) return set_error(SKA_EINVAL, "T >= 0, J >= 1, C >= 1");                     \
    if (T > 0 && (d_X == nullptr || d_R == nullptr || d_t == nullptr || d_K == nullptr))                     \
      return set_error(SKA_EINVAL, "d_X, d_R, d_t and d_K must not be NULL");                                \
    if (R_frame_stride != 0 && R_frame_stride != 9 * (int64_t)C) return set_error(SKA_EINVAL, "R frame stride must be 0 or 9*C"); \
    if (t_frame_stride != 0 && t_frame_stride != 3 * (int64_t)C) return set_error(SKA_EINVAL, "t frame stride must be 0 or 3*C"); \
    if (K_frame_stride != 0 && K_frame_stride != 9 * (int64_t)C) return set_error(SKA_EINVAL, "K frame stride must be 0 or 9*C"); \
  } while (0)

#define SKA_DEFINE_LOSS(SFX, S)                                                                                                   \
  int ska_project_points_##SFX(const S* d_X, int64_t T, int32_t J, int32_t C, const S* d_R, int64_t R_frame_stride, const S* d_t, \
                               int64_t t_frame_stride, const S* d_K, int64_t K_frame_stride, S* d_out, void* stream) {            \
    SKA_LOSS_CHECK();                                                                                                             \
    if (T > 0 && d_out == nullptr) return set_error(SKA_EINVAL, "d_out must not be NULL");                                        \
    return project_points<S>(d_X, T, J, C, d_R, R_frame_stride, d_t, t_frame_stride, d_K, K_frame_stride, d_out,                  \
                             (cudaStream_t)stream);                                                                               \
  }                                                                                                                               \
  int ska_reprojection_loss_##SFX(const S* d_X, int64_t T, int32_t J, int32_t C, const S* d_R, int64_t R_frame_stride,            \
                                  const S* d_t, int64_t t_frame_stride, const S* d_K, int64_t K_frame_stride, const S* d_x2d,     \
                                  const S* d_conf, double* d_sums, S* d_gX, S* d_gR, S* d_gt, S* d_gK, void* d_workspace,         \
                                  size_t ws_bytes, void* stream) {                                                                \
    SKA_LOSS_CHECK();                                                                                                             \
    if (d_sums == nullptr || d_workspace == nullptr) return set_error(SKA_EINVAL, "d_sums and d_workspace must not be NULL");     \
    if (T > 0 && d_x2d == nullptr) return set_error(SKA_EINVAL, "d_x2d must not be NULL");                                        \
    return reprojection_loss<S>(d_X, T, J, C, d_R, R_frame_stride, d_t, t_frame_stride, d_K, K_frame_stride, d_x2d, d_conf,       \
                                d_sums, d_gX, d_gR, d_gt, d_gK, d_workspace, ws_bytes, (cudaStream_t)stream);                     \
  }                                                                                                                               \
  int ska_pose_temporal_##SFX(const S* d_X, int64_t T, int32_t J, double* d_sum, S* d_gX, void* d_workspace, size_t ws_bytes,     \
                              void* stream) {                                                                                     \
    if (T < 0 || J < 1 || d_sum == nullptr || d_workspace == nullptr || (T > 0 && d_X == nullptr))                                \
      return set_error(SKA_EINVAL, "bad arguments");                                                                              \
    return pose_temporal<S>(d_X, T, J, d_sum, d_gX, d_workspace, ws_bytes, (cudaStream_t)stream);                                 \
  }                                                                                                                               \
  int ska_bone_length_##SFX(const S* d_X, int64_t T, int32_t J, const int32_t* bone_i, const int32_t* bone_j, int32_t n_bones,    \
                            const double* d_ref, double* d_sums, S* d_gX, void* d_workspace, size_t ws_bytes, void* stream) {     \
    if (T < 0 || J < 1 || d_sums == nullptr || d_workspace == nullptr || (T > 0 && d_X == nullptr) ||                             \
        (n_bones > 0 && (bone_i == nullptr || bone_j == nullptr)))                                                                \
      return set_error(SKA_EINVAL, "bad arguments");                                                                              \
    return bone_length<S>(d_X, T, J, bone_i, bone_j, n_bones, d_ref, d_sums, d_gX, d_workspace, ws_bytes, (cudaStream_t)stream);  \
  }                                                                                                                               \
  int ska_camera_centre_##SFX(const S* d_R, const S* d_t, int64_t n, S* d_C, void* stream) {                                      \
    if (n < 0 || (n > 0 && (d_R == nullptr || d_t == nullptr || d_C == nullptr))) return set_error(SKA_EINVAL, "bad arguments");  \
    return camera_centre<S>(d_R, d_t, n, d_C, (cudaStream_t)stream);                                                              \
  }                                                                                                                               \
  int ska_camera_smooth_##SFX(const S* d_R, const S* d_t, int64_t D0, int64_t M, double* d_sum, S* d_gR, S* d_gt,                 \
                              void* d_workspace, size_t ws_bytes, void* stream) {                                                 \
    if (D0 < 0 || M < 0 || d_sum == nullptr || d_workspace == nullptr || (D0 * M > 0 && (d_R == nullptr || d_t == nullptr)))      \
      return set_error(SKA_EINVAL, "bad arguments");                                                                              \
    return camera_smooth<S>(d_R, d_t, D0, M, d_sum, d_gR, d_gt, d_workspace, ws_bytes, (cudaStream_t)stream);                     \
  }                                                                                                                               \
  int ska_baseline_reg_##SFX(const S* d_R, const S* d_t, int64_t T, int32_t C, const double* d_mean, double* d_sum, S* d_gR,      \
                             S* d_gt, void* d_workspace, size_t ws_bytes, void* stream) {                                         \
    if (T < 0 || d_sum == nullptr || d_workspace == nullptr || (T > 0 && (d_R == nullptr || d_t == nullptr)))                     \
      return set_error(SKA_EINVAL, "bad arguments");                                                                              \
    return baseline_reg<S>(d_R, d_t, T, C, d_mean, d_sum, d_gR, d_gt, d_workspace, ws_bytes, (cudaStream_t)stream);               \
  }

SKA_DEFINE_LOSS(f32, float)
SKA_DEFINE_LOSS(f64, double)
#undef SKA_DEFINE_LOSS
#undef SKA_LOSS_CHECK

int ska_post_triage_f32(const SkaCamera* cams, const float* d_X, const float* d_kpts, const float* d_conf, int64_t T, int32_t J,
                        uint32_t flags, double conf_thr, double err_thresh_px, float* d_Xclean, float* d_em, uint8_t* d_flags,
                        void* stream) {
  if (cams == nullptr) return set_error(SKA_EINVAL, "cams must not be NULL");
  if (T < 0 || J < 1) return set_error(SKA_EINVAL, "T >= 0, J >= 1");
  if (flags > 3u) return set_error(SKA_EINVAL, "unknown flag bits");
  if (T == 0) return SKA_OK;
  if (d_X == nullptr || d_kpts == nullptr || d_Xclean == nullptr) return set_error(SKA_EINVAL, "d_X, d_kpts and d_Xclean must not be NULL");
  if (reinterpret_cast<uintptr_t>(d_kpts) % 8 != 0) return set_error(SKA_EALIGN, "d_kpts must be 8-byte aligned");
  return post_triage(cams, d_X, d_kpts, d_conf, T, J, flags, conf_thr, err_thresh_px, d_Xclean, d_em, d_flags, (cudaStream_t)stream);
}

int ska_frame_flag_counts_u8(const uint8_t* d_flags, int64_t T, int32_t J, int32_t* d_counts, void* stream) {
  if (T < 0 || J < 1) return set_error(SKA_EINVAL, "T >= 0, J >= 1");
  if (T == 0) return SKA_OK;
  if (d_flags == nullptr || d_counts == nullptr) return set_error(SKA_EINVAL, "d_flags and d_counts must not be NULL");
  if (reinterpret_cast<uintptr_t>(d_counts) % 16 != 0) return set_error(SKA_EALIGN, "d_counts must be 16-byte aligned");
  return flag_counts(d_flags, T, J, d_counts, (cudaStream_t)stream);
}

size_t ska_savgol_workspace_bytes(int64_t T, int32_t S) { return (T < 0 || S < 1) ? 0 : savgol_workspace_bytes(T, S); }

int ska_savgol_f32(const float* d_X, int64_t T, int32_t S, int32_t win, int32_t poly, float* d_out, void* d_workspace,
                   size_t ws_bytes, void* stream) {
  if (T < 0 || S < 1) return set_error(SKA_EINVAL, "T >= 0, S >= 1");
  if (T > 0 && (d_X == nullptr || d_out == nullptr || d_workspace == nullptr)) return set_error(SKA_EINVAL, "d_X, d_out and d_workspace must not be NULL");
  if (d_X == d_out && T > 0) return set_error(SKA_EINVAL, "d_out must not alias d_X");
  return savgol(d_X, T, S, win, poly, d_out, d_workspace, ws_bytes, (cudaStream_t)stream);
}

size_t ska_loss_workspace_bytes(int32_t C) { return C < 1 ? 0 : loss_workspace_bytes(C); }
size_t ska_reg_workspace_bytes(void) { return reg_workspace_bytes(); }

static int check_problem(const SkaBaProblem* p, bool need_points) {
  if (p == nullptr) return set_error(SKA_EINVAL, "problem must not be NULL");
  if (p->C < 2 || p->C > SKA_MAX_VIEWS) return set_error(SKA_EINVAL, "C must be in 2..SKA_MAX_VIEWS");
  if (p->T < 0 || p->J < 1) return set_error(SKA_EINVAL, "T must be >= 0 and J >= 1");
  if (p->T * (int64_t)p->J >= (int64_t)1 << 31) return set_error(SKA_EINVAL, "T*J must be < 2^31 per rank; shard the clip");
  if (p->layout != SKA_LAYOUT_VIEW_MAJOR && p->layout != SKA_LAYOUT_FRAME_MAJOR) return set_error(SKA_EINVAL, "bad layout");
  if (p->d_cams == nullptr || p->d_ctrl == nullptr || p->d_red == nullptr || p->d_red2 == nullptr || p->d_delta == nullptr)
    return set_error(SKA_EINVAL, "d_cams, d_ctrl, d_red, d_red2 and d_delta must not be NULL");
  if (need_points) {
    if (p->T > 0 && (p->d_x2d == nullptr || p->d_conf == nullptr || p->d_Xpp == nullptr))
      return set_error(SKA_EINVAL, "d_x2d, d_conf and d_Xpp must not be NULL");
    if (p->d_workspace == nullptr) return set_error(SKA_EINVAL, "d_workspace must not be NULL");
    if (reinterpret_cast<uintptr_t>(p->d_x2d) % 8 != 0) return set_error(SKA_EALIGN, "d_x2d must be 8-byte aligned");
    if (reinterpret_cast<uintptr_t>(p->d_workspace) % 16 != 0) return set_error(SKA_EALIGN, "d_workspace must be 16-byte aligned");
    // the loss is read by the per-observation kernels only (solve / control ignore it); they hold d and d^2 in fp32
    if (p->loss != SKA_BA_LOSS_L2 && p->loss != SKA_BA_LOSS_HUBER && p->loss != SKA_BA_LOSS_CAUCHY) return set_error(SKA_EINVAL, "unknown loss");
    if (p->loss != SKA_BA_LOSS_L2) {
      const float d = (float)p->loss_scale;
      if (!(isfinite(p->loss_scale) && p->loss_scale > 0.0 && isfinite(d * d) && d * d >= FLT_MIN))
        return set_error(SKA_EINVAL, "a robust loss needs a finite loss_scale > 0 whose square is a normal fp32 number");
    }
  }
  return SKA_OK;
}

int32_t ska_ba_red_doubles(int32_t C) { return (C < 2 || C > SKA_MAX_VIEWS) ? 0 : ba_red_size(C); }

size_t ska_ba_workspace_bytes(int32_t C) {
  if (C < 2 || C > SKA_MAX_VIEWS) return 0;
  return (size_t)ba_max_grid() * (size_t)ba_red_size(C) * sizeof(double);
}

int ska_ba_sum_f32(const float* d_x, int64_t count, double* d_out, void* d_workspace, size_t ws_bytes, void* stream) {
  if (d_out == nullptr || d_workspace == nullptr || count < 0 || (count > 0 && d_x == nullptr))
    return set_error(SKA_EINVAL, "d_x, d_out and d_workspace must not be NULL; count >= 0");
  return ba_sum(d_x, count, d_out, d_workspace, ws_bytes, stream);
}

int ska_ba_linearize_f32(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, true);
  if (rc != SKA_OK) return rc;
  return ba_linearize(*p, (cudaStream_t)stream);
}

int ska_ba_solve_f64(const SkaBaProblem* p, uint64_t free_mask, void* stream) {
  const int rc = check_problem(p, false);
  if (rc != SKA_OK) return rc;
  return ba_solve(p->C, free_mask, p->d_red, p->d_cams, p->d_ctrl, p->d_delta, p->peer, stream);
}

int ska_ba_backsub_f32(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, true);
  if (rc != SKA_OK) return rc;
  return ba_backsub(*p, (cudaStream_t)stream);
}

int ska_ba_control_f64(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, false);
  if (rc != SKA_OK) return rc;
  return ba_control(p->C, p->d_red, p->d_red2, p->d_cams, p->d_ctrl, p->d_hist, p->hist_rows, p->peer, stream);
}

size_t ska_ba_reg_workspace_bytes(int64_t T_local) { return T_local < 1 ? 0 : ba_reg_workspace_bytes(T_local); }
#define SKA_REG_ENTRY(call)                                                        \
  if (p == nullptr) return set_error(SKA_EINVAL, "problem pointer must not be NULL"); \
  return call
// the regularised LM's kernels are fp64: a robust scale needs a finite d > 0 whose square is a normal fp64 number
static int check_reg_loss(int32_t loss, double loss_scale) {
  if (loss != SKA_BA_LOSS_L2 && loss != SKA_BA_LOSS_HUBER && loss != SKA_BA_LOSS_CAUCHY) return set_error(SKA_EINVAL, "unknown loss");
  if (loss != SKA_BA_LOSS_L2 && !(isfinite(loss_scale) && loss_scale > 0.0 && isfinite(loss_scale * loss_scale) && loss_scale * loss_scale >= DBL_MIN))
    return set_error(SKA_EINVAL, "a robust loss needs a finite loss_scale > 0 whose square is a normal fp64 number");
  return SKA_OK;
}
#define SKA_REG_LOSS_ENTRY(call)                                                        \
  if (p == nullptr) return set_error(SKA_EINVAL, "problem pointer must not be NULL");   \
  if (const int rc = check_reg_loss(loss, loss_scale); rc != SKA_OK) return rc;        \
  return call
int ska_ba_reg_cost_robust_f64(const SkaBaRegProblem* p, int32_t which, int32_t loss, double loss_scale, void* stream) {
  SKA_REG_LOSS_ENTRY(ba_reg_cost(*p, which, loss, loss_scale, (cudaStream_t)stream));
}
int ska_ba_reg_linearize_robust_f64(const SkaBaRegProblem* p, int32_t loss, double loss_scale, void* stream) {
  SKA_REG_LOSS_ENTRY(ba_reg_linearize(*p, loss, loss_scale, (cudaStream_t)stream));
}
int ska_ba_reg_cg_robust_f64(const SkaBaRegProblem* p, int32_t op, int32_t loss, double loss_scale, void* stream) {
  SKA_REG_LOSS_ENTRY(ba_reg_cg(*p, op, loss, loss_scale, (cudaStream_t)stream));
}
#undef SKA_REG_LOSS_ENTRY
int ska_ba_reg_cost_f64(const SkaBaRegProblem* p, int32_t which, void* stream) { return ska_ba_reg_cost_robust_f64(p, which, SKA_BA_LOSS_L2, 0.0, stream); }
int ska_ba_reg_finish_cost_f64(const SkaBaRegProblem* p, int32_t which, void* stream) {
  SKA_REG_ENTRY(ba_reg_finish_cost(*p, which, (cudaStream_t)stream));
}
int ska_ba_reg_linearize_f64(const SkaBaRegProblem* p, void* stream) { return ska_ba_reg_linearize_robust_f64(p, SKA_BA_LOSS_L2, 0.0, stream); }
int ska_ba_reg_cg_f64(const SkaBaRegProblem* p, int32_t op, void* stream) { return ska_ba_reg_cg_robust_f64(p, op, SKA_BA_LOSS_L2, 0.0, stream); }
int ska_ba_reg_apply_f64(const SkaBaRegProblem* p, void* stream) { SKA_REG_ENTRY(ba_reg_apply(*p, (cudaStream_t)stream)); }
int ska_ba_reg_control_f64(const SkaBaRegProblem* p, void* stream) { SKA_REG_ENTRY(ba_reg_control(*p, (cudaStream_t)stream)); }
#undef SKA_REG_ENTRY

size_t ska_peer_region_bytes(int32_t world, int32_t slot_doubles) {
  if (world < 1 || world > SKA_MAX_PEERS || slot_doubles < 1) return 0;
  return (size_t)2 * world * slot_doubles * 2 * sizeof(uint64_t);  // [parity][sender][slot] x two tagged 64-bit words per double
}
int ska_peer_alloc(size_t bytes, void** d_ptr) { return peer_alloc(bytes, d_ptr); }
int ska_peer_free(void* d_ptr) { return peer_free(d_ptr); }
int ska_peer_export(void* d_ptr, unsigned char* handle64) {
  if (d_ptr == nullptr || handle64 == nullptr) return set_error(SKA_EINVAL, "pointers must not be NULL");
  return peer_export(d_ptr, handle64);
}
int ska_peer_import(const unsigned char* handle64, void** d_ptr) {
  if (d_ptr == nullptr || handle64 == nullptr) return set_error(SKA_EINVAL, "pointers must not be NULL");
  return peer_import(handle64, d_ptr);
}
int ska_peer_close(void* d_ptr) { return peer_close(d_ptr); }
int ska_peer_allreduce_f64(const SkaPeerComm* comm, double* d_buf, int32_t n, void* stream) {
  if (comm == nullptr) return set_error(SKA_EINVAL, "comm must not be NULL");
  return peer_allreduce(*comm, d_buf, n, (cudaStream_t)stream);
}
int ska_peer_allgather_f64(const SkaPeerComm* comm, const double* d_in, int32_t n, double* d_out, void* stream) {
  if (comm == nullptr) return set_error(SKA_EINVAL, "comm must not be NULL");
  return peer_allgather(*comm, d_in, n, d_out, (cudaStream_t)stream);
}

int32_t ska_ba_calib_red_doubles(int32_t C) { return C == 2 ? ba_calib_red_size(C) : 0; }

size_t ska_ba_calib_workspace_bytes(int32_t C) {
  if (C != 2) return 0;
  return (size_t)ba_max_grid() * (size_t)ba_calib_red_size(C) * sizeof(double);
}

int ska_ba_calib_linearize_f32(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, true);
  if (rc != SKA_OK) return rc;
  return ba_calib_linearize(*p, (cudaStream_t)stream);
}

int ska_ba_calib_solve_f64(const SkaBaProblem* p, uint64_t free_mask, const double* d_prior, void* stream) {
  const int rc = check_problem(p, false);
  if (rc != SKA_OK) return rc;
  return ba_calib_solve(p->C, free_mask, p->d_red, d_prior, p->d_cams, p->d_ctrl, p->d_delta, p->peer, stream);
}

int ska_ba_calib_backsub_f32(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, true);
  if (rc != SKA_OK) return rc;
  return ba_calib_backsub(*p, (cudaStream_t)stream);
}

int ska_ba_calib_control_f64(const SkaBaProblem* p, void* stream) {
  const int rc = check_problem(p, false);
  if (rc != SKA_OK) return rc;
  return ba_calib_control(p->C, p->d_red, p->d_red2, p->d_cams, p->d_ctrl, p->d_hist, p->hist_rows, p->peer, stream);
}

size_t ska_fuse_workspace_bytes(int64_t T) { return fuse_workspace_bytes(T); }

int ska_fuse_frames_f64(const double* d_Xl, const double* d_Xr, const double* d_Ul, const double* d_Ur, int64_t T, int32_t J,
                        const SkaFuseParams* prm, double* d_fused, double* d_ql, double* d_qr, double* d_aligned,
                        uint8_t* d_status, void* d_workspace, size_t ws_bytes, void* stream) {
  if (prm == nullptr) return set_error(SKA_EINVAL, "prm must not be NULL");
  if (T < 0 || J < 1 || J > 96) return set_error(SKA_EINVAL, "T must be >= 0 and 1 <= J <= 96");
  if (T > 0 && (d_Xl == nullptr || d_Xr == nullptr || d_Ul == nullptr || d_Ur == nullptr || d_fused == nullptr))
    return set_error(SKA_EINVAL, "d_Xl, d_Xr, d_Ul, d_Ur and d_fused must not be NULL");
  const int32_t key[5] = {prm->root, prm->lhip, prm->rhip, prm->lsho, prm->rsho};
  for (int k = 0; k < 5; ++k)
    if (key[k] < 0 || key[k] >= J) return set_error(SKA_EINVAL, "key joint index outside 0..J-1");
  if (prm->scale_mode != 0 && prm->scale_mode != 1) return set_error(SKA_EINVAL, "scale_mode must be 0 (hip) or 1 (torso)");
  if (prm->min_points < 1) return set_error(SKA_EINVAL, "min_points must be >= 1");
  return fuse_frames(d_Xl, d_Xr, d_Ul, d_Ur, T, J, *prm, d_fused, d_ql, d_qr, d_aligned, d_status, d_workspace, ws_bytes,
                     (cudaStream_t)stream);
}

int ska_rigid_fuse_f64(const double* d_L, const double* d_R, int64_t T, int32_t J, const int32_t* torso5, double tau,
                       const double* d_tau_j, int32_t allow_scale, const double* d_wL, const double* d_wR, int64_t w_frame_stride,
                       double* d_fused, double* d_Rts, double* d_diag, uint8_t* d_status, void* stream) {
  if (T < 0 || J < 1 || torso5 == nullptr) return set_error(SKA_EINVAL, "T >= 0, J >= 1, torso5 must not be NULL");
  for (int k = 0; k < 5; ++k)
    if (torso5[k] < 0 || torso5[k] >= J) return set_error(SKA_EINVAL, "torso joint index outside 0..J-1");
  if (T > 0 && (d_L == nullptr || d_R == nullptr || d_fused == nullptr || d_Rts == nullptr))
    return set_error(SKA_EINVAL, "d_L, d_R, d_fused and d_Rts must not be NULL");
  if (w_frame_stride != 0 && w_frame_stride != J) return set_error(SKA_EINVAL, "w_frame_stride must be 0 (per-joint weights) or J (per-frame)");
  return rigid_fuse(d_L, d_R, T, J, torso5, tau, d_tau_j, allow_scale, d_wL, d_wR, w_frame_stride, d_fused, d_Rts, d_diag, d_status,
                    (cudaStream_t)stream);
}

int ska_ema_f64(const double* d_X, int64_t T, int32_t J, const double* d_alpha_joint, int32_t adaptive, double alpha,
                double alpha_min, double alpha_max, double speed_gain, int64_t chunk, int32_t halo, double* d_Y, void* stream) {
  if (T < 0 || J < 1) return set_error(SKA_EINVAL, "T must be >= 0 and J >= 1");
  if (T > 0 && (d_X == nullptr || d_Y == nullptr || d_alpha_joint == nullptr))
    return set_error(SKA_EINVAL, "d_X, d_Y and d_alpha_joint must not be NULL");
  if (d_X == d_Y && T > 0) return set_error(SKA_EINVAL, "d_Y may not alias d_X");
  if (!(alpha_min <= alpha_max)) return set_error(SKA_EINVAL, "alpha_min must be <= alpha_max");
  return ema_smooth(d_X, T, J, d_alpha_joint, adaptive, alpha, alpha_min, alpha_max, speed_gain, chunk, halo, d_Y, (cudaStream_t)stream);
}

int ska_first_order_record_f64(double* d_k, double* d_scal, double* d_hist, int64_t max_rows, const double* const* sums5,
                               const double* d_den, const double* coef5, double lr, double beta1, double beta2, void* stream) {
  if (d_k == nullptr || d_scal == nullptr || sums5 == nullptr || coef5 == nullptr || max_rows < 0)
    return set_error(SKA_EINVAL, "d_k, d_scal, sums5 and coef5 must not be NULL; max_rows >= 0");
  return first_order_record(d_k, d_scal, d_hist, max_rows, sums5, d_den, coef5, lr, beta1, beta2, (cudaStream_t)stream);
}

#define SKA_OPTIM_ENTRY(SFX, S)                                                                                                   \
  int ska_adam_step_##SFX(S* d_p, const S* d_g, S* d_m, S* d_v, int64_t n, double step_size, double beta1, double beta2, double eps,  \
                          double inv_sqrt_bc2, S* d_step_out, const double* d_scalars, void* stream) {                             \
    if (n < 0 || (n > 0 && (d_g == nullptr || d_m == nullptr || d_v == nullptr || (d_p == nullptr && d_step_out == nullptr))))      \
      return set_error(SKA_EINVAL, "d_g, d_m, d_v and one of d_p / d_step_out must not be NULL; n >= 0");                          \
    return adam_step<S>(d_p, d_g, d_m, d_v, n, step_size, beta1, beta2, eps, inv_sqrt_bc2, d_step_out, d_scalars, nullptr, nullptr, \
                        1.0, 0.0, 0.0, (cudaStream_t)stream);                                                                       \
  }                                                                                                                                 \
  int ska_adam_step_terms_##SFX(S* d_p, const S* d_g0, double s0, const S* d_g1, double s1, const S* d_g2, double s2, S* d_m,       \
                                S* d_v, int64_t n, double beta1, double beta2, double eps, S* d_step_out, const double* d_scalars,  \
                                void* stream) {                                                                                     \
    if (n < 0 || (n > 0 && (d_g0 == nullptr || d_m == nullptr || d_v == nullptr || d_scalars == nullptr ||                         \
                            (d_p == nullptr && d_step_out == nullptr))))                                                            \
      return set_error(SKA_EINVAL, "d_g0, d_m, d_v, d_scalars and one of d_p / d_step_out must not be NULL; n >= 0");             \
    return adam_step<S>(d_p, d_g0, d_m, d_v, n, 0.0, beta1, beta2, eps, 1.0, d_step_out, d_scalars, d_g1, d_g2, s0, s1, s2,         \
                        (cudaStream_t)stream);                                                                                      \
  }                                                                                                                                 \
  int ska_so3_tangent_grad_##SFX(const S* d_R, const S* d_gR, int64_t n, S* d_gw, void* stream) {                                   \
    if (n < 0 || (n > 0 && (d_R == nullptr || d_gR == nullptr || d_gw == nullptr)))                                                 \
      return set_error(SKA_EINVAL, "d_R, d_gR and d_gw must not be NULL; n >= 0");                                                  \
    return so3_tangent_grad<S>(d_R, d_gR, n, d_gw, (cudaStream_t)stream);                                                           \
  }                                                                                                                                 \
  int ska_so3_retract_##SFX(S* d_R, const S* d_step, int64_t n, void* stream) {                                                     \
    if (n < 0 || (n > 0 && (d_R == nullptr || d_step == nullptr))) return set_error(SKA_EINVAL, "d_R and d_step must not be NULL"); \
    return so3_retract<S>(d_R, d_step, n, (cudaStream_t)stream);                                                                    \
  }
SKA_OPTIM_ENTRY(f32, float)
SKA_OPTIM_ENTRY(f64, double)
#undef SKA_OPTIM_ENTRY

#pragma GCC visibility pop
}  // extern "C"
