// ska_internal.h - shared between the translation units of libska.so (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ska.h"
#include "ska_prep.h"

namespace ska {

int set_error(int code, const char* msg);

struct TriArgs {
  const SkaCamera* cams;
  int32_t V;
  double centre[3];
  const double* Rt_frames;
  const float* kpts;
  const float* conf;
  int64_t T;
  int32_t J;
  int32_t layout;
  uint32_t flags;
  float* X;
  float* err;
  float* proj;
  uint8_t* status;
  void* stream;
  void* workspace;  // per-frame cameras only
  size_t ws_bytes;
};

int triangulate_dispatch(const TriArgs& a);
size_t tri_frames_workspace(int V, int64_t T);

// bundle adjustment (ska_ba.cu / ska_ba_wide.cu)
int ba_red_size(int C);
int ba_max_grid();
int ba_sum(const float* x, int64_t n, double* out, void* workspace, size_t ws_bytes, void* stream);
int ba_linearize(const SkaBaProblem& p, cudaStream_t s);
int ba_linearize_wide(const SkaBaProblem& p, cudaStream_t s);
int ba_backsub(const SkaBaProblem& p, cudaStream_t s);
int ba_solve(int C, uint64_t free_mask, double* red, double* cams, double* ctrl, double* delta, const SkaPeerComm* peer, void* stream);
int ba_control(int C, const double* red, double* red2, double* cams, double* ctrl, double* hist, int64_t hist_rows, const SkaPeerComm* peer,
               void* stream);
int launch_reduce(const double* partials, int rows, int ncol, double* out, cudaStream_t s);
// calibrating bundle adjustment: free intrinsics + distortion (ska_ba_calib.cu)
int ba_calib_red_size(int C);
int ba_calib_linearize(const SkaBaProblem& p, cudaStream_t s);
int ba_calib_backsub(const SkaBaProblem& p, cudaStream_t s);
int ba_calib_solve(int C, uint64_t free_mask, double* red, const double* prior, double* cams, double* ctrl, double* delta,
                   const SkaPeerComm* peer, void* stream);
int ba_calib_control(int C, const double* red, double* red2, double* cams, double* ctrl, double* hist, int64_t hist_rows,
                     const SkaPeerComm* peer, void* stream);

// regularised LM over the full configured objective, per-frame cameras (ska_ba_reg.cu)
size_t ba_reg_workspace_bytes(int64_t T_local);
int ba_reg_cost(const SkaBaRegProblem& p, int which, int loss, double loss_scale, cudaStream_t s);
int ba_reg_finish_cost(const SkaBaRegProblem& p, int which, cudaStream_t s);
int ba_reg_linearize(const SkaBaRegProblem& p, int loss, double loss_scale, cudaStream_t s);
int ba_reg_cg(const SkaBaRegProblem& p, int op, int loss, double loss_scale, cudaStream_t s);
int ba_reg_apply(const SkaBaRegProblem& p, cudaStream_t s);
int ba_reg_control(const SkaBaRegProblem& p, cudaStream_t s);
// exchange over NVLink peer memory (ska_peer.cu)
int peer_allreduce(const SkaPeerComm& c, double* buf, int n, cudaStream_t s);
int peer_allgather(const SkaPeerComm& c, const double* in, int n, double* out, cudaStream_t s);
int peer_alloc(size_t bytes, void** out);
int peer_free(void* p);
int peer_export(void* p, unsigned char* handle64);
int peer_import(const unsigned char* handle64, void** out);
int peer_close(void* p);

// standalone projection / losses (ska_project.cu, ska_losses.cu)
int project_cv(const SkaCamera* cams, int V, const float* X, const float* kpts, int64_t T, int J, int layout, float* proj,
               float* err, cudaStream_t s);
int frame_stats(const float* err, int64_t T, int J, int V, int layout, float* out, cudaStream_t s);
template <typename S>
int project_points(const S* X, int64_t T, int J, int C, const S* R, int64_t R_sT, const S* t, int64_t t_sT, const S* K,
                   int64_t K_sT, S* out, cudaStream_t s);
size_t loss_workspace_bytes(int C);
template <typename S>
int reprojection_loss(const S* X, int64_t T, int J, int C, const S* R, int64_t R_sT, const S* t, int64_t t_sT, const S* K,
                      int64_t K_sT, const S* x2d, const S* conf, double* sums, S* gX, S* gR, S* gt, S* gK, void* ws,
                      size_t ws_bytes, cudaStream_t s);
size_t reg_workspace_bytes();
template <typename S>
int pose_temporal(const S* X, int64_t T, int J, double* sum, S* gX, void* ws, size_t ws_bytes, cudaStream_t s);
template <typename S>
int bone_length(const S* X, int64_t T, int J, const int32_t* bi, const int32_t* bj, int nb, const double* ref, double* sums,
                S* gX, void* ws, size_t ws_bytes, cudaStream_t s);
template <typename S>
int camera_centre(const S* R, const S* t, int64_t n, S* C, cudaStream_t s);
template <typename S>
int camera_smooth(const S* R, const S* t, int64_t D0, int64_t M, double* sum, S* gR, S* gt, void* ws, size_t ws_bytes, cudaStream_t s);
template <typename S>
int baseline_reg(const S* R, const S* t, int64_t T, int Cn, const double* mean, double* sum, S* gR, S* gt, void* ws, size_t ws_bytes,
                 cudaStream_t s);


// post-triangulation triage + Savitzky-Golay smoothing (ska_post.cu)
int post_triage(const SkaCamera* cams, const float* X, const float* kpts, const float* conf, int64_t T, int J, uint32_t flags,
                double conf_thr, double err_thr, float* Xc, float* em, uint8_t* fl, cudaStream_t s);
int flag_counts(const uint8_t* flags, int64_t T, int J, int32_t* out, cudaStream_t s);
size_t savgol_workspace_bytes(int64_t T, int S);
int savgol(const float* X, int64_t T, int S, int win, int poly, float* out, void* ws, size_t ws_bytes, cudaStream_t s);

// first-order optimiser updates (ska_optim.cu)
template <typename S>
int adam_step(S* p, const S* g, S* m, S* v, int64_t n, double step_size, double b1, double b2, double eps, double inv_sqrt_bc2, S* step_out,
              const double* scalars, const S* g1, const S* g2, double s0, double s1, double s2, cudaStream_t s);
int first_order_record(double* k, double* scal, double* hist, int64_t max_rows, const double* const* sums, const double* den,
                       const double* coef, double lr, double b1, double b2, cudaStream_t s);
template <typename S>
int so3_tangent_grad(const S* R, const S* gR, int64_t n, S* gw, cudaStream_t s);
template <typename S>
int so3_retract(S* R, const S* step, int64_t n, cudaStream_t s);

// two-view 3D fusion + EMA (ska_fuse.cu)
size_t fuse_workspace_bytes(int64_t T);
int fuse_frames(const double* Xl, const double* Xr, const double* Ul, const double* Ur, int64_t T, int J, const SkaFuseParams& prm,
                double* fused, double* ql, double* qr, double* aligned, uint8_t* status, void* ws, size_t ws_bytes, cudaStream_t s);
int rigid_fuse(const double* L, const double* R, int64_t T, int J, const int32_t* torso5, double tau, const double* tau_j, int allow_scale,
               const double* wL, const double* wR, int64_t w_sT, double* fused, double* Rts, double* diag, uint8_t* status,
               cudaStream_t s);
int ema_smooth(const double* X, int64_t T, int J, const double* alpha_joint, int adaptive, double alpha, double alpha_min,
               double alpha_max, double speed_gain, int64_t chunk, int halo, double* Y, cudaStream_t s);

}  // namespace ska
