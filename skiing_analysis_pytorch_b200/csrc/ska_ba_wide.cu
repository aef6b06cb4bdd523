// ska_ba_wide.cu - BA linearisation for C >= 3 cameras (reduced system too large for per-thread
// registers): the Schur accumulation is a skinny SYRK, done warp-cooperatively from shared memory.
//
// Each warp owns 32 points per tile.
//   phase 1  thread = point: pass A over the cameras builds the damped 3x3 point block, its Cholesky
//            and dp0 = -Hd^-1 gp (the point's own step with the cameras frozen); pass B re-projects
//            each free camera c and
//              - writes Y_c = L^-1 W_c (3 x 6) transposed into the warp's staging buffer
//                Yt[col][3*lane + k] (the only shared-memory staging: 16.8 KB per warp at C = 8),
//              - forms the camera's 33 per-point sums-to-be (Hcc upper triangle 21, gc 6, bw 6) in
//                registers and reduces them over the 32 points with a TRANSPOSING butterfly: 5
//                exchange steps of 16/8/4/2/1 values leave lane i holding the warp total of value i
//                (31 shuffles for 32 values instead of 160).
//   phase 2  lane = one 6x6 block (a, b), a <= b, of Sw = sum Y^T Y: 36 fp32 accumulators, operands
//            read as 128-bit shared loads of 4 consecutive rows of one column (padded column stride:
//            conflict free), 144 FMA per 12 loads.
// Every kFlush tiles the per-lane fp32 accumulators are folded into the CTA's fp64 packed reduced
// system in shared memory in a fixed warp order (no atomics, deterministic); the CTA writes one
// fp64 partial row, ba_reduce_columns (ska_ba.cu) sums the rows in a fixed order.
//
// The same kernel also runs C == 2 (SKA_BA_FORCE_WIDE) so the two paths can be tested against
// each other.
#include <cuda_runtime.h>

#include "ska_ba.cuh"
#include "ska_internal.h"

namespace ska {

struct BaKernelArgsW {
  ObsLayout lay;
  int64_t N;
  int64_t n_tiles;
  uint32_t div_mul, div_shift;  // exact i / J (tensor-core form)
  const float* x2d;
  const float* conf;
  const double* cams;
  const double* ctrl;
  const float* Xpp;
  double* partials;
  int32_t loss;       // SKA_BA_LOSS_* (the kernel's Loss template argument selects the code)
  float loss_scale;   // robust scale d in pixels (unused by L2)
};

#ifndef SKA_BA_WIDE_WARPS
#define SKA_BA_WIDE_WARPS 12  // 384 threads x <= 168 registers = the whole register file, one CTA per SM
#endif

__device__ __forceinline__ void mbar_init_tc(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}

template <int C>
struct Wide {
  static constexpr int NC = C - 1, n = 6 * NC, nS = n * (n + 1) / 2;
  static constexpr int oBw = nS, oGc = nS + n, oHcc = nS + 2 * n, oCost = oHcc + 21 * NC, oClamp = oCost + 1, size = oClamp + 1;
  static constexpr int NP = NC * (NC + 1) / 2;              // 6x6 block pairs a <= b
  static constexpr int SL_A = largest_div(24, 32 / NP);     // row slices in phase 2 (24 chunks of 4 rows)
  static constexpr int CH_A = 24 / SL_A;
  static constexpr int W = SKA_BA_WIDE_WARPS;               // warps per CTA
  static constexpr int warp_floats = n * kYStride;
  static constexpr size_t smem = (size_t)W * warp_floats * sizeof(float) + (size_t)size * sizeof(double) + C * sizeof(CamF);
};

template <int C, int Loss>
__global__ void __launch_bounds__(32 * Wide<C>::W, 1) ba_linearize_wide_kernel(const BaKernelArgsW a) {
  using L = Wide<C>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_warp = reinterpret_cast<float*>(smem_raw);  // W * warp_floats, a multiple of 16 bytes
  double* s_red = reinterpret_cast<double*>(s_warp + (size_t)L::W * L::warp_floats);
  CamF* s_cam = reinterpret_cast<CamF*>(s_red + L::size);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* Yt = s_warp + (size_t)warp * L::warp_floats;

  if (threadIdx.x < C) load_cam(a.cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) s_red[k] = 0.0;
  __syncthreads();
  const float lam = (float)a.ctrl[kCtrlLambda];
  const int cur = (int)a.ctrl[kCtrlCur];
  const float* X = a.Xpp + (int64_t)cur * 3 * a.N;

  // phase-2 role: block pair and row slice
  int pa = 0, pb_ = 0;
  const int pair = lane % L::NP, slice_a = lane / L::NP;
  {
    int q = pair;
    for (int r = 0; r < L::NC; ++r) {
      const int len = L::NC - r;
      if (q < len) {
        pa = r;
        pb_ = r + q;
        break;
      }
      q -= len;
    }
  }
  const bool act_a = slice_a < L::SL_A;

  float accS[6][6], accH[L::NC], accX[L::NC];  // accH: lane i = entry i of the camera's 33 sums; accX: entry 32
#pragma unroll
  for (int k = 0; k < 6; ++k)
#pragma unroll
    for (int l = 0; l < 6; ++l) accS[k][l] = 0.f;
#pragma unroll
  for (int c = 0; c < L::NC; ++c) accH[c] = accX[c] = 0.f;
  float cost = 0.f, nclamp = 0.f;
  int since = 0;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t i = (tile * L::W + warp) * 32 + lane;
    const bool valid = i < a.N;
    // ---------------------------------------------------------------- phase 1
    float u[C], v[C], cw[C], Xp[3] = {0.f, 0.f, 1.f};
    if (valid) {
      int64_t koff, coff;
      obs_offsets(a.lay, i, koff, coff);
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
    } else {
#pragma unroll
      for (int c = 0; c < C; ++c) u[c] = v[c] = cw[c] = 0.f;
    }
    PointBlock pb;
    pb_zero(pb);
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ObsLin ol;
      project_lin(s_cam[c], Xp, u[c], v[c], ol);
      float au[3], av[3];
      point_rows(s_cam[c], ol, au, av);
      float rho, om;
      robust_loss<Loss>(fmaf(ol.eu, ol.eu, ol.ev * ol.ev), a.loss_scale, rho, om);
      cost = fmaf(cw[c], rho, cost);
      cw[c] *= om;  // pass B below re-projects the same state: it uses this weight
      pb_add(pb, cw[c], au, av, ol.eu, ol.ev);
      nclamp += (valid && ol.clamped) ? 1.f : 0.f;
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
    for (int c = 1; c < C; ++c) {
      ObsLin ol;
      project_lin(s_cam[c], Xp, u[c], v[c], ol);
      float au[3], av[3], bu[6], bv[6];
      point_rows(s_cam[c], ol, au, av);
      camera_rows(ol, bu, bv);
      const float w = cw[c];
      float s33[32], s32;
      const float adu = -fmaf(au[0], d0, fmaf(au[1], d1, au[2] * d2));
      const float adv = -fmaf(av[0], d0, fmaf(av[1], d1, av[2] * d2));
      int q = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        const float su = w * bu[r], sv = w * bv[r];
        float y0, y1, y2;  // a point without a factor has a zeroed one: Y = 0 without a branch
        chol3_fwd(f, fmaf(su, au[0], sv * av[0]), fmaf(su, au[1], sv * av[1]), fmaf(su, au[2], sv * av[2]), y0, y1, y2);
        float* yt = Yt + (6 * (c - 1) + r) * kYStride + 3 * lane;
        yt[0] = y0;
        yt[1] = y1;
        yt[2] = y2;
#pragma unroll
        for (int s2 = r; s2 < 6; ++s2, ++q) s33[q] = fmaf(su, bu[s2], sv * bv[s2]);  // Hcc upper triangle, 21 entries
        s33[21 + r] = fmaf(su, ol.eu, sv * ol.ev);                                   // gc
        if (r < 5) s33[27 + r] = fmaf(su, adu, sv * adv);                            // bw (entries 27..31)
        else s32 = fmaf(su, adu, sv * adv);                                          // bw[5] = entry 32
      }
      accH[c - 1] += transpose_reduce32(s33, lane);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s32 += __shfl_xor_sync(0xffffffffu, s32, o);
      accX[c - 1] += s32;
    }
    __syncwarp();
    // ---------------------------------------------------------------- phase 2: Sw block (pa, pb_)
    if (act_a) {
      // scalar FFMA on purpose: the packed form (rows 0-1 / 2-3 of a chunk in the halves of an F2, 6x3
      // half blocks) was measured 10 % slower - half as many independent accumulator chains
      const float* ya = Yt + (6 * pa) * kYStride + 4 * slice_a * L::CH_A;
      const float* yb = Yt + (6 * pb_) * kYStride + 4 * slice_a * L::CH_A;
#pragma unroll 2
      for (int ch = 0; ch < L::CH_A; ++ch) {
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
      double dc = (double)cost, dn = (double)nclamp;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        dc += __shfl_down_sync(0xffffffffu, dc, o);
        dn += __shfl_down_sync(0xffffffffu, dn, o);
      }
      cost = nclamp = 0.f;
      for (int w = 0; w < L::W; ++w) {
        __syncthreads();
        if (warp == w) {
          for (int sl = 0; sl < L::SL_A; ++sl) {
            if (act_a && slice_a == sl) {
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
          // lane i holds entry i of every camera's [Hcc (21) | gc (6) | bw (6)]; entry 32 is on every lane
          const int o33 = lane < 21 ? L::oHcc + lane : (lane < 27 ? L::oGc + (lane - 21) : L::oBw + (lane - 27));
          const int s33 = lane < 21 ? 21 : 6;
#pragma unroll
          for (int c = 0; c < L::NC; ++c) {
            s_red[o33 + s33 * c] += (double)accH[c];
            if (lane == 0) s_red[L::oBw + 6 * c + 5] += (double)accX[c];
          }
          if (lane == 0) {
            s_red[L::oCost] += dc;
            s_red[L::oClamp] += dn;
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int l = 0; l < 6; ++l) accS[k][l] = 0.f;
#pragma unroll
      for (int c = 0; c < L::NC; ++c) accH[c] = accX[c] = 0.f;
    }
  }
  __syncthreads();
  double* out = a.partials + (int64_t)blockIdx.x * L::size;
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) out[k] = s_red[k];
}

// ------------------------------------------------------------------------------------------------
// Tensor-core form for 5..8 cameras: ba_linearize_tc_kernel.
//
// The Schur accumulation Sw += Y^T Y is the one dense contraction of the path (42 x 42 x 3 per point at 8 cameras: 3 024
// of the 7 800 warp instructions per 32 points of the CUDA-core form above).  Here it runs on the 5th-generation tensor
// cores: Y is staged in shared memory in the K-major core-matrix layout tcgen05 reads (8 rows x 16 bytes per core
// matrix, no swizzle), split into a tf32-exact high part and the remainder, and ONE thread issues, per K = 8 step,
//     D_hh += Yhi^T Yhi,   D_hl += Yhi^T Ylo,   D_lh += Ylo^T Yhi        (tcgen05.mma kind::tf32, M = 64, N = 56, K = 8)
// for the K = 3 x 48 point rows of a CTA tile.  The three-product split keeps ~2^-20 relative accuracy, what the fp32
// FFMA form delivers.  MMAs into ONE accumulator retire ~100 cycles apart whatever their size (measured: 54 dependent
// N = 48 MMAs per tile kept the tensor pipe 23 % busy and the CUDA cores waiting), so the three products - and the even
// / odd K steps of each - go to SIX accumulators in tensor memory; they are summed and folded into the CTA's fp64
// reduced system every kTcFlush tiles (tcgen05.ld).  While the tensor pipe works on tile i the CUDA cores linearise
// tile i + 1 (two staging buffers; mbarriers: `staged` armed by the compute warps, `done` by tcgen05.commit).
//
// Staged layout: camera c's six columns are rows 8 (c - 1) + r of the operand (two zero rows per camera), point row
// (point p of the tile, coordinate j) is K index p + 48 j - so a thread's 18 values go to ONE base address plus
// compile-time offsets 16 r + 1536 j.
//
// The rest of the linearisation is re-cut so that a THREAD OWNS ONE (point, camera) OBSERVATION - 8 lanes per point:
// the projection and its Jacobians are formed once (the form above forms them twice), the 3 x 3 point block is summed
// over the point's lanes with a butterfly, every lane factors it, and the lane's camera keeps its 33 sums
// [Hcc | gc | bw] in registers across tiles (no per-tile transposing reduction).
constexpr int kTcWarps = 12;                    // compute warps: 48 points x 8 lanes per CTA tile; warp kTcWarps issues the MMAs
constexpr int kTcPts = 4 * kTcWarps;            // points per CTA tile
constexpr int kTcK = 3 * kTcPts;                // K extent of a tile: 144 point rows
constexpr int kTcN = 56;                        // staged operand rows: 7 cameras x 8 (6 used)
constexpr int kTcSBO = (kTcK / 4) * 128 + 16;   // bytes between 8-row groups: + 16 so that the seven cameras' rows of one K index fall into
                                                // different banks (a multiple of 128 puts a warp's 32 stores into 4 banks: measured 8-way conflicts)
constexpr int kTcBuf = (kTcN / 8) * kTcSBO;     // bytes of one staged operand (hi or lo)
constexpr int kTcAccStride = 64;                // tensor-memory columns per accumulator
constexpr int kTcTmemCols = 512;                // 6 accumulators x 64 columns -> the whole tensor memory (one CTA per SM)
constexpr int kTcFlush = 32;                    // tiles per fp32 accumulation window
static_assert(kTcK % 16 == 0, "a tile is a whole number of K = 8 MMA step pairs");

__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr) {
  // K-major, no swizzle: start address, leading (K-direction) byte offset 128, stride (8-row group) byte offset kTcSBO,
  // descriptor version 1 (all offsets in 16-byte units)
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(kTcSBO >> 4) << 32) | (1ull << 46);
}
constexpr uint32_t kTcIdesc = (1u << 4) /* D = f32 */ | (2u << 7) /* A = tf32 */ | (2u << 10) /* B = tf32 */ | ((uint32_t)(kTcN >> 3) << 17) | ((64u >> 4) << 24);

__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(kTcIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ bool tc_bar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  for (int spin = 0; spin < (1 << 16); ++spin) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done)
                 : "r"(a), "r"(parity)
                 : "memory");
    if (done) return true;
  }
  return false;  // never signalled: the caller traps instead of hanging the GPU
}
__device__ __forceinline__ void tc_bar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}

template <int C>
struct Tc {
  using W = Wide<C>;
  static constexpr size_t oRed = 4 * (size_t)kTcBuf + (size_t)kTcSBO;              // [buf0 hi | buf0 lo | buf1 hi | buf1 lo | pad]: an A operand
                                                                                   // descriptor spans 64 rows = 8 groups from its start
  static constexpr size_t oScr = oRed + (size_t)W::size * sizeof(double);
  static constexpr size_t oCam = oScr + (size_t)kTcWarps * 8 * 35 * sizeof(double);
  static constexpr size_t oBar = oCam + (size_t)C * sizeof(CamF) + 16;
  static constexpr size_t smem = oBar + 96;
};

struct TcObs {  // one lane's observation of a tile
  float u, v, cw, X[3];
};
// exact i / J for i < 2^31 (round-up method; mul == 0 encodes a power of two)
__device__ __forceinline__ uint32_t tc_div(uint32_t n, uint32_t mul, uint32_t shift) {
  return mul == 0 ? (n >> shift) : ((__umulhi(mul, n) + n) >> shift);
}
__device__ __forceinline__ TcObs tc_load(const BaKernelArgsW& a, const float* __restrict__ X, int64_t i, int cam, bool valid) {
  TcObs o;
  o.u = o.v = o.cw = 0.f;
  o.X[0] = o.X[1] = 0.f;
  o.X[2] = 1.f;
  if (valid) {
    const uint32_t t = tc_div((uint32_t)i, a.div_mul, a.div_shift);
    const uint32_t j = (uint32_t)i - t * (uint32_t)a.lay.J;
    const int64_t koff = (int64_t)t * a.lay.k_sT + 2 * (int64_t)j + cam * a.lay.k_sV;
    const int64_t coff = (int64_t)t * a.lay.c_sT + (int64_t)j + cam * a.lay.c_sV;
    const float2 q = __ldg(reinterpret_cast<const float2*>(a.x2d + koff));
    o.u = q.x;
    o.v = q.y;
    o.cw = __ldg(a.conf + coff);
    o.X[0] = __ldg(X + 3 * i);
    o.X[1] = __ldg(X + 3 * i + 1);
    o.X[2] = __ldg(X + 3 * i + 2);
  }
  return o;
}

template <int C>
__global__ void __launch_bounds__(32 * (kTcWarps + 1), 1) ba_linearize_tc_kernel(const BaKernelArgsW a) {
  using L = Wide<C>;
  using S = Tc<C>;
  constexpr int kCompute = 32 * kTcWarps;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* s_y = smem_raw;
  double* s_red = reinterpret_cast<double*>(smem_raw + S::oRed);
  double* s_scr = reinterpret_cast<double*>(smem_raw + S::oScr);
  CamF* s_cam = reinterpret_cast<CamF*>(smem_raw + S::oCam);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(smem_raw + S::oBar) + 15) & ~(uintptr_t)15);
  uint64_t* s_done = s_bar;        // [2] the MMAs that read staging buffer b have completed (tcgen05.commit)
  uint64_t* s_staged = s_bar + 2;  // [2] every compute warp has staged its rows of buffer b
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  if (threadIdx.x < C) load_cam(a.cams + threadIdx.x * kCamStride, s_cam[threadIdx.x]);
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) s_red[k] = 0.0;
  for (int k = threadIdx.x; k < (int)(S::oRed / 16); k += blockDim.x) reinterpret_cast<float4*>(s_y)[k] = make_float4(0.f, 0.f, 0.f, 0.f);  // pad rows stay zero
  if (threadIdx.x == 0) {
    mbar_init_tc(s_done, 1);
    mbar_init_tc(s_done + 1, 1);
    mbar_init_tc(s_staged, kTcWarps);
    mbar_init_tc(s_staged + 1, kTcWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(s_tmem)), "n"(kTcTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the zero fill, seen by the tensor pipe
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *s_tmem;
  const uint32_t y_base = (uint32_t)__cvta_generic_to_shared(s_y);
  const int64_t n_my = (a.n_tiles > blockIdx.x) ? (a.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;  // tiles of this CTA

  if (warp == kTcWarps) {
    // ---------------------------------------------------------------- MMA issuer: one thread
    bool fault = false;
    if (lane == 0) {
      for (int64_t it = 0; it < n_my; ++it) {
        const int buf = (int)(it & 1);
        if (!tc_bar_wait(s_staged + buf, (uint32_t)((it >> 1) & 1))) {
          fault = true;
          break;
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t first = (it % kTcFlush == 0) ? 1u : 0u;  // a new accumulation window: overwrite instead of add
        const uint32_t hi = y_base + (uint32_t)buf * 2u * (uint32_t)kTcBuf, lo = hi + (uint32_t)kTcBuf;
        uint64_t dh = tc_desc(hi), dl = tc_desc(lo);
#pragma unroll 1
        for (int ks = 0; ks < kTcK / 8; ks += 2) {  // even K steps -> accumulators 0..2, odd ones -> 3..5: six independent chains
          const uint32_t acc0 = (ks > 0 || !first) ? 1u : 0u;
          tc_mma(tmem + 0 * kTcAccStride, dh, dh, acc0);
          tc_mma(tmem + 1 * kTcAccStride, dh, dl, acc0);
          tc_mma(tmem + 2 * kTcAccStride, dl, dh, acc0);
          dh += 256 >> 4;  // next K = 8 step: two core matrices further (start address field, 16-byte units)
          dl += 256 >> 4;
          tc_mma(tmem + 3 * kTcAccStride, dh, dh, acc0);
          tc_mma(tmem + 4 * kTcAccStride, dh, dl, acc0);
          tc_mma(tmem + 5 * kTcAccStride, dl, dh, acc0);
          dh += 256 >> 4;
          dl += 256 >> 4;
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(s_done + buf)) : "memory");
      }
    }
    if (fault) __trap();
  } else {
    // ---------------------------------------------------------------- compute warps: a lane owns one (point, camera) observation
    const int cam = lane & 7, pl = lane >> 3;   // the lane's camera and its point within the warp
    const int pt = 4 * warp + pl;               // ... within the CTA tile
    const float lam = (float)a.ctrl[kCtrlLambda];
    const int cur = (int)a.ctrl[kCtrlCur];
    const float* X = a.Xpp + (int64_t)cur * 3 * a.N;
    const CamF cm = s_cam[cam < C ? cam : 0];
    const bool has_cols = cam >= 1 && cam < C;
    // the thread's 18 staged values: operand row 8 (cam - 1) + r, K index pt + 48 j -> base + 16 r + 1536 j
    const uint32_t st_off = has_cols ? (uint32_t)((cam - 1) * kTcSBO + (pt >> 2) * 128 + (pt & 3) * 4) : 0u;
    float acc[33];
#pragma unroll
    for (int q = 0; q < 33; ++q) acc[q] = 0.f;
    float cost = 0.f, nclamp = 0.f;
    bool fault = false;
    int64_t tile = blockIdx.x;
    TcObs nxt = tc_load(a, X, tile * kTcPts + pt, cam, (tile < a.n_tiles) && (tile * kTcPts + pt < a.N) && (cam < C));
    for (int64_t it = 0; it < n_my; ++it, tile += gridDim.x) {
      const int buf = (int)(it & 1);
      const TcObs ob = nxt;
      const bool valid = (tile * kTcPts + pt < a.N) && (cam < C);
      {  // the next tile's observation: in flight while this one is linearised
        const int64_t tn = tile + gridDim.x;
        nxt = tc_load(a, X, tn * kTcPts + pt, cam, (tn < a.n_tiles) && (tn * kTcPts + pt < a.N) && (cam < C));
      }
      ObsLin ol;
      project_lin(cm, ob.X, ob.u, ob.v, ol);
      float au[3], av[3];
      point_rows(cm, ol, au, av);
      PointBlock pb;
      pb_zero(pb);
      pb_add(pb, ob.cw, au, av, ol.eu, ol.ev);
      cost = fmaf(ob.cw, fmaf(ol.eu, ol.eu, ol.ev * ol.ev), cost);
      nclamp += (valid && ol.clamped) ? 1.f : 0.f;
      // ---- point block = sum over the point's 8 lanes (every lane ends with the total)
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        pb.h00 += __shfl_xor_sync(0xffffffffu, pb.h00, o);
        pb.h01 += __shfl_xor_sync(0xffffffffu, pb.h01, o);
        pb.h02 += __shfl_xor_sync(0xffffffffu, pb.h02, o);
        pb.h11 += __shfl_xor_sync(0xffffffffu, pb.h11, o);
        pb.h12 += __shfl_xor_sync(0xffffffffu, pb.h12, o);
        pb.h22 += __shfl_xor_sync(0xffffffffu, pb.h22, o);
        pb.g0 += __shfl_xor_sync(0xffffffffu, pb.g0, o);
        pb.g1 += __shfl_xor_sync(0xffffffffu, pb.g1, o);
        pb.g2 += __shfl_xor_sync(0xffffffffu, pb.g2, o);
      }
      const Chol3 f = chol3_damped(pb, lam);
      float d0, d1, d2;  // dp0 = -Hd^-1 gp
      {
        float y0, y1, y2;
        chol3_fwd(f, -pb.g0, -pb.g1, -pb.g2, y0, y1, y2);
        chol3_bwd(f, y0, y1, y2, d0, d1, d2);
      }
      float bu[6], bv[6];
      camera_rows(ol, bu, bv);
      const float w = (cam >= 1) ? ob.cw : 0.f;  // the gauge camera has no columns
      const float adu = -fmaf(au[0], d0, fmaf(au[1], d1, au[2] * d2));
      const float adv = -fmaf(av[0], d0, fmaf(av[1], d1, av[2] * d2));
      float y[6][3];
      {
        int q = 0;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          const float su = w * bu[r], sv = w * bv[r];
          chol3_fwd(f, fmaf(su, au[0], sv * av[0]), fmaf(su, au[1], sv * av[1]), fmaf(su, au[2], sv * av[2]), y[r][0], y[r][1], y[r][2]);
#pragma unroll
          for (int s2 = r; s2 < 6; ++s2, ++q) acc[q] = fmaf(su, bu[s2], fmaf(sv, bv[s2], acc[q]));  // Hcc upper triangle, 21 entries
          acc[21 + r] = fmaf(su, ol.eu, fmaf(sv, ol.ev, acc[21 + r]));                               // gc
          acc[27 + r] = fmaf(su, adu, fmaf(sv, adv, acc[27 + r]));                                   // bw
        }
      }
      // ---- stage Y_c = L^-1 W_c (hi / lo): the MMAs that read this buffer two tiles ago must be done
      if (it >= 2 && !tc_bar_wait(s_done + buf, (uint32_t)(((it >> 1) - 1) & 1))) fault = true;
      if (has_cols) {
        const uint32_t ad = y_base + (uint32_t)buf * 2u * (uint32_t)kTcBuf + st_off;
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const float hi = __uint_as_float(__float_as_uint(y[r][j]) & 0xFFFFE000u);  // exactly representable in tf32
            const float lo = y[r][j] - hi;
            const uint32_t off = (uint32_t)(16 * r + (kTcPts / 4) * 128 * j);  // compile-time after unrolling: folds into the store's immediate
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(ad + off), "f"(hi) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(ad + off + (uint32_t)kTcBuf), "f"(lo) : "memory");
          }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the staged rows become visible to the tensor pipe
      __syncwarp();
      if (lane == 0) tc_bar_arrive(s_staged + buf);
      // ---- periodic fp64 fold: tensor-memory accumulators and the per-lane camera sums
      const bool last = it + 1 == n_my;
      if ((it % kTcFlush) == kTcFlush - 1 || last) {
        // every MMA batch of the window must have landed (a commit covers all earlier MMAs)
        if (!tc_bar_wait(s_done + buf, (uint32_t)((it >> 1) & 1))) fault = true;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        double dv[35];
#pragma unroll
        for (int q = 0; q < 33; ++q) dv[q] = (double)acc[q];
        dv[33] = (double)cost;
        dv[34] = (double)nclamp;
#pragma unroll
        for (int q = 0; q < 35; ++q) {
          dv[q] += __shfl_xor_sync(0xffffffffu, dv[q], 8);
          dv[q] += __shfl_xor_sync(0xffffffffu, dv[q], 16);
        }
        if (lane < 8) {
#pragma unroll
          for (int q = 0; q < 35; ++q) s_scr[((size_t)warp * 8 + lane) * 35 + q] = dv[q];
        }
        // accumulator rows 16 w .. 16 w + 15 (cameras 2 w + 1, 2 w + 2) live in lanes 0..15 of tensor-memory subpartition w:
        // warps 0..3 sum the six accumulators and add their rows' upper-triangle entries to the fp64 system
        if (warp < 4) {
          float tot[kTcN];
#pragma unroll
          for (int c2 = 0; c2 < kTcN; ++c2) tot[c2] = 0.f;
          const uint32_t ta = tmem + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
          for (int ac = 0; ac < 6; ++ac) {
            uint32_t r[64];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
              asm volatile(
                  "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                  : "=r"(r[16 * cb + 0]), "=r"(r[16 * cb + 1]), "=r"(r[16 * cb + 2]), "=r"(r[16 * cb + 3]), "=r"(r[16 * cb + 4]), "=r"(r[16 * cb + 5]),
                    "=r"(r[16 * cb + 6]), "=r"(r[16 * cb + 7]), "=r"(r[16 * cb + 8]), "=r"(r[16 * cb + 9]), "=r"(r[16 * cb + 10]), "=r"(r[16 * cb + 11]),
                    "=r"(r[16 * cb + 12]), "=r"(r[16 * cb + 13]), "=r"(r[16 * cb + 14]), "=r"(r[16 * cb + 15])
                  : "r"(ta + (uint32_t)(ac * kTcAccStride) + 16u * cb)
                  : "memory");
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c2 = 0; c2 < kTcN; ++c2) tot[c2] += __uint_as_float(r[c2]);
          }
          const int orow = 16 * warp + lane;                  // operand row: camera slot orow >> 3, parameter orow & 7
          const int row = 6 * (orow >> 3) + (orow & 7);       // row of Sw
          if (lane < 16 && (orow & 7) < 6 && (orow >> 3) < C - 1) {
#pragma unroll
            for (int c2 = 0; c2 < kTcN; ++c2) {
              const int col = 6 * (c2 >> 3) + (c2 & 7);
              if ((c2 & 7) < 6 && (c2 >> 3) < C - 1 && col >= row) s_red[row * L::n - (row * (row - 1)) / 2 + (col - row)] += (double)tot[c2];
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(kCompute) : "memory");  // the compute warps only: the issuer never stops here
        // camera sums: thread (c, q) adds the warps' partials in warp order
        for (int idx = threadIdx.x; idx < (C - 1) * 33 + 2; idx += kCompute) {
          if (idx < (C - 1) * 33) {
            const int c = 1 + idx / 33, q = idx % 33;
            double sum = 0.0;
            for (int w2 = 0; w2 < kTcWarps; ++w2) sum += s_scr[((size_t)w2 * 8 + c) * 35 + q];
            const int o = q < 21 ? L::oHcc + 21 * (c - 1) + q : (q < 27 ? L::oGc + 6 * (c - 1) + (q - 21) : L::oBw + 6 * (c - 1) + (q - 27));
            s_red[o] += sum;
          } else {
            const int q = 33 + (idx - (C - 1) * 33);
            double sum = 0.0;
            for (int w2 = 0; w2 < kTcWarps; ++w2)
              for (int c = 0; c < 8; ++c) sum += s_scr[((size_t)w2 * 8 + c) * 35 + q];
            s_red[q == 33 ? L::oCost : L::oClamp] += sum;
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kCompute) : "memory");
#pragma unroll
        for (int q = 0; q < 33; ++q) acc[q] = 0.f;
        cost = nclamp = 0.f;
      }
    }
    if (fault) __trap();
  }
  __syncthreads();
  double* out = a.partials + (int64_t)blockIdx.x * L::size;
  for (int k = threadIdx.x; k < L::size; k += blockDim.x) out[k] = s_red[k];
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTcTmemCols) : "memory");
}

template <int C>
static int launch_tc(const SkaBaProblem& in, BaKernelArgsW& a, cudaStream_t s) {
  using L = Wide<C>;
  auto kern = ba_linearize_tc_kernel<C>;
  static bool attr_set[64] = {};
  int dev = 0, sms = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  if (dev < 64 && !attr_set[dev]) {
    ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc<C>::smem);
    if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
    attr_set[dev] = true;
  }
  a.n_tiles = (a.N + kTcPts - 1) / kTcPts;
  {
    const uint32_t d = (uint32_t)in.J;
    uint32_t sh = 0;
    while ((1u << sh) < d) ++sh;
    a.div_shift = sh;
    a.div_mul = ((1u << sh) == d) ? 0u : (uint32_t)((((uint64_t)1 << 32) * (((uint64_t)1 << sh) - d)) / d + 1);
  }
  int64_t grid = sms;  // one CTA per SM (its staging buffers take most of the shared memory)
  if (grid > a.n_tiles) grid = a.n_tiles;
  if (grid < 1) grid = 1;
  if (in.ws_bytes < (size_t)grid * L::size * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_workspace_bytes)");
  kern<<<(unsigned)grid, 32 * (kTcWarps + 1), Tc<C>::smem, s>>>(a);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, (int)grid, L::size, in.d_red, s);
}

template <int C, int Loss>
static int launch_wide(const SkaBaProblem& in, BaKernelArgsW& a, cudaStream_t s) {
  using L = Wide<C>;
  auto kern = ba_linearize_wide_kernel<C, Loss>;
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
  if (in.ws_bytes < (size_t)grid * L::size * sizeof(double)) return set_error(SKA_EWORKSPACE, "workspace too small (see ska_ba_workspace_bytes)");
  kern<<<(unsigned)grid, 32 * L::W, L::smem, s>>>(a);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return launch_reduce(a.partials, (int)grid, L::size, in.d_red, s);
}

template <int C>
static int launch_wide(const SkaBaProblem& in, BaKernelArgsW& a, cudaStream_t s) {
  switch (in.loss) {
    case SKA_BA_LOSS_HUBER: return launch_wide<C, kLossHuber>(in, a, s);
    case SKA_BA_LOSS_CAUCHY: return launch_wide<C, kLossCauchy>(in, a, s);
    default: return launch_wide<C, kLossL2>(in, a, s);
  }
}

int ba_linearize_wide(const SkaBaProblem& in, cudaStream_t s) {
  BaKernelArgsW a;
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
  a.Xpp = in.d_Xpp;
  a.partials = (double*)in.d_workspace;
  a.loss = in.loss;
  a.loss_scale = (float)in.loss_scale;
#ifndef SKA_BA_NO_TC
  if (in.C >= 5 && (in.flags & SKA_BA_TENSOR_CORE) && !(in.flags & SKA_BA_FORCE_WIDE)) {  // opt-in: measured slower than the CUDA-core form below
    if (in.loss != SKA_BA_LOSS_L2) return set_error(SKA_EUNSUPPORTED, "the tensor-core Schur form implements the L2 loss only");
    switch (in.C) {
      case 5: return launch_tc<5>(in, a, s);
      case 6: return launch_tc<6>(in, a, s);
      case 7: return launch_tc<7>(in, a, s);
      default: return launch_tc<8>(in, a, s);
    }
  }
#endif
  switch (in.C) {
    case 2: return launch_wide<2>(in, a, s);
    case 3: return launch_wide<3>(in, a, s);
    case 4: return launch_wide<4>(in, a, s);
    case 5: return launch_wide<5>(in, a, s);
    case 6: return launch_wide<6>(in, a, s);
    case 7: return launch_wide<7>(in, a, s);
    case 8: return launch_wide<8>(in, a, s);
    default: return set_error(SKA_EINVAL, "C must be in 2..8");
  }
}

}  // namespace ska
