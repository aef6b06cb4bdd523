// ska_triangulate_impl.cuh - fused weighted V-view DLT triangulation + reprojection scoring, sm_100a.
//
// Persistent kernel: grid = (#SMs x resident CTAs), each CTA walks tiles of kBlock*PTS points with
// a register prefetch of the NEXT tile's keypoints issued before the current tile is solved, so the
// HBM latency of the only loads hides behind ~800 instructions of arithmetic.  One thread owns PTS
// consecutive (frame, joint) points; a warp therefore owns a contiguous group of 32*PTS points
// whose keypoints are one 128-bit (PTS=2) or 64-bit (PTS=1) load per lane and view, coalesced.
// Cameras are compile-time-indexed kernel parameters (constant bank): every P'/K/distortion
// coefficient is an FFMA constant operand - no loads, no shared memory.  The 4x4 normal matrix,
// the secular iteration and the per-view scoring stay in registers; X is staged through shared
// memory per warp so the 12-byte/point output leaves as 128-bit stores.
// Traffic by design: 8V (+4V conf) bytes in, 12 + 4V bytes out per point, nothing re-read.
//
// Replaces: triangulation/triangulate.py:60-68,76-116; vggt/triangulate.py:19-34,64-71;
//           triangulation/reproject.py:49-83,243-244 (file:line in the reference checkout).
#pragma once
#include <cuda_runtime.h>
#ifdef SKA_CTA_WAIT_CLOCKS
#include <cstdio>
#endif

#include "ska_internal.h"
#include "ska_tri_point.cuh"

namespace ska {

template <int V>
struct TriParams {
  CamDev cam[V];
  CamPairDev camp[V / 2];  // the same cameras interleaved by view pairs (tri_point_vp, even V >= 4)
  double P64[V][12];
  float c[3];
  uint32_t weight_sqrt;
  uint32_t frame_major;  // 1: offsets need (t, j); 0: flat point index
  uint32_t x_vec;        // X base 16-byte aligned -> staged 128-bit stores
  int32_t J;
  int64_t N;             // T*J points
  int64_t n_tiles;
  int64_t k_sV, k_sT;    // kpts / proj strides in floats (view, frame)
  int64_t c_sV, c_sT;    // conf / err strides in floats
  const float* kpts;
  const float* conf;
  float* X;
  float* err;
  float* proj;
  uint8_t* status;
};

#ifndef SKA_VP_ROWS
#define SKA_VP_ROWS 2  // view-pair form: where the rows live between the two passes (kRowsRegs / kRowsRecomp / kRowsSmem)
#endif
#ifndef SKA_KBLOCK
#define SKA_KBLOCK 256
#endif
constexpr int kBlock = SKA_KBLOCK;

template <int V, int PTS, bool CONF>
struct TileInputs {
  float u[PTS][V], v[PTS][V], c[PTS][V];
};

// offsets (in floats) of this thread's first point of a tile, within view 0.  Point indices fit
// 32 bits (the C ABI rejects T*J >= 2^31), so the per-tile bookkeeping is 32-bit integer work.
template <int V, int PTS>
__device__ __forceinline__ void point_offsets(const TriParams<V>& prm, uint32_t i0, int64_t& koff, int64_t& coff) {
  if (prm.frame_major) {
    const uint32_t t = i0 / (uint32_t)prm.J;
    const uint32_t j = i0 - t * (uint32_t)prm.J;
    koff = (int64_t)t * prm.k_sT + 2 * (int64_t)j;
    coff = (int64_t)t * prm.c_sT + (int64_t)j;
  } else {
    koff = (int64_t)(2u * (uint64_t)i0);
    coff = (int64_t)i0;
  }
}

// first point of this thread in `tile`, clamped so out-of-range lanes recompute the last point(s)
// and every lane stays alive for the warp votes
template <int PTS>
__device__ __forceinline__ uint32_t thread_point(uint32_t tile, uint32_t N, bool& live) {
  const uint32_t i_raw = (tile * kBlock + threadIdx.x) * PTS;
  live = (i_raw + PTS <= N);
  return live ? i_raw : (N - PTS);
}

template <int V, int PTS, bool CONF>
__device__ __forceinline__ void load_tile(const TriParams<V>& prm, int64_t koff, int64_t coff, TileInputs<V, PTS, CONF>& in) {
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float* kp = prm.kpts + koff + (int64_t)k * prm.k_sV;
    if (PTS == 2) {
      const float4 q = __ldcs(reinterpret_cast<const float4*>(kp));
      in.u[0][k] = q.x; in.v[0][k] = q.y; in.u[PTS - 1][k] = q.z; in.v[PTS - 1][k] = q.w;
    } else {
      const float2 q = __ldcs(reinterpret_cast<const float2*>(kp));
      in.u[0][k] = q.x; in.v[0][k] = q.y;
    }
    if (CONF) {
      if (prm.conf != nullptr) {
        const float* cp = prm.conf + coff + (int64_t)k * prm.c_sV;
        if (PTS == 2) {
          const float2 q = __ldcs(reinterpret_cast<const float2*>(cp));
          in.c[0][k] = q.x; in.c[PTS - 1][k] = q.y;
        } else {
          in.c[0][k] = __ldcs(cp);
        }
      } else {
#pragma unroll
        for (int p = 0; p < PTS; ++p) in.c[p][k] = 1.0f;
      }
    }
  }
}

// LEAN: the common output set (X and err, no proj / status) compiled without the per-view pointer tests.
// (Alternating two prefetch buffers instead of copying `cur = nxt` was tried: the buffers went to local memory and
//  the 8-view shape slowed from 0.84 to 1.05 ms.)
template <int V, int PTS, uint32_t SOLVER, int DIST>
struct TriKernelTraits {
  static constexpr bool kVP = (PTS == 1) && (V >= 4) && (V % 2 == 0) && (DIST <= 1) && (SOLVER == kSolverSecular);
  static constexpr size_t kSlabBytes = (kVP && SKA_VP_ROWS == kRowsSmem) ? (size_t)kBlock * (8 * (V / 2)) * sizeof(F2) : 0;
};

template <int V, int PTS, bool CONF, int DIST, uint32_t SOLVER, int MINB, bool LEAN, bool SAMEK>
__global__ void __launch_bounds__(kBlock, MINB) tri_kernel(const __grid_constant__ TriParams<V> prm) {
  __shared__ __align__(16) float sX[kBlock / 32][32 * PTS * 3];
  extern __shared__ __align__(16) unsigned char tri_slab[];  // view-pair form with kRowsSmem: the rows of every thread
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t N = (uint32_t)prm.N, n_tiles = (uint32_t)prm.n_tiles;

  uint32_t tile = blockIdx.x;
  if (tile >= n_tiles) return;
  bool live;
  uint32_t i0 = thread_point<PTS>(tile, N, live);
  int64_t koff, coff;
  point_offsets<V, PTS>(prm, i0, koff, coff);
  TileInputs<V, PTS, CONF> cur;
  load_tile<V, PTS, CONF>(prm, koff, coff, cur);

  for (;;) {
    // ---- prefetch the next tile of this CTA into registers (loads stay in flight during the solve)
    const uint32_t ntile = tile + gridDim.x;
    const bool more = ntile < n_tiles;
    bool nlive = false;
    uint32_t ni0 = 0;
    int64_t nkoff = 0, ncoff = 0;
    TileInputs<V, PTS, CONF> nxt;
    if (more) {
      ni0 = thread_point<PTS>(ntile, N, nlive);
      point_offsets<V, PTS>(prm, ni0, nkoff, ncoff);
      load_tile<V, PTS, CONF>(prm, nkoff, ncoff, nxt);
    }

    float w2[PTS][V];
#pragma unroll
    for (int p = 0; p < PTS; ++p)
#pragma unroll
      for (int k = 0; k < V; ++k) w2[p][k] = CONF ? (prm.weight_sqrt ? cur.c[p][k] : cur.c[p][k] * cur.c[p][k]) : 1.0f;

    PointSource src;
    src.kpts = prm.kpts + koff;
    src.conf = (prm.conf != nullptr) ? prm.conf + coff : nullptr;
    src.k_sV = prm.k_sV;
    src.c_sV = prm.c_sV;
    src.weight_sqrt = prm.weight_sqrt;

    float X[PTS][3], du[PTS][V], dv[PTS][V];
    uint8_t st[PTS];
    constexpr bool kVP = TriKernelTraits<V, PTS, SOLVER, DIST>::kVP;
    if constexpr (kVP) {
      // many views: one point per thread, per-view work packed over pairs of views
      tri_point_vp<V, CONF, DIST, SKA_VP_ROWS, SAMEK>(prm.camp, prm.cam, prm.P64, prm.c[0], prm.c[1], prm.c[2], cur.u[0], cur.v[0], w2[0], src,
                                                      X[0], du[0], dv[0], st[0], reinterpret_cast<F2*>(tri_slab) + threadIdx.x, kBlock);
    } else {
      tri_points<V, PTS, CONF, DIST, SOLVER, 1, SAMEK>(prm.cam, prm.P64, prm.c[0], prm.c[1], prm.c[2], cur.u, cur.v, w2, src, X, du, dv, st);
    }

    // ---- per-view error / reprojection, coalesced
#pragma unroll
    for (int k = 0; k < V; ++k) {
      if ((LEAN || prm.err != nullptr) && live) {
        float* ep = prm.err + coff + (int64_t)k * prm.c_sV;
        const float e0 = sqrt_fast(fmaf(du[0][k], du[0][k], dv[0][k] * dv[0][k]));
        if (PTS == 2) {
          const float e1 = sqrt_fast(fmaf(du[PTS - 1][k], du[PTS - 1][k], dv[PTS - 1][k] * dv[PTS - 1][k]));
          __stcs(reinterpret_cast<float2*>(ep), make_float2(e0, e1));
        } else {
          __stcs(ep, e0);
        }
      }
      if (!LEAN && prm.proj != nullptr && live) {
        float* pp = prm.proj + koff + (int64_t)k * prm.k_sV;
        if (PTS == 2) {
          __stcs(reinterpret_cast<float4*>(pp),
                 make_float4(cur.u[0][k] + du[0][k], cur.v[0][k] + dv[0][k], cur.u[PTS - 1][k] + du[PTS - 1][k],
                             cur.v[PTS - 1][k] + dv[PTS - 1][k]));
        } else {
          __stcs(reinterpret_cast<float2*>(pp), make_float2(cur.u[0][k] + du[0][k], cur.v[0][k] + dv[0][k]));
        }
      }
    }
    if (!LEAN && prm.status != nullptr && live) {
#pragma unroll
      for (int p = 0; p < PTS; ++p) prm.status[i0 + p] = st[p];
    }

    // ---- X: (N,3) f32.  Stage the warp's 32*PTS*3 floats, then 128-bit stores.
    float* sx = sX[warp];
    __syncwarp();  // previous tile's readers are done with sx
#pragma unroll
    for (int p = 0; p < PTS; ++p) {
#pragma unroll
      for (int k = 0; k < 3; ++k) sx[(lane * PTS + p) * 3 + k] = X[p][k];
    }
    __syncwarp();
    const uint32_t warp_first = (tile * kBlock + warp * 32) * PTS;
    if (warp_first < N) {
      constexpr int kWarpFloats = 32 * PTS * 3, kWarpVec = kWarpFloats / 4;
      const uint32_t remain = N - warp_first;  // points of this warp that exist
      float* gx = prm.X + (int64_t)warp_first * 3;
      if (remain >= 32u * PTS && prm.x_vec) {
        // full warp, 16-byte aligned base (warp_first*3 floats is a multiple of 96 floats): straight-line
        // 128-bit stores, 1.5 (PTS=2) / 0.75 (PTS=1) per lane
#pragma unroll
        for (int r = 0; r < (kWarpVec + 31) / 32; ++r) {
          const int q = lane + 32 * r;
          if (q < kWarpVec) __stcs(reinterpret_cast<float4*>(gx) + q, reinterpret_cast<const float4*>(sx)[q]);
        }
      } else {
        const int nfl = (remain < 32u * PTS ? (int)remain : 32 * PTS) * 3;
        for (int q = lane; q < nfl; q += 32) gx[q] = sx[q];
      }
    }

    if (!more) break;
    tile = ntile;
    i0 = ni0;
    koff = nkoff;
    coff = ncoff;
    live = nlive;
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------
// Hot path (view-major layout, V <= 4, whole 64-point tiles): tri_kernel_cta.
//
// CTA = NW consumer warps + 1 producer warp, one CTA per SM, persistent.  The clip is cut into GROUPS of NW
// consecutive 64-point tiles; CTA b handles groups b, b + grid, ...  For one group the producer thread issues ONE
// bulk-asynchronous copy (TMA 1-D, cp.async.bulk) per view - NW x 512 contiguous bytes of keypoints, plus NW x 256
// bytes of confidences - into a ring of STAGES shared-memory stages; a `full` mbarrier per stage carries the byte
// count, an `empty` mbarrier collects one arrival per consumer warp.  Consumer warp w owns tile w of the group: it
// waits on `full`, reads its lane's two points with one 128-bit shared load per view, releases the stage and runs
// the two points as ONE packed (F2 -> FFMA2) computation.  Consumers issue no global loads and no load addressing;
// the producer costs ~2 instructions per tile (the first form of this kernel fed every consumer warp from its own
// producer lane: 22 serialised single-lane copies per group, ~40 issue slots per tile).
// (16 consumer warps - four per scheduler - with lane 0 of warp 0 as the producer, polling `empty` between its own
// tiles, was built and measured slower: 0.157 against 0.145 ms on config 2, profiles/r03_tri_cta_config2_bounds.log.)
//
// The arithmetic per pair is fast_stage<> (normal matrix, one LDL^T, secular step, certificate) -> ONE warp vote ->
// final row residuals -> scoring.  A warp in which any point fails the certificate (rare: near-degenerate geometry,
// non-finite input) finishes its tile in tri_pair_cold (general secular iteration + fp64 Jacobi), so the
// hot loop carries none of that state.  X leaves through a per-warp staging buffer as 128-bit stores, the per-view
// error as 64-bit stores.
#ifdef SKA_PLAIN_STORES  // measurement variant: default-policy stores instead of st.global.cs
#define SKA_ST(p, v) (*(p) = (v))
#else
#define SKA_ST(p, v) __stcs((p), (v))
#endif
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

#ifndef SKA_CTA_WARPS
#define SKA_CTA_WARPS 15  // consumer warps: (15 + 1) warps x 128 registers = the whole register file (registers are granted per
                          // warp in units of 512, so 14 warps could have 144 each, 12 warps 168); measured: 15 x 128 > 11 x 168
#endif
#ifndef SKA_CTA_STAGES
#define SKA_CTA_STAGES 4
#endif
#ifndef SKA_CTA_MAXREG
#define SKA_CTA_MAXREG 128
#endif
constexpr int kWarpPts = 64;  // points per warp tile (2 per lane)
constexpr int kColdCap = 32;  // per-warp list of tiles deferred to the cold loop

// (A group of NW + 1 tiles whose extra tile rotates over the consumer warps that share the producer warp's scheduler - so
// that every scheduler computes four tiles per group - was measured slower: 0.162 against 0.149 ms on config 2.)
template <int V, int NW, bool CONF, int STAGES>
struct CtaSmem {  // dynamic shared-memory layout of tri_kernel_cta
  static constexpr int kViewK = NW * kWarpPts * 2;           // floats of one view's keypoints in a stage
  static constexpr int kViewC = CONF ? NW * kWarpPts : 0;    // ... confidences
  static constexpr int kKptFloats = V * kViewK;
  static constexpr int kStageFloats = kKptFloats + V * kViewC;
  static constexpr size_t oX = (size_t)STAGES * kStageFloats * sizeof(float);
  static constexpr size_t oFull = oX + (size_t)NW * kWarpPts * 3 * sizeof(float);
  static constexpr size_t oEmpty = oFull + (size_t)STAGES * sizeof(uint64_t);
  static constexpr size_t oState = oEmpty + (size_t)STAGES * sizeof(uint64_t);
  static constexpr size_t oCold = oState + (size_t)NW * 2 * sizeof(uint32_t);
  static constexpr size_t bytes = oCold + (size_t)NW * kColdCap * sizeof(uint32_t);
};

// The rare tile: general secular iteration / fp64 fallback for each point of the lane's pair (the general tri_points<>
// one point at a time: the scalar kernel's arithmetic, in half the registers of the packed pair), results written where
// the hot path writes them.  Runs in the deferred cold loop of tri_kernel_cta, outside the hot loop.
template <int V, bool CONF, int DIST, bool SAMEK>
__device__ __forceinline__ void tri_pair_cold(const TriParams<V>& prm, uint32_t i0, float* sx6) {
#pragma unroll 1
  for (uint32_t i = i0; i < i0 + 2; ++i) {
    float u[1][V], v[1][V], w2[1][V], du[1][V], dv[1][V], X[1][3];
    uint8_t stt[1];
#pragma unroll
    for (int k = 0; k < V; ++k) {  // the stage was handed back: the point is read again from global memory
      const float2 q = *reinterpret_cast<const float2*>(prm.kpts + (int64_t)k * prm.k_sV + 2 * (int64_t)i);
      u[0][k] = q.x;
      v[0][k] = q.y;
      const float cf = CONF ? prm.conf[(int64_t)k * prm.c_sV + i] : 1.0f;
      w2[0][k] = CONF ? (prm.weight_sqrt ? cf : cf * cf) : 1.0f;
    }
    PointSource src;
    src.kpts = prm.kpts + 2 * (int64_t)i;
    src.conf = (CONF && prm.conf != nullptr) ? prm.conf + i : nullptr;
    src.k_sV = prm.k_sV;
    src.c_sV = prm.c_sV;
    src.weight_sqrt = prm.weight_sqrt;
    tri_points<V, 1, CONF, DIST, kSolverSecular, 1, SAMEK>(prm.cam, prm.P64, prm.c[0], prm.c[1], prm.c[2], u, v, w2, src, X, du, dv, stt);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      if (prm.err != nullptr) __stcs(prm.err + (int64_t)k * prm.c_sV + i, sqrt_fast(fmaf(du[0][k], du[0][k], dv[0][k] * dv[0][k])));
      if (prm.proj != nullptr)
        __stcs(reinterpret_cast<float2*>(prm.proj + (int64_t)k * prm.k_sV + 2 * (int64_t)i), make_float2(u[0][k] + du[0][k], v[0][k] + dv[0][k]));
    }
    if (prm.status != nullptr) prm.status[i] = stt[0];
#pragma unroll
    for (int k = 0; k < 3; ++k) sx6[(i - i0) * 3 + k] = X[0][k];
  }
}

// One group's bulk copies into `stage`: one per view (plus one per view of confidences), `full` expects their bytes.
template <int V, bool CONF, int NW, int STAGES>
__device__ __forceinline__ void cta_issue(const TriParams<V>& prm, float* stage, uint64_t* full, uint32_t g, uint32_t n_wt) {
  using L = CtaSmem<V, NW, CONF, STAGES>;
  const uint32_t t0 = g * NW;
  const uint32_t nt = (n_wt - t0 < (uint32_t)NW) ? (n_wt - t0) : (uint32_t)NW;
#ifdef SKA_CTA_L2_WINDOW  // measurement variant: copy from a 32-group window that stays in L2 (same instructions, no HBM reads)
  const uint32_t ts = (g % 32u) * NW;
#else
  const uint32_t ts = t0;
#endif
  mbar_expect_tx(full, (uint32_t)V * nt * (uint32_t)(kWarpPts * (CONF ? 12 : 8)));
#pragma unroll
  for (int k = 0; k < V; ++k) {
    bulk_g2s(stage + k * L::kViewK, prm.kpts + (int64_t)k * prm.k_sV + (int64_t)ts * (kWarpPts * 2), nt * (kWarpPts * 8), full);
    if (CONF)
      bulk_g2s(stage + L::kKptFloats + k * L::kViewC, prm.conf + (int64_t)k * prm.c_sV + (int64_t)ts * kWarpPts, nt * (kWarpPts * 4), full);
  }
}

#ifdef SKA_CTA_WAIT_CLOCKS  // measurement variant: clock64() spent waiting on `full`, summed over the launch and printed
__device__ unsigned long long g_cta_clocks[4];
#endif

// LEAN: the common output set (X and err, no proj / status, 16-byte aligned X) compiled without pointer tests.
//
// Loop state is one counter: k = how many of this CTA's groups were taken; the group is blockIdx.x + k * gridDim.x, its
// stage k % STAGES, the phase parity (k / STAGES) & 1.
template <int V, bool CONF, int DIST, int NW, int STAGES, bool SAMEK, bool LEAN>
__global__ void __maxnreg__(SKA_CTA_MAXREG) tri_kernel_cta(const __grid_constant__ TriParams<V> prm) {
  using L = CtaSmem<V, NW, CONF, STAGES>;
  extern __shared__ __align__(128) unsigned char cta_smem[];
  float* sK = reinterpret_cast<float*>(cta_smem);  // [STAGES][ V x NW x 128 kpts | V x NW x 64 conf ]
  float(*sX)[kWarpPts * 3] = reinterpret_cast<float(*)[kWarpPts * 3]>(cta_smem + L::oX);
  uint64_t* sFull = reinterpret_cast<uint64_t*>(cta_smem + L::oFull);
  uint64_t* sEmpty = reinterpret_cast<uint64_t*>(cta_smem + L::oEmpty);
  uint32_t* sState = reinterpret_cast<uint32_t*>(cta_smem + L::oState);  // per warp: k, n_cold during the cold loop
  uint32_t(*sCold)[kColdCap] = reinterpret_cast<uint32_t(*)[kColdCap]>(cta_smem + L::oCold);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t n_wt = (uint32_t)prm.n_tiles;  // whole 64-point tiles
  const uint32_t n_groups = (n_wt + NW - 1) / NW;
  const uint32_t n_mine = (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x;  // groups of this CTA (grid <= n_groups)
  if (threadIdx.x < STAGES) {
    mbar_init(sFull + threadIdx.x, 1);
    mbar_init(sEmpty + threadIdx.x, NW);  // one arrival per tile
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();  // the only CTA-wide barrier: barrier initialisation

  if (warp == NW) {
    // ---------------------------------------------------------------- producer: one thread
    if (lane == 0) {
      for (uint32_t p = 0; p < n_mine; ++p) {
        if (p >= STAGES) mbar_wait(sEmpty + p % STAGES, (p / STAGES - 1) & 1u);  // every tile of the stage's previous group was taken
        cta_issue<V, CONF, NW, STAGES>(prm, sK + (size_t)(p % STAGES) * L::kStageFloats, sFull + p % STAGES, blockIdx.x + p * gridDim.x, n_wt);
      }
    }
    return;
  }

  // ------------------------------------------------------------------ consumer warps
  float* sx = sX[warp];
  uint32_t* cold = sCold[warp];  // tiles of this warp that failed the certificate vote, finished after the hot loop
  const float cx = prm.c[0], cy = prm.c[1], cz = prm.c[2];
#ifdef SKA_CTA_WAIT_CLOCKS
  unsigned long long wait_clk = 0, n_hot = 0;
  const long long clk_start = clock64();
#endif
  uint32_t k = 0;
  for (;;) {
    uint32_t n_cold = 0;
    // ---- hot loop: certified tiles only
    while (k < n_mine && n_cold < (uint32_t)kColdCap) {
      const uint32_t st = k % STAGES;
      const uint32_t wt = (blockIdx.x + k * gridDim.x) * NW + (uint32_t)warp;
      if (wt >= n_wt) {  // last, partial group: nothing follows for this CTA
        k = n_mine;
        break;
      }
#ifdef SKA_CTA_WAIT_CLOCKS
      const long long w0 = clock64();
      mbar_wait(sFull + st, (k / STAGES) & 1u);
      wait_clk += clock64() - w0;
      ++n_hot;
#else
      mbar_wait(sFull + st, (k / STAGES) & 1u);
#endif
      const float* stage = sK + (size_t)st * L::kStageFloats;
      const uint32_t i0 = wt * kWarpPts + 2u * lane;
      F2 ut[V], vt[V], w2[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float4 q = *reinterpret_cast<const float4*>(stage + v * L::kViewK + warp * (kWarpPts * 2) + 4 * lane);
        ut[v] = mk2(q.x, q.z);
        vt[v] = mk2(q.y, q.w);
        if (CONF) {
          const float2 cf = *reinterpret_cast<const float2*>(stage + L::kKptFloats + v * L::kViewC + warp * kWarpPts + 2 * lane);
          w2[v] = prm.weight_sqrt ? mk2(cf.x, cf.y) : mk2(cf.x * cf.x, cf.y * cf.y);
        } else {
          w2[v] = mk2(1.f, 1.f);
        }
      }
      __syncwarp();                             // every lane holds its pair in registers
      if (lane == 0) mbar_arrive(sEmpty + st);  // this tile's share of the stage goes back to the producer
      ++k;
#ifdef SKA_CTA_NO_MATH  // measurement variant: the staging, the vote and the stores without the arithmetic
      F2 du[V], dv[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        du[v] = ut[v];
        dv[v] = vmul(vt[v], w2[v]);
      }
      const F2 Y0 = ut[0], Y1 = vt[0], Y2 = ut[V - 1];
      if (!__all_sync(0xffffffffu, Y0.x == Y0.x || Y0.y != Y0.y)) continue;
#else
      F2 a[V][4], b[V][4];
      Sym4T<F2> M;
      FastStage<F2> fs;
      fast_stage<V, CONF, 1, F2>(prm.cam, cx, cy, cz, ut, vt, w2, a, b, M, fs);
      // conv is false for non-finite inputs as well (every comparison with NaN fails): one vote decides the tile
      const bool good = mall(fs.conv) && mall(fs.well);
      if (!__all_sync(0xffffffffu, good)) {
        if (lane == 0) cold[n_cold] = wt;
        ++n_cold;
        continue;
      }
      F2 ra[V], rb[V], du[V], dv[V];
      row_residuals<V, F2>(a, b, fs.y0, fs.y1, fs.y2, ra, rb);
      score_views<V, DIST, SAMEK, F2>(prm.cam, fs.y0, fs.y1, fs.y2, ra, rb, ut, vt, du, dv);
      const F2 Y0 = fs.y0, Y1 = fs.y1, Y2 = fs.y2;
#endif
#pragma unroll
      for (int v = 0; v < V; ++v) {
        if (LEAN || prm.err != nullptr) {
          const F2 e = sqrt_fast(vfma(du[v], du[v], vmul(dv[v], dv[v])));
          SKA_ST(reinterpret_cast<float2*>(prm.err + (int64_t)v * prm.c_sV + i0), make_float2(e.x, e.y));
        }
        if (!LEAN && prm.proj != nullptr) {
          const F2 pu = vadd(ut[v], du[v]), pv = vadd(vt[v], dv[v]);
          SKA_ST(reinterpret_cast<float4*>(prm.proj + (int64_t)v * prm.k_sV + 2 * (int64_t)i0), make_float4(pu.x, pv.x, pu.y, pv.y));
        }
      }
      if (!LEAN && prm.status != nullptr) *reinterpret_cast<uchar2*>(prm.status + i0) = make_uchar2(0, 0);
      const F2 X0 = vadd(Y0, cx), X1 = vadd(Y1, cy), X2 = vadd(Y2, cz);
      *reinterpret_cast<float2*>(sx + lane * 6) = make_float2(X0.x, X1.x);
      *reinterpret_cast<float2*>(sx + lane * 6 + 2) = make_float2(X2.x, X0.y);
      *reinterpret_cast<float2*>(sx + lane * 6 + 4) = make_float2(X1.y, X2.y);
      // ---- X through shared memory: 192 floats per warp leave as 48 128-bit stores
      __syncwarp();
      float* gx = prm.X + (int64_t)wt * (kWarpPts * 3);
      if (LEAN || prm.x_vec) {
        SKA_ST(reinterpret_cast<float4*>(gx) + lane, reinterpret_cast<const float4*>(sx)[lane]);
        if (lane < 16) SKA_ST(reinterpret_cast<float4*>(gx) + 32 + lane, reinterpret_cast<const float4*>(sx)[32 + lane]);
      } else {
#pragma unroll
        for (int r = 0; r < 6; ++r) gx[lane + 32 * r] = sx[lane + 32 * r];
      }
      __syncwarp();  // sx is rewritten next iteration
    }
    // ---- cold loop (rare): the tiles the vote rejected, with the general per-point code.  The loop state waits in
    // shared memory (volatile: kept out of the registers the general solver needs, instead of a spill slot that the
    // hot loop would store to on every tile).
    volatile uint32_t* wstate = sState + 2 * warp;
    if (lane == 0) {
      wstate[0] = k;
      wstate[1] = n_cold;
    }
    __syncwarp();
#pragma unroll 1
    for (uint32_t ci = 0; ci < wstate[1]; ++ci) {
      const uint32_t wt = cold[ci];
      tri_pair_cold<V, CONF, DIST, SAMEK>(prm, wt * kWarpPts + 2u * lane, sx + lane * 6);
      __syncwarp();
      float* gx = prm.X + (int64_t)wt * (kWarpPts * 3);
      if (prm.x_vec) {
        __stcs(reinterpret_cast<float4*>(gx) + lane, reinterpret_cast<const float4*>(sx)[lane]);
        if (lane < 16) __stcs(reinterpret_cast<float4*>(gx) + 32 + lane, reinterpret_cast<const float4*>(sx)[32 + lane]);
      } else {
#pragma unroll
        for (int r = 0; r < 6; ++r) gx[lane + 32 * r] = sx[lane + 32 * r];
      }
      __syncwarp();
    }
    k = wstate[0];
    if (k >= n_mine) break;
  }
#ifdef SKA_CTA_WAIT_CLOCKS
  if (lane == 0) {
    atomicAdd(&g_cta_clocks[0], wait_clk);
    atomicAdd(&g_cta_clocks[1], n_hot);
    atomicAdd(&g_cta_clocks[2], (unsigned long long)(clock64() - clk_start));
    __threadfence();
    if (atomicAdd(&g_cta_clocks[3], 1ull) == (unsigned long long)gridDim.x * NW - 1) {  // the last consumer warp of the launch
      const unsigned long long w = g_cta_clocks[0], n = g_cta_clocks[1], t = g_cta_clocks[2];
      printf("tri_kernel_cta wait clocks: %llu tiles, full-barrier wait %.1f cycles/tile, warp lifetime %.1f cycles/tile (%.1f %% waiting)\n", n,
             (double)w / n, (double)t / n, 100.0 * w / t);
      for (int i = 0; i < 4; ++i) g_cta_clocks[i] = 0;
    }
  }
#endif
}

template <int V, bool CONF, int DIST, bool SAMEK, bool LEAN>
static cudaError_t launch_cta_impl(TriParams<V>& prm, cudaStream_t stream) {
  // with confidences a stage is 22.5 KB: the deeper-ring measurement variants keep 8 of them
  constexpr int NW = SKA_CTA_WARPS, STAGES = (CONF && SKA_CTA_STAGES > 8) ? 8 : SKA_CTA_STAGES, BLOCK = 32 * (NW + 1);
  auto kern = tri_kernel_cta<V, CONF, DIST, NW, STAGES, SAMEK, LEAN>;
  constexpr size_t smem = CtaSmem<V, NW, CONF, STAGES>::bytes;
  static_assert(smem <= 227 * 1024, "tri_kernel_cta staging does not fit the SM's shared memory");
  int dev = 0, sms = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  // idempotent
  if (ce != cudaSuccess) return ce;
  const int64_t n_groups = (prm.n_tiles + NW - 1) / NW;
  int64_t grid = sms;  // one persistent CTA per SM
  if (grid > n_groups) grid = n_groups;
  kern<<<(unsigned)grid, BLOCK, smem, stream>>>(prm);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// The same CTA organisation for many views (even V >= 6): tri_kernel_cta_vp.  A warp tile is 32 points, ONE point per
// lane, the per-view work packed over PAIRS OF VIEWS (vp_fast / vp_score of ska_tri_point.cuh).  The lane reads its
// observations from the stage straight into view-pair registers (no global-load addressing, no prefetch registers,
// no pair-assembling moves), parks the rows of the first pass in a shared-memory slab (kRowsSmem) or forms them a
// second time (kRowsRecomp), and the rare tile goes to the deferred cold loop like in tri_kernel_cta.
#ifndef SKA_CTA_VP_ROWS
#define SKA_CTA_VP_ROWS 1  // measured at 8 views: rows formed twice 0.490 ms, rows parked in a shared-memory slab 0.530 ms
#endif
#ifndef SKA_CTA_VP_STAGES
#define SKA_CTA_VP_STAGES 3
#endif
constexpr int kVpPts = 32;

template <int V, int NW, bool CONF, int STAGES, int ROWS>
struct CtaVpSmem {
  static constexpr int kViewK = NW * kVpPts * 2;
  static constexpr int kViewC = CONF ? NW * kVpPts : 0;
  static constexpr int kKptFloats = V * kViewK;
  static constexpr int kStageFloats = kKptFloats + V * kViewC;
  static constexpr int kSlabChunks = (ROWS == kRowsSmem) ? 8 * (V / 2) : 0;  // 8-byte chunks per thread
  static constexpr size_t oSlab = (size_t)STAGES * kStageFloats * sizeof(float);
  static constexpr size_t oX = oSlab + (size_t)NW * 32 * kSlabChunks * sizeof(F2);
  static constexpr size_t oFull = oX + (size_t)NW * kVpPts * 3 * sizeof(float);
  static constexpr size_t oEmpty = oFull + (size_t)STAGES * sizeof(uint64_t);
  static constexpr size_t oCold = oEmpty + (size_t)STAGES * sizeof(uint64_t);
  static constexpr size_t bytes = oCold + (size_t)NW * kColdCap * sizeof(uint32_t);
};

template <int V, bool CONF, int DIST, int NW, int STAGES, int ROWS, bool SAMEK, bool LEAN>
__global__ void __maxnreg__(SKA_CTA_MAXREG) tri_kernel_cta_vp(const __grid_constant__ TriParams<V> prm) {
  using L = CtaVpSmem<V, NW, CONF, STAGES, ROWS>;
  constexpr int H = V / 2;
  extern __shared__ __align__(128) unsigned char cta_smem[];
  float* sK = reinterpret_cast<float*>(cta_smem);
  F2* sSlab = reinterpret_cast<F2*>(cta_smem + L::oSlab);
  float(*sX)[kVpPts * 3] = reinterpret_cast<float(*)[kVpPts * 3]>(cta_smem + L::oX);
  uint64_t* sFull = reinterpret_cast<uint64_t*>(cta_smem + L::oFull);
  uint64_t* sEmpty = reinterpret_cast<uint64_t*>(cta_smem + L::oEmpty);
  uint32_t(*sCold)[kColdCap] = reinterpret_cast<uint32_t(*)[kColdCap]>(cta_smem + L::oCold);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t n_wt = (uint32_t)prm.n_tiles;  // whole 32-point tiles
  const uint32_t n_groups = (n_wt + NW - 1) / NW;
  if (threadIdx.x < STAGES) {
    mbar_init(sFull + threadIdx.x, 1);
    mbar_init(sEmpty + threadIdx.x, NW);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();

  if (warp == NW) {
    // ---------------------------------------------------------------- producer: one thread
    if (lane == 0) {
      int st = 0;
      uint32_t round = 0;
      for (uint32_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        if (round > 0) mbar_wait(sEmpty + st, (round - 1) & 1u);
        const uint32_t t0 = g * NW;
        const uint32_t nt = (n_wt - t0 < (uint32_t)NW) ? (n_wt - t0) : (uint32_t)NW;
        float* stage = sK + (size_t)st * L::kStageFloats;
        mbar_expect_tx(sFull + st, (uint32_t)V * nt * (uint32_t)(kVpPts * (CONF ? 12 : 8)));
#pragma unroll 1
        for (int k = 0; k < V; ++k) {
          bulk_g2s(stage + k * L::kViewK, prm.kpts + (int64_t)k * prm.k_sV + (int64_t)t0 * (kVpPts * 2), nt * (kVpPts * 8), sFull + st);
          if (CONF)
            bulk_g2s(stage + L::kKptFloats + k * L::kViewC, prm.conf + (int64_t)k * prm.c_sV + (int64_t)t0 * kVpPts, nt * (kVpPts * 4),
                     sFull + st);
        }
        if (++st == STAGES) {
          st = 0;
          ++round;
        }
      }
    }
    return;
  }

  // ------------------------------------------------------------------ consumer warps
  int st = 0;
  uint32_t par = 0;
  float* sx = sX[warp];
  uint32_t* cold = sCold[warp];
  F2* rowbuf = sSlab + (size_t)warp * 32 * L::kSlabChunks + lane;  // chunk c of this lane: rowbuf[32 c]
  const float cx = prm.c[0], cy = prm.c[1], cz = prm.c[2];
  uint32_t g = blockIdx.x;
  for (;;) {
    uint32_t n_cold = 0;
    // ---- hot loop: certified tiles only
    for (; g < n_groups && n_cold < (uint32_t)kColdCap; g += gridDim.x) {
      const uint32_t wt = g * NW + warp;
      if (wt >= n_wt) {
        g = n_groups;
        break;
      }
      mbar_wait(sFull + st, par);
      const float* stage = sK + (size_t)st * L::kStageFloats;
      const uint32_t i0 = wt * kVpPts + lane;
      float u[V], v[V];
      F2 w22[H];
#pragma unroll
      for (int k = 0; k < V; ++k) {
        const float2 q = *reinterpret_cast<const float2*>(stage + k * L::kViewK + warp * (kVpPts * 2) + 2 * lane);
        u[k] = q.x;
        v[k] = q.y;
      }
#pragma unroll
      for (int i = 0; i < H; ++i) {
        if (CONF) {
          const float* ca = stage + L::kKptFloats + (2 * i) * L::kViewC + warp * kVpPts + lane;
          const float c0 = ca[0], c1 = ca[L::kViewC];
          w22[i] = prm.weight_sqrt ? mk2(c0, c1) : mk2(c0 * c0, c1 * c1);
        } else {
          w22[i] = mk2(1.f, 1.f);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(sEmpty + st);
      if (++st == STAGES) {
        st = 0;
        par ^= 1u;
      }
      VpRows<V, ROWS> rows;
      Sym4 M;
      SecularState s;
      bool conv, well;
      vp_fast<V, CONF, ROWS>(prm.cam, cx, cy, cz, u, v, w22, rows, rowbuf, 32, M, s, conv, well);
      if (!__all_sync(0xffffffffu, conv && well)) {  // conv is false for non-finite inputs as well
        if (lane == 0) cold[n_cold] = wt;
        ++n_cold;
        continue;
      }
      const float Y[3] = {s.y0, s.y1, s.y2};
      F2 eu2[H], ev2[H];
      vp_score<V, DIST, ROWS, SAMEK>(prm.camp, prm.cam, Y, u, v, rows, rowbuf, 32, eu2, ev2);
#pragma unroll
      for (int i = 0; i < H; ++i) {
        if (LEAN || prm.err != nullptr) {
          const F2 e = sqrt_fast(vfma(eu2[i], eu2[i], vmul(ev2[i], ev2[i])));
          SKA_ST(prm.err + (int64_t)(2 * i) * prm.c_sV + i0, e.x);
          SKA_ST(prm.err + (int64_t)(2 * i + 1) * prm.c_sV + i0, e.y);
        }
        if (!LEAN && prm.proj != nullptr) {
          SKA_ST(reinterpret_cast<float2*>(prm.proj + (int64_t)(2 * i) * prm.k_sV + 2 * (int64_t)i0),
                 make_float2(u[2 * i] + eu2[i].x, v[2 * i] + ev2[i].x));
          SKA_ST(reinterpret_cast<float2*>(prm.proj + (int64_t)(2 * i + 1) * prm.k_sV + 2 * (int64_t)i0),
                 make_float2(u[2 * i + 1] + eu2[i].y, v[2 * i + 1] + ev2[i].y));
        }
      }
      if (!LEAN && prm.status != nullptr) prm.status[i0] = 0;
      sx[lane * 3 + 0] = Y[0] + cx;
      sx[lane * 3 + 1] = Y[1] + cy;
      sx[lane * 3 + 2] = Y[2] + cz;
      __syncwarp();
      float* gx = prm.X + (int64_t)wt * (kVpPts * 3);
      if (LEAN || prm.x_vec) {
        if (lane < 24) SKA_ST(reinterpret_cast<float4*>(gx) + lane, reinterpret_cast<const float4*>(sx)[lane]);
      } else {
#pragma unroll
        for (int r = 0; r < 3; ++r) gx[lane + 32 * r] = sx[lane + 32 * r];
      }
      __syncwarp();
    }
    // ---- cold loop (rare): the tiles the vote rejected, with the general per-point code
    __syncwarp();
#pragma unroll 1
    for (uint32_t ci = 0; ci < n_cold; ++ci) {
      const uint32_t wt = cold[ci];
      const uint32_t i0 = wt * kVpPts + lane;
      float u[V], v[V], w2[V], du[V], dv[V], Xp[3];
#pragma unroll
      for (int k = 0; k < V; ++k) {
        const float2 q = *reinterpret_cast<const float2*>(prm.kpts + (int64_t)k * prm.k_sV + 2 * (int64_t)i0);
        u[k] = q.x;
        v[k] = q.y;
        const float c = CONF ? prm.conf[(int64_t)k * prm.c_sV + i0] : 1.0f;
        w2[k] = prm.weight_sqrt ? c : c * c;
      }
      PointSource src;
      src.kpts = prm.kpts + 2 * (int64_t)i0;
      src.conf = CONF ? prm.conf + i0 : nullptr;
      src.k_sV = prm.k_sV;
      src.c_sV = prm.c_sV;
      src.weight_sqrt = prm.weight_sqrt;
      uint8_t stt;
      tri_point_vp<V, CONF, DIST, kRowsRecomp, SAMEK>(prm.camp, prm.cam, prm.P64, cx, cy, cz, u, v, w2, src, Xp, du, dv, stt);
#pragma unroll
      for (int k = 0; k < V; ++k) {
        if (prm.err != nullptr) prm.err[(int64_t)k * prm.c_sV + i0] = sqrt_fast(fmaf(du[k], du[k], dv[k] * dv[k]));
        if (prm.proj != nullptr)
          *reinterpret_cast<float2*>(prm.proj + (int64_t)k * prm.k_sV + 2 * (int64_t)i0) = make_float2(u[k] + du[k], v[k] + dv[k]);
      }
      if (prm.status != nullptr) prm.status[i0] = stt;
      sx[lane * 3 + 0] = Xp[0];
      sx[lane * 3 + 1] = Xp[1];
      sx[lane * 3 + 2] = Xp[2];
      __syncwarp();
      float* gx = prm.X + (int64_t)wt * (kVpPts * 3);
#pragma unroll
      for (int r = 0; r < 3; ++r) gx[lane + 32 * r] = sx[lane + 32 * r];
      __syncwarp();
    }
    if (g >= n_groups) break;
  }
}

// every view shares view 0's intrinsics and distortion bit for bit (the common rig: one camera model)
template <int V>
static bool same_intrinsics(const TriParams<V>& prm) {
  const CamDev& r = prm.cam[0];
  for (int k = 1; k < V; ++k) {
    const CamDev& c = prm.cam[k];
    bool same = c.fx == r.fx && c.fy == r.fy && c.skew == r.skew && c.ifx == r.ifx && c.ify == r.ify && c.ncx == r.ncx &&
                c.ncy == r.ncy && c.p1 == r.p1 && c.p2 == r.p2 && c.tp1 == r.tp1 && c.tp2 == r.tp2;
    for (int i = 0; i < 3; ++i) same = same && c.dk[i] == r.dk[i] && c.kd[i] == r.kd[i];
    for (int i = 0; i < 4; ++i) same = same && c.s[i] == r.s[i];
    if (!same) return false;
  }
  return true;
}

template <int V, bool CONF, int DIST>
static cudaError_t launch_cta(TriParams<V>& prm, cudaStream_t stream) {
  const bool lean = prm.err != nullptr && prm.proj == nullptr && prm.status == nullptr && prm.x_vec;
  if constexpr (DIST == 1) {
    if (same_intrinsics<V>(prm))
      return lean ? launch_cta_impl<V, CONF, DIST, true, true>(prm, stream) : launch_cta_impl<V, CONF, DIST, true, false>(prm, stream);
  }
  return lean ? launch_cta_impl<V, CONF, DIST, false, true>(prm, stream) : launch_cta_impl<V, CONF, DIST, false, false>(prm, stream);
}

template <int V, bool CONF, int DIST, bool SAMEK, bool LEAN>
static cudaError_t launch_cta_vp_impl(TriParams<V>& prm, cudaStream_t stream) {
  constexpr int NW = SKA_CTA_WARPS, STAGES = SKA_CTA_VP_STAGES, BLOCK = 32 * (NW + 1);
  auto kern = tri_kernel_cta_vp<V, CONF, DIST, NW, STAGES, SKA_CTA_VP_ROWS, SAMEK, LEAN>;
  constexpr size_t smem = CtaVpSmem<V, NW, CONF, STAGES, SKA_CTA_VP_ROWS>::bytes;
  static_assert(smem <= 227 * 1024, "tri_kernel_cta_vp staging does not fit the SM's shared memory");
  int dev = 0, sms = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  // idempotent
  if (ce != cudaSuccess) return ce;
  const int64_t n_groups = (prm.n_tiles + NW - 1) / NW;
  int64_t grid = sms;
  if (grid > n_groups) grid = n_groups;
  kern<<<(unsigned)grid, BLOCK, smem, stream>>>(prm);
  return cudaGetLastError();
}

template <int V, bool CONF, int DIST>
static cudaError_t launch_cta_vp(TriParams<V>& prm, cudaStream_t stream) {
  const bool lean = prm.err != nullptr && prm.proj == nullptr && prm.status == nullptr && prm.x_vec;
  if constexpr (DIST == 1) {
    if (same_intrinsics<V>(prm))
      return lean ? launch_cta_vp_impl<V, CONF, DIST, true, true>(prm, stream) : launch_cta_vp_impl<V, CONF, DIST, true, false>(prm, stream);
  }
  return lean ? launch_cta_vp_impl<V, CONF, DIST, false, true>(prm, stream) : launch_cta_vp_impl<V, CONF, DIST, false, false>(prm, stream);
}

}  // namespace ska

#include "ska_tri_frames.cuh"

namespace ska {

#ifndef SKA_MINB_SMALL
#define SKA_MINB_SMALL 2  // V <= 4: resident CTAs per SM the register allocator must allow
#endif
#ifndef SKA_MINB_LARGE
#define SKA_MINB_LARGE 2  // V >= 5: 2 x 256 threads x 128 registers with the rows recomputed (SKA_VP_RECOMP); 1 x 256 x 206 with the rows kept
#endif
template <int V, int PTS, bool CONF, int DIST, uint32_t SOLVER = kSolverSecular, int MINB = (V <= 4 ? SKA_MINB_SMALL : SKA_MINB_LARGE)>
static cudaError_t launch(TriParams<V>& prm, cudaStream_t stream) {
  // the hot path gets a lean-output instantiation (X and err only: measured 0.84 -> 0.70 ms on the 8-view shape - the
  // per-view pointer tests cost a BSSY/BSYNC pair and a scheduling barrier each); everything else the general one
  constexpr bool kHasLean = (V >= 5) && (SOLVER == kSolverSecular) && (DIST <= 1);  // V <= 4: this kernel only sees tails and odd layouts
  constexpr bool kHasSameK = kHasLean && (DIST == 1) && (V % 2 == 0);                // view-pair form: shared intrinsics loaded once
  const bool lean = kHasLean && prm.err != nullptr && prm.proj == nullptr && prm.status == nullptr;
  void (*kern)(TriParams<V>) = tri_kernel<V, PTS, CONF, DIST, SOLVER, MINB, false, false>;
  if constexpr (kHasLean) {
    if (lean) kern = tri_kernel<V, PTS, CONF, DIST, SOLVER, MINB, true, false>;
  }
  if constexpr (kHasSameK) {
    if (same_intrinsics<V>(prm)) {
      kern = tri_kernel<V, PTS, CONF, DIST, SOLVER, MINB, false, true>;
      if (lean) kern = tri_kernel<V, PTS, CONF, DIST, SOLVER, MINB, true, true>;
    }
  }
  constexpr size_t slab = TriKernelTraits<V, PTS, SOLVER, DIST>::kSlabBytes;
  if (slab > 48 * 1024 - sizeof(float) * kBlock * PTS * 3) {
    const cudaError_t ca = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slab);  // idempotent
    if (ca != cudaSuccess) return ca;
  }
  const int64_t per_tile = (int64_t)kBlock * PTS;
  prm.n_tiles = (prm.N + per_tile - 1) / per_tile;
  int dev = 0, sms = 0, per_sm = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ce != cudaSuccess) return ce;
  ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBlock, slab);
  if (ce != cudaSuccess) return ce;
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)sms * per_sm;  // one wave of resident CTAs, each walks tiles
  if (grid > prm.n_tiles) grid = prm.n_tiles;
  kern<<<(unsigned)grid, kBlock, slab, stream>>>(prm);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Per-frame extrinsics (process_triangulate passes R[i], T[i] per frame: triangulate.py:76-82).
// tri_prep_frames: one thread per frame turns the frame's fp64 [R|t] (T,V,12) into the same
// kernel-side camera the static path prepares on the host (prep_camera / default_centre, identical
// code) and stores it in the caller's workspace; tri_frames_kernel then runs the very same
// tri_points<> arithmetic with cameras read through L1 (the ~J threads of a frame share them).
template <int V>
struct FrameCams {
  CamDev cam[V];
  double P64[V][12];
  float c[4];
};

template <int V>
struct StaticCams {
  SkaCamera cam[V];
};

constexpr int kPrepThreads = 64;

// Each thread builds its frame's cameras in SHARED memory; the block then writes its kPrepThreads structs as one
// contiguous run of 8-byte words.  (Writing the 632-byte structs straight from their threads scattered every store over 32
// sectors: 1 150 B of DRAM writes per 632-byte struct and 0.88 ms per 1 M frames at 6 % issue utilisation.)
template <int V>
__global__ void __launch_bounds__(kPrepThreads) tri_prep_frames(const __grid_constant__ StaticCams<V> st, const double* __restrict__ Rt,
                                                               int64_t T, uint32_t pinhole, FrameCams<V>* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char prep_smem[];
  static_assert(sizeof(FrameCams<V>) % 8 == 0, "block copy moves 8-byte words");
  FrameCams<V>* loc = reinterpret_cast<FrameCams<V>*>(prep_smem);
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x;
  const int64_t t = t0 + threadIdx.x;
  if (t < T) {
    SkaCamera cams[V];
#pragma unroll 1
    for (int v = 0; v < V; ++v) {
      cams[v] = st.cam[v];
      const double* s = Rt + (t * V + v) * 12;
      for (int k = 0; k < 9; ++k) cams[v].R[k] = s[k];
      for (int k = 0; k < 3; ++k) cams[v].t[k] = s[9 + k];
    }
    double c[3];
    default_centre(cams, V, c);
    FrameCams<V>& o = loc[threadIdx.x];
#pragma unroll 1
    for (int v = 0; v < V; ++v) {
      int d = 0;
      const char* why = "";
      CamDev cd;
      double P[12];
      prep_camera(cams[v], c, pinhole != 0, cd, P, d, &why);  // K / dist were validated on the host
      o.cam[v] = cd;
      for (int k = 0; k < 12; ++k) o.P64[v][k] = P[k];
    }
    o.c[0] = (float)c[0];
    o.c[1] = (float)c[1];
    o.c[2] = (float)c[2];
    o.c[3] = 0.f;
  }
  __syncthreads();
  const int64_t left = T - t0;
  const int nvalid = (int)(left < (int64_t)blockDim.x ? left : (int64_t)blockDim.x);
  const int words = nvalid * (int)(sizeof(FrameCams<V>) / 8);
  const uint2* src = reinterpret_cast<const uint2*>(prep_smem);
  uint2* dst = reinterpret_cast<uint2*>(out + t0);
  for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
}

template <int V>
struct TriFrameParams {
  const FrameCams<V>* frames;
  uint32_t weight_sqrt, frame_major;
  int32_t J;
  int64_t N;
  int64_t k_sV, k_sT, c_sV, c_sT;
  const float* kpts;
  const float* conf;
  float* X;
  float* err;
  float* proj;
  uint8_t* status;
};

template <int V>
__global__ void __launch_bounds__(128) tri_frames_kernel(const TriFrameParams<V> prm) {
  const int64_t i_raw = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i_raw < prm.N;
  const int64_t i = live ? i_raw : prm.N - 1;  // every lane stays alive for the warp votes
  const uint32_t t = (uint32_t)i / (uint32_t)prm.J;
  const uint32_t j = (uint32_t)i - t * (uint32_t)prm.J;
  int64_t koff, coff;
  if (prm.frame_major) {
    koff = (int64_t)t * prm.k_sT + 2 * (int64_t)j;
    coff = (int64_t)t * prm.c_sT + (int64_t)j;
  } else {
    koff = 2 * i;
    coff = i;
  }
  float u[1][V], v[1][V], w2[1][V];
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float2 q = __ldg(reinterpret_cast<const float2*>(prm.kpts + koff + (int64_t)k * prm.k_sV));
    u[0][k] = q.x;
    v[0][k] = q.y;
    float c = 1.0f;
    if (prm.conf != nullptr) c = __ldg(prm.conf + coff + (int64_t)k * prm.c_sV);
    w2[0][k] = prm.weight_sqrt ? c : c * c;
  }
  PointSource src;
  src.kpts = prm.kpts + koff;
  src.conf = (prm.conf != nullptr) ? prm.conf + coff : nullptr;
  src.k_sV = prm.k_sV;
  src.c_sV = prm.c_sV;
  src.weight_sqrt = prm.weight_sqrt;
  const FrameCams<V>& fc = prm.frames[t];
  float X[1][3], du[1][V], dv[1][V];
  uint8_t st[1];
  tri_points<V, 1, true, 2, kSolverSecular>(fc.cam, fc.P64, fc.c[0], fc.c[1], fc.c[2], u, v, w2, src, X, du, dv, st);
  if (!live) return;
  prm.X[3 * i] = X[0][0];
  prm.X[3 * i + 1] = X[0][1];
  prm.X[3 * i + 2] = X[0][2];
#pragma unroll
  for (int k = 0; k < V; ++k) {
    if (prm.err != nullptr) prm.err[coff + (int64_t)k * prm.c_sV] = sqrt_fast(fmaf(du[0][k], du[0][k], dv[0][k] * dv[0][k]));
    if (prm.proj != nullptr)
      *reinterpret_cast<float2*>(prm.proj + koff + (int64_t)k * prm.k_sV) = make_float2(u[0][k] + du[0][k], v[0][k] + dv[0][k]);
  }
  if (prm.status != nullptr) prm.status[i] = st[0];
}

// fused path: view-major layout, V <= 4, no skew / thin prism, 16-byte aligned streams, skeletons of >= 8 joints
template <int V>
static int dispatch_frames_fused(const TriArgs& a, bool& taken) {
  taken = false;
  if constexpr (V <= 4) {
    const bool fm = (a.layout == SKA_LAYOUT_FRAME_MAJOR);
    const int64_t N = a.T * (int64_t)a.J;
    auto al = [](const void* p, uintptr_t n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; };
    const bool conf = (a.conf != nullptr);
    if (fm || N < 64 || !al(a.kpts, 16) || !al(a.X, 16) || !al(a.err, 8) || !al(a.proj, 16) || (N % 2 != 0) ||
        (conf && (!al(a.conf, 16) || N % 4 != 0)) || !frames_table_fits<SKA_FR_WARPS>(a.J))
      return SKA_OK;
    TriFramesParams<V> prm;
    int dist = 0;
    const double origin[3] = {0.0, 0.0, 0.0};
    for (int v = 0; v < V; ++v) {
      double P[12];
      int d = 0;
      const char* why = "";
      SkaCamera cam = a.cams[v];
      for (int k = 0; k < 9; ++k) cam.R[k] = (k % 4 == 0) ? 1.0 : 0.0;
      cam.t[0] = cam.t[1] = cam.t[2] = 0.0;
      const int rc = prep_camera(cam, origin, (a.flags & SKA_PINHOLE_REPROJ) != 0, prm.ck[v], P, d, &why);
      if (rc != SKA_OK) return set_error(rc, why);
      dist = d > dist ? d : dist;
      const double k22 = a.cams[v].K[8];
      prm.Kn[v][0] = a.cams[v].K[0] / k22;
      prm.Kn[v][1] = a.cams[v].K[1] / k22;
      prm.Kn[v][2] = a.cams[v].K[2] / k22;
      prm.Kn[v][3] = a.cams[v].K[4] / k22;
      prm.Kn[v][4] = a.cams[v].K[5] / k22;
      prm.cams[v] = a.cams[v];
    }
    if (dist >= 2) return SKA_OK;
    prm.Rt = a.Rt_frames;
    prm.weight_sqrt = (a.flags & SKA_WEIGHT_SQRT) ? 1u : 0u;
    prm.pinhole = (a.flags & SKA_PINHOLE_REPROJ) ? 1u : 0u;
    prm.J = a.J;
    prm.divJ = make_fastdiv((uint32_t)a.J);
    prm.N = N;
    prm.n_tiles = N / 64;
    prm.k_sV = 2 * N;
    prm.c_sV = N;
    prm.kpts = a.kpts;
    prm.conf = a.conf;
    prm.X = a.X;
    prm.err = a.err;
    prm.proj = a.proj;
    prm.status = a.status;
    cudaStream_t s = (cudaStream_t)a.stream;
    const bool lean = a.err != nullptr && a.proj == nullptr && a.status == nullptr;
    cudaError_t ce;
#define SKA_FR(CONF, DIST) (lean ? launch_frames_impl<V, CONF, DIST, true>(prm, s) : launch_frames_impl<V, CONF, DIST, false>(prm, s))
    ce = conf ? (dist ? SKA_FR(true, 1) : SKA_FR(true, 0)) : (dist ? SKA_FR(false, 1) : SKA_FR(false, 0));
#undef SKA_FR
    if (ce == cudaSuccess && prm.n_tiles * 64 < N) {
      const uint32_t first = (uint32_t)(prm.n_tiles * 64);
      if (conf) tri_frames_tail_kernel<V, true><<<1, 64, 0, s>>>(prm, first);
      else tri_frames_tail_kernel<V, false><<<1, 64, 0, s>>>(prm, first);
      ce = cudaGetLastError();
    }
    if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
    taken = true;
  }
  return SKA_OK;
}

template <int V>
static int dispatch_frames(const TriArgs& a) {
#ifndef SKA_NO_FRAMES_FUSED
  {
    bool taken = false;
    const int rc = dispatch_frames_fused<V>(a, taken);
    if (rc != SKA_OK || taken) return rc;
  }
#endif
  if (a.ws_bytes < (size_t)a.T * sizeof(FrameCams<V>) || a.workspace == nullptr)
    return set_error(SKA_EWORKSPACE, "workspace too small (see ska_tri_frames_workspace_bytes)");
  if (reinterpret_cast<uintptr_t>(a.workspace) % 16 != 0) return set_error(SKA_EALIGN, "workspace must be 16-byte aligned");
  StaticCams<V> st;
  const double origin[3] = {0.0, 0.0, 0.0};
  for (int v = 0; v < V; ++v) {  // validate K / dist once on the host (R, t are per frame)
    CamDev tmp;
    double P[12];
    int d = 0;
    const char* why = "";
    const int rc = prep_camera(a.cams[v], origin, (a.flags & SKA_PINHOLE_REPROJ) != 0, tmp, P, d, &why);
    if (rc != SKA_OK) return set_error(rc, why);
    st.cam[v] = a.cams[v];
  }
  cudaStream_t s = (cudaStream_t)a.stream;
  FrameCams<V>* frames = reinterpret_cast<FrameCams<V>*>(a.workspace);
  {
    const size_t smem = (size_t)kPrepThreads * sizeof(FrameCams<V>);
    static bool attr_set[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev < 64 && !attr_set[dev] && smem > 48 * 1024) {  // idempotent; a benign race sets it twice
      const cudaError_t ca = cudaFuncSetAttribute(tri_prep_frames<V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (ca != cudaSuccess) return set_error((int)ca, cudaGetErrorString(ca));
      attr_set[dev] = true;
    }
    tri_prep_frames<V><<<(unsigned)((a.T + kPrepThreads - 1) / kPrepThreads), kPrepThreads, smem, s>>>(
        st, a.Rt_frames, a.T, (a.flags & SKA_PINHOLE_REPROJ) ? 1u : 0u, frames);
  }
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  TriFrameParams<V> prm;
  prm.frames = frames;
  prm.weight_sqrt = (a.flags & SKA_WEIGHT_SQRT) ? 1u : 0u;
  prm.J = a.J;
  prm.N = a.T * (int64_t)a.J;
  const bool fm = (a.layout == SKA_LAYOUT_FRAME_MAJOR);
  prm.frame_major = fm ? 1u : 0u;
  if (fm) {
    prm.k_sV = 2 * (int64_t)a.J;
    prm.k_sT = 2 * (int64_t)a.J * V;
    prm.c_sV = a.J;
    prm.c_sT = (int64_t)a.J * V;
  } else {
    prm.k_sV = 2 * prm.N;
    prm.k_sT = 2 * (int64_t)a.J;
    prm.c_sV = prm.N;
    prm.c_sT = a.J;
  }
  prm.kpts = a.kpts;
  prm.conf = a.conf;
  prm.X = a.X;
  prm.err = a.err;
  prm.proj = a.proj;
  prm.status = a.status;
  tri_frames_kernel<V><<<(unsigned)((prm.N + 127) / 128), 128, 0, s>>>(prm);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return SKA_OK;
}

template <int V>
static size_t frames_ws_bytes(int64_t T) {
  return (size_t)T * sizeof(FrameCams<V>);
}

template <int V>
static int dispatch(const TriArgs& a) {
  if (a.Rt_frames != nullptr) return dispatch_frames<V>(a);
  TriParams<V> prm;
  int dist = 0;  // max distortion level over the views: 0 pinhole, 1 rational+tangential, 2 prism/skew
  for (int v = 0; v < V; ++v) {
    int d = 0;
    const char* why = "";
    const int rc = prep_camera(a.cams[v], a.centre, (a.flags & SKA_PINHOLE_REPROJ) != 0, prm.cam[v], prm.P64[v], d, &why);
    if (rc != SKA_OK) return set_error(rc, why);
    dist = d > dist ? d : dist;
  }
  for (int k = 0; k < 3; ++k) prm.c[k] = (float)a.centre[k];
  for (int i = 0; i < V / 2; ++i) make_cam_pair(prm.cam[2 * i], prm.cam[2 * i + 1], prm.camp[i]);
  const uint32_t solver = a.flags & SKA_SOLVER_MASK;
  prm.weight_sqrt = (a.flags & SKA_WEIGHT_SQRT) ? 1u : 0u;
  prm.J = a.J;
  prm.N = a.T * (int64_t)a.J;
  const bool fm = (a.layout == SKA_LAYOUT_FRAME_MAJOR);
  prm.frame_major = fm ? 1u : 0u;
  if (fm) {
    prm.k_sV = 2 * (int64_t)a.J;
    prm.k_sT = 2 * (int64_t)a.J * V;
    prm.c_sV = a.J;
    prm.c_sT = (int64_t)a.J * V;
  } else {
    prm.k_sV = 2 * prm.N;
    prm.k_sT = 2 * (int64_t)a.J;
    prm.c_sV = prm.N;
    prm.c_sT = a.J;
  }
  prm.kpts = a.kpts;
  prm.conf = a.conf;
  prm.X = a.X;
  prm.err = a.err;
  prm.proj = a.proj;
  prm.status = a.status;
  auto al = [](const void* p, uintptr_t n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; };
  prm.x_vec = al(a.X, 16) ? 1u : 0u;
  const bool conf = (a.conf != nullptr);
  // pair path: flat point index, even point count, vector-aligned streams
  const bool pair_ok = !fm && (prm.N % 2 == 0) && al(a.kpts, 16) && al(a.conf, 8) && al(a.err, 8) && al(a.proj, 16);
  // V <= 4: tri_kernel_cta (bulk-staged whole 64-point tiles, point pairs packed, rows in registers) + tri_kernel for
  //         the < 64-point tail and everything the pair path cannot take.
  // V >= 5: tri_kernel, one point per thread; for even V its per-view work is packed over view pairs (tri_point_vp).
  // Forms that were built, measured slower and removed: a producer LANE per consumer warp (22 single-lane copies per
  // group), the bulk-staged kernel for V = 6, 8, a streaming three-pass form (profiles/r01_tri_kernel_variants.txt).
  // the bulk copies need 16-byte aligned view bases: the confidence plane of view k starts at k * N floats
  const bool cta_ok = (V <= 4) && pair_ok && (!conf || (al(a.conf, 16) && prm.N % 4 == 0));
  cudaError_t ce;
  cudaStream_t s = (cudaStream_t)a.stream;
#define SKA_GO(PTS)                                                                      \
  (conf ? (dist ? launch<V, PTS, true, 1>(prm, s) : launch<V, PTS, true, 0>(prm, s))     \
        : (dist ? launch<V, PTS, false, 1>(prm, s) : launch<V, PTS, false, 0>(prm, s)))
  if (solver == kSolverJacobi64) {
    // exact / measurement solvers: one generic instantiation (weights and full distortion always on)
    ce = launch<V, 1, true, 2, kSolverJacobi64, 1>(prm, s);
  } else if (solver == kSolverJacobi32) {
    ce = launch<V, 1, true, 2, kSolverJacobi32, 1>(prm, s);
  } else if (dist >= 2) {
    ce = launch<V, 1, true, 2, kSolverSecular, 1>(prm, s);  // thin prism / skew: rare, one generic instantiation
  } else if constexpr (V <= 4) {
    if (cta_ok) {
      // whole 64-point tiles -> bulk-staged kernel; the < 64-point tail -> tri_kernel
      const int64_t n_full = prm.N / kWarpPts, done = n_full * kWarpPts;
      ce = cudaSuccess;
      if (n_full > 0) {
        TriParams<V> q = prm;
        q.n_tiles = n_full;
        ce = conf ? (dist ? launch_cta<V, true, 1>(q, s) : launch_cta<V, true, 0>(q, s))
                  : (dist ? launch_cta<V, false, 1>(q, s) : launch_cta<V, false, 0>(q, s));
      }
      if (ce == cudaSuccess && done < prm.N) {
        prm.N -= done;  // strides keep describing the whole clip
        prm.kpts += 2 * done;
        if (prm.conf != nullptr) prm.conf += done;
        prm.X += 3 * done;
        if (prm.err != nullptr) prm.err += done;
        if (prm.proj != nullptr) prm.proj += 2 * done;
        if (prm.status != nullptr) prm.status += done;
        ce = SKA_GO(2);
      }
    } else {
      ce = pair_ok ? SKA_GO(2) : SKA_GO(1);
    }
  } else if constexpr (V % 2 == 0) {
    // even V >= 6: whole 32-point tiles -> bulk-staged view-pair kernel; the tail and unaligned / frame-major input -> tri_kernel
    const bool vp_ok = !fm && al(a.kpts, 16) && (prm.N % 2 == 0) && al(a.X, 16) && al(a.proj, 8) && (!conf || (al(a.conf, 16) && prm.N % 4 == 0));
#ifdef SKA_NO_CTA_VP
    const bool use_vp = false;
#else
    const bool use_vp = vp_ok;
#endif
    if (use_vp) {
      const int64_t n_full = prm.N / kVpPts, done = n_full * kVpPts;
      ce = cudaSuccess;
      if (n_full > 0) {
        TriParams<V> q = prm;
        q.n_tiles = n_full;
        ce = conf ? (dist ? launch_cta_vp<V, true, 1>(q, s) : launch_cta_vp<V, true, 0>(q, s))
                  : (dist ? launch_cta_vp<V, false, 1>(q, s) : launch_cta_vp<V, false, 0>(q, s));
      }
      if (ce == cudaSuccess && done < prm.N) {
        prm.N -= done;
        prm.kpts += 2 * done;
        if (prm.conf != nullptr) prm.conf += done;
        prm.X += 3 * done;
        if (prm.err != nullptr) prm.err += done;
        if (prm.proj != nullptr) prm.proj += 2 * done;
        if (prm.status != nullptr) prm.status += done;
        ce = SKA_GO(1);
      }
    } else {
      ce = SKA_GO(1);
    }
  } else {
    ce = SKA_GO(1);
  }
#undef SKA_GO
  if (ce != cudaSuccess) return set_error((int)ce, cudaGetErrorString(ce));
  return SKA_OK;
}

}  // namespace ska
