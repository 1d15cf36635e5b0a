// common.cuh -- parameter blocks, the handle, and small device helpers shared by the kernels of libuavsim.so.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/uavsim.h"
#include "philox.cuh"

#define PMI_NT 256   // threads per CTA, PMI kernel
#define STAT_W 8     // doubles per statistics slot

static thread_local char g_err[512] = "";
#define SET_ERR(...) snprintf(g_err, sizeof(g_err), __VA_ARGS__)
#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      SET_ERR("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                                      \
    }                                                                                      \
  } while (0)

// ------------------------------------------------------------------------------------------------
// kernel-side parameter block
// ------------------------------------------------------------------------------------------------
struct GuardK {
  float t2_up, t2_dn, c1, c0;
};

// Decision bands of the tile step kernel for environments whose entities stay within r of the map centre: per radius
// the centre C of the guard band and its half width H (a pair with |s_f - C| <= H is decided in fp64).
struct TileBand {
  float r, Cp, Hp, Cd, Hd, Cc, Hc, pad;
};

struct KParams {
  int n, m, na, num_steps;
  int64_t E;                  // environments of this handle (plane stride of rew4 is E*n)
  int64_t env_id_offset;      // global id of env 0 (RNG key only)
  double x_max, y_max;
  double dtv_u, dtv_t;        // dt*v_max of UAVs / targets (Python evaluates dt*v_max first)
  double dt, uav_h_max;       // for actions outside the precomputed table
  double dc, dp, two_dp;      // two_dp = radio*dp, radio = 2 (src/agent/uav.py:214)
  double tv, uv;              // target / uav v_max
  double tv_over_uv;
  double s_dp_le, s_dp_lt, s_dc_le, s_2dp_le;  // exact squared thresholds
  double alpha, beta, gamma;
  double tt_hi;               // 2*m_targets            (src/environment.py:207-208)
  double dup_lo;              // -e/2*n_uav             (src/environment.py:209-210)
  double inv_dp, inv_dc, inv_na, inv_tt_hi, inv_dup_span;  // reciprocals for fp32-bound outputs
  // fp32 prefilter: map centre, validity radius, guarded squared thresholds (thr^2 + fp32 error bound)
  double cx, cy, rmax;
  float f_dp, f_dcmv;         // targets: dp; UAVs: max(dc + dt*v_max, 2 dp) (old position bounded through the new one)
  // fp32 classification of the fast step kernel (step_fast_kernel.cuh): per radius the squared threshold rounded up /
  // down to fp32 and the two coefficients of the guard g(R) = c1 R + c0 (R = largest |coordinate - centre| of the
  // environment).  s_f <= t2_dn - g: certainly inside; s_f > t2_up + g: certainly outside; between: decided in fp64.
  GuardK g_dp, g_2dp, g_dc, g_pf;
  float r_fast;   // the fast kernel serves environments whose entities stay within this distance of the map centre
  float r_tile;   // the same for the tile kernel (its fp16 hi + lo operands carry ~22 bits of a coordinate)
  TileBand tb[2]; // bands for a swarm inside / around the map, and for anything up to r_tile
  // fp32 copies of the constants the fast kernel's fp32 output arithmetic uses (no per-iteration conversions)
  float dp_f, inv_dp_f, inv_dc_f, inv_na_f, tt_hi_f, inv_tt_hi_f, dup_lo_f, inv_dup_span_f, alpha_f, beta_f, gamma_f;
  float k_ex1_f, tv_over_uv_f, cx_f, cy_f;
  float dtv_u_f;  // dt*v_max of the UAVs in fp32
  const double *sincos_tab;  // [FM_TAB_SIZE][2] sine / cosine of k pi/32 (fast_math.cuh), device memory
  int stat_slots;            // slots per region of the statistics array
  int *fast_ctr;             // counter-scheduled kernels (fast / generic step, PMI tensor): {next unit of work beyond the first
                             // wave, CTAs that have left}; zero between launches (the last CTA to leave rewinds it); launches of one
                             // handle are stream-ordered, so one pair serves all of them
};

struct PmiDev {
  int H;
  const float *w0, *b0, *w1t, *b1, *w2;  // w1t = fc1 weight transposed to [3H,H]
  float b2;
};

typedef void (*StepKernelFn)(const KParams, const UavSimBuffers, const double *, int64_t, int64_t, int, int, double,
                             int, double *);
struct ActEntry;
typedef void (*FastKernelFn)(const KParams, const UavSimBuffers, const ActEntry *, int64_t, int64_t, int, double, int,
                             double *);

typedef void (*SmallKernelFn)(const KParams, const UavSimBuffers, const ActEntry *, int64_t, int64_t, int, double, int,
                              double *, int, uint64_t, uint32_t);

struct PmiTcDev;

struct uavsim {
  UavSimParams hp;
  KParams kp;
  UavSimBuffers buf;
  bool bound;
  int device, sm_count;
  int64_t E;
  double *d_dth;      // [3*na] dt * heading-rate per action (src/agent/uav.py:73-81,96), its cos and sin
  double *d_stats;    // [3][slots][STAT_W] per-CTA partial sums (step kernel | pmi kernel | fast step kernel: int64 counts of 2^-22)
  double *d_stats8;   // [8] reduced
  double *h_stats8;   // pinned
  int stat_slots;
  int epb, grid_max, nt;   // environments per CTA, resident CTAs, threads per CTA of the step kernel
  StepKernelFn step_fn[2];  // [MASKS]
  size_t smem_step;
  // fast step kernel (64 x 64): [0] plain, [1] with masks / per-target counts
  bool has_fast;
  int step_path;            // 0 auto, 1 generic kernel, 2 per-UAV fast kernel, 3 tile kernel, 4 small-swarm kernel (2-4: error if unusable)
  FastKernelFn fast_fn[2];
  size_t smem_fast[2];
  int fast_grid_max[2];
  // small-swarm step kernel (n, m <= 16, step_small_kernel.cuh): groups of environments in two-warp CTAs
  bool has_small;
  SmallKernelFn small_fn[2];
  int small_grid_max[2];
  // tile step kernel (64 x 64, step_tile_kernel.cuh): [0] plain, [1] with masks / per-target counts
  FastKernelFn tile_fn[2];
  size_t smem_tile[2];
  int tile_grid_max[2];
  ActEntry *d_act;          // [na] per action: dt * rate (fp64), cos / sin of it (fp32)
  double *d_sctab;          // sine / cosine table of the fast kernel's heading routine
  int *d_fast_ctr;          // work counter of the counter-scheduled kernels (KParams::fast_ctr)
  // pmi
  bool has_pmi;
  PmiDev pmi;
  float *d_pmi_blob;
  int pmi_g, pmi_pmax, pmi_tm, pmi_grid_max;
  // tensor-core path (H = 128): fc1 pre-split into UMMA tiles
  bool has_tc;
  bool tc_range;  // the rebalanced weights fit the tensor path's fp16 operands (false: hidden 64 / 128 served by CUDA cores)
  bool has_cc;   // the fp32 CUDA-core PMI kernel fits this shape (its pair buffer is 8 192 rows; n > 91 needs the tensor path)
  int pmi_path;        // 0 auto, 1 CUDA cores, 2 tensor cores
  float *d_tc_tiles;   // [12][2][128*32]
  int tc_g;
  float tc_x_safe;     // largest |input| of a pair row the tensor path's fp16 activations hold (rows beyond are counted)
  size_t smem_pmi;
  // host-buffer pipeline
  cudaStream_t s_in, s_comp, s_out;
  cudaEvent_t ev_user, ev_in[16], ev_comp[16], ev_out[16], ev_done[2];
  int host_chunks;            // chunk count of the host-buffer steps queued so far (0: none yet)
  int64_t host_steps_queued;  // tickets issued by uavsim_step_host / _async
  int64_t t, launches;
};

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
#define PI_D 3.141592653589793

// Python float `%` with a positive divisor (CPython float_rem): fmod, then shift negatives up.
__device__ __forceinline__ double pymod_pos(double a, double b) {
  double r = fmod(a, b);
  if (r < 0.0) r += b;
  return r;
}

// src/utils/data_util.py:43-56 clip_and_normalize, choice 0 with floor 0
__device__ __forceinline__ double clipnorm_0(double v, double hi) {
  v = fmin(fmax(v, 0.0), hi);
  return (v - 0.0) / (hi - 0.0);
}
// choice -1 with ceil 0: (v-floor)/(0-floor) - 1
__device__ __forceinline__ double clipnorm_m1(double v, double lo) {
  v = fmin(fmax(v, lo), 0.0);
  return (v - lo) / (0.0 - lo) - 1.0;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_down_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide reduction of per-thread statistics into this CTA's slot (accumulating across launches;
// one writer per slot, no atomics, so the totals are reproducible for a fixed launch geometry).
// Statistics of kernels whose CTAs draw their work from a launch-wide counter (KParams::fast_ctr): which CTA steps
// which environment depends on timing, so the reward sums are kept as integer counts of 2^-22 -- exact, hence the same
// totals whatever the grouping.  A value in [-1, 1] as such a count: v + 3 lies in [2, 4], where consecutive floats are
// 2^-22 apart and the bit pattern is linear in the value (round to nearest even): FADD + IADD3.
__device__ __forceinline__ int sf_fx(float v) { return __float_as_int(v + 3.0f) - 0x40400000; }

// the four reward sums as 64-bit fixed-point counts
__device__ inline void block_stats_commit_fx(long long *red /*smem [warps][4]*/, long long *slot, long long v0, long long v1, long long v2,
                                             long long v3) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    v0 += __shfl_xor_sync(0xffffffffu, v0, o); v1 += __shfl_xor_sync(0xffffffffu, v1, o);
    v2 += __shfl_xor_sync(0xffffffffu, v2, o); v3 += __shfl_xor_sync(0xffffffffu, v3, o);
  }
  __syncthreads();
  const int nw = (int)(blockDim.x >> 5);   // (red holds [nw][4]: the callers' 64-entry buffers serve up to 16 warps)
  if (lane == 0) { red[wid * 4 + 0] = v0; red[wid * 4 + 1] = v1; red[wid * 4 + 2] = v2; red[wid * 4 + 3] = v3; }
  __syncthreads();
  if (threadIdx.x < 4) {
    long long a = 0;
    for (int w = 0; w < nw; w++) a += red[w * 4 + threadIdx.x];
    slot[threadIdx.x] += a;
  }
  __syncthreads();
}

__device__ void block_stats_commit(double *red /*smem [nwarps*7], at most 64 doubles: 9 warps*/, double *slot, double v0, double v1, double v2,
                                   double v3, double v4, int vmax, double v6, int nthreads) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = nthreads >> 5;
  v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3 = warp_sum(v3); v4 = warp_sum(v4);
  v6 = warp_sum(v6);
  vmax = warp_max(vmax);
  __syncthreads();
  if (lane == 0) {
    red[wid * 7 + 0] = v0; red[wid * 7 + 1] = v1; red[wid * 7 + 2] = v2; red[wid * 7 + 3] = v3;
    red[wid * 7 + 4] = v4; red[wid * 7 + 5] = (double)vmax; red[wid * 7 + 6] = v6;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int w = 0; w < nw; w++) {
      for (int k = 0; k < 5; k++) a[k] += red[w * 7 + k];
      a[5] = fmax(a[5], red[w * 7 + 5]);
      a[6] += red[w * 7 + 6];
    }
    for (int k = 0; k < 5; k++) slot[k] += a[k];
    slot[5] = fmax(slot[5], a[5]);
    slot[6] += a[6];
  }
}

