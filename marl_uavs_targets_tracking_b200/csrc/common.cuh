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

// Fields of a statistics slot (int64): 0-3 the four reward planes as sf_fx counts of the fp32 values written to rew4,
// then covered targets (sum), their maximum, env-steps and the PMI pair rows beyond the tensor path's fp16 range.
enum { ST_REW, ST_TT, ST_BP, ST_DUP, ST_COV, ST_CMAX, ST_ENVS, ST_PMI_OOR, STAT_W };

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
  int *fast_ctr;             // counter-scheduled kernels (fast / generic step, PMI tensor): {next unit of work beyond the first
                             // wave, CTAs that have left}; zero between launches (work_counter_leave rewinds it); launches of one
                             // handle are stream-ordered, so one pair serves all of them
};

struct PmiDev {
  int H;
  const float *w0, *b0, *w1t, *b1, *w2;  // w1t = fc1 weight transposed to [3H,H]
  float b2;
};

typedef void (*StepKernelFn)(const KParams, const UavSimBuffers, const double *, int64_t, int64_t, int, int, double,
                             int, long long *);
struct ActEntry;
typedef void (*FastKernelFn)(const KParams, const UavSimBuffers, const ActEntry *, int64_t, int64_t, int, double, int,
                             long long *);

typedef void (*SmallKernelFn)(const KParams, const UavSimBuffers, const ActEntry *, int64_t, int64_t, int, double, int,
                              long long *, int, uint64_t, uint32_t);

struct PmiTcDev;

struct uavsim {
  UavSimParams hp;
  KParams kp;
  UavSimBuffers buf;
  bool bound;
  int device, sm_count;
  int64_t E;
  double *d_dth;      // [3*na] dt * heading-rate per action (src/agent/uav.py:73-81,96), its cos and sin
  long long *d_stats; // [stat_slots][STAT_W] per-CTA statistics, slot = block index (every step and PMI kernel)
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

// Episode statistics.  Which CTA steps which environment depends on timing wherever the work comes from a launch-wide
// counter (KParams::fast_ctr), so every kernel keeps its statistics as integers: the reward values as counts of 2^-22,
// covered targets and env-steps as plain counts.  Integer sums are exact in any order, hence the totals are the same
// whatever the grouping and whichever kernel served a step.  A value in [-1, 1] as such a count: v + 3 lies in [2, 4],
// where consecutive floats are 2^-22 apart and the bit pattern is linear in the value (round to nearest even): FADD + IADD3.
__device__ __forceinline__ int sf_fx(float v) { return __float_as_int(v + 3.0f) - 0x40400000; }

// Adds the statistics of the calling warp's lanes to `slot` (the CTA's slot of the statistics array, accumulating across
// launches).  Every lane of the warp calls; lanes and fields without a value pass 0.  Lane 0 adds the warp's totals with
// 64-bit atomics (the maximum for ST_CMAX), skipping zeros: no shared memory, no barrier.
__device__ __forceinline__ void stats_commit(long long *slot, long long rew, long long tt, long long bp, long long dup,
                                             long long cov, long long cmax, long long envs, long long pmi_oor = 0) {
  long long v[STAT_W] = {rew, tt, bp, dup, cov, cmax, envs, pmi_oor};
#pragma unroll
  for (int k = 0; k < STAT_W; k++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const long long w = __shfl_xor_sync(0xffffffffu, v[k], o);
      v[k] = (k == ST_CMAX) ? max(v[k], w) : v[k] + w;
    }
  if ((threadIdx.x & 31) != 0) return;
#pragma unroll
  for (int k = 0; k < STAT_W; k++) {
    if (v[k] == 0) continue;
    if (k == ST_CMAX) atomicMax(slot + k, v[k]);
    else atomicAdd(reinterpret_cast<unsigned long long *>(slot + k), (unsigned long long)v[k]);
  }
}

// End of a counter-scheduled launch (KParams::fast_ctr): thread 0 of every CTA signs out after its last unit of work,
// and the last CTA to leave rewinds the counter for the next launch.
__device__ __forceinline__ void work_counter_leave(int *ctr) {
  if (threadIdx.x != 0) return;
  __threadfence();
  if (atomicAdd(ctr + 1, 1) == (int)gridDim.x - 1) { ctr[0] = 0; ctr[1] = 0; __threadfence(); }
}
