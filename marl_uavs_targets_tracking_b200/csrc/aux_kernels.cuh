// aux_kernels.cuh -- reset / begin-episode / random-policy / statistics kernels.
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// reset / begin-episode / random-policy / statistics kernels
// ------------------------------------------------------------------------------------------------
// pre-step observation: lists empty -> -1 blocks, self part x/dc, y/dc, a/Na (src/agent/uav.py:156-190)
__device__ __forceinline__ void write_initial_obs(float *ob, double x, double y, int a, double dc, int na) {
#pragma unroll
  for (int k = 0; k < 9; k++) ob[k] = -1.f;
  ob[9] = (float)(x / dc);
  ob[10] = (float)(y / dc);
  ob[11] = (float)((double)a / (double)na);
}

// Environment.reset (src/environment.py:45-107) with Philox draws instead of Python's `random`.
__global__ void uavsim_reset_kernel(const KParams P, const UavSimBuffers B, uint64_t seed) {
  const int64_t total_u = P.E * P.n, total_t = P.E * P.m;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total_u + total_t; k += stride) {
    if (k < total_u) {
      const int64_t e = k / P.n;
      const int i = (int)(k - e * P.n);
      const uint32_t g = (uint32_t)(P.env_id_offset + e);
      const Philox4 r = philox4x32_10((uint32_t)i, UAVSIM_RNG_UAV_RESET, g, 0u, seed);
      // x_i = i * x_max / (n_uav + 1), i = 1..n ; y = y_max / 2  (environment.py:105-107)
      const double x = (double)(i + 1) * P.x_max / (double)(P.n + 1);
      const double y = P.y_max / 2;
      const double h = -PI_D + (PI_D - (-PI_D)) * philox_u53(r.v[0], r.v[1]);  // random.uniform(-pi, pi)
      const int a = (int)philox_below(r.v[2], (uint32_t)P.na);                   // random.randint(0, na-1)
      B.ux[k] = x; B.uy[k] = y; B.uh[k] = h; B.ua[k] = a;
      write_initial_obs(B.obs + k * 12, x, y, a, P.dc, P.na);
    } else {
      const int64_t kt = k - total_u;
      const int64_t e = kt / P.m;
      const int t = (int)(kt - e * P.m);
      const uint32_t g = (uint32_t)(P.env_id_offset + e);
      const Philox4 r = philox4x32_10((uint32_t)t, UAVSIM_RNG_TGT_POS, g, 0u, seed);
      const Philox4 r2 = philox4x32_10((uint32_t)t, UAVSIM_RNG_TGT_HEAD, g, 0u, seed);
      B.tx[kt] = 0 + (P.x_max - 0) * philox_u53(r.v[0], r.v[1]);   // random.uniform(0, x_max)
      B.ty[kt] = 0 + (P.y_max - 0) * philox_u53(r.v[2], r.v[3]);
      B.th[kt] = -PI_D + (PI_D - (-PI_D)) * philox_u53(r2.v[0], r2.v[1]);
      // r2.v[2..3] is the unused a0 draw (environment.py:81)
    }
  }
}

__global__ void uavsim_initial_obs_kernel(const KParams P, const UavSimBuffers B) {
  const int64_t total_u = P.E * P.n;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total_u; k += stride)
    write_initial_obs(B.obs + k * 12, B.ux[k], B.uy[k], B.ua[k], P.dc, P.na);
}

__global__ void uavsim_random_actions_kernel(const KParams P, int32_t *__restrict__ actions, uint64_t seed,
                                             uint32_t step) {
  const int64_t total_u = P.E * P.n;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total_u; k += stride) {
    const int64_t e = k / P.n;
    const int i = (int)(k - e * P.n);
    const Philox4 r = philox4x32_10((uint32_t)i, UAVSIM_RNG_ACTION, (uint32_t)(P.env_id_offset + e), step, seed);
    actions[k] = (int32_t)philox_below(r.v[0], (uint32_t)P.na);
  }
}

__global__ void uavsim_stats_clear_kernel(long long *stats, int count) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) stats[k] = 0;
}

// Combines the per-CTA slots (common.cuh: ST_*) in one CTA: integer sums and a maximum, exact in any order; the four
// reward counts scale by 2^-22.
__global__ void uavsim_stats_reduce_kernel(const long long *__restrict__ stats, int slots, double *__restrict__ out) {
  __shared__ long long tot[STAT_W];
  if (threadIdx.x < STAT_W) tot[threadIdx.x] = 0;
  __syncthreads();
  long long a[STAT_W] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int s = threadIdx.x; s < slots; s += blockDim.x)
    for (int k = 0; k < STAT_W; k++) {
      const long long v = stats[(size_t)s * STAT_W + k];
      a[k] = (k == ST_CMAX) ? max(a[k], v) : a[k] + v;
    }
  for (int k = 0; k < STAT_W; k++) {
    if (k == ST_CMAX) atomicMax(&tot[k], a[k]);
    else atomicAdd(reinterpret_cast<unsigned long long *>(&tot[k]), (unsigned long long)a[k]);
  }
  __syncthreads();
  if (threadIdx.x < STAT_W) out[threadIdx.x] = (double)tot[threadIdx.x] * (threadIdx.x <= ST_DUP ? 1.0 / 4194304.0 : 1.0);
}
