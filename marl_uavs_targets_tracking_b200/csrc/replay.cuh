// replay.cuh -- prioritized replay on the device (SURVEY.md section 8f, row f-2).
//
// Semantics of the reference's PrioritizedReplayBuffer (src/train.py:73-139), restated for whole batches:
//   add      every inserted transition gets the current maximum priority (1.0 for an empty buffer) at ring position
//            pos, pos+1, ...; the maximum is invariant during an add because every value written equals it
//            (train.py:88-98).  Only the last `capacity` transitions of a longer batch survive, like the deque.
//   sample   p = priority^alpha / sum (float32, train.py:109-110); indices by numpy's choice(p=...): float64 inclusive
//            scan of p, normalised by its last element, searchsorted(cdf, u, side='right') (train.py:112);
//            weights (size * p[idx])^-beta / max (train.py:116-118).
//   update   priorities[idx[k]] = new[k] in order k = 0, 1, ...: for a repeated index the LAST write wins
//            (train.py:134-136).
// The reference keeps python objects in a deque and calls priorities.max() once per inserted transition
// (O(capacity) each); here the transitions stay in HBM as structure-of-arrays rows and every call is a few launches.
#pragma once
#include "common.cuh"
#include "philox.cuh"

#define REPLAY_NT 256
#define REPLAY_SCAN_ELEMS 2048  // elements per block of the scan (8 per thread)

struct uavsim_replay {
  int device;
  int64_t capacity, size, pos;
  int state_dim;
  float alpha;
  float *states, *next_states, *rewards, *priorities;  // [C,D] [C,D] [C] [C]
  int32_t *actions;                                    // [C]
  int32_t *owner;                                      // [C] scratch of update (-1 when idle)
  float *prob;                                         // [C] priority^alpha, then normalised
  double *cdf;                                         // [C] inclusive scan of prob
  double *block_sums;                                  // [ceil(C / REPLAY_SCAN_ELEMS) + 1]
  float *scalars;                                      // [0] max priority, [1] sum of p^alpha, [2] max weight
  int64_t launches;
};

// ---- add ---------------------------------------------------------------------------------------
// As signed integers, non-negative floats order like their values and -0.0f (0x80000000, INT_MIN) ranks below +0.0f,
// so `out` (cleared to +0.0f) ends at priorities.max() whichever zero fmaxf returns for a slot holding -0.0f.
__global__ void replay_max_kernel(const float *__restrict__ pri, int64_t n, float *__restrict__ out) {
  float m = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, pri[i]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int *>(out), __float_as_int(m));
}

// rows [skip, count) of the batch go to ring slots (pos + k) % capacity; one thread per float of a row
__global__ void replay_add_kernel(uavsim_replay R, const float *__restrict__ s, const int32_t *__restrict__ a,
                                  const float *__restrict__ r, const float *__restrict__ s2, int64_t skip, int64_t count,
                                  int empty) {
  const int D = R.state_dim;
  const int64_t total = (count - skip) * D;
  const float maxp = empty ? 1.0f : R.scalars[0];
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = skip + t / D;
    const int d = (int)(t % D);
    const int64_t slot = (R.pos + k) % R.capacity;
    R.states[slot * D + d] = s[k * D + d];
    R.next_states[slot * D + d] = s2[k * D + d];
    if (d == 0) {
      R.actions[slot] = a[k];
      R.rewards[slot] = r[k];
      R.priorities[slot] = maxp;
    }
  }
}

// ---- sample ------------------------------------------------------------------------------------
// q = priority^alpha and per-block fp64 partial sums (fixed order: deterministic)
__global__ void replay_pow_kernel(uavsim_replay R, int64_t n) {
  __shared__ double red[REPLAY_NT / 32];
  const int64_t base = (int64_t)blockIdx.x * REPLAY_SCAN_ELEMS;
  double acc = 0;
  for (int k = threadIdx.x; k < REPLAY_SCAN_ELEMS; k += REPLAY_NT) {
    const int64_t i = base + k;
    if (i < n) {
      const float q = powf(R.priorities[i], R.alpha);
      R.prob[i] = q;
      acc += (double)q;
    }
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int w = 0; w < REPLAY_NT / 32; w++) s += red[w];
    R.block_sums[blockIdx.x] = s;
  }
}

// one block: total = sum of the block sums -> scalars[1] (float32, like numpy's float32 sum up to rounding)
__global__ void replay_total_kernel(uavsim_replay R, int nblocks) {
  if (threadIdx.x == 0) {
    double s = 0;
    for (int b = 0; b < nblocks; b++) s += R.block_sums[b];
    R.scalars[1] = (float)s;
    R.scalars[2] = 0.f;
  }
}

// p = q / total (float32 division, train.py:110) and the per-block sums of p in fp64
__global__ void replay_norm_kernel(uavsim_replay R, int64_t n) {
  __shared__ double red[REPLAY_NT / 32];
  const int64_t base = (int64_t)blockIdx.x * REPLAY_SCAN_ELEMS;
  const float total = R.scalars[1];
  double acc = 0;
  for (int k = threadIdx.x; k < REPLAY_SCAN_ELEMS; k += REPLAY_NT) {
    const int64_t i = base + k;
    if (i < n) {
      const float p = R.prob[i] / total;
      R.prob[i] = p;
      acc += (double)p;
    }
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int w = 0; w < REPLAY_NT / 32; w++) s += red[w];
    R.block_sums[blockIdx.x] = s;
  }
}

// one block: exclusive scan of the block sums in place (nblocks <= a few thousand); block_sums[nblocks] = the total
__global__ void replay_scan_blocks_kernel(uavsim_replay R, int nblocks) {
  if (threadIdx.x == 0) {
    double run = 0;
    for (int b = 0; b < nblocks; b++) { const double v = R.block_sums[b]; R.block_sums[b] = run; run += v; }
    R.block_sums[nblocks] = run;
  }
}

// Inclusive fp64 scan of each block of REPLAY_SCAN_ELEMS slots, placed between the block's offsets B_b = block_sums[b]
// and B_{b+1} = fl(B_b + S_b) (replay_scan_blocks_kernel).  The in-block sums x_i (the thread's running sum on its offset
// in the block) round differently from S_b and from the next thread's offset, so written as they are they could step
// down at a thread, warp or block start and give a slot with p = 0 an interval an ulp wide.  Instead
//   cdf_i = B_{b+1}                          from the block's last slot with p > 0 on,
//   cdf_i = min(fl(B_b + M_i), B_{b+1})      before it, M_i = max of x_j over the block's slots j <= i with p_j > 0 (0 if none).
// The maximum is exact in any order and fl(B_b + .) is monotone, so the CDF never steps down, and a slot with p = 0
// repeats the value before it (B_b at a block's start, the previous block's last value): its interval is empty and the
// search never returns it.  Every cdf_i stays within the rounding of the chains that made x_i, B_b and B_{b+1}.
__global__ void replay_scan_kernel(uavsim_replay R, int64_t n) {
  __shared__ double warp_tot[REPLAY_NT / 32], warp_max[REPLAY_NT / 32];
  __shared__ int warp_last[REPLAY_NT / 32];
  constexpr int PER = REPLAY_SCAN_ELEMS / REPLAY_NT;
  const int64_t base = (int64_t)blockIdx.x * REPLAY_SCAN_ELEMS + (int64_t)threadIdx.x * PER;
  double v[PER], run = 0;
  unsigned pos = 0;  // bit k: slot base + k has p > 0
#pragma unroll
  for (int k = 0; k < PER; k++) {
    const float p = (base + k < n) ? R.prob[base + k] : 0.f;
    run += (double)p;
    v[k] = run;
    if (p > 0.f) pos |= 1u << k;
  }
  double inc = run;  // inclusive scan of the per-thread totals across the block
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  double off = 0;
  for (int w = 0; w < wid; w++) off += warp_tot[w];
  off += inc - run;
  double m = 0;  // running maximum of x over the thread's slots with p > 0
#pragma unroll
  for (int k = 0; k < PER; k++) { if (pos >> k & 1) m = fmax(m, off + v[k]); v[k] = m; }
  double mi = m;  // inclusive maximum over the warp's threads
  for (int o = 1; o < 32; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, mi, o); if (lane >= o) mi = fmax(mi, u); }
  double before = __shfl_up_sync(0xffffffffu, mi, 1);  // maximum over the block's earlier threads
  if (lane == 0) before = 0;
  const int wlast = __reduce_max_sync(0xffffffffu, pos ? (int)threadIdx.x * PER + 31 - __clz(pos) : -1);
  if (lane == 31) warp_max[wid] = mi;
  if (lane == 0) warp_last[wid] = wlast;
  __syncthreads();
  int last = -1;  // the block's last slot with p > 0
  for (int w = 0; w < REPLAY_NT / 32; w++) { last = max(last, warp_last[w]); if (w < wid) before = fmax(before, warp_max[w]); }
  const double b0 = R.block_sums[blockIdx.x], b1 = R.block_sums[blockIdx.x + 1];
#pragma unroll
  for (int k = 0; k < PER; k++)
    if (base + k < n) R.cdf[base + k] = (int)threadIdx.x * PER + k >= last ? b1 : fmin(b0 + fmax(before, v[k]), b1);
}

// one thread per drawn sample: u -> index (searchsorted right on cdf / cdf[n-1]), gather the row, raw weight
__global__ void replay_draw_kernel(uavsim_replay R, int64_t n, int64_t batch, float beta, const double *__restrict__ uniforms,
                                   uint64_t seed, uint64_t counter, float *__restrict__ o_s, int32_t *__restrict__ o_a,
                                   float *__restrict__ o_r, float *__restrict__ o_s2, int64_t *__restrict__ o_idx,
                                   float *__restrict__ o_w) {
  const int D = R.state_dim;
  const double last = R.cdf[n - 1];
  float wmax = 0.f;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < batch; k += (int64_t)gridDim.x * blockDim.x) {
    double u;
    if (uniforms) {
      u = uniforms[k];
    } else {
      const Philox4 x = philox4x32_10((uint32_t)k, (uint32_t)(k >> 32), (uint32_t)counter, (uint32_t)(counter >> 32), seed);
      u = philox_u53(x.v[0], x.v[1]);
    }
    int64_t lo = 0, hi = n;  // first index with cdf[i] / last > u
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (R.cdf[mid] / last <= u) lo = mid + 1; else hi = mid;
    }
    const int64_t idx = lo < n ? lo : n - 1;
    o_idx[k] = idx;
    for (int d = 0; d < D; d++) { o_s[k * D + d] = R.states[idx * D + d]; o_s2[k * D + d] = R.next_states[idx * D + d]; }
    o_a[k] = R.actions[idx];
    o_r[k] = R.rewards[idx];
    const float w = powf((float)n * R.prob[idx], -beta);
    o_w[k] = w;
    wmax = fmaxf(wmax, w);
  }
  for (int o = 16; o; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int *>(R.scalars + 2), __float_as_uint(wmax));
}

__global__ void replay_weight_norm_kernel(uavsim_replay R, int64_t batch, float *__restrict__ o_w) {
  const float m = R.scalars[2];
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < batch; k += (int64_t)gridDim.x * blockDim.x) o_w[k] = o_w[k] / m;
}

// ---- update_priorities: last write wins ----------------------------------------------------------
__global__ void replay_claim_kernel(uavsim_replay R, const int64_t *__restrict__ idx, int64_t count) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < count; k += (int64_t)gridDim.x * blockDim.x)
    atomicMax(R.owner + idx[k], (int32_t)k);
}
__global__ void replay_write_kernel(uavsim_replay R, const int64_t *__restrict__ idx, const float *__restrict__ pri, int64_t count) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < count; k += (int64_t)gridDim.x * blockDim.x)
    if (R.owner[idx[k]] == (int32_t)k) R.priorities[idx[k]] = pri[k];
}
__global__ void replay_release_kernel(uavsim_replay R, const int64_t *__restrict__ idx, int64_t count) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < count; k += (int64_t)gridDim.x * blockDim.x) R.owner[idx[k]] = -1;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int replay_grid(int64_t work) {
  int64_t b = (work + REPLAY_NT - 1) / REPLAY_NT;
  return (int)(b < 1 ? 1 : (b > 148 * 8 ? 148 * 8 : b));
}

extern "C" int uavsim_replay_create(int64_t capacity, int state_dim, double alpha, int device, uavsim_replay_t **out) {
  if (!out || capacity <= 0 || capacity > (1ll << 31) - 1 || state_dim <= 0) { SET_ERR("uavsim_replay_create: bad argument"); return UAVSIM_ERR_ARG; }
  *out = nullptr;
  CUDA_TRY(cudaSetDevice(device));
  uavsim_replay *h = (uavsim_replay *)calloc(1, sizeof(uavsim_replay));
  if (!h) { SET_ERR("uavsim_replay_create: out of host memory"); return UAVSIM_ERR_ARG; }
  h->device = device; h->capacity = capacity; h->state_dim = state_dim; h->alpha = (float)alpha;
  const size_t C = (size_t)capacity, nb = (C + REPLAY_SCAN_ELEMS - 1) / REPLAY_SCAN_ELEMS + 1;
  int rc = 0;
#define REPLAY_ALLOC(p, bytes) if (!rc) { cudaError_t e_ = cudaMalloc((void **)&(p), (bytes)); if (e_ != cudaSuccess) { SET_ERR("uavsim_replay_create: cudaMalloc: %s", cudaGetErrorString(e_)); rc = (int)e_; } }
  REPLAY_ALLOC(h->states, C * state_dim * 4) REPLAY_ALLOC(h->next_states, C * state_dim * 4)
  REPLAY_ALLOC(h->rewards, C * 4) REPLAY_ALLOC(h->priorities, C * 4) REPLAY_ALLOC(h->actions, C * 4)
  REPLAY_ALLOC(h->owner, C * 4) REPLAY_ALLOC(h->prob, C * 4) REPLAY_ALLOC(h->cdf, C * 8)
  REPLAY_ALLOC(h->block_sums, nb * 8) REPLAY_ALLOC(h->scalars, 16)
#undef REPLAY_ALLOC
  if (!rc) {
    cudaError_t e = cudaMemset(h->priorities, 0, C * 4);
    if (e == cudaSuccess) e = cudaMemset(h->owner, 0xff, C * 4);
    if (e == cudaSuccess) e = cudaMemset(h->scalars, 0, 16);
    if (e != cudaSuccess) { SET_ERR("uavsim_replay_create: cudaMemset: %s", cudaGetErrorString(e)); rc = (int)e; }
  }
  if (rc) { uavsim_replay_destroy(h); return rc; }
  *out = h;
  return 0;
}

extern "C" int uavsim_replay_destroy(uavsim_replay_t *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  void *ptrs[] = {h->states, h->next_states, h->rewards, h->priorities, h->actions, h->owner, h->prob, h->cdf, h->block_sums, h->scalars};
  for (void *p : ptrs) if (p) cudaFree(p);
  free(h);
  return 0;
}

extern "C" int64_t uavsim_replay_size(const uavsim_replay_t *h) { return h ? h->size : 0; }
extern "C" int64_t uavsim_replay_pos(const uavsim_replay_t *h) { return h ? h->pos : 0; }
extern "C" int64_t uavsim_replay_launch_count(const uavsim_replay_t *h) { return h ? h->launches : 0; }

extern "C" int uavsim_replay_add(uavsim_replay_t *h, const float *states, const int32_t *actions, const float *rewards,
                                 const float *next_states, int64_t count, void *stream) {
  if (!h || count < 0 || (count > 0 && (!states || !actions || !rewards || !next_states))) { SET_ERR("uavsim_replay_add: bad argument"); return UAVSIM_ERR_ARG; }
  if (count == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->device));
  const int empty = h->size == 0;
  if (!empty) {
    CUDA_TRY(cudaMemsetAsync(h->scalars, 0, 4, st));
    replay_max_kernel<<<replay_grid(h->capacity), REPLAY_NT, 0, st>>>(h->priorities, h->capacity, h->scalars);
    h->launches++;
  }
  const int64_t skip = count > h->capacity ? count - h->capacity : 0;
  replay_add_kernel<<<replay_grid((count - skip) * h->state_dim), REPLAY_NT, 0, st>>>(*h, states, actions, rewards, next_states, skip, count, empty);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  h->pos = (h->pos + count) % h->capacity;
  h->size = h->size + count > h->capacity ? h->capacity : h->size + count;
  return 0;
}

extern "C" int uavsim_replay_sample(uavsim_replay_t *h, int64_t batch, double beta, const double *uniforms, uint64_t seed,
                                    uint64_t counter, float *o_states, int32_t *o_actions, float *o_rewards,
                                    float *o_next_states, int64_t *o_indices, float *o_weights, int64_t *n_out, void *stream) {
  if (!h || !n_out || batch < 0) { SET_ERR("uavsim_replay_sample: bad argument"); return UAVSIM_ERR_ARG; }
  const int64_t n = h->size;
  const int64_t b = batch < n ? batch : n;  // min(batch_size, len(buffer)), train.py:112
  *n_out = b;
  if (b == 0) return 0;
  if (!o_states || !o_actions || !o_rewards || !o_next_states || !o_indices || !o_weights) { SET_ERR("uavsim_replay_sample: NULL output"); return UAVSIM_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->device));
  const int nblocks = (int)((n + REPLAY_SCAN_ELEMS - 1) / REPLAY_SCAN_ELEMS);
  replay_pow_kernel<<<nblocks, REPLAY_NT, 0, st>>>(*h, n);
  replay_total_kernel<<<1, 32, 0, st>>>(*h, nblocks);
  replay_norm_kernel<<<nblocks, REPLAY_NT, 0, st>>>(*h, n);
  replay_scan_blocks_kernel<<<1, 32, 0, st>>>(*h, nblocks);
  replay_scan_kernel<<<nblocks, REPLAY_NT, 0, st>>>(*h, n);
  replay_draw_kernel<<<replay_grid(b), REPLAY_NT, 0, st>>>(*h, n, b, (float)beta, uniforms, seed, counter, o_states, o_actions,
                                                          o_rewards, o_next_states, o_indices, o_weights);
  replay_weight_norm_kernel<<<replay_grid(b), REPLAY_NT, 0, st>>>(*h, b, o_weights);
  CUDA_TRY(cudaGetLastError());
  h->launches += 7;
  return 0;
}

extern "C" int uavsim_replay_update_priorities(uavsim_replay_t *h, const int64_t *indices, const float *priorities, int64_t count, void *stream) {
  if (!h || count < 0 || (count > 0 && (!indices || !priorities))) { SET_ERR("uavsim_replay_update_priorities: bad argument"); return UAVSIM_ERR_ARG; }
  if (count == 0) return 0;
  if (count > (1ll << 31) - 1) { SET_ERR("uavsim_replay_update_priorities: count too large"); return UAVSIM_ERR_UNSUPPORTED; }
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->device));
  const int g = replay_grid(count);
  replay_claim_kernel<<<g, REPLAY_NT, 0, st>>>(*h, indices, count);
  replay_write_kernel<<<g, REPLAY_NT, 0, st>>>(*h, indices, priorities, count);
  replay_release_kernel<<<g, REPLAY_NT, 0, st>>>(*h, indices, count);
  CUDA_TRY(cudaGetLastError());
  h->launches += 3;
  return 0;
}

// checkpoint / test access: copy the ring (slots [0, size)) and the priorities [capacity] to HOST buffers; any may be NULL
extern "C" int uavsim_replay_export(uavsim_replay_t *h, float *states, int32_t *actions, float *rewards, float *next_states,
                                    float *priorities, float *probabilities, void *stream) {
  if (!h) { SET_ERR("uavsim_replay_export: NULL handle"); return UAVSIM_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t n = (size_t)h->size, D = (size_t)h->state_dim;
  if (states && n) CUDA_TRY(cudaMemcpyAsync(states, h->states, n * D * 4, cudaMemcpyDeviceToHost, st));
  if (next_states && n) CUDA_TRY(cudaMemcpyAsync(next_states, h->next_states, n * D * 4, cudaMemcpyDeviceToHost, st));
  if (actions && n) CUDA_TRY(cudaMemcpyAsync(actions, h->actions, n * 4, cudaMemcpyDeviceToHost, st));
  if (rewards && n) CUDA_TRY(cudaMemcpyAsync(rewards, h->rewards, n * 4, cudaMemcpyDeviceToHost, st));
  if (priorities) CUDA_TRY(cudaMemcpyAsync(priorities, h->priorities, (size_t)h->capacity * 4, cudaMemcpyDeviceToHost, st));
  if (probabilities && n) CUDA_TRY(cudaMemcpyAsync(probabilities, h->prob, n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}
