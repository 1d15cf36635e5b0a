// policy.cuh -- fused policy step for the batched rollout (SURVEY.md section 8f, row f-1).
//
// The reference draws one action per agent with a batch-of-one actor forward, `Categorical(probs).sample()` and an
// `.item()` sync (src/models/actor_critic.py:138-148, src/train.py:160-176).  With the environment resident on the GPU
// the policy step of a rollout is `probs = softmax(fc2(relu(fc1(obs))))` over all E*n rows followed by one categorical
// draw per row (src/models/actor_critic.py:85-99): six small library kernels in stock PyTorch, which at 10x10 cost
// twice the environment step.  Here it is ONE launch: a thread owns four rows; the two halves of Blackwell's f32x2
// instructions carry two HIDDEN UNITS (j, j+1) of one row, so the weights arrive from shared memory already paired
// (one broadcast LDS.128 = the pair's fc1 weights for two inputs, or its fc2 weights for two actions) and serve the
// thread's four rows, while the row's inputs enter as scalar-broadcast operands -- no register shuffling in front of
// the FFMA2s.  The hidden activation is never materialised: a unit pair is consumed by the logit accumulators (kept
// as even-unit / odd-unit partial sums) as soon as it is computed; softmax, inverse-CDF draw (Philox4x32-10 keyed
// (seed; row, counter)) and the optional probability output happen in registers.  fp32 throughout, like the torch
// module (the summation order differs: 2e-6 on the probabilities).
#pragma once
#include "common.cuh"
#include "philox.cuh"

#define POLICY_NT 128        // threads per CTA
#define POLICY_ROWS 4        // rows per thread
#define POLICY_IN 12         // state_dim (src/environment.py:29)
#define POLICY_AMAX 16       // max actions (reference: na = 12)
#define POLICY_HMAX 512      // max hidden units (reference: 128, src/configs/*.yaml actor_critic.hidden_dim)

struct PolicyDev {
  const float *w1, *b1, *w2, *b2;  // fc1.weight [H,12], fc1.bias [H], fc2.weight [A,H], fc2.bias [A]  (torch layouts)
  int H, A;
};

__device__ __forceinline__ uint64_t pol_pack2(float lo, float hi) {
  return (uint64_t)__float_as_uint(lo) | ((uint64_t)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ uint64_t pol_fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ float pol_lo(uint64_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float pol_hi(uint64_t v) { return __uint_as_float((uint32_t)(v >> 32)); }

// shared memory: per hidden-unit pair (j, j+1) a record of 64 floats:
//   [ 0..23]  {w1[j][k], w1[j+1][k]} for k = 0..11        [24..25] {b1[j], b1[j+1]}   [26..31] 0
//   [32..63]  {w2[a][j], w2[a][j+1]} for a = 0..AP-1 (0 beyond the action count)
// AP = number of actions rounded up to a multiple of 4; the padding logits are -inf (probability 0)
// PDL: the form uavsim_run_policy launches with programmatic dependent launch.  The weights are constant for the whole
// call, so they are staged before griddepcontrol.wait and that overlaps the previous step kernel's tail; nothing else
// touches global memory before the wait.  Launched without the attribute, the wait passes straight through.
// GREEDY: the deterministic action rule of evaluation.  The same logits and softmax; the action is the smallest index
// among the maximal probabilities as this kernel computes them (lg[a] * (1 / sum), the values the probs output holds), so
// it equals torch.argmax of that output.  No Philox draw: seed and counter are ignored.
template <int AP, bool PDL, bool GREEDY>
__device__ __forceinline__ void policy_rows(const float *__restrict__ obs, int64_t rows, const PolicyDev W, uint64_t seed,
                                            uint64_t counter, int32_t *__restrict__ actions, float *__restrict__ probs) {
  extern __shared__ __align__(16) float s_w[];
  const int H = W.H, A = W.A, HP = (H + 1) / 2;  // unit pairs (an odd H gets a zero unit: relu(0) * 0 adds nothing)
  for (int k = threadIdx.x; k < HP * 64; k += POLICY_NT) {
    const int jp = k >> 6, e = k & 63, j = 2 * jp + (e & 1);
    float v = 0.f;
    if (j < H) {
      if (e < 24) v = W.w1[j * POLICY_IN + (e >> 1)];
      else if (e < 26) v = W.b1[j];
      else if (e >= 32 && ((e - 32) >> 1) < A) v = W.w2[((e - 32) >> 1) * H + j];
    }
    s_w[k] = v;
  }
  __syncthreads();
  if (PDL) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }

  const int64_t stride = (int64_t)gridDim.x * POLICY_NT * POLICY_ROWS;
  for (int64_t r0 = ((int64_t)blockIdx.x * POLICY_NT + threadIdx.x) * POLICY_ROWS; r0 < rows; r0 += stride) {
    float x[POLICY_ROWS][POLICY_IN];  // rows r0 .. r0+3 (clamped reads; stores are guarded)
#pragma unroll
    for (int q = 0; q < POLICY_ROWS; q++) {
      const float4 *p = reinterpret_cast<const float4 *>(obs + min(r0 + q, rows - 1) * POLICY_IN);
#pragma unroll
      for (int v = 0; v < POLICY_IN / 4; v++) {
        const float4 t = p[v];
        x[q][4 * v] = t.x; x[q][4 * v + 1] = t.y; x[q][4 * v + 2] = t.z; x[q][4 * v + 3] = t.w;
      }
    }
    uint64_t lg2[POLICY_ROWS][AP];  // logit partial sums {over even units, over odd units}
#pragma unroll
    for (int q = 0; q < POLICY_ROWS; q++)
#pragma unroll
      for (int a = 0; a < AP; a++) lg2[q][a] = 0ull;

#pragma unroll 1
    for (int jp = 0; jp < HP; jp++) {
      const ulonglong2 *wj = reinterpret_cast<const ulonglong2 *>(s_w + jp * 64);
      uint64_t w1p[POLICY_IN], w2p[AP];
#pragma unroll
      for (int v = 0; v < POLICY_IN / 2; v++) { const ulonglong2 t = wj[v]; w1p[2 * v] = t.x; w1p[2 * v + 1] = t.y; }
      const uint64_t bp = wj[6].x;
#pragma unroll
      for (int v = 0; v < AP / 2; v++) { const ulonglong2 t = wj[8 + v]; w2p[2 * v] = t.x; w2p[2 * v + 1] = t.y; }
#pragma unroll
      for (int q = 0; q < POLICY_ROWS; q++) {
        uint64_t h = bp;
#pragma unroll
        for (int k = 0; k < POLICY_IN; k++) h = pol_fma2(w1p[k], pol_pack2(x[q][k], x[q][k]), h);
        h = pol_pack2(fmaxf(pol_lo(h), 0.f), fmaxf(pol_hi(h), 0.f));  // ReLU of units j, j+1
#pragma unroll
        for (int a = 0; a < AP; a++) lg2[q][a] = pol_fma2(w2p[a], h, lg2[q][a]);
      }
    }

    // softmax + one categorical draw per row (inverse CDF on the unnormalised weights)
#pragma unroll
    for (int q = 0; q < POLICY_ROWS; q++) {
      const int64_t r = r0 + q;
      if (r >= rows) break;
      float lg[AP];
#pragma unroll
      for (int a = 0; a < AP; a++) lg[a] = a < A ? (pol_lo(lg2[q][a]) + pol_hi(lg2[q][a])) + W.b2[a] : -INFINITY;
      float mx = lg[0];
#pragma unroll
      for (int a = 1; a < AP; a++) mx = fmaxf(mx, lg[a]);
      float sum = 0.f;
#pragma unroll
      for (int a = 0; a < AP; a++) { lg[a] = expf(lg[a] - mx); sum += lg[a]; }
      int act = 0;
      if constexpr (GREEDY) {
        const float inv = 1.0f / sum;
        float best = lg[0] * inv;
#pragma unroll
        for (int a = 1; a < AP; a++) {
          const float p = lg[a] * inv;
          if (a < A && p > best) { best = p; act = a; }  // strictly greater: a tie keeps the first index
        }
      } else {
        const Philox4 rn = philox4x32_10((uint32_t)r, (uint32_t)(r >> 32), (uint32_t)counter, (uint32_t)(counter >> 32), seed);
        // (the 53-bit uniform can round UP to 1.0f: clamped below 1, or a zero-probability last action could be drawn)
        const float u = fminf((float)philox_u53(rn.v[0], rn.v[1]), 0x1.fffffep-1f) * sum;
        // inverse CDF: the action is the number of prefix sums that do not exceed u, capped at the last action
        float run = 0.f;
#pragma unroll
        for (int a = 0; a < AP - 1; a++) { run += lg[a]; act += (run <= u && a < A - 1) ? 1 : 0; }
      }
      actions[r] = act;
      if (probs) {
        const float inv = 1.0f / sum;
#pragma unroll
        for (int a = 0; a < AP; a++) if (a < A) probs[r * A + a] = lg[a] * inv;
      }
    }
  }
}

template <int AP, bool PDL = false>
__global__ void __launch_bounds__(POLICY_NT)
uavsim_policy_kernel(const float *__restrict__ obs, int64_t rows, const PolicyDev W, uint64_t seed, uint64_t counter,
                     int32_t *__restrict__ actions, float *__restrict__ probs) {
  policy_rows<AP, PDL, false>(obs, rows, W, seed, counter, actions, probs);
}

// The greedy form: a kernel of its own name, so that traces and profiles tell the two action rules apart.
template <int AP, bool PDL = false>
__global__ void __launch_bounds__(POLICY_NT)
uavsim_policy_greedy_kernel(const float *__restrict__ obs, int64_t rows, const PolicyDev W, uint64_t seed,
                            uint64_t counter, int32_t *__restrict__ actions, float *__restrict__ probs) {
  policy_rows<AP, PDL, true>(obs, rows, W, seed, counter, actions, probs);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef void (*PolicyKernelFn)(const float *, int64_t, const PolicyDev, uint64_t, uint64_t, int32_t *, float *);

// One policy launch over `rows` rows: the kernel instance, its dynamic shared memory and grid.
struct PolicyLaunch {
  PolicyKernelFn fn;
  size_t smem;
  int blocks;
};

// The weight rules of the fused policy kernel (shared by uavsim_policy_sample and uavsim_run_policy).
static int policy_check_weights(const UavSimPolicyWeights *w, const char *who) {
  if (!w || !w->w1 || !w->b1 || !w->w2 || !w->b2) { SET_ERR("%s: NULL argument", who); return UAVSIM_ERR_ARG; }
  if (w->state_dim != POLICY_IN || w->hidden < 1 || w->hidden > POLICY_HMAX || w->n_actions < 2 || w->n_actions > POLICY_AMAX) {
    SET_ERR("%s: supports state_dim = %d, hidden <= %d, 2 <= n_actions <= %d (got %d, %d, %d)", who, POLICY_IN,
            POLICY_HMAX, POLICY_AMAX, w->state_dim, w->hidden, w->n_actions);
    return UAVSIM_ERR_UNSUPPORTED;
  }
  return 0;
}

static PolicyDev policy_dev(const UavSimPolicyWeights *w) {
  PolicyDev W;
  W.w1 = w->w1; W.b1 = w->b1; W.w2 = w->w2; W.b2 = w->b2; W.H = w->hidden; W.A = w->n_actions;
  return W;
}

// (weights already checked by policy_check_weights; needs the current device set)
static int policy_plan(int64_t rows, const PolicyDev &W, bool pdl, bool greedy, int device, PolicyLaunch *L) {
  if (greedy) {
    switch ((W.A + 3) / 4) {
      case 1: L->fn = pdl ? uavsim_policy_greedy_kernel<4, true> : uavsim_policy_greedy_kernel<4>; break;
      case 2: L->fn = pdl ? uavsim_policy_greedy_kernel<8, true> : uavsim_policy_greedy_kernel<8>; break;
      case 3: L->fn = pdl ? uavsim_policy_greedy_kernel<12, true> : uavsim_policy_greedy_kernel<12>; break;
      default: L->fn = pdl ? uavsim_policy_greedy_kernel<16, true> : uavsim_policy_greedy_kernel<16>; break;
    }
  } else {
    switch ((W.A + 3) / 4) {
      case 1: L->fn = pdl ? uavsim_policy_kernel<4, true> : uavsim_policy_kernel<4>; break;
      case 2: L->fn = pdl ? uavsim_policy_kernel<8, true> : uavsim_policy_kernel<8>; break;
      case 3: L->fn = pdl ? uavsim_policy_kernel<12, true> : uavsim_policy_kernel<12>; break;
      default: L->fn = pdl ? uavsim_policy_kernel<16, true> : uavsim_policy_kernel<16>; break;
    }
  }
  L->smem = (size_t)((W.H + 1) / 2) * 64 * sizeof(float);
  int rc = raise_dynamic_smem((const void *)L->fn, device, L->smem);
  if (rc) return rc;
  int sms = 148, occ = 1;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, L->fn, POLICY_NT, L->smem);
  if (occ < 1) occ = 1;
  // persistent, balanced grid: every CTA stages the weights once and runs the same number of 512-row iterations
  // (a grid of "one CTA per iteration" pays the staging per iteration and ends in a mostly idle last wave)
  const int64_t iters = (rows + (int64_t)POLICY_NT * POLICY_ROWS - 1) / ((int64_t)POLICY_NT * POLICY_ROWS);
  const int64_t resident = (int64_t)sms * occ;
  const int64_t per_cta = (iters + resident - 1) / resident;
  int64_t blocks = (iters + per_cta - 1) / (per_cta > 0 ? per_cta : 1);
  L->blocks = (int)(blocks < 1 ? 1 : blocks);
  return 0;
}

// uavsim_policy_sample / uavsim_policy_greedy: every argument is checked before the device is touched
static int policy_launch_rows(const float *obs, int64_t rows, const UavSimPolicyWeights *w, bool greedy, uint64_t seed,
                              uint64_t counter, int32_t *actions, float *probs, int device, void *stream,
                              const char *who) {
  if (!w || rows < 0 || (rows > 0 && (!obs || !actions))) {
    SET_ERR("%s: NULL argument", who);
    return UAVSIM_ERR_ARG;
  }
  int rc = policy_check_weights(w, who);
  if (rc) return rc;
  if (rows == 0) return 0;
  if ((reinterpret_cast<uintptr_t>(obs) & 15) != 0) {  // the kernel reads each row with three float4 loads
    SET_ERR("%s: obs must be 16-byte aligned", who);
    return UAVSIM_ERR_ARG;
  }
  CUDA_TRY(cudaSetDevice(device));
  const PolicyDev W = policy_dev(w);
  PolicyLaunch L;
  rc = policy_plan(rows, W, false, greedy, device, &L);
  if (rc) return rc;
  L.fn<<<L.blocks, POLICY_NT, L.smem, (cudaStream_t)stream>>>(obs, rows, W, seed, counter, actions, probs);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

extern "C" int uavsim_policy_sample(const float *obs, int64_t rows, const UavSimPolicyWeights *w, uint64_t seed,
                                    uint64_t counter, int32_t *actions, float *probs, int device, void *stream) {
  return policy_launch_rows(obs, rows, w, false, seed, counter, actions, probs, device, stream, "uavsim_policy_sample");
}

extern "C" int uavsim_policy_greedy(const float *obs, int64_t rows, const UavSimPolicyWeights *w, int32_t *actions,
                                    float *probs, int device, void *stream) {
  return policy_launch_rows(obs, rows, w, true, 0, 0, actions, probs, device, stream, "uavsim_policy_greedy");
}
