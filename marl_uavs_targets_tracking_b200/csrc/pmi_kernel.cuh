// pmi_kernel.cuh -- PMI reciprocal reward: fp32 CUDA-core implementation (the exact-fp32 parity path).
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// PMI reciprocal reward (src/agent/uav.py:262-291 + src/models/PMINet.py:41-72), fp32 CUDA-core GEMM.
// CTA = G environments: enumerate neighbour pairs, run the folded MLP over tiles of TM pair rows
// (layer 0 block-diagonal 12->3H, layer 1 3H->H as a register-tiled SGEMM with fc1^T streamed
// through shared memory, layer 2 H->1 as a shuffle reduction), then the per-UAV softmax and mix.
// ------------------------------------------------------------------------------------------------
#define PMI_KC 32  // k-chunk of fc1 streamed per iteration

struct PmiSmem {
  float *obs;       // [G*n*12]
  double *raw;      // [G*n]
  uint32_t *off;    // [G*n+1]
  uint32_t *pair;   // [pmax]  (a << 16) | b, local UAV indices in the group
  float *logit;     // [pmax]
  float *x;         // [TM*12]
  float *h0;        // [TM*(3H+4)]
  float *wchunk;    // [PMI_KC*H]
  float *w0, *b0, *b1, *w2;  // [3H*5] [3H] [H] [H]
};

static size_t pmi_smem_bytes(int n, int H, int G, int pmax, int TM) {
  size_t b = 0;
  b += (size_t)G * n * 8;                          // raw (doubles first)
  b += (size_t)G * n * 12 * 4;                     // obs
  b += ((size_t)G * n + 1 + 3) / 4 * 4 * 4;        // off (padded)
  b += (size_t)pmax * 8;                           // pair + logit
  b += (size_t)TM * 12 * 4 + (size_t)TM * (3 * H + 4) * 4 + (size_t)PMI_KC * H * 4;
  b += (size_t)(3 * H * 5 + 3 * H + H + H) * 4;
  return b + 32;
}

__device__ __forceinline__ PmiSmem pmi_carve(unsigned char *base, int n, int H, int G, int pmax, int TM) {
  PmiSmem s;
  double *d = reinterpret_cast<double *>(base);
  s.raw = d; d += (size_t)G * n;
  float *f = reinterpret_cast<float *>(d);
  s.obs = f; f += (size_t)G * n * 12;
  s.off = reinterpret_cast<uint32_t *>(f); f += ((size_t)G * n + 1 + 3) / 4 * 4;
  s.pair = reinterpret_cast<uint32_t *>(f); f += pmax;
  s.logit = f; f += pmax;
  s.x = f; f += (size_t)TM * 12;
  s.h0 = f; f += (size_t)TM * (3 * H + 4);
  s.wchunk = f; f += (size_t)PMI_KC * H;
  s.w0 = f; f += 3 * H * 5;
  s.b0 = f; f += 3 * H;
  s.b1 = f; f += H;
  s.w2 = f; f += H;
  return s;
}

template <int CPT, int TM>  // H = 16*CPT output columns; TM rows per tile (TM/16 rows per thread)
__global__ void __launch_bounds__(PMI_NT)
uavsim_pmi_kernel(const KParams P, const UavSimBuffers B, const PmiDev W, int64_t env_begin, int64_t env_count,
                  int G, int pmax, double coop, long long *__restrict__ stats) {
  constexpr int H = 16 * CPT, H3 = 3 * H, LD0 = H3 + 4, RPT = TM / 16;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = P.n, tid = threadIdx.x;
  const PmiSmem S = pmi_carve(smem_raw, n, H, G, pmax, TM);

  for (int k = tid; k < H3 * 5; k += PMI_NT) S.w0[k] = W.w0[k];
  for (int k = tid; k < H3; k += PMI_NT) S.b0[k] = W.b0[k];
  for (int k = tid; k < H; k += PMI_NT) { S.b1[k] = W.b1[k]; S.w2[k] = W.w2[k]; }

  const int ty = tid >> 4, tx = tid & 15;
  const int64_t ngroups = (env_count + G - 1) / G;
  long long fx_r = 0;  // reward statistic (common.cuh: sf_fx)

  for (int64_t grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int64_t e0 = env_begin + grp * G;
    const int ne = (int)min((int64_t)G, env_begin + env_count - e0);
    const int A = ne * n;  // UAVs in this group (<= PMI_NT)
    __syncthreads();
    for (int k = tid; k < A * 12; k += PMI_NT) S.obs[k] = B.obs[e0 * n * 12 + k];
    uint64_t nb0 = 0, nb1 = 0;
    if (tid < A) {
      S.raw[tid] = B.raw[e0 * n + tid];
      nb0 = B.nbr_bits[(e0 * n + tid) * 2];
      nb1 = B.nbr_bits[(e0 * n + tid) * 2 + 1];
      S.off[tid + 1] = __popcll(nb0) + __popcll(nb1);
    }
    __syncthreads();
    if (tid == 0) {  // exclusive scan of the neighbour counts (A <= 256)
      uint32_t acc = 0;
      S.off[0] = 0;
      for (int a = 0; a < A; a++) { acc += S.off[a + 1]; S.off[a + 1] = acc; }
    }
    __syncthreads();
    const int npairs = (int)S.off[A];
    if (tid < A) {  // neighbours in ascending index order, like the reference's loop (uav.py:277-282)
      const int base = (tid / n) * n;
      uint32_t p = S.off[tid];
      uint64_t w = nb0;
      while (w) { const int j = __ffsll((long long)w) - 1; w &= w - 1; S.pair[p++] = ((uint32_t)tid << 16) | (uint32_t)(base + j); }
      w = nb1;
      while (w) { const int j = __ffsll((long long)w) - 1; w &= w - 1; S.pair[p++] = ((uint32_t)tid << 16) | (uint32_t)(base + 64 + j); }
    }
    __syncthreads();

    for (int p0 = 0; p0 < npairs; p0 += TM) {
      const int rows = min(TM, npairs - p0);
      // input rows: la_i * la_j (uav.py:280-281), fp32
      for (int k = tid; k < TM * 12; k += PMI_NT) {
        const int r = k / 12, c = k - r * 12;
        float v = 0.f;
        if (r < rows) {
          const uint32_t pr = S.pair[p0 + r];
          v = S.obs[(pr >> 16) * 12 + c] * S.obs[(pr & 0xffffu) * 12 + c];
        }
        S.x[k] = v;
      }
      __syncthreads();
      // layer 0: three branch Linear+BN(folded)+ReLU, concatenated (PMINet.py:45-58)
      for (int k = tid; k < TM * H3; k += PMI_NT) {
        const int r = k / H3, u = k - r * H3;
        const int b = u / H;
        const int off = (b == 0) ? 0 : (b == 1 ? 5 : 9);
        const int dim = (b == 0) ? 5 : (b == 1 ? 4 : 3);
        const float *xr = S.x + r * 12 + off, *wr = S.w0 + u * 5;
        float acc = S.b0[u];
        for (int c = 0; c < dim; c++) acc = fmaf(wr[c], xr[c], acc);
        S.h0[r * LD0 + u] = fmaxf(acc, 0.f);
      }
      // layer 1: [TM,3H] x [3H,H]
      float acc[RPT][CPT];
#pragma unroll
      for (int a = 0; a < RPT; a++)
#pragma unroll
        for (int c = 0; c < CPT; c++) acc[a][c] = 0.f;
      for (int kc = 0; kc < H3; kc += PMI_KC) {
        __syncthreads();  // h0 complete (first pass) / previous chunk consumed
        for (int k = tid; k < PMI_KC * H; k += PMI_NT) S.wchunk[k] = W.w1t[(size_t)kc * H + k];
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < PMI_KC; k++) {
          float av[RPT], bv[CPT];
#pragma unroll
          for (int a = 0; a < RPT; a++) av[a] = S.h0[(ty + 16 * a) * LD0 + kc + k];
#pragma unroll
          for (int c = 0; c < CPT; c++) bv[c] = S.wchunk[k * H + tx + 16 * c];
#pragma unroll
          for (int a = 0; a < RPT; a++)
#pragma unroll
            for (int c = 0; c < CPT; c++) acc[a][c] = fmaf(av[a], bv[c], acc[a][c]);
        }
      }
      // bias + ReLU, then layer 2 (PMINet.py:59-62): dot with fc2 across the 16 column threads
#pragma unroll
      for (int a = 0; a < RPT; a++) {
        float part = 0.f;
#pragma unroll
        for (int c = 0; c < CPT; c++) {
          const int col = tx + 16 * c;
          part = fmaf(S.w2[col], fmaxf(acc[a][c] + S.b1[col], 0.f), part);
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        const int r = ty + 16 * a;
        if (tx == 0 && r < rows) S.logit[p0 + r] = part + W.b2;
      }
      __syncthreads();
    }
    __syncthreads();

    // softmax over each UAV's neighbours (scipy.special.softmax on float32) and the mix (uav.py:284-290)
    if (tid < A) {
      const uint32_t lo = S.off[tid], hi = S.off[tid + 1];
      const double raw = S.raw[tid];
      double r;
      if (hi > lo) {
        float mx = S.logit[lo];
        for (uint32_t p = lo + 1; p < hi; p++) mx = fmaxf(mx, S.logit[p]);
        float ssum = 0.f;
        for (uint32_t p = lo; p < hi; p++) ssum += expf(S.logit[p] - mx);
        double s = 0;
        for (uint32_t p = lo; p < hi; p++) {
          const float wgt = expf(S.logit[p] - mx) / ssum;
          s += S.raw[S.pair[p] & 0xffffu] * (double)wgt;
        }
        r = (1 - coop) * raw + coop * s;
      } else {
        r = (1 - coop) * raw;
      }
      r = fmin(fmax(r, -1.0), 1.0);
      B.rew4[e0 * n + tid] = (float)r;
      fx_r += sf_fx((float)r);
    }
  }
  stats_commit(stats + (size_t)blockIdx.x * STAT_W, fx_r, 0, 0, 0, 0, 0, 0);
}

