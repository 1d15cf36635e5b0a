// step_tile_kernel.cuh -- the fused environment step for swarms of 64 UAVs x 64 targets (Environment.step,
// src/environment.py:120-164) as an ALL-PAIRS TILE kernel: one environment per 128-thread CTA, persistent over
// environments, every pair test and every masked sum evaluated with all 32 lanes of a warp converged.
//
// How the pair phase is laid out (what differs from step_fast_kernel.cuh, which keeps one UAV per lane and walks
// per-UAV candidate lists at 20-25 active lanes):
//   * Warp w owns the 16 UAVs 16w .. 16w+15 (the rows of a 16 x 16 tile) and sweeps the 64 partners in four column
//     tiles.  Inside a tile a thread holds the eight pairs that the A fragment of mma.sync.m16n8k16 assigns to it:
//     rows g and g+8 (g = lane / 4) x columns {2q, 2q+1, 2q+8, 2q+9} (q = lane % 4), two adjacent partners per
//     packed f32x2 instruction.
//   * A pair test is u = fp32 squared distance - C (C = centre of the guard band of that radius).  The SIGN of u is
//     the decision; |u| <= H (half width of the band: the proven fp32 error bound, KParams::GuardK) marks a pair that
//     fp32 cannot decide, and exactly those pairs -- about one in 10^5 -- are re-decided on the spot in fp64 with
//     the reference's arithmetic (tile_fix).  No row or environment is re-evaluated because of one ambiguous pair.
//   * The 0 / 1 decision of a pair becomes an fp16 weight (PRMT replicates the two sign bits over the two halves of
//     a register, one AND turns them into 1.0h / 0) IN THE REGISTER LAYOUT OF THE A OPERAND, and the masked sums of
//     the local state (src/agent/uav.py:101-147, :156-197: sum of partner x, y, cos h, sin h, action, count) are one
//     or two mma.sync per tile against a B operand that holds the partners' features split into fp16 hi + lo parts
//     (the 0 / 1 operand is exact, so hi + lo gives ~22 bits; the accumulators are fp32).  The Gauss-Seidel
//     observation order (partner j < i at its new state, j > i at its old state, src/environment.py:133-138) is the
//     tile position: column tiles left of the diagonal use the partners' NEW records, tiles right of it the OLD
//     ones, and the diagonal tile splits per half-register with two constant masks.
//   * What is not linear in the partner -- sum of distances to tracked targets (uav.py:199-212), sum of
//     exp((2dp - d) / 2dp) over UAVs within 2 dp (uav.py:214-229) -- is evaluated per pair (MUFU) under the sign of
//     u; column tiles without any pair inside 2 dp are skipped by a warp vote.
//   * The neighbour set d <= dp (uav.py:305) stays as one bit per pair in a register; the neighbour mean of MAAC-G
//     (uav.py:293-310) is again an mma.sync (rebuilt weights x {raw hi, raw lo, 1}).
// Environments that the fp32 tile path does not serve (an entity far from the map, a UAV inside the 4 m x 4 m
// origin corner where the row weights of uav.py:162-186 differ from 1, a distance exactly on dp, huge action
// indices) take tile_agent_exact for every UAV: the reference's arithmetic in fp64, pair by pair.
// Data movement is the fast kernel's: cp.async.bulk for the eight input arrays (double-buffered behind the pair
// phase) and for all outputs.
#pragma once
#include "step_fast_kernel.cuh"
#include <cuda_fp16.h>

#define TILE_NT 128
#ifndef TILE_CTAS_PER_SM
#define TILE_CTAS_PER_SM 5
#endif
#define TILE_SUM_W 28  // floats per UAV in the sums array (112 B rows: conflict-free 128-bit reads)

struct __align__(16) TileFeat {
  float c, s, a, pad;  // cos h, sin h, action index
};

template <bool AUX>
struct __align__(128) TileSmem {
  // inputs of the current environment (bulk-loaded)
  double ux[64], uy[64], uh[64];
  double tx[64], ty[64], th[64];
  int32_t ua[64], act[64];
  // new state (bulk-stored)
  double oux[64], ouy[64], ouh[64];
  double otx[64], oty[64], oth[64];
  int32_t oua[64];
  double xo[64], yo[64];                  // UAV positions before the move (fp64: exact decisions)
  float4 npos[32], opos[32], tpos[32];    // fp32 positions relative to the map centre, {x_c, x_c+1, y_c, y_c+1}
  TileFeat nfe[64], ofe[64];              // fp32 records after / before the move
  float2 tfe[64];                         // target heading terms (cos h, sin h) * tv / uv
  float2 own[64];                         // what fp32 dropped of the own position
  // B operands: one 16-byte row of eight fp16 per entity {f0 hi, f0 lo, f1 hi, f1 lo, ...}.  After the pair phase
  // the same bytes stage the outputs (observations [64][12], four reward planes [4][64]).
  uint4 bt1[64];                          // targets: x, y, vx, vy
  uint4 bn1[64], bn2[64];                 // UAVs after the move: {x, y, cos, sin}, {1, a, 0 ...}
  uint4 bo1[64], bo2[64];                 // UAVs before the move
  float sums[64][TILE_SUM_W];             // per UAV: masked sums out of the pair phase
  uint4 braw[64];                         // {raw hi, raw lo, 1, 0 ...}: B operand of the neighbour mean
  float raw[64];
  uint32_t nbw[64][2];                    // neighbour sets in natural bit order (PMI hand-over, exact path)
  int32_t tcnt[AUX ? 64 : 1];
  uint32_t cover[4][2];
  uint32_t rmax[4];
  int32_t slow;
  unsigned long long mbar;
};

// ---- small wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ ulonglong2 tl_lds128(const void *p) { return *reinterpret_cast<const ulonglong2 *>(p); }
// squared distances of two adjacent partners {x0, x1}, {y0, y1} to a row position held as broadcast pairs
__device__ __forceinline__ uint64_t tl_sq(const ulonglong2 P, uint64_t xr, uint64_t yr) {
  const uint64_t dx = f2_sub(P.x, xr), dy = f2_sub(P.y, yr);
  return f2_fma(dx, dx, f2_mul(dy, dy));
}
// the same minus the band centre, fused: dx^2 + (dy^2 - C)
__device__ __forceinline__ uint64_t tl_sqc(const ulonglong2 P, uint64_t xr, uint64_t yr, uint64_t negC) {
  const uint64_t dx = f2_sub(P.x, xr), dy = f2_sub(P.y, yr);
  return f2_fma(dx, dx, f2_fma(dy, dy, negC));
}
// 0xFFFF in the half whose source is negative: {sign(lo), sign(hi)}
__device__ __forceinline__ uint32_t tl_signs(uint64_t u) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, 0xffbb;" : "=r"(r) : "r"((uint32_t)u), "r"((uint32_t)(u >> 32)));
  return r;
}
__device__ __forceinline__ float tl_min3abs(float a, float b, float c) {
  float r;
  asm("min.abs.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float tl_min3(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// smallest |value| of four packed pairs
__device__ __forceinline__ float tl_band4(uint64_t u0, uint64_t u1, uint64_t u2, uint64_t u3) {
  float m = tl_min3abs(f2_lo(u0), f2_hi(u0), f2_lo(u1));
  m = tl_min3abs(m, f2_hi(u1), f2_lo(u2));
  m = tl_min3abs(m, f2_hi(u2), f2_lo(u3));
  return fminf(m, fabsf(f2_hi(u3)));
}
__device__ __forceinline__ void tl_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// B fragments of a 16-partner column tile from rows of eight fp16 (k-major): two / four transposed 8 x 8 loads
__device__ __forceinline__ void tl_ldb2(uint32_t addr, uint32_t &b0, uint32_t &b1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(addr));
}
__device__ __forceinline__ void tl_ldb4(uint32_t addr, uint32_t &b0, uint32_t &b1, uint32_t &b2, uint32_t &b3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
}
// (a, b) = hi + lo in fp16: {a hi, b hi} and {a lo, b lo}, one packed conversion each
__device__ __forceinline__ void tl_split2(float a, float b, uint32_t &hi2, uint32_t &lo2) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 back = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - back.x, b - back.y);
  hi2 = *reinterpret_cast<const uint32_t *>(&h);
  lo2 = *reinterpret_cast<const uint32_t *>(&l);
}
// one B row {a hi, b hi, a lo, b lo, c hi, d hi, c lo, d lo}: the sums of hi and lo parts land in neighbouring quads of the
// accumulator and are added when the UAV is finished
__device__ __forceinline__ uint4 tl_brow(float a, float b, float c, float d) {
  uint4 r;
  tl_split2(a, b, r.x, r.y);
  tl_split2(c, d, r.z, r.w);
  return r;
}
__device__ __forceinline__ uint64_t tl_set_half(uint64_t u, int half, float v) {
  const uint64_t b = (uint64_t)__float_as_uint(v);
  return half ? ((u & 0x00000000ffffffffull) | (b << 32)) : ((u & 0xffffffff00000000ull) | b);
}

// ------------------------------------------------------------------------------------------------
// Pairs inside the guard band: decided in fp64 exactly as the reference does (d2 = dx*dx + dy*dy, no contraction;
// d2 <= s* with s* the largest double whose square root passes the reference's comparison).  u[k] holds the pairs
// (row0 + 8 (k & 1), col0 + 8 (k >> 1) + {0, 1}); a decided pair leaves with |u| = 2 H and the right sign.  `s_lt`
// is the strict threshold where the caller also needs d < thr (coverage): a distance exactly on the radius cannot be
// expressed by one sign, the environment is flagged for the exact path.  `kmask`: which of the four u[k] are in use.
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ void tile_fix(const double *rx, const double *ry, const double *cx, const double *cy, int row0,
                                      int col0, double s_le, double s_lt, float H, int kmask, uint64_t *u, int32_t *slow) {
  const float out = 2.0f * H + 1e-30f;
  for (int k = 0; k < 4; k++) {
    if (!((kmask >> k) & 1)) continue;
    for (int h = 0; h < 2; h++) {
      const float v = h ? f2_hi(u[k]) : f2_lo(u[k]);
      if (!(fabsf(v) <= H)) continue;
      const int row = row0 + 8 * (k & 1), col = col0 + 8 * (k >> 1) + h;
      const double dx = cx[col] - rx[row], dy = cy[col] - ry[row];
      const double d2 = dx * dx + dy * dy;
      const bool hit = d2 <= s_le;
      if (hit != (d2 <= s_lt)) *slow = 1;
      u[k] = tl_set_half(u[k], h, hit ? -out : out);
    }
  }
}

// inverse of the fp16 value of bit 10 + J (0x0400, 0x0800, 0x1000, 0x2000 = 2^-14, 2^-13, 2^-11, 2^-7)
__device__ __forceinline__ float tl_nscale(int J) { return J == 0 ? 16384.f : (J == 1 ? 8192.f : (J == 2 ? 2048.f : 128.f)); }

// what the exact path produces for one UAV
struct TileAgent {
  float ob[9];
  float tt, dup;
  uint32_t nb[2];   // neighbour set d <= dp, natural bit order
  uint32_t cov[2];  // targets strictly inside dp, natural bit order
};
struct TileMaskPtrs {
  uint8_t *obs_mask, *comm_mask, *nbr_mask, *dup_mask, *cover_mask;
};

// ------------------------------------------------------------------------------------------------
// exact path: the reference's arithmetic pair by pair in fp64, including the min(dist, 1) row weights of
// src/agent/uav.py:162-186 (same routine as fast_agent_exact, on this kernel's shared-memory layout).
// ------------------------------------------------------------------------------------------------
template <bool AUX>
__device__ __noinline__ void tile_agent_exact(const ExactK P, const TileMaskPtrs B, const TileSmem<AUX> *Sp, int i,
                                              int64_t mrow_t, int64_t mrow_u, TileAgent *Op) {
  const TileSmem<AUX> &S = *Sp;
  const double xi = S.oux[i], yi = S.ouy[i];
  const double chi = (double)S.nfe[i].c, shi = (double)S.nfe[i].s;
  const int ai = S.oua[i];
  double tt = 0, o0 = 0, o1 = 0, o2 = 0, o3 = 0;
  int nobs = 0;
  uint32_t cov[2] = {0, 0};
  for (int t = 0; t < 64; t++) {
    const double dx = S.otx[t] - xi, dy = S.oty[t] - yi;
    const double d2 = dx * dx + dy * dy;
    const bool hit = d2 <= P.s_dp_le, cv = d2 <= P.s_dp_lt;
    if (AUX && B.obs_mask) { B.obs_mask[mrow_t + t] = hit; B.cover_mask[mrow_t + t] = cv; }
    if (cv) cov[t >> 5] |= 1u << (t & 31);
    if (hit) {
      const double d = sqrt(d2);
      tt += 1 + (P.dp - d) / P.dp;  // uav.py:208
      double rx = dx / P.dp, ry = dy / P.dp, vx = (double)S.tfe[t].x - chi, vy = (double)S.tfe[t].y - shi;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;  // uav.py:174-180
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; }
      o0 += rx; o1 += ry; o2 += vx; o3 += vy;
      nobs++;
    }
  }
  double dup = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
  int ncomm = 0;
  uint32_t nb[2] = {0, 0};
  for (int j = 0; j < 64; j++) {
    if (j == i) {
      if (AUX && B.obs_mask) { B.comm_mask[mrow_u + j] = 0; B.nbr_mask[mrow_u + j] = 0; B.dup_mask[mrow_u + j] = 0; }
      continue;
    }
    const double dxn = S.oux[j] - xi, dyn = S.ouy[j] - yi;
    const double d2n = dxn * dxn + dyn * dyn;
    const bool hit_dup = d2n <= P.s_2dp_le, hit_nbr = d2n <= P.s_dp_le;
    if (hit_dup) { const double d = sqrt(d2n); dup += -0.5 * exp((P.two_dp - d) / P.two_dp); }  // uav.py:226
    if (hit_nbr) nb[j >> 5] |= 1u << (j & 31);
    double dxc, dyc, d2c;
    TileFeat rj;  // partner's record: after its move if it moved first, before it otherwise
    if (j < i) { dxc = dxn; dyc = dyn; d2c = d2n; rj = S.nfe[j]; }
    else { dxc = S.xo[j] - xi; dyc = S.yo[j] - yi; d2c = dxc * dxc + dyc * dyc; rj = S.ofe[j]; }
    const bool hit_c = d2c <= P.s_dc_le;
    if (AUX && B.obs_mask) { B.comm_mask[mrow_u + j] = hit_c; B.nbr_mask[mrow_u + j] = hit_nbr; B.dup_mask[mrow_u + j] = hit_dup; }
    if (hit_c) {
      double rx = dxc / P.dc, ry = dyc / P.dc, vx = (double)rj.c - chi, vy = (double)rj.s - shi;
      double da = ((double)rj.a - (double)ai) / (double)P.na;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; da /= w; }
      c0 += rx; c1 += ry; c2 += vx; c3 += vy; c4 += da;
      ncomm++;
    }
  }
  TileAgent &O = *Op;
  if (ncomm) {
    const double k = (double)ncomm;
    O.ob[0] = (float)(c0 / k); O.ob[1] = (float)(c1 / k); O.ob[2] = (float)(c2 / k); O.ob[3] = (float)(c3 / k); O.ob[4] = (float)(c4 / k);
  } else {
    O.ob[0] = O.ob[1] = O.ob[2] = O.ob[3] = O.ob[4] = -1.f;
  }
  if (nobs) {
    const double k = (double)nobs;
    O.ob[5] = (float)(o0 / k); O.ob[6] = (float)(o1 / k); O.ob[7] = (float)(o2 / k); O.ob[8] = (float)(o3 / k);
  } else {
    O.ob[5] = O.ob[6] = O.ob[7] = O.ob[8] = -1.f;
  }
  O.tt = (float)tt; O.dup = (float)dup;
  O.nb[0] = nb[0]; O.nb[1] = nb[1];
  O.cov[0] = cov[0]; O.cov[1] = cov[1];
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
template <bool AUX>
__global__ void __launch_bounds__(TILE_NT, TILE_CTAS_PER_SM)
uavsim_step_tile_kernel(const KParams P, const UavSimBuffers B, const ActEntry *__restrict__ act_tab, int64_t env_begin,
                        int64_t env_count, int mode, double coop, int done_flag, long long *__restrict__ stats) {
  constexpr int N = 64, M = 64;
  typedef TileSmem<AUX> SmemT;
  static_assert(offsetof(SmemT, bo2) + sizeof(uint4) * 64 - offsetof(SmemT, bt1) >= sizeof(float) * (12 * N + 4 * N), "output staging");
  extern __shared__ __align__(128) unsigned char tile_smem_raw[];
  SmemT &S = *reinterpret_cast<SmemT *>(tile_smem_raw);
  float *const s_obs = reinterpret_cast<float *>(S.bt1);            // [N][12], after the pair phase
  float *const s_rew = s_obs + 12 * N;                              // [4][N]
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int g = lane >> 2, q = lane & 3;
  const uint32_t bar = sf_smem(&S.mbar);
  constexpr uint32_t IN_BYTES = 3 * N * 8 + 3 * M * 8 + 2 * N * 4;
  const bool pmi_pending = (mode == UAVSIM_MODE_PMI) && (coop != 0.0);
  const bool mean_mode = (mode == UAVSIM_MODE_MEAN) && (coop != 0.0);
  const bool aux_on = AUX && (B.obs_mask != nullptr);
  const bool need_nbr = pmi_pending || mean_mode || aux_on;

  auto issue_loads = [&](int64_t e) {
    sf_expect_tx(bar, IN_BYTES);
    sf_bulk_g2s(sf_smem(S.ux), B.ux + e * N, N * 8, bar);
    sf_bulk_g2s(sf_smem(S.uy), B.uy + e * N, N * 8, bar);
    sf_bulk_g2s(sf_smem(S.uh), B.uh + e * N, N * 8, bar);
    sf_bulk_g2s(sf_smem(S.tx), B.tx + e * M, M * 8, bar);
    sf_bulk_g2s(sf_smem(S.ty), B.ty + e * M, M * 8, bar);
    sf_bulk_g2s(sf_smem(S.th), B.th + e * M, M * 8, bar);
    sf_bulk_g2s(sf_smem(S.ua), B.ua + e * N, N * 4, bar);
    sf_bulk_g2s(sf_smem(S.act), B.actions + e * N, N * 4, bar);
  };

  if (t == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == 0 && (int64_t)blockIdx.x < env_count) {
    if (elect_one()) issue_loads(env_begin + blockIdx.x);
  }

  const int64_t plane = P.E * N;
  const float inv_dp_f = P.inv_dp_f, inv_dc_f = P.inv_dc_f, inv_na_f = P.inv_na_f;
  const float k_ex0 = 1.4426950408889634f, k_ex1 = P.k_ex1_f;
  long long fx_r = 0, fx_tt = 0, fx_bp = 0, fx_dup = 0, st_cov = 0, st_envs = 0;  // statistics (common.cuh: sf_fx)
  int st_cmax = 0;
  uint32_t parity = 0;

  // rows of this thread in the tile of its warp, and the constant masks of the diagonal tile: half h of the register
  // (row g, columns 2q + h) lies left of the diagonal iff 2q + h < g (partner moved first: NEW record), right of
  // it iff 2q + h > g (OLD record); 2q + h == g is the UAV itself.
  const int r0 = 16 * warp + g, r1 = r0 + 8;
  constexpr uint32_t ONE2 = 0x3C003C00u;  // {1.0h, 1.0h}
  const uint32_t mL = ((2 * q < g) ? 0x00003C00u : 0u) | ((2 * q + 1 < g) ? 0x3C000000u : 0u);
  const uint32_t mU = ((2 * q > g) ? 0x00003C00u : 0u) | ((2 * q + 1 > g) ? 0x3C000000u : 0u);
  const uint32_t ones_b = (g == 0) ? ONE2 : 0u;  // B operand {1, 0, ...} of the target count
  // ldmatrix row addresses: lane l supplies row (l & 7) of matrix l >> 3
  const uint32_t ldm_row = (uint32_t)((lane & 7) + ((lane >> 3) & 1) * 8) * 16u;
  const uint32_t ldm_sel = (uint32_t)(lane >> 4);  // 0: first array, 1: second array (x4 loads)

  for (int64_t k = blockIdx.x; k < env_count; k += gridDim.x) {
    const int64_t e = env_begin + k;
    if (warp == 0) {
      if (elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    if (t == 0) S.slow = 0;
    __syncthreads();
    sf_mbar_wait(bar, parity);
    parity ^= 1;

    float rabs;
    if (t >= 64) {
      // ---- phase 0a: target j (src/agent/target.py:27-60) ----
      const int j = t - 64;
      double x = S.tx[j], y = S.ty[j], h = S.th[j];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);
      x += P.dtv_t * ch;
      y += P.dtv_t * sh;
      if (0 > y || y > P.y_max) { h = -h; sh = -sh; }
      else if (x < 0 || x > P.x_max) { h = (h > 0) ? (PI_D - h) : (-PI_D - h); ch = -ch; }
      S.otx[j] = x; S.oty[j] = y; S.oth[j] = h;
      const float txf = (float)(x - P.cx), tyf = (float)(y - P.cy);
      const float vx = (float)ch * P.tv_over_uv_f, vy = (float)sh * P.tv_over_uv_f;
      float *ts = reinterpret_cast<float *>(&S.tpos[j >> 1]) + (j & 1);
      ts[0] = txf; ts[2] = tyf;
      S.tfe[j] = make_float2(vx, vy);
      S.bt1[j] = tl_brow(txf, tyf, vx, vy);
      rabs = fmaxf(fabsf(txf), fabsf(tyf));
      if (AUX) S.tcnt[j] = 0;
    } else {
      // ---- phase 0b: UAV t (src/agent/uav.py:73-99) ----
      double x = S.ux[t], y = S.uy[t], h = S.uh[t];
      const int a_old = S.ua[t], act = S.act[t];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);
      const float cof = (float)ch, sof = (float)sh;
      const float xof = (float)(x - P.cx), yof = (float)(y - P.cy);
      S.xo[t] = x; S.yo[t] = y;
      float *so = reinterpret_cast<float *>(&S.opos[t >> 1]) + (t & 1);
      so[0] = xof; so[2] = yof;
      S.ofe[t] = TileFeat{cof, sof, (float)a_old, 0.f};
      S.bo1[t] = tl_brow(xof, yof, cof, sof);
      S.bo2[t] = make_uint4(0x3C00u | ((uint32_t)__half_as_ushort(__float2half_rn((float)a_old)) << 16), 0u, 0u, 0u);
      x += P.dtv_u * ch;
      y += P.dtv_u * sh;
      double dh;
      float cd, sd;
      if ((unsigned)act < (unsigned)P.na) {
        const ActEntry en = act_tab[act];
        dh = en.dth; cd = en.cd; sd = en.sd;
      } else {  // the reference's formula accepts any integer (uav.py:73-81)
        dh = P.dt * ((double)(2 * (act + 1) - P.na - 1) * P.uav_h_max / (double)(P.na - 1));
        double sd_, cd_;
        sincos_shared(dh, &sd_, &cd_);
        cd = (float)cd_; sd = (float)sd_;
      }
      h = wrap_heading(h + dh);
      const float chf = fmaf(cof, cd, -(sof * sd));
      const float shf = fmaf(sof, cd, cof * sd);
      const float xf = (float)(x - P.cx), yf = (float)(y - P.cy);
      S.own[t] = make_float2((float)((x - P.cx) - (double)xf), (float)((y - P.cy) - (double)yf));
      S.oux[t] = x; S.ouy[t] = y; S.ouh[t] = h; S.oua[t] = act;
      float *sn = reinterpret_cast<float *>(&S.npos[t >> 1]) + (t & 1);
      sn[0] = xf; sn[2] = yf;
      S.nfe[t] = TileFeat{chf, shf, (float)act, 0.f};
      S.bn1[t] = tl_brow(xf, yf, chf, shf);
      S.bn2[t] = make_uint4(0x3C00u | ((uint32_t)__half_as_ushort(__float2half_rn((float)act)) << 16), 0u, 0u, 0u);
      rabs = fmaxf(fmaxf(fabsf(xf), fabsf(yf)), fmaxf(fabsf(xof), fabsf(yof)));
      // fp16 carries action indices exactly up to 2048: anything else takes the exact path
      if ((unsigned)act >= 2048u || (unsigned)a_old >= 2048u) rabs = __int_as_float(0x7f800000);
      // the only place a row weight (uav.py:162-186) differs from 1
      if (fabs(x) < 2.0 && fabs(y) < 2.0) rabs = __int_as_float(0x7f800000);
    }
    if (!(rabs == rabs)) rabs = __int_as_float(0x7f800000);
    {
      const uint32_t rm = __reduce_max_sync(0xffffffffu, __float_as_uint(rabs));
      if (lane == 0) S.rmax[warp] = rm;
    }
    __syncthreads();
    if (warp == 0 && k + gridDim.x < env_count) {  // next environment, behind the pair phase
      if (elect_one()) issue_loads(e + gridDim.x);
    }

    const float R = __uint_as_float(max(max(S.rmax[0], S.rmax[1]), max(S.rmax[2], S.rmax[3])));
    const bool slow0 = !(R <= P.r_tile);
    // neighbour decisions of this thread's pairs: register kk (the A-fragment slot), column tile J -> bit 10 + J of
    // each half.  Read as fp16 these single bits are the weights 2^-14, 2^-13, 2^-11, 2^-7: the B rows of column tile J
    // carry the inverse factor (tl_nscale), so the neighbour mean needs no rebuilt weights.
    uint32_t nw[4] = {0u, 0u, 0u, 0u};

    if (!slow0) {
      // ================= phase 1: all pairs of the 16 rows of this warp =================
      // band centre and half width per radius: certainly inside below C - H, certainly outside above C + H
      const TileBand &TB = P.tb[(R <= P.tb[0].r) ? 0 : 1];
      const float Cp = TB.Cp, Hp = TB.Hp, Cd = TB.Cd, Hd = TB.Hd, Cc = TB.Cc, Hc = TB.Hc;
      const uint64_t nCp2 = pack2(-Cp, -Cp), nCd2 = pack2(-Cd, -Cd), nCc2 = pack2(-Cc, -Cc), Cp2 = pack2(Cp, Cp);
      uint64_t xr0, yr0, xr1, yr1;
      {
        const float *p0 = reinterpret_cast<const float *>(&S.npos[r0 >> 1]) + (r0 & 1);
        const float *p1 = reinterpret_cast<const float *>(&S.npos[r1 >> 1]) + (r1 & 1);
        xr0 = pack2(p0[0], p0[0]); yr0 = pack2(p0[2], p0[2]);
        xr1 = pack2(p1[0], p1[0]); yr1 = pack2(p1[2], p1[2]);
      }
      const int64_t mrow0_t = (e * N + r0) * M, mrow1_t = (e * N + r1) * M;  // N == M: also the rows of the UAV masks

      // ---- targets: observe_target (uav.py:101-122), tracking reward (uav.py:199-212), coverage (environment.py:246-253)
      float ct1[4] = {0.f, 0.f, 0.f, 0.f}, ct2[4] = {0.f, 0.f, 0.f, 0.f};
      float tt0 = 0.f, tt1 = 0.f;
      uint32_t covA = 0, covB = 0;
#pragma unroll 1
      for (int J = 0; J < 4; J++) {
        const ulonglong2 P0 = tl_lds128(&S.tpos[8 * J + q]), P1 = tl_lds128(&S.tpos[8 * J + q + 4]);
        uint64_t u0 = tl_sqc(P0, xr0, yr0, nCp2), u1 = tl_sqc(P0, xr1, yr1, nCp2);
        uint64_t u2 = tl_sqc(P1, xr0, yr0, nCp2), u3 = tl_sqc(P1, xr1, yr1, nCp2);
        if (tl_band4(u0, u1, u2, u3) <= Hp) {
          uint64_t uu[4] = {u0, u1, u2, u3};
          tile_fix(S.oux, S.ouy, S.otx, S.oty, r0, 16 * J + 2 * q, P.s_dp_le, P.s_dp_lt, Hp, 15, uu, &S.slow);
          u0 = uu[0]; u1 = uu[1]; u2 = uu[2]; u3 = uu[3];
        }
        uint32_t a[4];
        a[0] = tl_signs(u0) & ONE2; a[1] = tl_signs(u1) & ONE2; a[2] = tl_signs(u2) & ONE2; a[3] = tl_signs(u3) & ONE2;
        const uint32_t KJ = 0x04000400u << J;  // bits 10..13 of each half are set in a hit: one of them per column tile
        covA |= (a[0] | a[1]) & KJ;
        covB |= (a[2] | a[3]) & KJ;
        uint32_t b0, b1;
        tl_ldb2(sf_smem(S.bt1) + (uint32_t)J * 256u + ldm_row, b0, b1);
        tl_mma(ct1, a, b0, b1);
        tl_mma(ct2, a, ones_b, ones_b);
        {  // sum of distances to the tracked targets
          const uint64_t s0 = f2_add(u0, Cp2), s1 = f2_add(u1, Cp2), s2 = f2_add(u2, Cp2), s3 = f2_add(u3, Cp2);
          const float d00 = fast_sqrtf(f2_lo(s0)), d01 = fast_sqrtf(f2_hi(s0)), d10 = fast_sqrtf(f2_lo(s1)), d11 = fast_sqrtf(f2_hi(s1));
          const float d20 = fast_sqrtf(f2_lo(s2)), d21 = fast_sqrtf(f2_hi(s2)), d30 = fast_sqrtf(f2_lo(s3)), d31 = fast_sqrtf(f2_hi(s3));
          if (f2_lo(u0) < 0.f) tt0 += d00;
          if (f2_hi(u0) < 0.f) tt0 += d01;
          if (f2_lo(u2) < 0.f) tt0 += d20;
          if (f2_hi(u2) < 0.f) tt0 += d21;
          if (f2_lo(u1) < 0.f) tt1 += d10;
          if (f2_hi(u1) < 0.f) tt1 += d11;
          if (f2_lo(u3) < 0.f) tt1 += d30;
          if (f2_hi(u3) < 0.f) tt1 += d31;
        }
        if (AUX) {
          const uint64_t uu[4] = {u0, u1, u2, u3};
#pragma unroll
          for (int kk = 0; kk < 4; kk++) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
              const bool hit = (h ? f2_hi(uu[kk]) : f2_lo(uu[kk])) < 0.f;
              const int col = 16 * J + 2 * q + 8 * (kk >> 1) + h;
              if (aux_on) {
                const int64_t o = ((kk & 1) ? mrow1_t : mrow0_t) + col;
                B.obs_mask[o] = hit; B.cover_mask[o] = hit;
              }
              if (hit && B.tracker_cnt) atomicAdd(&S.tcnt[col], 1);
            }
          }
        }
      }

      // ---- UAV partners: communication (uav.py:124-147), duplicate tracking (uav.py:214-229), neighbours (uav.py:305)
      float cc1[4] = {0.f, 0.f, 0.f, 0.f}, cc2[4] = {0.f, 0.f, 0.f, 0.f};
      float dup0 = 0.f, dup1 = 0.f;
#pragma unroll 1
      for (int J = 0; J < 4; J++) {
        const int col0 = 16 * J + 2 * q;
        const ulonglong2 N0 = tl_lds128(&S.npos[8 * J + q]), N1 = tl_lds128(&S.npos[8 * J + q + 4]);
        // new-new squared distances: duplicate tracking and neighbours everywhere, communication left of the diagonal
        const uint64_t s0 = tl_sq(N0, xr0, yr0), s1 = tl_sq(N0, xr1, yr1), s2 = tl_sq(N1, xr0, yr0), s3 = tl_sq(N1, xr1, yr1);
        uint32_t a[4];
        uint32_t cmask[4] = {0, 0, 0, 0};  // AUX: communication decisions as sign halves
        if (J < warp) {  // partners moved first: their new records
          uint64_t u0 = f2_add(s0, nCc2), u1 = f2_add(s1, nCc2), u2 = f2_add(s2, nCc2), u3 = f2_add(s3, nCc2);
          if (tl_band4(u0, u1, u2, u3) <= Hc) {
            uint64_t uu[4] = {u0, u1, u2, u3};
            tile_fix(S.oux, S.ouy, S.oux, S.ouy, r0, col0, P.s_dc_le, P.s_dc_le, Hc, 15, uu, &S.slow);
            u0 = uu[0]; u1 = uu[1]; u2 = uu[2]; u3 = uu[3];
          }
          a[0] = tl_signs(u0) & ONE2; a[1] = tl_signs(u1) & ONE2; a[2] = tl_signs(u2) & ONE2; a[3] = tl_signs(u3) & ONE2;
          uint32_t b0, b1, b2, b3;
          tl_ldb4(sf_smem(S.bn1) + ldm_sel * (uint32_t)(sizeof(uint4) * 64) + (uint32_t)J * 256u + ldm_row, b0, b1, b2, b3);
          tl_mma(cc1, a, b0, b1);
          tl_mma(cc2, a, b2, b3);
          if (AUX) { cmask[0] = a[0]; cmask[1] = a[1]; cmask[2] = a[2]; cmask[3] = a[3]; }
        } else {
          const ulonglong2 O0 = tl_lds128(&S.opos[8 * J + q]), O1 = tl_lds128(&S.opos[8 * J + q + 4]);
          if (J > warp) {  // partners move later: their old records
            uint64_t u0 = tl_sqc(O0, xr0, yr0, nCc2), u1 = tl_sqc(O0, xr1, yr1, nCc2);
            uint64_t u2 = tl_sqc(O1, xr0, yr0, nCc2), u3 = tl_sqc(O1, xr1, yr1, nCc2);
            if (tl_band4(u0, u1, u2, u3) <= Hc) {
              uint64_t uu[4] = {u0, u1, u2, u3};
              tile_fix(S.oux, S.ouy, S.xo, S.yo, r0, col0, P.s_dc_le, P.s_dc_le, Hc, 15, uu, &S.slow);
              u0 = uu[0]; u1 = uu[1]; u2 = uu[2]; u3 = uu[3];
            }
            a[0] = tl_signs(u0) & ONE2; a[1] = tl_signs(u1) & ONE2; a[2] = tl_signs(u2) & ONE2; a[3] = tl_signs(u3) & ONE2;
            uint32_t b0, b1, b2, b3;
            tl_ldb4(sf_smem(S.bo1) + ldm_sel * (uint32_t)(sizeof(uint4) * 64) + (uint32_t)J * 256u + ldm_row, b0, b1, b2, b3);
            tl_mma(cc1, a, b0, b1);
            tl_mma(cc2, a, b2, b3);
            if (AUX) { cmask[0] = a[0]; cmask[1] = a[1]; cmask[2] = a[2]; cmask[3] = a[3]; }
          } else {
            // diagonal tile.  Register 1 (rows g+8, columns < 8) lies entirely left of the diagonal, register 2
            // (rows g, columns >= 8) entirely right of it; registers 0 and 3 straddle it.
            uint64_t n0 = f2_add(s0, nCc2), n1 = f2_add(s1, nCc2), n3 = f2_add(s3, nCc2);
            uint64_t o0 = tl_sqc(O0, xr0, yr0, nCc2), o2 = tl_sqc(O1, xr0, yr0, nCc2), o3 = tl_sqc(O1, xr1, yr1, nCc2);
            if (fminf(tl_band4(n0, n1, n1, n3), tl_band4(o0, o2, o2, o3)) <= Hc) {
              uint64_t un[4] = {n0, n1, n1, n3}, uo[4] = {o0, o0, o2, o3};
              tile_fix(S.oux, S.ouy, S.oux, S.ouy, r0, col0, P.s_dc_le, P.s_dc_le, Hc, 11, un, &S.slow);
              tile_fix(S.oux, S.ouy, S.xo, S.yo, r0, col0, P.s_dc_le, P.s_dc_le, Hc, 13, uo, &S.slow);
              n0 = un[0]; n1 = un[1]; n3 = un[3];
              o0 = uo[0]; o2 = uo[2]; o3 = uo[3];
            }
            uint32_t an[4], ao[4];
            an[0] = tl_signs(n0) & mL; an[1] = tl_signs(n1) & ONE2; an[2] = 0u; an[3] = tl_signs(n3) & mL;
            ao[0] = tl_signs(o0) & mU; ao[1] = 0u; ao[2] = tl_signs(o2) & ONE2; ao[3] = tl_signs(o3) & mU;
            uint32_t b0, b1, b2, b3;
            tl_ldb4(sf_smem(S.bn1) + ldm_sel * (uint32_t)(sizeof(uint4) * 64) + (uint32_t)J * 256u + ldm_row, b0, b1, b2, b3);
            tl_mma(cc1, an, b0, b1);
            tl_mma(cc2, an, b2, b3);
            tl_ldb4(sf_smem(S.bo1) + ldm_sel * (uint32_t)(sizeof(uint4) * 64) + (uint32_t)J * 256u + ldm_row, b0, b1, b2, b3);
            tl_mma(cc1, ao, b0, b1);
            tl_mma(cc2, ao, b2, b3);
            if (AUX) { cmask[0] = an[0] | ao[0]; cmask[1] = an[1]; cmask[2] = ao[2]; cmask[3] = an[3] | ao[3]; }
          }
        }
        // duplicate tracking / neighbours on the new-new distances
        uint64_t d0 = f2_add(s0, nCd2), d1 = f2_add(s1, nCd2), d2 = f2_add(s2, nCd2), d3 = f2_add(s3, nCd2);
        if (tl_band4(d0, d1, d2, d3) <= Hd) {
          uint64_t uu[4] = {d0, d1, d2, d3};
          tile_fix(S.oux, S.ouy, S.oux, S.ouy, r0, col0, P.s_2dp_le, P.s_2dp_le, Hd, 15, uu, &S.slow);
          d0 = uu[0]; d1 = uu[1]; d2 = uu[2]; d3 = uu[3];
        }
        float anyd = tl_min3(f2_lo(d0), f2_hi(d0), f2_lo(d1));
        anyd = tl_min3(anyd, f2_hi(d1), f2_lo(d2));
        anyd = tl_min3(anyd, f2_hi(d2), f2_lo(d3));
        anyd = fminf(anyd, f2_hi(d3));
        uint32_t nsig[4] = {0, 0, 0, 0};
        if (__any_sync(0xffffffffu, anyd < 0.f)) {
          const float e00 = fast_ex2f(fmaf(fast_sqrtf(f2_lo(s0)), k_ex1, k_ex0)), e01 = fast_ex2f(fmaf(fast_sqrtf(f2_hi(s0)), k_ex1, k_ex0));
          const float e10 = fast_ex2f(fmaf(fast_sqrtf(f2_lo(s1)), k_ex1, k_ex0)), e11 = fast_ex2f(fmaf(fast_sqrtf(f2_hi(s1)), k_ex1, k_ex0));
          const float e20 = fast_ex2f(fmaf(fast_sqrtf(f2_lo(s2)), k_ex1, k_ex0)), e21 = fast_ex2f(fmaf(fast_sqrtf(f2_hi(s2)), k_ex1, k_ex0));
          const float e30 = fast_ex2f(fmaf(fast_sqrtf(f2_lo(s3)), k_ex1, k_ex0)), e31 = fast_ex2f(fmaf(fast_sqrtf(f2_hi(s3)), k_ex1, k_ex0));
          if (f2_lo(d0) < 0.f) dup0 += e00;
          if (f2_hi(d0) < 0.f) dup0 += e01;
          if (f2_lo(d2) < 0.f) dup0 += e20;
          if (f2_hi(d2) < 0.f) dup0 += e21;
          if (f2_lo(d1) < 0.f) dup1 += e10;
          if (f2_hi(d1) < 0.f) dup1 += e11;
          if (f2_lo(d3) < 0.f) dup1 += e30;
          if (f2_hi(d3) < 0.f) dup1 += e31;
          if (need_nbr) {
            uint64_t p0 = f2_add(s0, nCp2), p1 = f2_add(s1, nCp2), p2 = f2_add(s2, nCp2), p3 = f2_add(s3, nCp2);
            if (tl_band4(p0, p1, p2, p3) <= Hp) {
              uint64_t uu[4] = {p0, p1, p2, p3};
              tile_fix(S.oux, S.ouy, S.oux, S.ouy, r0, col0, P.s_dp_le, P.s_dp_le, Hp, 15, uu, &S.slow);
              p0 = uu[0]; p1 = uu[1]; p2 = uu[2]; p3 = uu[3];
            }
            nsig[0] = tl_signs(p0); nsig[1] = tl_signs(p1); nsig[2] = tl_signs(p2); nsig[3] = tl_signs(p3);
            const uint32_t KJ = 0x04000400u << J;
            nw[0] |= nsig[0] & KJ; nw[1] |= nsig[1] & KJ; nw[2] |= nsig[2] & KJ; nw[3] |= nsig[3] & KJ;
          }
        }
        if (AUX && aux_on) {
          const uint32_t dsig[4] = {tl_signs(d0), tl_signs(d1), tl_signs(d2), tl_signs(d3)};
#pragma unroll
          for (int kk = 0; kk < 4; kk++) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
              const int col = col0 + 8 * (kk >> 1) + h, row = (kk & 1) ? r1 : r0;
              const int64_t o = ((kk & 1) ? mrow1_t : mrow0_t) + col;
              const bool self = (col == row);
              B.comm_mask[o] = (uint8_t)(((cmask[kk] >> (16 * h)) & 0xffffu) != 0u);
              B.dup_mask[o] = (uint8_t)(!self && ((dsig[kk] >> (16 * h)) & 1u));
              B.nbr_mask[o] = (uint8_t)(!self && ((nsig[kk] >> (16 * h)) & 1u));
            }
          }
        }
      }

      // ---- hand the sums of the 16 rows to the threads that finish the UAVs ----
      tt0 += __shfl_xor_sync(0xffffffffu, tt0, 1); tt1 += __shfl_xor_sync(0xffffffffu, tt1, 1);
      dup0 += __shfl_xor_sync(0xffffffffu, dup0, 1); dup1 += __shfl_xor_sync(0xffffffffu, dup1, 1);
      tt0 += __shfl_xor_sync(0xffffffffu, tt0, 2); tt1 += __shfl_xor_sync(0xffffffffu, tt1, 2);
      dup0 += __shfl_xor_sync(0xffffffffu, dup0, 2); dup1 += __shfl_xor_sync(0xffffffffu, dup1, 2);
      // quad q holds columns 2q, 2q+1 of the accumulators: {x hi, y hi}, {x lo, y lo}, {f2 hi, f3 hi}, {f2 lo, f3 lo}
      *reinterpret_cast<float2 *>(&S.sums[r0][2 * q]) = make_float2(ct1[0], ct1[1]);
      *reinterpret_cast<float2 *>(&S.sums[r1][2 * q]) = make_float2(ct1[2], ct1[3]);
      *reinterpret_cast<float2 *>(&S.sums[r0][8 + 2 * q]) = make_float2(cc1[0], cc1[1]);
      *reinterpret_cast<float2 *>(&S.sums[r1][8 + 2 * q]) = make_float2(cc1[2], cc1[3]);
      if (q == 0) {
        *reinterpret_cast<float4 *>(&S.sums[r0][16]) = make_float4(ct2[0], tt0, dup0, 0.f);
        *reinterpret_cast<float4 *>(&S.sums[r1][16]) = make_float4(ct2[2], tt1, dup1, 0.f);
        *reinterpret_cast<float2 *>(&S.sums[r0][20]) = make_float2(cc2[0], cc2[1]);
        *reinterpret_cast<float2 *>(&S.sums[r1][20]) = make_float2(cc2[2], cc2[3]);
      }
      {  // coverage: OR over the rows of this warp; bit (10 + J) of half h of covA / covB = column 16 J + 2 q (+ 8) + h
        const uint32_t ca = ((covA >> 10) & 0xFu) | ((covA >> 22) & 0xF0u), cb = ((covB >> 10) & 0xFu) | ((covB >> 22) & 0xF0u);
        const uint32_t wa = __reduce_or_sync(0xffffffffu, ca << (8 * q)), wb = __reduce_or_sync(0xffffffffu, cb << (8 * q));
        if (lane == 0) { S.cover[warp][0] = wa; S.cover[warp][1] = wb; }
      }
      if (pmi_pending) {  // neighbour sets in natural bit order for the PMI kernel
        uint32_t w0[2] = {0, 0}, w1[2] = {0, 0};
#pragma unroll
        for (int J = 0; J < 4; J++) {
#pragma unroll
          for (int kk = 0; kk < 4; kk++) {
            const uint32_t two = ((nw[kk] >> (10 + J)) & 1u) | (((nw[kk] >> (26 + J)) & 1u) << 1);
            const int col = 16 * J + 2 * q + 8 * (kk >> 1);
            if (kk & 1) w1[col >> 5] |= two << (col & 31); else w0[col >> 5] |= two << (col & 31);
          }
        }
        // not its own neighbour
        w0[r0 >> 5] &= ~(1u << (r0 & 31)); w1[r1 >> 5] &= ~(1u << (r1 & 31));
#pragma unroll
        for (int wd = 0; wd < 2; wd++) {
          uint32_t v0 = w0[wd], v1 = w1[wd];
          v0 |= __shfl_xor_sync(0xffffffffu, v0, 1); v1 |= __shfl_xor_sync(0xffffffffu, v1, 1);
          v0 |= __shfl_xor_sync(0xffffffffu, v0, 2); v1 |= __shfl_xor_sync(0xffffffffu, v1, 2);
          if (q == 0) { S.nbw[r0][wd] = v0; S.nbw[r1][wd] = v1; }
        }
      }
    }
    __syncthreads();  // sums complete; the B operands become the output staging

    // ================= finish the UAVs (threads 0 .. 63, one UAV each) =================
    const bool slow = slow0 || (S.slow != 0);
    float raw = 0.f, ttn = 0.f, bpn = 0.f, dupn = 0.f;
    uint32_t nb0 = 0, nb1 = 0;  // exact path: neighbour set in natural order
    if (t < 64) {
      const double xi = S.oux[t], yi = S.ouy[t];
      const int ai = S.oua[t];
      const float *pp = reinterpret_cast<const float *>(&S.npos[t >> 1]) + (t & 1);
      const float xf = pp[0], yf = pp[2];
      float o0, o1, o2, o3, o4, o5, o6, o7, o8, tt_f, dup_f;
      if (!slow) {
        const float chf = S.nfe[t].c, shf = S.nfe[t].s;
        const float2 ol = S.own[t];
        const float4 ta = *reinterpret_cast<const float4 *>(&S.sums[t][0]), tb4 = *reinterpret_cast<const float4 *>(&S.sums[t][4]);
        const float4 ca = *reinterpret_cast<const float4 *>(&S.sums[t][8]), cb4 = *reinterpret_cast<const float4 *>(&S.sums[t][12]);
        const float4 s4 = *reinterpret_cast<const float4 *>(&S.sums[t][16]);
        const float2 s12 = *reinterpret_cast<const float2 *>(&S.sums[t][20]);
        const float4 st = make_float4(ta.x + ta.z, ta.y + ta.w, tb4.x + tb4.z, tb4.y + tb4.w);   // hi + lo
        const float4 sc = make_float4(ca.x + ca.z, ca.y + ca.w, cb4.x + cb4.z, cb4.y + cb4.w);
        if (s4.x > 0.5f) {
          const float rk = sf_rcp(s4.x);
          o5 = (fmaf(st.x, rk, -xf) - ol.x) * inv_dp_f;
          o6 = (fmaf(st.y, rk, -yf) - ol.y) * inv_dp_f;
          o7 = fmaf(st.z, rk, -chf);
          o8 = fmaf(st.w, rk, -shf);
          tt_f = fmaf(2.0f, s4.x, -s4.y * inv_dp_f);  // sum of 1 + (dp - d)/dp
        } else {
          o5 = o6 = o7 = o8 = -1.f;
          tt_f = 0.f;
        }
        if (s12.x > 0.5f) {
          const float rk = sf_rcp(s12.x);
          o0 = (fmaf(sc.x, rk, -xf) - ol.x) * inv_dc_f;
          o1 = (fmaf(sc.y, rk, -yf) - ol.y) * inv_dc_f;
          o2 = fmaf(sc.z, rk, -chf);
          o3 = fmaf(sc.w, rk, -shf);
          o4 = fmaf(s12.y, rk, -(float)ai) * inv_na_f;
        } else {
          o0 = o1 = o2 = o3 = o4 = -1.f;
        }
        // the diagonal pair (the UAV itself, distance 0) went through the duplicate-tracking sum: taken out again
        dup_f = -0.5f * (s4.z - fast_ex2f(fmaf(fast_sqrtf(0.f), k_ex1, k_ex0)));
      } else {
        const ExactK XK = {P.s_dp_le, P.s_dp_lt, P.s_2dp_le, P.s_dc_le, P.dp, P.dc, P.two_dp, P.na};
        const TileMaskPtrs MP = {B.obs_mask, B.comm_mask, B.nbr_mask, B.dup_mask, B.cover_mask};
        TileAgent X;
        tile_agent_exact<AUX>(XK, MP, &S, t, (e * N + t) * M, (e * N + t) * N, &X);
        o0 = X.ob[0]; o1 = X.ob[1]; o2 = X.ob[2]; o3 = X.ob[3]; o4 = X.ob[4];
        o5 = X.ob[5]; o6 = X.ob[6]; o7 = X.ob[7]; o8 = X.ob[8];
        tt_f = X.tt; dup_f = X.dup;
        nb0 = X.nb[0]; nb1 = X.nb[1];
        S.nbw[t][0] = nb0; S.nbw[t][1] = nb1;
        const uint32_t c0 = __reduce_or_sync(0xffffffffu, X.cov[0]), c1 = __reduce_or_sync(0xffffffffu, X.cov[1]);
        if (lane == 0) { S.cover[warp][0] = c0; S.cover[warp][1] = c1; S.cover[warp + 2][0] = 0u; S.cover[warp + 2][1] = 0u; }
        if (AUX && B.tracker_cnt) {
          if (t == 0) for (int j = 0; j < 64; j++) S.tcnt[j] = 0;  // (fix-ups may have flagged the environment after a partial count)
          __syncwarp();
        }
      }
      {
        // boundary punishment (uav.py:231-250); the inside / outside decision (closed interval, uav.py:239) falls
        // back to fp64 within a millimetre of a wall
        const float dbdr = fminf(P.cx_f - fabsf(xf), P.cy_f - fabsf(yf));
        bool inside = dbdr > 0.f;
        if (fabsf(dbdr) < 1e-3f) inside = 0 <= xi && xi <= P.x_max && 0 <= yi && yi <= P.y_max;
        const float bp = inside ? ((dbdr < P.dp_f) ? (-0.5f * (P.dp_f - dbdr) * inv_dp_f) : 0.0f) : -0.5f;
        // normalise + weights (environment.py:206-220)
        ttn = fminf(fmaxf(tt_f, 0.0f), P.tt_hi_f) * P.inv_tt_hi_f;
        dupn = (fminf(fmaxf(dup_f, P.dup_lo_f), 0.0f) - P.dup_lo_f) * P.inv_dup_span_f - 1.0f;
        bpn = (fminf(fmaxf(bp, -0.5f), 0.0f) + 0.5f) * 2.0f - 1.0f;
        raw = fmaf(P.alpha_f, ttn, fmaf(P.beta_f, bpn, P.gamma_f * dupn));
        S.raw[t] = raw;
        {  // B row of the neighbour mean: {raw hi, scale, raw lo, 0, ...} times the factor of the UAV's column tile
          const float sc = tl_nscale(t >> 4);
          uint4 br = make_uint4(0u, 0u, 0u, 0u);
          tl_split2(raw * sc, sc, br.x, br.y);
          S.braw[t] = br;
        }
      }
      float *ob = s_obs + t * 12;
      reinterpret_cast<float4 *>(ob)[0] = make_float4(o0, o1, o2, o3);
      reinterpret_cast<float4 *>(ob)[1] = make_float4(o4, o5, o6, o7);
      reinterpret_cast<float4 *>(ob)[2] = make_float4(o8, (float)(xi * P.inv_dc), (float)(yi * P.inv_dc), (float)ai * inv_na_f);
      s_rew[N + t] = ttn;
      s_rew[2 * N + t] = bpn;
      s_rew[3 * N + t] = dupn;
      fx_tt += sf_fx(ttn); fx_bp += sf_fx(bpn); fx_dup += sf_fx(dupn);
    }
    if (slow && AUX && B.tracker_cnt) {
      __syncthreads();
      if (t < 64) {  // per-target tracker counts of the exact path
        const double xi = S.oux[t], yi = S.ouy[t];
        for (int j = 0; j < 64; j++) {
          const double dx = S.otx[j] - xi, dy = S.oty[j] - yi;
          if (dx * dx + dy * dy <= P.s_dp_lt) atomicAdd(&S.tcnt[j], 1);
        }
      }
    }
    __syncthreads();  // raw rewards of every UAV

    // ================= cooperative reward (environment.py:222-227) =================
    if (!mean_mode || slow) {
      if (t < 64) {
        float r;
        if (mode == UAVSIM_MODE_SELF || coop == 0.0) {
          r = raw;  // uav.py:271-272 / :300-301
        } else if (mode == UAVSIM_MODE_MEAN) {
          // uav.py:293-310 -- the conditional expression covers the whole sum: no neighbour -> 0
          float s = 0;
          const int cnt = __popc(nb0) + __popc(nb1);
          uint32_t w = nb0;
          while (w) { const int b = __ffs(w) - 1; w &= w - 1; s += S.raw[b]; }
          w = nb1;
          while (w) { const int b = __ffs(w) - 1; w &= w - 1; s += S.raw[32 + b]; }
          const float cf = (float)coop;
          r = cnt ? fmaf(1.0f - cf, raw, cf * s * sf_rcp((float)cnt)) : 0.0f;
        } else {
          r = 0.0f;  // finished by the PMI kernel
          const int64_t gi = e * N + t;
          B.raw[gi] = (double)raw;
          B.nbr_bits[gi * 2] = (uint64_t)S.nbw[t][0] | ((uint64_t)S.nbw[t][1] << 32);
          B.nbr_bits[gi * 2 + 1] = 0;
        }
        r = fminf(fmaxf(r, -1.0f), 1.0f);  // clip_and_normalize(reward, -1, 1) is a plain clip
        s_rew[t] = r;
        if (!pmi_pending) fx_r += sf_fx(r);
      }
    } else {
      // neighbour mean as one more masked sum: the neighbour bits of column tile J, read as fp16, x {raw hi, 1, raw lo} x scale
      float cr[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int J = 0; J < 4; J++) {
        const uint32_t KJ = 0x04000400u << J;
        uint32_t a[4];
#pragma unroll
        for (int kk = 0; kk < 4; kk++) a[kk] = nw[kk] & KJ;
        uint32_t b0, b1;
        tl_ldb2(sf_smem(S.braw) + (uint32_t)J * 256u + ldm_row, b0, b1);
        tl_mma(cr, a, b0, b1);
      }
      // thread q = 0 of a quad holds {sum raw hi, count}, thread q = 1 {sum raw lo, 0}
      const float lo0 = __shfl_sync(0xffffffffu, cr[0], (lane & ~3) | 1), lo1 = __shfl_sync(0xffffffffu, cr[2], (lane & ~3) | 1);
      if (q == 0) {
        const float cf = (float)coop;
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
          const int row = rr ? r1 : r0;
          const float rw = S.raw[row];
          // the UAV itself (distance 0) is in the set: taken out of sum and count
          const float s = (rr ? (cr[2] + lo1) : (cr[0] + lo0)) - rw, cnt = (rr ? cr[3] : cr[1]) - 1.0f;
          float r = (cnt > 0.5f) ? fmaf(1.0f - cf, rw, cf * s * sf_rcp(cnt)) : 0.0f;
          r = fminf(fmaxf(r, -1.0f), 1.0f);
          s_rew[row] = r;
          fx_r += sf_fx(r);
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk copies
    __syncthreads();
    if (warp == 0) {
      if (elect_one()) {
        sf_bulk_s2g(B.ux + e * N, sf_smem(S.oux), N * 8);
        sf_bulk_s2g(B.uy + e * N, sf_smem(S.ouy), N * 8);
        sf_bulk_s2g(B.uh + e * N, sf_smem(S.ouh), N * 8);
        sf_bulk_s2g(B.ua + e * N, sf_smem(S.oua), N * 4);
        sf_bulk_s2g(B.tx + e * M, sf_smem(S.otx), M * 8);
        sf_bulk_s2g(B.ty + e * M, sf_smem(S.oty), M * 8);
        sf_bulk_s2g(B.th + e * M, sf_smem(S.oth), M * 8);
        sf_bulk_s2g(B.obs + e * N * 12, sf_smem(s_obs), N * 48);
        if (!pmi_pending) sf_bulk_s2g(B.rew4 + e * N, sf_smem(s_rew), N * 4);
        sf_bulk_s2g(B.rew4 + plane + e * N, sf_smem(s_rew + N), N * 4);
        sf_bulk_s2g(B.rew4 + 2 * plane + e * N, sf_smem(s_rew + 2 * N), N * 4);
        sf_bulk_s2g(B.rew4 + 3 * plane + e * N, sf_smem(s_rew + 3 * N), N * 4);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (AUX && B.tracker_cnt && t < 64) B.tracker_cnt[e * M + t] = S.tcnt[t];
    if (t == 0) {
      const int c = __popc(S.cover[0][0] | S.cover[1][0] | S.cover[2][0] | S.cover[3][0]) +
                    __popc(S.cover[0][1] | S.cover[1][1] | S.cover[2][1] | S.cover[3][1]);
      B.covered[e] = c;
      if (B.done) B.done[e] = done_flag;
      st_cov += c;
      st_cmax = max(st_cmax, c);
      st_envs++;
    }
  }
  __syncwarp();
  if (warp == 0) {
    if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // outputs complete before the CTA retires
  }
  stats_commit(stats + (size_t)blockIdx.x * STAT_W, fx_r, fx_tt, fx_bp, fx_dup, st_cov, st_cmax, st_envs);
}
