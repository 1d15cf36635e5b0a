// step_fast_kernel.cuh -- the fused environment step for swarms of 64 UAVs x 64 targets (Environment.step,
// src/environment.py:120-164), one environment per 64-thread CTA, persistent over environments.
//
// What differs from the generic kernel (step_kernel.cuh), and why:
//   * Work distribution.  Every resident CTA starts on the environment of its block index and draws each further one
//     from a launch-wide counter (KParams::fast_ctr; the last CTA to leave rewinds it).  With a fixed stride the warp
//     schedulers' preference for some CTAs let those finish early and the SMs ran at 24 of 28 resident warps; the
//     counter was worth 10 %.  The reward statistics are therefore integer sums (sf_fx): order-independent.
//   * Data movement.  The eight state / action arrays of an environment (3.5 KB) arrive by cp.async.bulk (TMA engine,
//     mbarrier complete_tx) while the previous environment is computed, and the outputs (new state, observations,
//     four reward planes: 7.4 KB) leave by bulk shared -> global copies; no thread issues a global load or store
//     on the hot path and there is no per-thread 64-bit address arithmetic.
//   * Pair arithmetic in fp32 with a TWO-SIDED guard.  Positions are staged as fp32 relative to the map centre.
//     With g(R) a proven bound on the fp32 error of a squared distance (R = largest |coordinate - centre| of the
//     environment, KParams::GuardK): s_f <= thr^2 - g is certainly inside the radius, s_f > thr^2 + g certainly
//     outside, and only a pair in the band between the two (about one pair in 10^5) is AMBIGUOUS.  Every walk
//     tracks the largest squared distance it accepted; a UAV whose list held an ambiguous pair walks THAT LIST once
//     more through a checked twin (sf_*_checked) that decides the pairs inside the band in fp64 with the reference's
//     arithmetic, so every mask, count and coverage bit is decided exactly as before -- but the candidates of an
//     ordinary UAV never touch the fp64 pipe.  (Until round 2 such a UAV re-evaluated its whole row -- all three
//     lists, fp64 sums and all -- which took 13 % of the issued instructions.)
//     The observation sums are fp32 (outputs are fp32, contract 1e-5; measured ~2e-7).
//   * Candidate walks.  A sign-bit prefilter (packed f32x2 FMAs, as in the generic kernel) marks the partners inside
//     each guarded radius; two walks consume them: targets (observation + tracking reward + coverage), and ONE walk
//     over the UAV slots for communication partners (new record if the partner moved first, old record otherwise:
//     src/agent/uav.py:124-147 in the update order of src/environment.py:133-138), duplicate-tracking and neighbour
//     partners (src/agent/uav.py:214-229, :305).  UAV records are stored two per SLOT (partners 2b and 2b+1 side by side in
//     the halves of the packed fp32 registers): the UAV walks visit slots, not partners, and evaluate both partners
//     of a slot with f32x2 arithmetic and 0/1 weights -- a swarm that flies in formation has its partners in runs of
//     consecutive indices, so the trips nearly halve exactly when the candidate lists are long.
//   * fp64 sine / cosine of the headings by fm_sincos_small (fast_math.cuh) instead of the library call.
// Everything that is not a pair test (kinematics, reflection, boundary term, normalisation, cooperative reward,
// statistics) follows the generic kernel line by line.
#pragma once
#include "common.cuh"
#include "fast_math.cuh"
#include <stddef.h>
#include "step_kernel.cuh"

#define FAST_NT 64  // threads per CTA = UAVs = targets of an environment

// per action: dt * heading-rate (src/agent/uav.py:73-81, :96) and the fp32 cosine / sine of that angle
struct ActEntry {
  double dth;
  float cd, sd;
};

// two UAVs (2b, 2b+1) side by side: the halves of the packed f32x2 operands
struct __align__(16) SlotRec {
  float4 pos;  // {x0, x1, y0, y1} relative to the map centre
  float4 hd;   // {cos h0, cos h1, sin h0, sin h1}
  float2 a;    // action index as float
  float2 pad;
};
// two targets: positions, then cos / sin of the heading times tv / uv (src/agent/uav.py:115-116)
struct __align__(16) TSlot {
  float4 pos;  // {x0, x1, y0, y1}
  float4 vel;  // {vx0, vx1, vy0, vy1}
};

template <int N, int M, bool AUX>
struct __align__(128) FastSmem {
  // inputs of the current environment (bulk-loaded)
  double ux[N], uy[N], uh[N];
  double tx[M], ty[M], th[M];
  int32_t ua[N], act[N];
  // new state (bulk-stored)
  double oux[N], ouy[N], ouh[N];
  double otx[M], oty[M], oth[M];
  int32_t oua[N];
  // working set of the pair phase (fp32, positions relative to the map centre).  Once the pair phase is over
  // (second CTA barrier) the same bytes stage the outputs: observations [N][12] over the UAV slots, the four reward
  // planes [4][N] over the target slots.
  SlotRec slotn[N / 2];  // UAVs after their move
  SlotRec sloto[N / 2];  // UAVs before their move (sloto - slotn is a compile-time offset)
  TSlot tslot[M / 2];
  double xo[N], yo[N];   // fp64 positions before the move (exact path only)
  float raw[N];          // weighted raw reward of every UAV (neighbour mean)
  int32_t tcnt[AUX ? M : 1];
  uint32_t cover[2][2];  // per warp: targets with a UAV strictly inside dp (even / odd word)
  uint32_t rmax[2];      // per warp: largest |coordinate - centre| as float bits
  unsigned long long mbar;
  long long next_k;      // the environment this CTA takes next (drawn from the launch-wide counter)
};
static_assert(sizeof(SlotRec) == 48 && sizeof(TSlot) == 32, "slot layout");

// ---- single-thread async-copy instructions.  They are issued from `if (warp == 0) if (elect_one())`: ptxas
//      recognises a branch on the predicate of ELECT as a single-thread region and emits the copies back to back on
//      the uniform datapath.  Under `if (t == 0)`, or predicated on an elected lane inside the asm, every copy was
//      wrapped in a VOTEU / ELECT / BRA.U.ANY waterfall of ~14 instructions (profiles/r2_* history). ----
__device__ __forceinline__ void sf_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sf_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void sf_bulk_s2g(void *dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t sf_smem(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sf_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; spin++) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    if (spin > (1u << 22)) __trap();  // a copy that never lands traps instead of hanging the GPU
  }
}

__device__ __forceinline__ uint64_t f2_sub(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float f2_lo(uint64_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float f2_hi(uint64_t v) { return __uint_as_float((uint32_t)(v >> 32)); }
// Packed 0 / 1 weights {a0 <= b, a1 <= b}.  (Written with setp / selp on the bit patterns: with `set.le.f32.f32`
// feeding the low half of a packed operand, ptxas 12.9 turned the set into FSETP + SEL ..., 0x1 -- the INTEGER one, a
// denormal as a float -- and every even partner lost its weight.  tools/sass_lines.py --listing shows the encoding.)
__device__ __forceinline__ uint64_t sf_le2(float a0, float a1, float b) {
  uint32_t lo, hi;
  asm("{\n\t.reg .pred p, q;\n\t"
      "setp.le.f32 p, %2, %4;\n\t"
      "setp.le.f32 q, %3, %4;\n\t"
      "selp.b32 %0, 0x3f800000, 0, p;\n\t"
      "selp.b32 %1, 0x3f800000, 0, q;\n\t}"
      : "=r"(lo), "=r"(hi) : "f"(a0), "f"(a1), "f"(b));
  return (uint64_t)lo | ((uint64_t)hi << 32);
}
__device__ __forceinline__ float sf_le(float a, float b) { return (a <= b) ? 1.0f : 0.0f; }
__device__ __forceinline__ int sf_msb(uint32_t w) {  // index of the highest set bit (w != 0): one FLO
  int r;
  asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(w));
  return r;
}
__device__ __forceinline__ float sf_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Candidate sets are kept as an EVEN and an ODD word: bit b of the even word is partner 2b, of the odd word partner
// 2b+1 (the two partners of slot b).
//
// Sign-bit prefilter over 64 partner positions (32 pairs {x0, x1, y0, y1}, `stride` bytes apart) against one or two
// guarded squared radii: the partner's bit is set iff fma(dx, dx, fma(dy, dy, -thr)) < 0.
template <bool TWO, int STRIDE>
__device__ __forceinline__ void prefilter64(const void *__restrict__ pf, float xf, float yf, float thrA, float thrB,
                                            uint32_t &aE, uint32_t &aO, uint32_t &bE, uint32_t &bO) {
  const uint64_t xf2 = pack2(xf, xf), yf2 = pack2(yf, yf), nA = pack2(-thrA, -thrA), nB = pack2(-thrB, -thrB);
  const unsigned char *base = reinterpret_cast<const unsigned char *>(pf);
  uint32_t ae = 0, ao = 0, be = 0, bo = 0;
#ifndef FAST_PF_UNROLL
#define FAST_PF_UNROLL 8   // slots per loop trip (measured: 4 -> 8 -1 %, 16 no further gain)
#endif
#pragma unroll 1
  for (int k = 0; k < 32; k += FAST_PF_UNROLL) {
#pragma unroll
    for (int u = 0; u < FAST_PF_UNROLL; u++) {
      const ulonglong2 p = *reinterpret_cast<const ulonglong2 *>(base + (k + u) * STRIDE);
      const uint64_t dx = f2_sub(p.x, xf2), dy = f2_sub(p.y, yf2);
      const uint64_t tA = f2_fma(dx, dx, f2_fma(dy, dy, nA));
      ae = __funnelshift_l((uint32_t)tA, ae, 1);
      ao = __funnelshift_l((uint32_t)(tA >> 32), ao, 1);
      if (TWO) {
        const uint64_t tB = f2_fma(dx, dx, f2_fma(dy, dy, nB));
        be = __funnelshift_l((uint32_t)tB, be, 1);
        bo = __funnelshift_l((uint32_t)(tB >> 32), bo, 1);
      }
    }
  }
  aE = __brev(ae); aO = __brev(ao);  // pair 0 went in first and sits in bit 31
  bE = __brev(be); bO = __brev(bo);
}

// even / odd words -> the natural 64-bit set (bit j = partner j): only the PMI hand-over needs it
__device__ __forceinline__ uint64_t sf_interleave(uint32_t e, uint32_t o) {
  auto spread = [](uint32_t v) {
    uint64_t x = v;
    x = (x | (x << 16)) & 0x0000FFFF0000FFFFull;
    x = (x | (x << 8)) & 0x00FF00FF00FF00FFull;
    x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0Full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    x = (x | (x << 1)) & 0x5555555555555555ull;
    return x;
  };
  return spread(e) | (spread(o) << 1);
}

// what the pair phase produces for one UAV
struct FastAgent {
  float ob[9];        // communication part (5) and observation part (4) of the local state
  float tt, dup;      // raw tracking reward, raw duplicate punishment
  uint32_t nb[2];     // neighbour set d <= dp (even / odd word)
  uint32_t cov[2];    // targets strictly inside dp (even / odd word)
};

// ------------------------------------------------------------------------------------------------
// exact path: the reference's arithmetic pair by pair in fp64, including the min(dist, 1) row weights of
// src/agent/uav.py:162-186.  Taken by UAVs within 2 m of the origin in both
// coordinates (the only place where a row weight differs from 1) and by every UAV of an environment with an
// entity outside the radius the fast path serves.  Cold: never inlined; its constants and mask pointers travel by
// value (a reference to the kernel's parameter block would force a copy of the whole block into local memory at
// kernel entry) and the result lands in a struct that only the cold branch of the caller touches.
// ------------------------------------------------------------------------------------------------
struct ExactK {
  double s_dp_le, s_dp_lt, s_2dp_le, s_dc_le, dp, dc, two_dp;
  int na;
};
struct MaskPtrs {
  uint8_t *obs_mask, *comm_mask, *nbr_mask, *dup_mask, *cover_mask;
};
template <int N, int M, bool AUX>
__device__ __noinline__ void fast_agent_exact(const ExactK P, const MaskPtrs B, const FastSmem<N, M, AUX> &S, int i,
                                              int64_t mrow_t, int64_t mrow_u, FastAgent *Op) {
  const double xi = S.oux[i], yi = S.ouy[i];
  const float *own = reinterpret_cast<const float *>(&S.slotn[i >> 1]) + (i & 1);
  const double chi = (double)own[4], shi = (double)own[6];
  const int ai = S.oua[i];
  double tt = 0, o0 = 0, o1 = 0, o2 = 0, o3 = 0;
  int nobs = 0;
  uint32_t cov[2] = {0, 0};
  for (int t = 0; t < M; t++) {
    const double dx = S.otx[t] - xi, dy = S.oty[t] - yi;
    const double d2 = dx * dx + dy * dy;
    const bool hit = d2 <= P.s_dp_le, cv = d2 <= P.s_dp_lt;
    if (AUX && B.obs_mask) { B.obs_mask[mrow_t + t] = hit; B.cover_mask[mrow_t + t] = cv; }
    if (cv) cov[t & 1] |= 1u << (t >> 1);
    if (hit) {
      const double d = sqrt(d2);
      tt += 1 + (P.dp - d) / P.dp;  // uav.py:208
      const float *tr = reinterpret_cast<const float *>(&S.tslot[t >> 1]) + (t & 1);
      double rx = dx / P.dp, ry = dy / P.dp, vx = (double)tr[4] - chi, vy = (double)tr[6] - shi;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;  // uav.py:174-180
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; }
      o0 += rx; o1 += ry; o2 += vx; o3 += vy;
      nobs++;
    }
  }
  double dup = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
  int ncomm = 0;
  uint32_t nb[2] = {0, 0};
  for (int j = 0; j < N; j++) {
    if (j == i) {
      if (AUX && B.obs_mask) { B.comm_mask[mrow_u + j] = 0; B.nbr_mask[mrow_u + j] = 0; B.dup_mask[mrow_u + j] = 0; }
      continue;
    }
    const double dxn = S.oux[j] - xi, dyn = S.ouy[j] - yi;
    const double d2n = dxn * dxn + dyn * dyn;
    const bool hit_dup = d2n <= P.s_2dp_le, hit_nbr = d2n <= P.s_dp_le;
    if (hit_dup) { const double d = sqrt(d2n); dup += -0.5 * exp((P.two_dp - d) / P.two_dp); }  // uav.py:226
    if (hit_nbr) nb[j & 1] |= 1u << (j >> 1);
    double dxc, dyc, d2c;
    const float *rj;  // partner's record: after its move if it moved first, before it otherwise
    if (j < i) { dxc = dxn; dyc = dyn; d2c = d2n; rj = reinterpret_cast<const float *>(&S.slotn[j >> 1]) + (j & 1); }
    else { dxc = S.xo[j] - xi; dyc = S.yo[j] - yi; d2c = dxc * dxc + dyc * dyc; rj = reinterpret_cast<const float *>(&S.sloto[j >> 1]) + (j & 1); }
    const bool hit_c = d2c <= P.s_dc_le;
    if (AUX && B.obs_mask) { B.comm_mask[mrow_u + j] = hit_c; B.nbr_mask[mrow_u + j] = hit_nbr; B.dup_mask[mrow_u + j] = hit_dup; }
    if (hit_c) {
      double rx = dxc / P.dc, ry = dyc / P.dc, vx = (double)rj[4] - chi, vy = (double)rj[6] - shi;
      double da = ((double)rj[8] - (double)ai) / (double)P.na;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; da /= w; }
      c0 += rx; c1 += ry; c2 += vx; c3 += vy; c4 += da;
      ncomm++;
    }
  }
  FastAgent &O = *Op;
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
// Checked twins of the three candidate walks.  A walk that accepted a squared distance inside the guard band hands
// its list to the twin, which repeats the walk and decides every pair inside the band as the reference does:
// d2 = dx*dx + dy*dy in fp64 (no contraction) against the exact squared threshold.  Cold (about one list in a
// hundred); never inlined, results through a struct that only the cold branch of the caller touches.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int sf_exact_pair(double bx, double by, double ax, double ay, double s_le, double s_lt) {
  const double dx = bx - ax, dy = by - ay;
  const double d2 = dx * dx + dy * dy;
  return (d2 <= s_le ? 1 : 0) | (d2 <= s_lt ? 2 : 0);  // bit 0: d <= thr, bit 1: d < thr
}
struct WalkOwn {     // the walking UAV
  double xi, yi;
  float xf, yf;
  int t;
};
struct TgtOut { float ox, oy, ovx, ovy, ttacc; uint32_t cvE, cvO, ncE, ncO; };
template <int N, int M, bool AUX>
__device__ __noinline__ void sf_targets_checked(const FastSmem<N, M, AUX> *Sp, const WalkOwn W, float T_lo, double s_le,
                                                double s_lt, float inv_dp_f, uint32_t cvE, uint32_t cvO, TgtOut *O) {
  const FastSmem<N, M, AUX> &S = *Sp;
  float ox = 0, oy = 0, ovx = 0, ovy = 0, ttacc = 0;
  uint32_t ncE = 0, ncO = 0;
  for (int par = 0; par < 2; par++) {
    uint32_t w = par ? cvO : cvE;
    const float *rec = reinterpret_cast<const float *>(S.tslot) + par;
    while (w) {
      const int b = sf_msb(w);
      const uint32_t bit = 1u << b;
      w ^= bit;
      const float *r = rec + 8 * b;
      const float dx = r[0] - W.xf, dy = r[2] - W.yf;
      const float s = fmaf(dx, dx, dy * dy);
      if (s > T_lo) {
        const int dec = sf_exact_pair(S.otx[2 * b + par], S.oty[2 * b + par], W.xi, W.yi, s_le, s_lt);
        if (!(dec & 1)) { if (par) cvO ^= bit; else cvE ^= bit; continue; }
        if (!(dec & 2)) { if (par) ncO |= bit; else ncE |= bit; }  // d == dp: observed and tracked, not covered
      }
      ox += dx; oy += dy; ovx += r[4]; ovy += r[6];
      ttacc = fmaf(fast_sqrtf(s), -inv_dp_f, ttacc);
    }
  }
  O->ox = ox; O->oy = oy; O->ovx = ovx; O->ovy = ovy; O->ttacc = ttacc;
  O->cvE = cvE; O->cvO = cvO; O->ncE = ncE; O->ncO = ncO;
}
struct CommOut { float sx, sy, sc, ss, sa, cn; uint32_t cmE, cmO; };
template <int N, int M, bool AUX>
__device__ __noinline__ void sf_comm_checked(const FastSmem<N, M, AUX> *Sp, const WalkOwn W, float T_lo, float T_hi,
                                             double s_le, int ihx, uint32_t w, CommOut *O) {
  const FastSmem<N, M, AUX> &S = *Sp;
  float sx = 0, sy = 0, sc = 0, ss = 0, sa = 0, cn = 0;
  uint32_t cmE = 0, cmO = 0;
  while (w) {
    const int b = sf_msb(w);
    const uint32_t bit = 1u << b;
    w ^= bit;
    const bool moved = b < ihx;  // the partner's record after its move, or before it
    const SlotRec &rec = moved ? S.slotn[b] : S.sloto[b];
    const double *px = moved ? S.oux : S.xo, *py = moved ? S.ouy : S.yo;
    const float *f = reinterpret_cast<const float *>(&rec);
    for (int h = 0; h < 2; h++) {
      const float dx = f[h] - W.xf, dy = f[2 + h] - W.yf;
      const float s = fmaf(dx, dx, dy * dy);
      bool hit = s <= T_hi;
      // (the UAV's own entry stays on the fp32 test: the caller takes it out again with the same test)
      if (hit && s > T_lo && 2 * b + h != W.t) hit = sf_exact_pair(px[2 * b + h], py[2 * b + h], W.xi, W.yi, s_le, s_le) & 1;
      if (hit) {
        sx += dx; sy += dy; sc += f[4 + h]; ss += f[6 + h]; sa += f[8 + h]; cn += 1.0f;
        if (h) cmO |= bit; else cmE |= bit;
      }
    }
  }
  O->sx = sx; O->sy = sy; O->sc = sc; O->ss = ss; O->sa = sa; O->cn = cn; O->cmE = cmE; O->cmO = cmO;
}
struct DupOut { float dup; uint32_t nbE, nbO, dpE, dpO; };
template <int N, int M, bool AUX>
__device__ __noinline__ void sf_dup_checked(const FastSmem<N, M, AUX> *Sp, const WalkOwn W, float T2_lo, float T2_hi,
                                            float Tp_lo, float Tp_hi, double s_2dp_le, double s_dp_le, float k_ex0,
                                            float k_ex1, uint32_t cdE, uint32_t cdO, DupOut *O) {
  const FastSmem<N, M, AUX> &S = *Sp;
  float dup = 0;
  uint32_t nb[2] = {0, 0}, dp[2] = {0, 0};
  for (int par = 0; par < 2; par++) {
    uint32_t w = par ? cdO : cdE;
    const unsigned char *rec = reinterpret_cast<const unsigned char *>(S.slotn) + 4 * par;
    while (w) {
      const int b = sf_msb(w);
      const uint32_t bit = 1u << b;
      w ^= bit;
      const float *r = reinterpret_cast<const float *>(rec + 48 * b);
      const float dx = r[0] - W.xf, dy = r[2] - W.yf;
      const float s = fmaf(dx, dx, dy * dy);
      if (s > T2_hi) continue;  // (cdE / cdO hold every partner of the walked slots)
      if (s > T2_lo && !(sf_exact_pair(S.oux[2 * b + par], S.ouy[2 * b + par], W.xi, W.yi, s_2dp_le, s_2dp_le) & 1)) continue;
      dp[par] |= bit;
      dup += fast_ex2f(fmaf(fast_sqrtf(s), k_ex1, k_ex0));
      if (s <= Tp_hi) {
        bool in = true;
        if (s > Tp_lo) in = sf_exact_pair(S.oux[2 * b + par], S.ouy[2 * b + par], W.xi, W.yi, s_dp_le, s_dp_le) & 1;
        if (in) nb[par] |= bit;
      }
    }
  }
  O->dup = dup; O->nbE = nb[0]; O->nbO = nb[1]; O->dpE = dp[0]; O->dpO = dp[1];
}


// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
#ifndef FAST_LOAD_WARP
#define FAST_LOAD_WARP 1   // the warp whose elected thread draws the next environment and issues its bulk loads
#endif
#ifndef FAST_COV_THREAD
#define FAST_COV_THREAD 32  // the thread that writes the covered count / done flag of an environment (warp 1: warp 0 issues the stores)
#endif
#ifndef FAST_CTAS_PER_SM
#define FAST_CTAS_PER_SM 14
#endif
template <int N, int M, bool AUX>
__global__ void __launch_bounds__(FAST_NT, FAST_CTAS_PER_SM)
uavsim_step_fast_kernel(const KParams P, const UavSimBuffers B, const ActEntry *__restrict__ act_tab, int64_t env_begin,
                        int64_t env_count, int mode, double coop, int done_flag, long long *__restrict__ stats) {
  static_assert(N == 64 && M == 64 && FAST_NT == 64, "one thread per UAV and per target");
  typedef FastSmem<N, M, AUX> SmemT;
  static_assert(offsetof(SmemT, sloto) - offsetof(SmemT, slotn) == sizeof(SlotRec) * (N / 2), "record offset");
  static_assert(sizeof(SlotRec) * N >= sizeof(float) * 12 * N && sizeof(TSlot) * (M / 2) >= sizeof(float) * 4 * N, "output staging");
  extern __shared__ __align__(128) unsigned char fast_smem_raw[];
  SmemT &S = *reinterpret_cast<SmemT *>(fast_smem_raw);
  float *const s_obs = reinterpret_cast<float *>(S.slotn);   // [N][12], after the pair phase
  float *const s_rew = reinterpret_cast<float *>(S.tslot);   // [4][N],  after the pair phase
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint32_t bar = sf_smem(&S.mbar);
  constexpr uint32_t IN_BYTES = 3 * N * 8 + 3 * M * 8 + 2 * N * 4;
  constexpr uint32_t OLD_OFF = (uint32_t)(sizeof(SlotRec) * (N / 2));
  const bool pmi_pending = (mode == UAVSIM_MODE_PMI) && (coop != 0.0);

  // one elected thread of warp 0: the eight input arrays of environment e
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
  // statistics (common.cuh: sf_fx); the reward counts are summed in 32 bits for up to 256 environments
  int fx_r = 0, fx_tt = 0, fx_bp = 0, fx_dup = 0;                 // at most 2^22 per environment
  long long fxs_r = 0, fxs_tt = 0, fxs_bp = 0, fxs_dup = 0;
  long long st_cov = 0, st_envs = 0;
  int st_cmax = 0;
  uint32_t trips = 0;
  uint32_t parity = 0;
  const int ih = t >> 1, ic = t & 1;   // own slot and place in it
  // Slots below ihx hold partners that moved before this UAV (their NEW records are observed), slots from ihx on
  // partners that move after it (OLD records); the own slot follows its other occupant (2 ih < t iff t is odd).
  const int ihx = ih + ic;

  // Environments beyond the first wave are handed out by a launch-wide counter: CTAs that the warp schedulers favour
  // take more of them, and all CTAs of an SM finish together (with a fixed stride the resident warps thinned out over
  // the last quarter of the launch: 24 of 28 warps per SM on average).
  for (int64_t k = blockIdx.x, k_next = 0; k < env_count; k = k_next) {
    const int64_t e = env_begin + k;
    sf_mbar_wait(bar, parity);  // the inputs of this environment have landed
    parity ^= 1;

    // Phase 0 is split into arithmetic (registers only, reads the input arrays) and stores: everything phase 0 writes
    // is also a source of the previous environment's bulk stores, and the ~300 instructions of arithmetic hide the
    // time the copy engine takes to read them out of shared memory (the wait sat at the loop top until round 2:
    // every thread of the CTA idled there behind the elected thread).
    // ---- phase 0a: target t (src/agent/target.py:27-60) ----
    double t_x = S.tx[t], t_y = S.ty[t], t_h = S.th[t];
    float t_vx, t_vy;
    {
      double sh, ch;
      heading_sincos(t_h, P.sincos_tab, sh, ch);
      t_x += P.dtv_t * ch;
      t_y += P.dtv_t * sh;
      // reflection (target.py:52-58); cos(-h) = cos h, sin(-h) = -sin h, cos(+-pi - h) = -cos h, sin(+-pi - h) = sin h
      if (0 > t_y || t_y > P.y_max) { t_h = -t_h; sh = -sh; }
      else if (t_x < 0 || t_x > P.x_max) { t_h = (t_h > 0) ? (PI_D - t_h) : (-PI_D - t_h); ch = -ch; }
      t_vx = (float)ch * P.tv_over_uv_f; t_vy = (float)sh * P.tv_over_uv_f;
    }
    const float txf = (float)(t_x - P.cx), tyf = (float)(t_y - P.cy);
    float rabs = fmaxf(fabsf(txf), fabsf(tyf));
    // ---- phase 0b: UAV t (src/agent/uav.py:73-99) ----
    double xi, yi, hi;      // state after the move
    float xf, yf, chf, shf, xl, yl;  // own fp32 position relative to the centre, heading, and what fp32 dropped of the position
    const double xo_d = S.ux[t], yo_d = S.uy[t];
    const int a_old = S.ua[t], ai = S.act[t];
    float xof, yof, cof, sof;
    {
      double h = S.uh[t];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);
      cof = (float)ch; sof = (float)sh;
      xof = (float)(xo_d - P.cx); yof = (float)(yo_d - P.cy);
      xi = xo_d + P.dtv_u * ch;
      yi = yo_d + P.dtv_u * sh;
      double dh;
      float cd, sd;
      if ((unsigned)ai < (unsigned)P.na) {
        const ActEntry en = act_tab[ai];
        dh = en.dth; cd = en.cd; sd = en.sd;
      } else {  // the reference's formula accepts any integer (uav.py:73-81)
        dh = P.dt * ((double)(2 * (ai + 1) - P.na - 1) * P.uav_h_max / (double)(P.na - 1));
        double sd_, cd_;
        sincos_shared(dh, &sd_, &cd_);
        cd = (float)cd_; sd = (float)sd_;
      }
      hi = wrap_heading(h + dh);
      // cos / sin of the new heading by angle addition in fp32: they only feed the observation (the next step
      // evaluates the stored heading again)
      chf = fmaf(cof, cd, -(sof * sd));
      shf = fmaf(sof, cd, cof * sd);
      xf = (float)(xi - P.cx); yf = (float)(yi - P.cy);
      xl = (float)((xi - P.cx) - (double)xf); yl = (float)((yi - P.cy) - (double)yf);
      rabs = fmaxf(fmaxf(rabs, fmaxf(fabsf(xf), fabsf(yf))), fmaxf(fabsf(xof), fabsf(yof)));
      // fp32 sums of action indices are exact only for small integers: anything else takes the exact path
      if ((unsigned)ai >= 4096u || (unsigned)a_old >= 4096u) rabs = __int_as_float(0x7f800000);
      if (!(rabs == rabs)) rabs = __int_as_float(0x7f800000);
    }
    // The thread that committed the previous outputs waits until they have left shared memory.  (Bulk groups belong
    // to the issuing thread: elect.sync with a full mask picks the same lane every time.)
    if (warp == 0) {
      if (elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    __syncthreads();
    {
      S.otx[t] = t_x; S.oty[t] = t_y; S.oth[t] = t_h;
      float *ts = reinterpret_cast<float *>(&S.tslot[ih]) + ic;
      ts[0] = txf; ts[2] = tyf; ts[4] = t_vx; ts[6] = t_vy;
      if (AUX) S.tcnt[t] = 0;
      S.xo[t] = xo_d; S.yo[t] = yo_d;
      float *so = reinterpret_cast<float *>(&S.sloto[ih]) + ic;
      so[0] = xof; so[2] = yof; so[4] = cof; so[6] = sof; so[8] = (float)a_old;
      S.oux[t] = xi; S.ouy[t] = yi; S.ouh[t] = hi; S.oua[t] = ai;
      float *sn = reinterpret_cast<float *>(&S.slotn[ih]) + ic;
      sn[0] = xf; sn[2] = yf; sn[4] = chf; sn[6] = shf; sn[8] = (float)ai;
    }
    {
      const uint32_t rm = __reduce_max_sync(0xffffffffu, __float_as_uint(rabs));
      if (lane == 0) S.rmax[warp] = rm;
    }
    __syncthreads();
    if (warp == FAST_LOAD_WARP) {  // next environment, behind the pair phase (warp 0 issues the twelve stores: the duties are split)
      if (elect_one()) {
        const int64_t kn = (int64_t)gridDim.x + (int64_t)atomicAdd(P.fast_ctr, 1);
        S.next_k = kn;
        if (kn < env_count) issue_loads(env_begin + kn);
      }
    }

    // ---- phase 1: pair tests, observation, raw reward ----
    const float R = __uint_as_float(max(S.rmax[0], S.rmax[1]));
    const bool far_env = !(R <= P.r_fast);
    const bool near_origin = fabs(xi) < 2.0 && fabs(yi) < 2.0;  // the only place a row weight differs from 1
    const int64_t mrow_t = (e * N + t) * M, mrow_u = (e * N + t) * N;
    // results of the pair phase: nine list entries of the local state, raw tracking / duplicate terms, the
    // neighbour set d <= dp and the targets strictly inside dp (even / odd words)
    float o0, o1, o2, o3, o4, o5, o6, o7, o8, tt_f, dup_f;
    uint32_t nbE = 0, nbO = 0, cvE = 0, cvO = 0;
    uint32_t ncE = 0, ncO = 0;  // targets at distance exactly dp: observed and tracked, not covered
    uint32_t cmE = 0, cmO = 0, dpE = 0, dpO = 0;  // AUX: communication / duplicate sets for the mask outputs
#ifdef FAST_ABL_NOPAIRS
    // profiling switch (tools/gpu_round.sh): no pair work at all -- what phase 0, the finishing code and the copies cost
    const bool exact = false;
    o0 = o1 = o2 = o3 = o4 = o5 = o6 = o7 = o8 = -1.f; tt_f = 0.f; dup_f = 0.f;
    if (far_env && near_origin) {
#else
    const bool exact = far_env || near_origin;
    if (!exact) {
#endif
      const float g_dp = fmaf(R, P.g_dp.c1, P.g_dp.c0), g_2dp = fmaf(R, P.g_2dp.c1, P.g_2dp.c0);
      // An old position rebuilt from the new one carries the rounding of the new coordinate, of the cosine and of the
      // FMA: at most u (2R + dt v) instead of u R, so the offset's error grows from 2uR to u (3R + dt v) <= twice the
      // modelled one plus the guard's slope times dt v.
      const float ndtv_f = -P.dtv_u_f;
      const float g_dc = 2.0f * fmaf(R, P.g_dc.c1, P.g_dc.c0) + P.g_dc.c1 * fabsf(P.dtv_u_f);
      const float g_pf = fmaf(R, P.g_pf.c1, P.g_pf.c0);
      const float Tp_hi = __fadd_ru(P.g_dp.t2_up, g_dp), Tp_lo = __fadd_rd(P.g_dp.t2_dn, -g_dp);
      const float T2_hi = __fadd_ru(P.g_2dp.t2_up, g_2dp), T2_lo = __fadd_rd(P.g_2dp.t2_dn, -g_2dp);
      const float Tc_hi = __fadd_ru(P.g_dc.t2_up, g_dc), Tc_lo = __fadd_rd(P.g_dc.t2_dn, -g_dc);
      const float Tf_hi = __fadd_ru(P.g_pf.t2_up, g_pf);
      const uint64_t xf2 = pack2(xf, xf), yf2 = pack2(yf, yf);
      const WalkOwn WO = {xi, yi, xf, yf, t};

      uint32_t ccE, ccO;  // UAV candidate slots (even / odd partner)
      // -- targets: observe_target (uav.py:101-122), tracking reward (uav.py:199-212), coverage (environment.py:246-253)
      {
        uint32_t d0, d1;
        prefilter64<false, (int)sizeof(TSlot)>(S.tslot, xf, yf, Tp_hi, 0.f, cvE, cvO, d0, d1);
        float ox = 0, oy = 0, ovx = 0, ovy = 0, ttacc = 0, smax_t = 0;
#pragma unroll
        for (int par = 0; par < 2; par++) {
          uint32_t w = par ? cvO : cvE;
          const float *rec = reinterpret_cast<const float *>(S.tslot) + par;
#pragma unroll 1
          while (w) {
            const int b = sf_msb(w);
            w ^= 1u << b;
            const float *r = rec + 8 * b;
            const float dx = r[0] - xf, dy = r[2] - yf;
            const float s = fmaf(dx, dx, dy * dy);
            smax_t = fmaxf(smax_t, s);  // every candidate is accepted: unambiguous iff all of them are below the lower guard
            ox += dx; oy += dy; ovx += r[4]; ovy += r[6];
            ttacc = fmaf(fast_sqrtf(s), -inv_dp_f, ttacc);  // sum of (dp - d)/dp - 1
          }
        }
        if (smax_t > Tp_lo) {  // a pair inside the guard band: this list once more, checked
          TgtOut X;
          sf_targets_checked<N, M, AUX>(&S, WO, Tp_lo, P.s_dp_le, P.s_dp_lt, inv_dp_f, cvE, cvO, &X);
          ox = X.ox; oy = X.oy; ovx = X.ovx; ovy = X.ovy; ttacc = X.ttacc;
          cvE = X.cvE; cvO = X.cvO; ncE = X.ncE; ncO = X.ncO;
        }
        const int nobs = __popc(cvE) + __popc(cvO);
        if (nobs) {
          const float kf = (float)nobs, rk = sf_rcp(kf);
          // the own coordinate's fp32 rounding is common to every row: taken out of the mean exactly
          o5 = fmaf(ox, rk, -xl) * inv_dp_f;
          o6 = fmaf(oy, rk, -yl) * inv_dp_f;
          o7 = fmaf(ovx, rk, -chf);
          o8 = fmaf(ovy, rk, -shf);
          tt_f = fmaf(2.0f, kf, ttacc);  // sum of 1 + (dp - d)/dp
        } else {
          o5 = o6 = o7 = o8 = -1.f;
          tt_f = 0.f;
        }
      }

      // -- UAV partners.  ONE prefilter on the NEW positions against the widest radius any UAV-UAV test can reach:
      //    the communication radius widened by one move (a partner that moves after this UAV is tested at its old
      //    position, at most dt*v from the new one) or the duplicate-tracking radius 2 dp, whichever is larger
      //    (KParams::g_pf).  The own bit is always set (distance 0): the own slot is walked like any other and the own
      //    contributions, known in closed form, are taken out afterwards.
      uint32_t d0_, d1_;
      prefilter64<false, (int)sizeof(SlotRec)>(S.slotn, xf, yf, Tf_hi, 0.f, ccE, ccO, d0_, d1_);
      const unsigned char *slot_new = reinterpret_cast<const unsigned char *>(S.slotn);
      const unsigned char *slot_old = reinterpret_cast<const unsigned char *>(S.sloto);
      // -- ONE walk over the candidate slots, two partners per trip, for the three UAV-UAV lists:
      //    communication (uav.py:124-147; the partner's record after its move if it moved first, before it otherwise),
      //    duplicate-tracking punishment (uav.py:214-229) and the neighbour set (uav.py:305), both at NEW positions.
      //    Weights 1 / 0 from the upper guards; per list one running extreme (largest accepted squared distance, or the
      //    smallest |n - T| for the neighbour bits) tells afterwards whether a pair sat inside the band.  (Until round 2
      //    the duplicate / neighbour list had its own prefilter radius and its own walk, one partner per trip: 27 trips
      //    of 22 instructions on top of the 20 communication trips; here it rides on the communication trips.  The trip
      //    is 52 instructions with two 16-byte loads and one 8-byte load: tools/loop_count.py.)
      {
        uint64_t sx = 0, sy = 0, sc = 0, ss = 0, sa = 0, cn = 0, dp2 = 0;
        float smax_c = 0.f, smax_d = 0.f, dmin_n = 3.0e38f;
        const float Tp_nx = __uint_as_float(__float_as_uint(Tp_hi) + 1u);   // the float above Tp_hi (positive)
        const uint64_t tpn2 = pack2(Tp_nx, Tp_nx);
        // |n - T| <= T - Tp_lo covers Tp_lo <= n <= Tp_hi (and as much above T); never narrower than a few ulp of T
        const float nb_band = fmaxf(__fadd_ru(Tp_nx, -Tp_lo), 4.0f * (Tp_nx - Tp_hi));
        const uint64_t kx1 = pack2(k_ex1, k_ex1), kx0 = pack2(k_ex0, k_ex0);
        uint32_t w = ccE | ccO;
#pragma unroll 1
        while (w) {
          const int b = sf_msb(w);
          const uint32_t bit = 1u << b;
          w ^= bit;
          const unsigned char *rn = slot_new + 48 * b;
          const bool moved = b < ihx;
          const unsigned char *rp = (moved ? slot_new : slot_old) + 48 * b;  // (one select and one multiply-add)
          const ulonglong2 hd = *reinterpret_cast<const ulonglong2 *>(rp + 16);   // {cos0, cos1}, {sin0, sin1}
          const uint64_t aa = *reinterpret_cast<const uint64_t *>(rp + 32);       // {a0, a1}
          const ulonglong2 pn = *reinterpret_cast<const ulonglong2 *>(rn);        // positions after the move
          // offsets at the new positions (duplicate tracking / neighbours), and from them the offsets the communication
          // test needs: the partner's position BEFORE its move is the one after it minus dt v (cos h, sin h) of the OLD
          // heading (uav.py:88-94), so one packed FMA per axis replaces a third 16-byte load and a subtraction; the
          // communication guard carries the extra rounding
          const uint64_t ex = f2_sub(pn.x, xf2), ey = f2_sub(pn.y, yf2);
          const float mv = moved ? 0.0f : ndtv_f;
          const uint64_t mv2 = pack2(mv, mv);
          const uint64_t dx = f2_fma(hd.x, mv2, ex), dy = f2_fma(hd.y, mv2, ey);
          const uint64_t s2 = f2_fma(dx, dx, f2_mul(dy, dy));
          const float s0 = f2_lo(s2), s1 = f2_hi(s2);
          const bool h0 = s0 <= Tc_hi, h1 = s1 <= Tc_hi;
          const uint64_t wh = pack2(h0 ? 1.0f : 0.0f, h1 ? 1.0f : 0.0f);
          {  // largest accepted squared distance through the weights: one packed product and one three-way maximum
            const uint64_t sw = f2_mul(s2, wh);
            smax_c = fmaxf(fmaxf(smax_c, f2_lo(sw)), f2_hi(sw));
          }
          sx = f2_fma(wh, dx, sx); sy = f2_fma(wh, dy, sy);
          sc = f2_fma(wh, hd.x, sc); ss = f2_fma(wh, hd.y, ss);
          sa = f2_fma(wh, aa, sa);
          cn = f2_add(cn, wh);
          if (AUX) { if (h0) cmE |= bit; if (h1) cmO |= bit; }
          // duplicate tracking / neighbours at the new positions
          const uint64_t n2 = f2_fma(ex, ex, f2_mul(ey, ey));
          const float n0 = f2_lo(n2), n1 = f2_hi(n2);
          const bool g0 = n0 <= T2_hi, g1 = n1 <= T2_hi;
          const uint64_t wg = pack2(g0 ? 1.0f : 0.0f, g1 ? 1.0f : 0.0f);
          {
            const uint64_t nw = f2_mul(n2, wg);
            smax_d = fmaxf(fmaxf(smax_d, f2_lo(nw)), f2_hi(nw));
          }
          const uint64_t arg = f2_fma(pack2(fast_sqrtf(n0), fast_sqrtf(n1)), kx1, kx0);
          dp2 = f2_fma(wg, pack2(fast_ex2f(f2_lo(arg)), fast_ex2f(f2_hi(arg))), dp2);  // exp((2dp - d)/(2dp))
          if (AUX) { if (g0) dpE |= bit; if (g1) dpO |= bit; }
          {  // Neighbour bits from the SIGN of n - T (T = the float above Tp_hi: n <= Tp_hi iff n - T < 0), spread over the
             // word by an arithmetic shift; the smallest |n - T| seen tells afterwards whether any partner sat in the
             // band around the radius (either side of it: a few more checked walks, never a wrong bit).
            const uint64_t dn = f2_sub(n2, tpn2);
            const uint32_t m0 = (uint32_t)((int32_t)(uint32_t)dn >> 31), m1 = (uint32_t)((int32_t)(uint32_t)(dn >> 32) >> 31);
            nbE |= m0 & bit; nbO |= m1 & bit;
            dmin_n = fminf(fminf(dmin_n, fabsf(f2_lo(dn))), fabsf(f2_hi(dn)));
          }
        }
        // own entry of the own slot: the record that was read there (new if this UAV sits in the odd place, else old)
        // (the own entry also went into smax_c: its distance is 0 or one move, far from the band unless dt*v ~ dc; the
        // checked twin keeps it on this same fp32 test)
        float own_w, own_dx, own_dy, own_c, own_s, own_a;
        {
          const float *r = reinterpret_cast<const float *>(slot_new + (ic ? 0u : OLD_OFF) + 48 * ih) + ic;
          own_c = r[4]; own_s = r[6]; own_a = r[8];
          // the same arithmetic as the walk: 0 in the odd place (new record), one move back in the even place
          own_dx = own_c * (ic ? 0.0f : ndtv_f); own_dy = own_s * (ic ? 0.0f : ndtv_f);  // fma(c, mv, xf - xf)
          const float s_own = fmaf(own_dx, own_dx, own_dy * own_dy);
          own_w = sf_le(s_own, Tc_hi);
        }
        float tsx = f2_lo(sx) + f2_hi(sx), tsy = f2_lo(sy) + f2_hi(sy), tsc = f2_lo(sc) + f2_hi(sc);
        float tss = f2_lo(ss) + f2_hi(ss), tsa = f2_lo(sa) + f2_hi(sa), tcn = f2_lo(cn) + f2_hi(cn);
        if (smax_c > Tc_lo) {  // a pair inside the guard band: this list once more, checked
          CommOut X;
          sf_comm_checked<N, M, AUX>(&S, WO, Tc_lo, Tc_hi, P.s_dc_le, ihx, ccE | ccO, &X);
          tsx = X.sx; tsy = X.sy; tsc = X.sc; tss = X.ss; tsa = X.sa; tcn = X.cn;
          if (AUX) { cmE = X.cmE; cmO = X.cmO; }
        }
        const float cntf = tcn - own_w;
        if (AUX) { if (ic) cmO &= ~(1u << ih); else cmE &= ~(1u << ih); }
        if (cntf > 0.5f) {
          const float rk = sf_rcp(cntf);
          o0 = fmaf(tsx - own_w * own_dx, rk, -xl) * inv_dc_f;
          o1 = fmaf(tsy - own_w * own_dy, rk, -yl) * inv_dc_f;
          o2 = fmaf(tsc - own_w * own_c, rk, -chf);
          o3 = fmaf(tss - own_w * own_s, rk, -shf);
          o4 = ((tsa - own_w * own_a) - cntf * (float)ai) * (rk * inv_na_f);
        } else {
          o0 = o1 = o2 = o3 = o4 = -1.f;
        }
        // the UAV itself (distance 0 after the move) went through the duplicate / neighbour tests: taken out again
        const uint32_t ownE = ic ? 0u : (1u << ih), ownO = ic ? (1u << ih) : 0u;
        float dup = (f2_lo(dp2) + f2_hi(dp2)) - fast_ex2f(fmaf(fast_sqrtf(0.f), k_ex1, k_ex0));
        nbE &= ~ownE; nbO &= ~ownO;
        if (AUX) { dpE &= ~ownE; dpO &= ~ownO; }
        if ((smax_d > T2_lo) || (dmin_n <= nb_band)) {  // a pair inside a guard band: this list once more, checked
          DupOut X;
          sf_dup_checked<N, M, AUX>(&S, WO, T2_lo, T2_hi, Tp_lo, Tp_hi, P.s_2dp_le, P.s_dp_le, k_ex0, k_ex1, (ccE | ccO) & ~ownE,
                                    (ccE | ccO) & ~ownO, &X);
          dup = X.dup; nbE = X.nbE; nbO = X.nbO;
          if (AUX) { dpE = X.dpE; dpO = X.dpO; }
        }
        dup_f = -0.5f * dup;
      }
    }
    if (exact) {
      const ExactK XK = {P.s_dp_le, P.s_dp_lt, P.s_2dp_le, P.s_dc_le, P.dp, P.dc, P.two_dp, P.na};
      const MaskPtrs MP = {B.obs_mask, B.comm_mask, B.nbr_mask, B.dup_mask, B.cover_mask};
      FastAgent X;
      fast_agent_exact<N, M, AUX>(XK, MP, S, t, mrow_t, mrow_u, &X);
      o0 = X.ob[0]; o1 = X.ob[1]; o2 = X.ob[2]; o3 = X.ob[3]; o4 = X.ob[4];
      o5 = X.ob[5]; o6 = X.ob[6]; o7 = X.ob[7]; o8 = X.ob[8];
      tt_f = X.tt; dup_f = X.dup;
      nbE = X.nb[0]; nbO = X.nb[1]; cvE = X.cov[0]; cvO = X.cov[1];
    } else if (AUX && B.obs_mask) {
      for (int j = 0; j < 64; j++) {
        const int b = j >> 1;
        const uint8_t v = (((j & 1) ? cvO : cvE) >> b) & 1u;
        B.obs_mask[mrow_t + j] = v; B.cover_mask[mrow_t + j] = v & ~((((j & 1) ? ncO : ncE) >> b) & 1u);
        B.comm_mask[mrow_u + j] = (((j & 1) ? cmO : cmE) >> b) & 1u;
        B.nbr_mask[mrow_u + j] = (((j & 1) ? nbO : nbE) >> b) & 1u;
        B.dup_mask[mrow_u + j] = (((j & 1) ? dpO : dpE) >> b) & 1u;
      }
    }
    cvE &= ~ncE; cvO &= ~ncO;  // from here on: the targets strictly inside dp
    if (AUX && B.tracker_cnt) {
#pragma unroll
      for (int par = 0; par < 2; par++) {
        uint32_t w = par ? cvO : cvE;
        while (w) { const int b = sf_msb(w); w ^= 1u << b; atomicAdd(&S.tcnt[2 * b + par], 1); }
      }
    }
    {  // coverage: targets with at least one UAV strictly inside dp (environment.py:246-253), OR over the warp
      const uint32_t c0 = __reduce_or_sync(0xffffffffu, cvE), c1 = __reduce_or_sync(0xffffffffu, cvO);
      if (lane == 0) { S.cover[warp][0] = c0; S.cover[warp][1] = c1; }
    }

    // The terms below only feed fp32 outputs (and the statistics of those outputs): evaluated in fp32.  The one
    // decision among them, inside / outside the map (uav.py:239), stays in fp64.
    float raw, ttn, bpn, dupn;
    {
      // boundary punishment (uav.py:231-250).  Distance to the nearest wall from the centred fp32 coordinates; the
      // inside / outside decision (closed interval, uav.py:239) falls back to fp64 within a millimetre of a wall.
      // (The value is continuous across the wall, -1/2 on both sides; the decision only has to be consistent.)
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
    }
    __syncthreads();  // every walk is over: the slot areas become the output staging
    k_next = S.next_k;

    // ---- phase 2: cooperative reward (environment.py:222-227), coverage count, outputs ----
    {
      float *ob = s_obs + t * 12;
      reinterpret_cast<float4 *>(ob)[0] = make_float4(o0, o1, o2, o3);
      reinterpret_cast<float4 *>(ob)[1] = make_float4(o4, o5, o6, o7);
      reinterpret_cast<float4 *>(ob)[2] = make_float4(o8, (float)(xi * P.inv_dc), (float)(yi * P.inv_dc), (float)ai * inv_na_f);
      float r;
      const int64_t gi = e * N + t;
      if (mode == UAVSIM_MODE_SELF || coop == 0.0) {
        r = raw;  // uav.py:271-272 / :300-301
      } else if (mode == UAVSIM_MODE_MEAN) {
        // uav.py:293-310 -- the conditional expression covers the whole sum: no neighbour -> 0
        float s = 0;
        const int cnt = __popc(nbE) + __popc(nbO);
        {  // one trip per slot with a neighbour: both raw rewards of the slot in one 8-byte load
          uint32_t u = nbE | nbO;
          float s1 = 0;
          while (u) {
            const int b = sf_msb(u);
            const uint32_t bit = 1u << b;
            u ^= bit;
            const float2 rr = *reinterpret_cast<const float2 *>(&S.raw[2 * b]);
            s += (nbE & bit) ? rr.x : 0.0f;
            s1 += (nbO & bit) ? rr.y : 0.0f;
          }
          s += s1;
        }
        const float cf = (float)coop;
        r = cnt ? fmaf(1.0f - cf, raw, cf * s * sf_rcp((float)cnt)) : 0.0f;
      } else {
        r = 0.0f;  // finished by the PMI kernel
        B.raw[gi] = (double)raw;
        B.nbr_bits[gi * 2] = sf_interleave(nbE, nbO);
        B.nbr_bits[gi * 2 + 1] = 0;
      }
      r = fminf(fmaxf(r, -1.0f), 1.0f);  // clip_and_normalize(reward, -1, 1) is a plain clip
      s_rew[t] = r;
      s_rew[N + t] = ttn;
      s_rew[2 * N + t] = bpn;
      s_rew[3 * N + t] = dupn;
      if (!pmi_pending) fx_r += sf_fx(r);
      fx_tt += sf_fx(ttn); fx_bp += sf_fx(bpn); fx_dup += sf_fx(dupn);
      if ((++trips & 255u) == 0u) {  // 256 environments fill 31 bits: move the sums on to 64 bits
        fxs_r += fx_r; fxs_tt += fx_tt; fxs_bp += fx_bp; fxs_dup += fx_dup;
        fx_r = fx_tt = fx_bp = fx_dup = 0;
      }
      if (AUX && B.tracker_cnt) B.tracker_cnt[e * M + t] = S.tcnt[t];
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
    if (t == FAST_COV_THREAD) {
      const int c = __popc(S.cover[0][0] | S.cover[1][0]) + __popc(S.cover[0][1] | S.cover[1][1]);
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
  work_counter_leave(P.fast_ctr);
  stats_commit(stats + (size_t)blockIdx.x * STAT_W, fxs_r + fx_r, fxs_tt + fx_tt, fxs_bp + fx_bp, fxs_dup + fx_dup, st_cov,
               st_cmax, st_envs);
}
