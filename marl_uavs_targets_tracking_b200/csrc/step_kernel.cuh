// step_kernel.cuh -- the fused environment step kernel (Environment.step, src/environment.py:120-164).
//
// CTA = epb environments, thread q = (env q / n, UAV q % n), epb * n <= NT.  Per step:
//   phase 0  targets move and reflect (src/agent/target.py:27-60), UAVs integrate their heading-rate action
//            (src/agent/uav.py:73-99); old and new UAV records are staged in shared memory (one block per
//            environment, double2 records read with broadcast 128-bit loads, plus fp32 shadows of the
//            positions relative to the map centre).
//   phase 1  one thread per UAV, partners in chunks of 32.  (A) an fp32 prefilter walks every partner of the
//            chunk (4 flops + compares) and keeps a candidate bit when the fp32 squared distance is below the
//            threshold PLUS a guard band that bounds the fp32 error; (B) only the candidates are re-evaluated
//            in fp64 on the exact squared thresholds, which decide every mask; hits accumulate the observation
//            sums, tracking / duplicate terms, neighbour bits and per-target tracker counts.  Then the boundary
//            term, normalisation and weights.
//   phase 2  cooperative reward (self / neighbour mean; PMI is finished by uavsim_pmi_kernel), coverage
//            count, coalesced output stores, per-CTA episode statistics.
//
// Precision plan.  Everything that decides an integer output (the five range masks, coverage) is fp64 in
// the reference's evaluation order; the fp32 prefilter is only ever conservative (KParams::f_*, see
// prefilter_threshold in uavsim.cu) and is bypassed for an environment whose entities left the radius the
// error bound assumes.  The observation sums are fp64 but LINEAR: mean_j((x_j - x_i)/dc) is accumulated as
// sum(x_j - x_i) and scaled once -- valid because the reference's per-row weight min(||(rx,ry) - (x,y)||, 1)
// (src/agent/uav.py:162-186) is exactly 1 unless |x| < 2 and |y| < 2; UAVs inside that 4 m x 4 m corner
// take the exact per-row path (agent_exact).  The transcendental parts of the tracking and duplicate terms
// (sqrt, exp on hits) are evaluated in fp32: they only feed fp32 outputs that are normalised by 2m and
// e/2*n (error <= ~1e-7 against the 1e-5 bar).
#pragma once
#include "common.cuh"
#include "fast_math.cuh"

// tuning knobs (overridable with -D for experiments)
#ifndef UAVSIM_NT64
#define UAVSIM_NT64 64   // threads per CTA of the 64x64 kernel
#endif

// ------------------------------------------------------------------------------------------------
// shared memory: one block per environment (byte offsets below), then CTA-wide arrays
// ------------------------------------------------------------------------------------------------
struct EnvLayout {
  int tpos, tvel, npos, nhd, opos, ohd, tposf, nposf, na_, oa, stride;
};

__host__ __device__ constexpr EnvLayout env_layout(int n, int m) {
  EnvLayout L{};
  int o = 0;
  L.tpos = o; o += 16 * m;   // double2 (x, y) after the move
  L.tvel = o; o += 16 * m;   // double2 (cos h, sin h) * tv / uv
  L.npos = o; o += 16 * n;   // double2 UAV (x, y) after the move
  L.nhd = o; o += 16 * n;    // double2 (cos h, sin h) after the move
  L.opos = o; o += 16 * n;   // before the move
  L.ohd = o; o += 16 * n;
  L.tposf = o; o += 16 * ((m + 1) / 2);  // fp32 target positions relative to the map centre, two per float4 {x0, x1, y0, y1}
  L.nposf = o; o += 16 * ((n + 1) / 2);  // fp32 new UAV positions, same pairing (operands of the packed f32x2 prefilter)
  L.na_ = o; o += 4 * n;     // new action index
  L.oa = o; o += 4 * n;      // previous action index
  L.stride = (o + 15) & ~15;
  return L;
}

struct CtaSmem {
  unsigned char *env;  // [epb] environment blocks
  double *raw;         // [epb*n]
  double *dth;         // [3*na] per action: dt*rate, cos(dt*rate), sin(dt*rate)
  long long *next;     // the group this CTA steps next (drawn by thread 0)
  float *obs;          // [epb*n*12]
  int *tcnt;           // [epb*m] UAVs strictly within dp of each target
  int *far;            // [epb] 1 if an entity is farther than KParams::rmax from the map centre
  int *cov;            // [epb] covered targets
};

static size_t step_smem_bytes(int n, int m, int na, int epb) {
  const EnvLayout L = env_layout(n, m);
  size_t b = (size_t)epb * L.stride;
  b += ((size_t)epb * n + 1) * 8 + 8;           // raw, next (+ pad)
  b += (size_t)epb * n * 12 * 4;                // obs
  b += ((size_t)epb * m + 2 * (size_t)epb) * 4 + 4;  // tcnt, far, cov (+ pad)
  b += 3 * (size_t)na * 8;                      // dth
  return b + 16;
}

// The per-action table (the only run-time sized array) comes last, so with compile-time n, m and epb every other
// offset is a constant.
__device__ __forceinline__ CtaSmem carve(unsigned char *base, int n, int m, int na, int epb, int stride) {
  CtaSmem s;
  s.env = base;
  double *d = reinterpret_cast<double *>(base + (size_t)epb * stride);  // stride is a multiple of 16
  s.raw = d; d += (size_t)epb * n;
  s.next = reinterpret_cast<long long *>(d); d += 1;
  d += ((size_t)epb * n + 1) & 1;  // keep obs 16-byte aligned (plain pointer arithmetic: stays shared)
  s.obs = reinterpret_cast<float *>(d);
  int *ip = reinterpret_cast<int *>(s.obs + (size_t)epb * n * 12);
  s.tcnt = ip; ip += (size_t)epb * m;
  s.far = ip; ip += epb;
  s.cov = ip; ip += epb;
  ip += ((size_t)epb * m) & 1;  // 8-byte alignment for the doubles that follow
  s.dth = reinterpret_cast<double *>(ip);
  (void)na;
  return s;
}

// typed views into one environment block
struct EnvView {
  unsigned char *b;
  EnvLayout L;
  __device__ __forceinline__ double2 *tpos() const { return reinterpret_cast<double2 *>(b + L.tpos); }
  __device__ __forceinline__ double2 *tvel() const { return reinterpret_cast<double2 *>(b + L.tvel); }
  __device__ __forceinline__ double2 *npos() const { return reinterpret_cast<double2 *>(b + L.npos); }
  __device__ __forceinline__ double2 *nhd() const { return reinterpret_cast<double2 *>(b + L.nhd); }
  __device__ __forceinline__ double2 *opos() const { return reinterpret_cast<double2 *>(b + L.opos); }
  __device__ __forceinline__ double2 *ohd() const { return reinterpret_cast<double2 *>(b + L.ohd); }
  __device__ __forceinline__ float4 *tposf() const { return reinterpret_cast<float4 *>(b + L.tposf); }
  __device__ __forceinline__ float4 *nposf() const { return reinterpret_cast<float4 *>(b + L.nposf); }
  // entity j of a paired array: pair j/2, slot j%2 (x at float slot, y two floats later)
  __device__ __forceinline__ static void put_pair(float4 *arr, int j, float x, float y) {
    float *f = reinterpret_cast<float *>(arr + (j >> 1)) + (j & 1);
    f[0] = x; f[2] = y;
  }
  __device__ __forceinline__ static float2 get_pair(const float4 *arr, int j) {
    const float *f = reinterpret_cast<const float *>(arr + (j >> 1)) + (j & 1);
    return make_float2(f[0], f[2]);
  }
  __device__ __forceinline__ int *na_() const { return reinterpret_cast<int *>(b + L.na_); }
  __device__ __forceinline__ int *oa() const { return reinterpret_cast<int *>(b + L.oa); }
};

// one copy of the fp64 sincos code for both call sites (instruction-fetch footprint)
__device__ __noinline__ void sincos_shared(double h, double *s, double *c) { sincos(h, s, c); }

// sin / cos of a heading: the wrapped range takes the inline routine, anything else the library one (whose pointer
// arguments stay inside the cold branch)
__device__ __forceinline__ void heading_sincos(double h, const double *tab, double &s, double &c) {
  if (fabs(h) < 3.3) {
    double s1, c1;
    fm_sincos_tab(h, tab, &s1, &c1);
    s = s1; c = c1;
  } else {
    double s2, c2;
    sincos_shared(h, &s2, &c2);
    s = s2; c = c2;
  }
}

// (h + pi) % (2 pi) - pi with Python's float % (uav.py:97).  For h + pi in [-2pi, 4pi) -- always, unless dt * rate
// exceeds a full turn -- the fmod is one exact subtraction (Sterbenz) or, below zero, the same single addition
// CPython performs after fmod; otherwise the general routine.
__device__ __forceinline__ double wrap_heading(double h) {
  const double TWO_PI = 2 * PI_D;
  double x = h + PI_D;
  if (x >= 0.0 && x < TWO_PI) { /* fmod is the identity */ }
  else if (x >= TWO_PI && x < 2 * TWO_PI) x -= TWO_PI;
  else if (x < 0.0 && x > -TWO_PI) x += TWO_PI;
  else x = pymod_pos(x, TWO_PI);
  return x - PI_D;
}

// Hot-loop loads through an explicit 32-bit shared address.  With C++ pointers the compiler re-derives the base of the
// dynamic shared array (S2UR SR_CgaCtaId + UMOV + ULEA + IMAD.U32) next to almost every access instead of keeping it
// in a register -- ~5 % of the issued instructions, twice per trip of the candidate loops; an address that went through
// an opaque asm once has to stay in its register.
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) { asm volatile("mov.b32 %0, %0;" : "+r"(v)); return v; }
__device__ __forceinline__ double2 lds_d2(uint32_t a) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ int lds_i32(uint32_t a) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}

// what phase 1 produces for one UAV
struct AgentOut {
  double tt, dup;         // raw tracking reward / duplicate punishment (before normalisation)
  uint32_t nb[4];         // neighbour set d <= dp, bit j of word j/32
};

// approximate fp32 sqrt / exp2 (one MUFU each, ~2 ulp): they only feed fp32 reward terms
__device__ __forceinline__ float fast_sqrtf(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fast_ex2f(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ------------------------------------------------------------------------------------------------
// exact per-row path: the reference's arithmetic hit by hit, including the min(dist,1) row weights.
// Taken by UAVs within 2 m of the origin in both coordinates (never inlined: it is cold).
// ------------------------------------------------------------------------------------------------
template <bool MASKS>
__device__ __noinline__ void agent_exact(const KParams &P, const UavSimBuffers &B, const EnvView V, int *tcnt, int i,
                                         int n, int m, float *ob, int64_t mrow_t, int64_t mrow_u, AgentOut *Op) {
  const double2 me = V.npos()[i], mh = V.nhd()[i];
  const double xi = me.x, yi = me.y, chi = mh.x, shi = mh.y;
  const int ai = V.na_()[i];
  const double2 *tpos = V.tpos(), *tvel = V.tvel(), *npos = V.npos(), *nhd = V.nhd(), *opos = V.opos(), *ohd = V.ohd();
  const int *na_ = V.na_(), *oa = V.oa();
  double tt = 0, o0 = 0, o1 = 0, o2 = 0, o3 = 0;
  int nobs = 0;
  for (int t = 0; t < m; t++) {
    const double2 tp = tpos[t];
    const double dx = tp.x - xi, dy = tp.y - yi;
    const double d2 = dx * dx + dy * dy;
    const bool hit = d2 <= P.s_dp_le, cov = d2 <= P.s_dp_lt;
    if (MASKS) { B.obs_mask[mrow_t + t] = hit; B.cover_mask[mrow_t + t] = cov; }
    if (hit) {
      const double d = sqrt(d2);
      tt += 1 + (P.dp - d) / P.dp;  // uav.py:208
      const double2 tv = tvel[t];
      double rx = dx / P.dp, ry = dy / P.dp, vx = tv.x - chi, vy = tv.y - shi;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;  // uav.py:174-180
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; }
      o0 += rx; o1 += ry; o2 += vx; o3 += vy;
      nobs++;
      if (cov) atomicAdd(&tcnt[t], 1);
    }
  }
  double dup = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
  int ncomm = 0;
  uint32_t nb[4] = {0, 0, 0, 0};
  for (int j = 0; j < n; j++) {
    if (j == i) {
      if (MASKS) { B.comm_mask[mrow_u + j] = 0; B.nbr_mask[mrow_u + j] = 0; B.dup_mask[mrow_u + j] = 0; }
      continue;
    }
    const double2 np = npos[j];
    const double dxn = np.x - xi, dyn = np.y - yi;
    const double d2n = dxn * dxn + dyn * dyn;
    const bool hit_dup = d2n <= P.s_2dp_le, hit_nbr = d2n <= P.s_dp_le;
    if (hit_dup) { const double d = sqrt(d2n); dup += -0.5 * exp((P.two_dp - d) / P.two_dp); }  // uav.py:226
    if (hit_nbr) nb[j >> 5] |= 1u << (j & 31);
    double dxc, dyc, d2c;
    double2 hd;
    int aj;
    if (j < i) { dxc = dxn; dyc = dyn; d2c = d2n; hd = nhd[j]; aj = na_[j]; }
    else { const double2 op = opos[j]; dxc = op.x - xi; dyc = op.y - yi; d2c = dxc * dxc + dyc * dyc; hd = ohd[j]; aj = oa[j]; }
    const bool hit_c = d2c <= P.s_dc_le;
    if (MASKS) { B.comm_mask[mrow_u + j] = hit_c; B.nbr_mask[mrow_u + j] = hit_nbr; B.dup_mask[mrow_u + j] = hit_dup; }
    if (hit_c) {
      double rx = dxc / P.dc, ry = dyc / P.dc, vx = hd.x - chi, vy = hd.y - shi;
      double da = (double)(aj - ai) / (double)P.na;
      const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;
      if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; da /= w; }
      c0 += rx; c1 += ry; c2 += vx; c3 += vy; c4 += da;
      ncomm++;
    }
  }
  if (ncomm) {
    const double k = (double)ncomm;
    ob[0] = (float)(c0 / k); ob[1] = (float)(c1 / k); ob[2] = (float)(c2 / k); ob[3] = (float)(c3 / k); ob[4] = (float)(c4 / k);
  } else {
    ob[0] = ob[1] = ob[2] = ob[3] = ob[4] = -1.f;
  }
  if (nobs) {
    const double k = (double)nobs;
    ob[5] = (float)(o0 / k); ob[6] = (float)(o1 / k); ob[7] = (float)(o2 / k); ob[8] = (float)(o3 / k);
  } else {
    ob[5] = ob[6] = ob[7] = ob[8] = -1.f;
  }
  Op->tt = tt; Op->dup = dup;
  Op->nb[0] = nb[0]; Op->nb[1] = nb[1]; Op->nb[2] = nb[2]; Op->nb[3] = nb[3];
}

// ------------------------------------------------------------------------------------------------
// fast path
// ------------------------------------------------------------------------------------------------
struct CommAcc {
  double sx, sy, sc, ss;
  int sa, cnt;
};

__device__ __forceinline__ uint32_t low_bits(int len) { return len >= 32 ? 0xffffffffu : ((1u << len) - 1u); }

// (A) fp32 prefilter over one chunk of partner positions: candidate mask for a guarded squared threshold.
// Blackwell's packed fp32 pipe does two partners per instruction (sub/mul/fma.f32x2 -> FADD2 / FMUL2 / FFMA2, each
// half an ordinary IEEE fp32 operation, so the error bound behind the guard is unchanged); partners are stored two
// per float4 {x0, x1, y0, y1}.  `pf` points at the pair holding partner 0 of the chunk (chunks start on even
// indices); a trailing odd slot holds +huge and can never pass.  Code size matters (the kernel is
// instruction-fetch sensitive): UAVSIM_PF_UNROLL partners per loop trip with compile-time bits.
#ifndef UAVSIM_PF_UNROLL
#define UAVSIM_PF_UNROLL 16
#endif
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  return (uint64_t)__float_as_uint(lo) | ((uint64_t)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ uint32_t prefilter(const float4 *__restrict__ pf, int len, float xf, float yf, float thr) {
  constexpr int U = UAVSIM_PF_UNROLL;
  const uint64_t xf2 = pack2(xf, xf), yf2 = pack2(yf, yf), nthr2 = pack2(-thr, -thr);
  // t = dx*dx + (dy*dy - thr) as two packed FMAs: negative exactly when the pair is a candidate (the two roundings,
  // <= 2 ulp of thr, are inside the 3 ulp the guard of prefilter_threshold() reserves for the arithmetic, and the
  // guard is doubled on top).  The sign bit is shifted into the mask with one funnel shift per partner -- no compare,
  // no select; the first partner ends up in the highest bit, undone by one bit reversal per chunk.
  uint32_t mask = 0;
  auto pair_bits = [&](int k) {  // partners 2k, 2k+1 of the chunk
    const ulonglong2 p = reinterpret_cast<const ulonglong2 *>(pf)[k];  // {x0, x1}, {y0, y1}: one 128-bit load
    uint64_t dx, dy, t;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(dx) : "l"(p.x), "l"(xf2));
    asm("sub.f32x2 %0, %1, %2;" : "=l"(dy) : "l"(p.y), "l"(yf2));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(t) : "l"(dy), "l"(nthr2));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(t) : "l"(dx), "l"(t));
    mask = __funnelshift_l((uint32_t)t, mask, 1);
    mask = __funnelshift_l((uint32_t)(t >> 32), mask, 1);
  };
  int jj = 0;
#pragma unroll 1
  for (; jj + U <= len; jj += U) {
#pragma unroll
    for (int u = 0; u < U / 2; u++) pair_bits(jj / 2 + u);
  }
#pragma unroll 1
  for (; jj < len; jj += 2) pair_bits(jj / 2);
  // jj partners went through (len rounded up to even; the odd trailing slot holds +huge: t = +inf, bit 0)
  return jj ? (__brev(mask) >> (32 - jj)) & low_bits(len) : 0u;
}

// One chunk of up to 32 partner UAVs j = jb .. jb+len-1 for UAV i.  Partners with j < i moved before i: their
// new state serves the reward tests and communication; partners with j > i move after i: new-new distance for
// the rewards, new-old distance for communication (uav.py:124-147 with the update order of environment.py:133-138).
// Candidates: `cn` = evaluate j's NEW position exactly (needed up to dc if j moved first, else up to 2dp);
// `co` = evaluate j's OLD position exactly (j > i, communication range dc).  The old position is within dt*v of
// the new one, so co is prefiltered on the NEW position with the threshold dc + dt*v.
// One generic routine for every chunk (kept small on purpose).  Returns the neighbour bits (d <= dp).
template <bool MASKS>
__device__ __forceinline__ uint32_t pair_chunk(const KParams &P, const UavSimBuffers &B, const EnvView V, uint32_t sb, int jb, int len,
                                               int i, double xi, double yi, float xf, float yf, bool far_env,
                                               float k_ex0, float k_ex1, CommAcc &A, double &dup, int64_t mrow_u) {
  const int sj = i - jb;                                   // bits below sj moved before i, bits above move after
  const uint32_t lt = sj <= 0 ? 0u : low_bits(sj);
  const uint32_t self = (sj >= 0 && sj < 32) ? (1u << sj) : 0u;
  uint32_t cn, co;
  if (far_env) {
    cn = co = low_bits(len);
  } else {
    // ONE guarded threshold, max(dc + dt*v, 2 dp), for both lists: finer masks (exactly dc for moved partners, 2dp for the
    // reward-only evaluations) saved fewer exact evaluations than their extra compare + select cost on every pair
    cn = co = prefilter(V.nposf() + jb / 2, len, xf, yf, P.f_dcmv);
  }
  cn &= ~self;
  co &= ~(lt | self);
  if (MASKS)
    for (int jj = 0; jj < len; jj++) { B.comm_mask[mrow_u + jb + jj] = 0; B.nbr_mask[mrow_u + jb + jj] = 0; B.dup_mask[mrow_u + jb + jj] = 0; }

  // (B) exact fp64 evaluation of the candidates only.  Each lane walks its own bits (ascending j, like the
  // reference's loops); the warp runs max-over-lanes trips, so the two lists get two lean loops instead of one
  // fat one.  Sums over the two lists commute up to fp64 rounding of the (order-dependent) additions.
  const uint32_t a_npos = sb + V.L.npos, a_nhd = sb + V.L.nhd, a_opos = sb + V.L.opos, a_ohd = sb + V.L.ohd;
  const uint32_t a_na = sb + V.L.na_, a_oa = sb + V.L.oa;
  uint32_t nbits = 0;
#pragma unroll 1
  while (cn) {  // partner's NEW position: duplicate term, neighbour bit, and communication if it moved first
    const int jj = __ffs((int)cn) - 1;
    const uint32_t rest = cn & (cn - 1), bit = cn ^ rest;  // bit = 1 << jj without the shift
    cn = rest;
    const int j = jb + jj;
    const double2 np = lds_d2(a_npos + 16u * (uint32_t)j);
    const double dxn = np.x - xi, dyn = np.y - yi;
    const double d2n = dxn * dxn + dyn * dyn;
    const bool hd = d2n <= P.s_2dp_le;  // uav.py:225
    const bool hn = d2n <= P.s_dp_le;   // uav.py:305
    const bool hc = (bit & lt) && (d2n <= P.s_dc_le);  // uav.py:135, partner already at its new state (jj < sj)
    if (hd) dup += (double)fast_ex2f(fmaf(fast_sqrtf((float)d2n), k_ex1, k_ex0));  // exp((2dp - d)/(2dp))
    if (hn) nbits |= bit;
    if (hc) {
      const double2 h = lds_d2(a_nhd + 16u * (uint32_t)j);
      A.sx += dxn; A.sy += dyn; A.sc += h.x; A.ss += h.y; A.sa += lds_i32(a_na + 4u * (uint32_t)j); A.cnt++;
    }
    if (MASKS) { B.nbr_mask[mrow_u + j] = hn; B.dup_mask[mrow_u + j] = hd; if (hc) B.comm_mask[mrow_u + j] = 1; }
  }
#pragma unroll 1
  while (co) {  // partner's OLD position (it moves after i): communication only
    const int jj = __ffs((int)co) - 1;
    co &= co - 1;
    const int j = jb + jj;
    const double2 op = lds_d2(a_opos + 16u * (uint32_t)j);
    const double dxo = op.x - xi, dyo = op.y - yi;
    const double d2o = dxo * dxo + dyo * dyo;
    if (d2o <= P.s_dc_le) {
      const double2 h = lds_d2(a_ohd + 16u * (uint32_t)j);
      A.sx += dxo; A.sy += dyo; A.sc += h.x; A.ss += h.y; A.sa += lds_i32(a_oa + 4u * (uint32_t)j); A.cnt++;
      if (MASKS) B.comm_mask[mrow_u + j] = 1;
    }
  }
  return nbits;
}

template <int CN, int CM, bool WARP_ENV, bool MASKS>
__device__ __forceinline__ void agent_fast(const KParams &P, const UavSimBuffers &B, const EnvView V, uint32_t sb, int *tcnt, int i,
                                           int n_rt, int m_rt, bool far_env, float *ob, int64_t mrow_t, int64_t mrow_u,
                                           AgentOut &O) {
  const int n = CN ? CN : n_rt, m = CM ? CM : m_rt;
  const double2 me = V.npos()[i], mh = V.nhd()[i];
  const double xi = me.x, yi = me.y, chi = mh.x, shi = mh.y;
  const float2 mef = EnvView::get_pair(V.nposf(), i);
  const float xf = mef.x, yf = mef.y;

  // ---- targets: observe_target (uav.py:101-122), tracking reward (uav.py:199-212), coverage (environment.py:246-253)
  {
    const float inv_dp_f = (float)(1.0 / P.dp);
    double ox = 0, oy = 0, ovx = 0, ovy = 0, tt = 0;
    int nobs = 0;
    const uint32_t a_tpos = sb + V.L.tpos, a_tvel = sb + V.L.tvel;
#pragma unroll 1
    for (int tb = 0; tb < m; tb += 32) {
      const int len = min(32, m - tb);
      const uint32_t ct0 = far_env ? low_bits(len) : prefilter(V.tposf() + tb / 2, len, xf, yf, P.f_dp);
      uint32_t ct = ct0;
      if (MASKS)
        for (int jj = 0; jj < len; jj++) { B.obs_mask[mrow_t + tb + jj] = 0; B.cover_mask[mrow_t + tb + jj] = 0; }
#pragma unroll 1
      while (ct) {
        const int jj = __ffs((int)ct) - 1;
        ct &= ct - 1;
        const int t = tb + jj;
        const double2 tp = lds_d2(a_tpos + 16u * (uint32_t)t);
        const double dx = tp.x - xi, dy = tp.y - yi;
        const double d2 = dx * dx + dy * dy;
        const bool hit = d2 <= P.s_dp_le;
        if (MASKS) { B.obs_mask[mrow_t + t] = hit; B.cover_mask[mrow_t + t] = (d2 <= P.s_dp_lt); }
        if (hit) {
          const double2 tv = lds_d2(a_tvel + 16u * (uint32_t)t);
          ox += dx; oy += dy; ovx += tv.x; ovy += tv.y;
          nobs++;
          tt += (double)(2.0f - fast_sqrtf((float)d2) * inv_dp_f);  // 1 + (dp - d)/dp
          if (d2 <= P.s_dp_lt) atomicAdd(&tcnt[t], 1);
        }
      }
    }
    // observation part of the local state (uav.py:176-186; row weights are all 1 here), -1 block when empty
    if (nobs) {
      const double k = (double)nobs, rk = 1.0 / k, rs = rk * P.inv_dp;  // outputs are fp32: reciprocals are exact enough
      ob[5] = (float)(ox * rs);
      ob[6] = (float)(oy * rs);
      ob[7] = (float)((ovx - k * chi) * rk);
      ob[8] = (float)((ovy - k * shi) * rk);
    } else {
      ob[5] = ob[6] = ob[7] = ob[8] = -1.f;
    }
    O.tt = tt;
  }

  // ---- UAVs: observe_uav in the sequential update order (uav.py:124-147, environment.py:133-138),
  //      duplicate-tracking punishment (uav.py:214-229), neighbour set (uav.py:305)
  const float k_ex0 = 1.4426950408889634f, k_ex1 = (float)(-1.4426950408889634 / P.two_dp);
  CommAcc A = {0, 0, 0, 0, 0, 0};
  double dup = 0;
#pragma unroll 1
  for (int c = 0; c < 4; c++) {
    const int jb = 32 * c;
    uint32_t nbits = 0;
    if (jb < n) nbits = pair_chunk<MASKS>(P, B, V, sb, jb, min(32, n - jb), i, xi, yi, xf, yf, far_env, k_ex0, k_ex1, A, dup, mrow_u);
    O.nb[c] = nbits;
  }

  // ---- communication part of the local state (uav.py:162-172)
  if (A.cnt) {
    const double k = (double)A.cnt, rk = 1.0 / k, rs = rk * P.inv_dc;
    const int ai = V.na_()[i];
    ob[0] = (float)(A.sx * rs);
    ob[1] = (float)(A.sy * rs);
    ob[2] = (float)((A.sc - k * chi) * rk);
    ob[3] = (float)((A.ss - k * shi) * rk);
    ob[4] = (float)((double)(A.sa - A.cnt * ai) * P.inv_na * rk);
  } else {
    ob[0] = ob[1] = ob[2] = ob[3] = ob[4] = -1.f;
  }
  O.dup = -0.5 * dup;
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
#ifndef UAVSIM_WARPS_PER_SM
#define UAVSIM_WARPS_PER_SM 32   // 64 registers per thread: measured best of 16 / 20 / 24 / 32 resident warps per SM
#endif
template <int CN, int CM, bool MASKS, int NT>
__global__ void __launch_bounds__(NT, UAVSIM_WARPS_PER_SM * 32 / NT)
uavsim_step_kernel(const KParams P, const UavSimBuffers B, const double *__restrict__ g_dth, int64_t env_begin,
                   int64_t env_count, int epb_rt, int mode, double coop, int done_flag,
                   long long *__restrict__ stats) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = CN ? CN : P.n, m = CM ? CM : P.m;
  const int epb = CN ? NT / CN : epb_rt;  // environments per CTA: the host passes NT / n, a constant when n is
  constexpr bool WARP_ENV = (CN > 0) && (CN % 32 == 0);
  const EnvLayout L = (CN && CM) ? env_layout(CN, CM) : env_layout(n, m);
  const int tid = threadIdx.x;
  const CtaSmem S = carve(smem_raw, n, m, P.na, epb, L.stride);
  const int64_t plane = P.E * n;  // rew4 plane stride
  const uint32_t s_env0 = opaque_u32((uint32_t)__cvta_generic_to_shared(S.env));

  for (int k = tid; k < 3 * P.na; k += NT) S.dth[k] = g_dth[k];
  for (int k = tid; k < epb; k += NT) {  // odd trailing slots of the paired fp32 arrays: never a candidate
    const EnvView V0{S.env + (size_t)k * L.stride, L};
    if (m & 1) EnvView::put_pair(V0.tposf(), m, 3.0e18f, 3.0e18f);
    if (n & 1) EnvView::put_pair(V0.nposf(), n, 3.0e18f, 3.0e18f);
  }

  const int64_t ngroups = (env_count + epb - 1) / epb;
  // per-thread statistics, reduced once at the end (src/train.py:181-192)
  long long fx_r = 0, fx_tt = 0, fx_bp = 0, fx_dup = 0;
  long long st_cov = 0, st_envs = 0;
  int st_cmax = 0;

  // Groups beyond the first wave are handed out by a launch-wide counter, as in the fast kernel: the warp schedulers
  // favour some CTAs, and with a fixed stride the favoured ones retire early and leave their SM under-occupied.
  long long drawn = 0;
  if (tid == 0 && (int64_t)blockIdx.x < ngroups) drawn = (long long)gridDim.x + (long long)atomicAdd(P.fast_ctr, 1);
  for (int64_t grp = blockIdx.x, grp_next = 0; grp < ngroups; grp = grp_next) {
    const int64_t e0 = env_begin + grp * epb;
    const int ne = (int)min((int64_t)epb, env_begin + env_count - e0);
    if (tid < epb) { S.far[tid] = 0; S.cov[tid] = 0; }  // (their readers of the previous iteration have passed a barrier)
    if (tid == 0) *S.next = drawn;
    __syncthreads();                // previous iteration's readers are done; dth table visible
    grp_next = *S.next;
#ifdef GENERIC_STATIC_STRIDE   // A/B switch: the fixed stride of round 1
    grp_next = grp + gridDim.x;
#endif
    // (thread 0 draws one group ahead: the atomic's round trip is over by the time the next iteration asks for it)
    if (tid == 0 && grp_next < ngroups) drawn = (long long)gridDim.x + (long long)atomicAdd(P.fast_ctr, 1);
    if (!WARP_ENV) {
      // Small-swarm instances are bound by global-load latency, not by issue slots (10x10: long-scoreboard stalls
      // dominate): pull the state of this CTA's NEXT group of environments into L2 while this one is computed, one
      // prefetch per 128-byte line.  (The 64x64 instance is issue-bound; there the extra instructions cost more than
      // the latency they hide.)
      const int64_t grp_n = grp_next;
      if (grp_n < ngroups) {
        const int64_t e0n = env_begin + grp_n * epb;
        const int nen = (int)min((int64_t)epb, env_begin + env_count - e0n);  // the last group may be partial: stay inside the arrays
        auto pf = [](const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); };
        for (int q = tid * 16; q < nen * n; q += NT * 16) { pf(B.ux + e0n * n + q); pf(B.uy + e0n * n + q); pf(B.uh + e0n * n + q); }
        for (int q = tid * 32; q < nen * n; q += NT * 32) { pf(B.ua + e0n * n + q); pf(B.actions + e0n * n + q); }
        for (int q = tid * 16; q < nen * m; q += NT * 16) { pf(B.tx + e0n * m + q); pf(B.ty + e0n * m + q); pf(B.th + e0n * m + q); }
      }
    }

    // ---- phase 0a: targets (src/agent/target.py:27-60) ----
    for (int q = tid; q < ne * m; q += NT) {
      const int64_t gi = e0 * m + q;
      const int te = q / m, t = q - te * m;
      const EnvView V{S.env + (size_t)te * L.stride, L};
      double x = B.tx[gi], y = B.ty[gi], h = B.th[gi];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);  // (< 1 ulp table routine; the library call took 83 instructions per heading)
      x += P.dtv_t * ch;
      y += P.dtv_t * sh;
      // reflection (target.py:52-58); cos/sin of the reflected heading follow from the identities
      // cos(-h) = cos h, sin(-h) = -sin h, cos(+-pi - h) = -cos h, sin(+-pi - h) = sin h (they feed the observation only)
      if (0 > y || y > P.y_max) {
        h = -h; sh = -sh; B.th[gi] = h;
      } else if (x < 0 || x > P.x_max) {
        h = (h > 0) ? (PI_D - h) : (-PI_D - h); ch = -ch; B.th[gi] = h;
      }
      B.tx[gi] = x; B.ty[gi] = y;
      V.tpos()[t] = make_double2(x, y);
      // cos(target.h) * target.v_max / self.v_max  (src/agent/uav.py:115-116)
      V.tvel()[t] = make_double2(ch * P.tv_over_uv, sh * P.tv_over_uv);  // fp32 outputs: the ratio is exact enough
      EnvView::put_pair(V.tposf(), t, (float)(x - P.cx), (float)(y - P.cy));
      if (!(fabs(x - P.cx) <= P.rmax && fabs(y - P.cy) <= P.rmax)) S.far[te] = 1;
      S.tcnt[q] = 0;
    }
    // ---- phase 0b: UAV kinematics (src/agent/uav.py:73-99) ----
    const int q = tid;
    const bool active = q < ne * n;
    const int el = active ? q / n : 0, i = q - el * n;
    const int64_t ge = e0 + el, gi = e0 * n + q;
    const EnvView V{S.env + (size_t)el * L.stride, L};
    if (active) {
      double x = B.ux[gi], y = B.uy[gi], h = B.uh[gi];
      const int a_old = B.ua[gi], act = B.actions[gi];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);
      V.opos()[i] = make_double2(x, y); V.ohd()[i] = make_double2(ch, sh); V.oa()[i] = a_old;
      x += P.dtv_u * ch;
      y += P.dtv_u * sh;
      // cos/sin of the new heading by angle addition (|error| ~ 3e-16; they only feed the observation).
      // The next step re-evaluates sincos from the stored heading, so the trajectory is unaffected.
      double dh, cd, sd;
      if ((unsigned)act < (unsigned)P.na) {
        dh = S.dth[3 * act]; cd = S.dth[3 * act + 1]; sd = S.dth[3 * act + 2];
      } else {  // the reference's formula accepts any integer (uav.py:73-81); off-table actions take it literally
        dh = P.dt * ((double)(2 * (act + 1) - P.na - 1) * P.uav_h_max / (double)(P.na - 1));
        sincos_shared(dh, &sd, &cd);
      }
      h += dh;
      h = wrap_heading(h);
      V.npos()[i] = make_double2(x, y);
      V.nhd()[i] = make_double2(ch * cd - sh * sd, sh * cd + ch * sd);
      V.na_()[i] = act;
      EnvView::put_pair(V.nposf(), i, (float)(x - P.cx), (float)(y - P.cy));
      // the prefilter's error bound assumes every entity within rmax of the map centre
      if (!(fabs(x - P.cx) <= P.rmax && fabs(y - P.cy) <= P.rmax)) S.far[el] = 1;
      B.ux[gi] = x; B.uy[gi] = y; B.uh[gi] = h; B.ua[gi] = act;
    }
    __syncthreads();

    // ---- phase 1: all-pairs tests, observation, raw reward ----
    AgentOut O;
    O.tt = 0; O.dup = 0; O.nb[0] = O.nb[1] = O.nb[2] = O.nb[3] = 0;
    double raw = 0, ttn = 0, bpn = 0, dupn = 0;
    if (active) {
      const double2 me = V.npos()[i];
      const double xi = me.x, yi = me.y;
      const int ai = V.na_()[i];
      float *ob = S.obs + (size_t)q * 12;
      const int64_t mrow_t = (ge * n + i) * m, mrow_u = (ge * n + i) * n;
      // row weights differ from 1 only if |x| < 2 and |y| < 2 (|rx|,|ry| <= 1 for any row in range)
      const bool near_origin = fabs(xi) < 2.0 && fabs(yi) < 2.0;
      if (near_origin) agent_exact<MASKS>(P, B, V, S.tcnt + el * m, i, n, m, ob, mrow_t, mrow_u, &O);
      else agent_fast<CN, CM, WARP_ENV, MASKS>(P, B, V, s_env0 + (uint32_t)el * (uint32_t)L.stride, S.tcnt + el * m, i, n, m, S.far[el] != 0, ob, mrow_t, mrow_u, O);
      if (MASKS) { B.comm_mask[mrow_u + i] = 0; B.nbr_mask[mrow_u + i] = 0; B.dup_mask[mrow_u + i] = 0; }
      ob[9] = (float)(xi * P.inv_dc);
      ob[10] = (float)(yi * P.inv_dc);
      ob[11] = (float)((double)ai * P.inv_na);

      // boundary punishment (uav.py:231-250)
      const double dbdr = fmin(fmin(xi - 0, P.x_max - xi), fmin(yi - 0, P.y_max - yi));
      double bp;
      if (0 <= xi && xi <= P.x_max && 0 <= yi && yi <= P.y_max)
        bp = (dbdr < P.dp) ? (-0.5 * (P.dp - dbdr) * P.inv_dp) : 0.0;
      else
        bp = -0.5;
      // normalise + weights (environment.py:206-220)
      ttn = fmin(fmax(O.tt, 0.0), P.tt_hi) * P.inv_tt_hi;                      // choice 0: (v - 0)/(2m - 0)
      dupn = (fmin(fmax(O.dup, P.dup_lo), 0.0) - P.dup_lo) * P.inv_dup_span - 1.0;  // choice -1: (v - lo)/(0 - lo) - 1
      bpn = (fmin(fmax(bp, -0.5), 0.0) + 0.5) * 2.0 - 1.0;
      raw = P.alpha * ttn + P.beta * bpn + P.gamma * dupn;
      S.raw[q] = raw;
    }
    __syncthreads();

    // ---- phase 2: cooperative reward (environment.py:222-227), coverage, outputs ----
    if (active) {
      double r;
      const bool pmi_pending = (mode == UAVSIM_MODE_PMI) && (coop != 0.0);
      if (mode == UAVSIM_MODE_SELF || coop == 0.0) {
        r = raw;  // uav.py:271-272 / :300-301
      } else if (mode == UAVSIM_MODE_MEAN) {
        // uav.py:293-310 -- the conditional expression covers the whole sum: no neighbour -> 0
        const double *R = S.raw + el * n;
        double s = 0;
        int cnt = 0;
#pragma unroll
        for (int c = 0; c < 4; c++) {
          uint32_t w = O.nb[c];
          while (w) { const int j = __ffs((int)w) - 1; w &= w - 1; s += R[32 * c + j]; cnt++; }
        }
        r = cnt ? ((1 - coop) * raw + coop * s / (double)cnt) : 0.0;
      } else {
        r = 0.0;  // finished by uavsim_pmi_kernel
        B.raw[gi] = raw;
        B.nbr_bits[gi * 2] = (uint64_t)O.nb[0] | ((uint64_t)O.nb[1] << 32);
        B.nbr_bits[gi * 2 + 1] = (uint64_t)O.nb[2] | ((uint64_t)O.nb[3] << 32);
      }
      r = fmin(fmax(r, -1.0), 1.0);  // clip_and_normalize(reward, -1, 1) is a plain clip
      if (!pmi_pending) { B.rew4[gi] = (float)r; fx_r += sf_fx((float)r); }
      B.rew4[plane + gi] = (float)ttn;
      B.rew4[2 * plane + gi] = (float)bpn;
      B.rew4[3 * plane + gi] = (float)dupn;
      fx_tt += sf_fx((float)ttn); fx_bp += sf_fx((float)bpn); fx_dup += sf_fx((float)dupn);
    }
    // environment.py:246-253: targets with at least one UAV strictly within dp, counted cooperatively
    for (int k = tid; k < ne * m; k += NT) {
      const int c = S.tcnt[k];
      if (c > 0) atomicAdd(&S.cov[k / m], 1);
      if (B.tracker_cnt) B.tracker_cnt[e0 * m + k] = c;
    }
    {  // coalesced observation write: ne*n*12 floats = ne*n*3 float4, contiguous in global memory
      const float4 *src = reinterpret_cast<const float4 *>(S.obs);
      float4 *dst = reinterpret_cast<float4 *>(B.obs + e0 * n * 12);
      for (int k = tid; k < ne * n * 3; k += NT) dst[k] = src[k];
    }
    __syncthreads();
    if (tid < ne) {
      const int c = S.cov[tid];
      B.covered[e0 + tid] = c;
      if (B.done) B.done[e0 + tid] = done_flag;
      st_cov += c;
      st_cmax = max(st_cmax, c);
      st_envs++;
    }
  }
  work_counter_leave(P.fast_ctr);
  stats_commit(stats + (size_t)blockIdx.x * STAT_W, fx_r, fx_tt, fx_bp, fx_dup, st_cov, st_cmax, st_envs);
}
