// step_small_kernel.cuh -- the fused environment step for SMALL swarms (n_uav <= 16, m_targets <= 16; the shipped
// scenario is 10 x 10): Environment.step, src/environment.py:120-164, in two-warp CTAs.
//
// Why a separate kernel.  With one thread per UAV and a few thousand environments (BASELINE configs[1]: 4 096
// environments of 10 x 10) the generic kernel is a single partial wave whose duration is the dependency chain of one
// thread -- ~1 950 instructions at ~18 cycles each, 17 us -- whatever the batch size.  Here a CTA of 64 threads takes a
// group of G = min(32 / n, 32 / m, 8) environments and the chain is cut in two:
//   * warp 0, lane (g, i): UAV i of environment g -- kinematics, then its UAV partners (communication, duplicate
//     tracking, neighbours), then everything that finishes the UAV;
//   * warp 1, lane (g, j): target j of environment g -- motion and reflection; then, as lane (g, i), the TARGETS of UAV i
//     (observation part, tracking reward, coverage), handed to warp 0 through shared memory.
// Both warps keep their lanes dense (30 of 32 at 10 x 10).  No prefilter (with <= 16 partners the exact fp64 test of
// every pair is cheaper than selecting candidates), no per-thread copy of the parameter block, table sine / cosine.
// (A first version with one environment per warp kept 11 lanes of 32 busy: three times the warp instructions, no
// faster than the generic kernel.)
// Every range decision is the reference's: d2 = dx*dx + dy*dy in fp64 (no contraction) against the exact squared
// thresholds; sums are fp64, transcendental reward terms fp32 (they feed fp32 outputs), the min(dist, 1) row weights of
// src/agent/uav.py:162-186 are applied hit by hit for a UAV inside the 4 m x 4 m origin corner.
#pragma once
#include "step_fast_kernel.cuh"

#define SMALL_NT 64           // warp 0: UAV lanes, warp 1: target lanes
#define SMALL_MAX 16          // UAVs / targets per environment
#define SMALL_G 8             // environments per CTA iteration at most
#ifndef SMALL_CTAS_PER_SM
#define SMALL_CTAS_PER_SM 12
#endif

struct __align__(16) SmallRec {   // one UAV, after or before its move
  double x, y;
  float c, s;                     // cos / sin of the heading
  int a, pad;                     // action index
};
struct __align__(16) SmallTgt {
  double x, y;
  float vx, vy;                   // (cos h, sin h) * tv / uv  (src/agent/uav.py:115-116)
  float pad0, pad1;
};
struct __align__(16) SmallHand {  // what the target walk of one UAV hands to the lane that finishes the UAV
  float tb0, tb1, tb2, tb3;       // observation part of the local state
  float tt, pad0, pad1, pad2;     // raw tracking reward
};
struct SmallEnv {
  SmallRec un[SMALL_MAX], uo[SMALL_MAX];
  SmallTgt tg[SMALL_MAX];
};
struct SmallSmem {
  SmallEnv env[SMALL_G];
  SmallHand hand[32];
  double raw[32];
  uint32_t cov[SMALL_G];
  int32_t tcnt[SMALL_G][SMALL_MAX];
};

__host__ __device__ inline int small_group(int n, int m) {
  int g = 32 / (n > m ? n : m);
  return g > SMALL_G ? SMALL_G : g;
}

template <bool AUX>
__global__ void __launch_bounds__(SMALL_NT, SMALL_CTAS_PER_SM)
uavsim_step_small_kernel(const KParams P, const UavSimBuffers B, const ActEntry *__restrict__ act_tab, int64_t env_begin,
                         int64_t env_count, int mode, double coop, int done_flag, long long *__restrict__ stats,
                         int rng_on, uint64_t rng_seed, uint32_t rng_step) {
  __shared__ SmallSmem S;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = P.n, m = P.m, G = small_group(n, m);
  const int64_t ngroups = (env_count + G - 1) / G;
  const int64_t plane = P.E * n;
  const bool pmi_pending = (mode == UAVSIM_MODE_PMI) && (coop != 0.0);
  const bool mean_mode = (mode == UAVSIM_MODE_MEAN) && (coop != 0.0);
  const bool aux_on = AUX && (B.obs_mask != nullptr);
  // (environment of the group, UAV) of this lane, and (environment, target) in warp 1's phase 0.  lane < 32 and n, m <= 16:
  // the quotient through one fp32 multiplication is exact
  const int gu = (int)(((float)lane + 0.5f) * __frcp_rn((float)n)), iu = lane - gu * n;
  const int gt = (int)(((float)lane + 0.5f) * __frcp_rn((float)m)), jt = lane - gt * m;
  const float k_ex0 = 1.4426950408889634f, k_ex1 = P.k_ex1_f;
  long long fx_r = 0, fx_tt = 0, fx_bp = 0, fx_dup = 0, st_cov = 0, st_envs = 0;  // statistics (common.cuh: sf_fx)
  int st_cmax = 0;
  // Programmatic dependent launch: when the steps of a rollout are queued back to back (uavsim_run_random_policy) this
  // grid may start while its predecessor drains -- everything above (parameters, lane roles) overlaps the predecessor's
  // tail; nothing below touches global memory before the predecessor has completed.  A plain launch passes straight through.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  for (int64_t grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int64_t e0 = env_begin + grp * G;
    const int ne = (int)min((int64_t)G, env_begin + env_count - e0);  // the last group may be partial
    const bool uav_lane = gu < ne;     // warp 0: moves and finishes UAV (gu, iu); warp 1: walks its targets
    const int64_t e = e0 + gu, gi = e * n + iu;
    __syncthreads();  // the previous group's records, hand-over and counts are no longer read
    if (threadIdx.x < SMALL_G) S.cov[threadIdx.x] = 0;   // (first touched again after the next barrier)
    if (B.tracker_cnt && threadIdx.x < SMALL_G * 2) {
#pragma unroll
      for (int q = 0; q < SMALL_MAX / 2; q++) S.tcnt[threadIdx.x >> 1][(threadIdx.x & 1) * (SMALL_MAX / 2) + q] = 0;
    }

    // ---- phase 0: UAV kinematics (src/agent/uav.py:73-99) | target motion (src/agent/target.py:27-60) ----
    if (warp == 0) {
      if (uav_lane) {
        double x = B.ux[gi], y = B.uy[gi], h = B.uh[gi];
        const int a_old = B.ua[gi];
        int act;
        if (rng_on) {  // random policy drawn in place (the draw of uavsim_random_actions_kernel, aux_kernels.cuh)
          const Philox4 rr = philox4x32_10((uint32_t)iu, UAVSIM_RNG_ACTION, (uint32_t)(P.env_id_offset + e), rng_step, rng_seed);
          act = (int)philox_below(rr.v[0], (uint32_t)P.na);
          B.actions[gi] = act;
        } else {
          act = B.actions[gi];
        }
        double sh, ch;
        heading_sincos(h, P.sincos_tab, sh, ch);
        const float cof = (float)ch, sof = (float)sh;
        S.env[gu].uo[iu] = SmallRec{x, y, cof, sof, a_old, 0};
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
        // cos / sin of the new heading by angle addition: they only feed the observation
        S.env[gu].un[iu] = SmallRec{x, y, fmaf(cof, cd, -(sof * sd)), fmaf(sof, cd, cof * sd), act, 0};
        B.ux[gi] = x; B.uy[gi] = y; B.uh[gi] = h; B.ua[gi] = act;
      }
    } else if (gt < ne) {
      const int64_t gq = (e0 + gt) * m + jt;
      double x = B.tx[gq], y = B.ty[gq], h = B.th[gq];
      double sh, ch;
      heading_sincos(h, P.sincos_tab, sh, ch);
      x += P.dtv_t * ch;
      y += P.dtv_t * sh;
      // reflection (target.py:52-58); cos(-h) = cos h, sin(-h) = -sin h, cos(+-pi - h) = -cos h, sin(+-pi - h) = sin h
      if (0 > y || y > P.y_max) { h = -h; sh = -sh; B.th[gq] = h; }
      else if (x < 0 || x > P.x_max) { h = (h > 0) ? (PI_D - h) : (-PI_D - h); ch = -ch; B.th[gq] = h; }
      B.tx[gq] = x; B.ty[gq] = y;
      S.env[gt].tg[jt] = SmallTgt{x, y, (float)ch * P.tv_over_uv_f, (float)sh * P.tv_over_uv_f, 0.f, 0.f};
    }
    __syncthreads();

    // ---- phase 1: warp 0: the UAV partners of UAV (gu, iu); warp 1: its targets ----
    float ob0 = -1.f, ob1 = -1.f, ob2 = -1.f, ob3 = -1.f, ob4 = -1.f;      // communication part of the local state
    float dup_f = 0.f;
    uint32_t nb = 0;
    double xi = 0, yi = 0;
    int ai = 0;
    if (uav_lane) {
      const SmallEnv &V = S.env[gu];
      const int i = iu;
      const SmallRec me = V.un[i];
      xi = me.x; yi = me.y; ai = me.a;
      const double chi = (double)me.c, shi = (double)me.s;
      // the only place a row weight (uav.py:162-186) differs from 1
      const bool near_origin = fabs(xi) < 2.0 && fabs(yi) < 2.0;
      if (warp == 0) {
        // observe_uav in the sequential update order (uav.py:124-147, environment.py:133-138): partner j < i at its new
        // state, j > i at its old state; duplicate-tracking punishment (uav.py:214-229) and the neighbour set
        // (uav.py:305) at the new positions
        const int64_t mrow_u = (e * n + i) * n;
        double sx = 0, sy = 0, sc = 0, ss = 0, sa = 0, dup = 0;
        int cnt = 0;
#pragma unroll 1
        for (int j = 0; j < n; j++) {
          if (j == i) {
            if (AUX && aux_on) { B.comm_mask[mrow_u + j] = 0; B.nbr_mask[mrow_u + j] = 0; B.dup_mask[mrow_u + j] = 0; }
            continue;
          }
          const SmallRec nj = V.un[j];
          const double dxn = nj.x - xi, dyn = nj.y - yi;
          const double d2n = dxn * dxn + dyn * dyn;
          const bool hd = d2n <= P.s_2dp_le, hn = d2n <= P.s_dp_le;
          if (hd) dup += (double)fast_ex2f(fmaf(fast_sqrtf((float)d2n), k_ex1, k_ex0));  // exp((2dp - d)/(2dp)), uav.py:226
          if (hn) nb |= 1u << j;
          double dxc = dxn, dyc = dyn, d2c = d2n;
          float cj = nj.c, sj = nj.s;
          int aj = nj.a;
          if (j > i) {
            const SmallRec oj = V.uo[j];
            dxc = oj.x - xi; dyc = oj.y - yi; d2c = dxc * dxc + dyc * dyc;
            cj = oj.c; sj = oj.s; aj = oj.a;
          }
          const bool hc = d2c <= P.s_dc_le;
          if (AUX && aux_on) { B.comm_mask[mrow_u + j] = hc; B.nbr_mask[mrow_u + j] = hn; B.dup_mask[mrow_u + j] = hd; }
          if (hc) {
            if (!near_origin) {  // row weights are 1: linear sums, scaled once
              sx += dxc; sy += dyc; sc += (double)cj; ss += (double)sj; sa += (double)aj;
            } else {             // uav.py:162-172 row by row
              double rx = dxc / P.dc, ry = dyc / P.dc, vx = (double)cj - chi, vy = (double)sj - shi;
              double da = ((double)aj - (double)ai) / (double)P.na;
              const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;
              if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; da /= w; }
              sx += rx; sy += ry; sc += vx; ss += vy; sa += da;
            }
            cnt++;
          }
        }
        if (cnt) {
          const double kq = (double)cnt, rk = 1.0 / kq;
          if (!near_origin) {
            const double rs = rk * P.inv_dc;  // outputs are fp32: reciprocals are exact enough
            ob0 = (float)(sx * rs); ob1 = (float)(sy * rs);
            ob2 = (float)((sc - kq * chi) * rk); ob3 = (float)((ss - kq * shi) * rk);
            ob4 = (float)((sa - kq * (double)ai) * P.inv_na * rk);
          } else {
            ob0 = (float)(sx / kq); ob1 = (float)(sy / kq); ob2 = (float)(sc / kq); ob3 = (float)(ss / kq); ob4 = (float)(sa / kq);
          }
        }
        dup_f = (float)(-0.5 * dup);
      } else {
        // observe_target (uav.py:101-122), tracking reward (uav.py:199-212), coverage (environment.py:246-253)
        float tb0 = -1.f, tb1 = -1.f, tb2 = -1.f, tb3 = -1.f;
        uint32_t cov = 0;
        const int64_t mrow_t = (e * n + i) * m;
        double ox = 0, oy = 0, ovx = 0, ovy = 0, tt = 0;
        int nobs = 0;
#pragma unroll 1
        for (int t = 0; t < m; t++) {
          const SmallTgt tp = V.tg[t];
          const double dx = tp.x - xi, dy = tp.y - yi;
          const double d2 = dx * dx + dy * dy;
          const bool hit = d2 <= P.s_dp_le, cv = d2 <= P.s_dp_lt;
          if (AUX && aux_on) { B.obs_mask[mrow_t + t] = hit; B.cover_mask[mrow_t + t] = cv; }
          if (cv) cov |= 1u << t;
          if (hit) {
            tt += (double)(2.0f - fast_sqrtf((float)d2) * P.inv_dp_f);  // 1 + (dp - d)/dp, uav.py:208
            if (!near_origin) {
              ox += dx; oy += dy; ovx += (double)tp.vx; ovy += (double)tp.vy;
            } else {  // uav.py:174-186 row by row
              double rx = dx / P.dp, ry = dy / P.dp, vx = (double)tp.vx - chi, vy = (double)tp.vy - shi;
              const double wx = rx - xi, wy = ry - yi, w2 = wx * wx + wy * wy;
              if (w2 < 1.0) { const double w = sqrt(w2); rx /= w; ry /= w; vx /= w; vy /= w; }
              ox += rx; oy += ry; ovx += vx; ovy += vy;
            }
            nobs++;
          }
        }
        if (nobs) {
          const double kq = (double)nobs, rk = 1.0 / kq;
          if (!near_origin) {
            const double rs = rk * P.inv_dp;
            tb0 = (float)(ox * rs); tb1 = (float)(oy * rs);
            tb2 = (float)((ovx - kq * chi) * rk); tb3 = (float)((ovy - kq * shi) * rk);
          } else {
            tb0 = (float)(ox / kq); tb1 = (float)(oy / kq); tb2 = (float)(ovx / kq); tb3 = (float)(ovy / kq);
          }
        }
        S.hand[lane] = SmallHand{tb0, tb1, tb2, tb3, (float)tt, 0.f, 0.f, 0.f};
        if (cov) atomicOr(&S.cov[gu], cov);
        if (B.tracker_cnt) {
          uint32_t w = cov;
          while (w) { const int t = __ffs((int)w) - 1; w &= w - 1; atomicAdd(&S.tcnt[gu][t], 1); }
        }
      }
    }
    __syncthreads();  // the target halves are handed over; coverage sets complete

    if (warp == 0) {
      // ---- boundary punishment (uav.py:231-250), normalisation and weights (environment.py:206-220) ----
      double raw = 0, ttn = 0, bpn = 0, dupn = 0;
      SmallHand H = SmallHand{-1.f, -1.f, -1.f, -1.f, 0.f, 0.f, 0.f, 0.f};
      if (uav_lane) {
        H = S.hand[lane];
        const double dbdr = fmin(fmin(xi - 0, P.x_max - xi), fmin(yi - 0, P.y_max - yi));
        double bp;
        if (0 <= xi && xi <= P.x_max && 0 <= yi && yi <= P.y_max) bp = (dbdr < P.dp) ? (-0.5 * (P.dp - dbdr) * P.inv_dp) : 0.0;
        else bp = -0.5;
        ttn = fmin(fmax((double)H.tt, 0.0), P.tt_hi) * P.inv_tt_hi;
        dupn = (fmin(fmax((double)dup_f, P.dup_lo), 0.0) - P.dup_lo) * P.inv_dup_span - 1.0;
        bpn = (fmin(fmax(bp, -0.5), 0.0) + 0.5) * 2.0 - 1.0;
        raw = P.alpha * ttn + P.beta * bpn + P.gamma * dupn;
      }
      // ---- cooperative reward (environment.py:222-227) ----
      double r = raw;  // uav.py:271-272 / :300-301
      if (mean_mode) {
        // uav.py:293-310 -- the conditional expression covers the whole sum: no neighbour -> 0
        S.raw[lane] = raw;
        __syncwarp();
        double s_ = 0;
        uint32_t w = nb;
        while (w) { const int j = __ffs((int)w) - 1; w &= w - 1; s_ += S.raw[gu * n + j]; }
        const int cnt = __popc(nb);
        r = cnt ? ((1 - coop) * raw + coop * s_ / (double)cnt) : 0.0;
      }
      if (uav_lane) {
        if (pmi_pending) {
          r = 0.0;  // finished by the PMI kernel
          B.raw[gi] = raw;
          B.nbr_bits[gi * 2] = (uint64_t)nb;
          B.nbr_bits[gi * 2 + 1] = 0;
        }
        r = fmin(fmax(r, -1.0), 1.0);  // clip_and_normalize(reward, -1, 1) is a plain clip
        if (!pmi_pending) { B.rew4[gi] = (float)r; fx_r += sf_fx((float)r); }
        B.rew4[plane + gi] = (float)ttn;
        B.rew4[2 * plane + gi] = (float)bpn;
        B.rew4[3 * plane + gi] = (float)dupn;
        fx_tt += sf_fx((float)ttn); fx_bp += sf_fx((float)bpn); fx_dup += sf_fx((float)dupn);
        float4 *ob = reinterpret_cast<float4 *>(B.obs + gi * 12);
        ob[0] = make_float4(ob0, ob1, ob2, ob3);
        ob[1] = make_float4(ob4, H.tb0, H.tb1, H.tb2);
        ob[2] = make_float4(H.tb3, (float)(xi * P.inv_dc), (float)(yi * P.inv_dc), (float)((double)ai * P.inv_na));
      }
      if (lane < ne) {  // one lane per environment: targets with a UAV strictly inside dp (environment.py:246-253)
        const int c = __popc(S.cov[lane]);
        B.covered[e0 + lane] = c;
        if (B.done) B.done[e0 + lane] = done_flag;
        st_cov += c;
        st_cmax = max(st_cmax, c);
        st_envs++;
      }
    } else if (B.tracker_cnt && gt < ne) {
      B.tracker_cnt[(e0 + gt) * m + jt] = S.tcnt[gt][jt];
    }
  }
  // warp 0 holds all statistics of the CTA
  if (warp == 0) stats_commit(stats + (size_t)blockIdx.x * STAT_W, fx_r, fx_tt, fx_bp, fx_dup, st_cov, st_cmax, st_envs);
}
