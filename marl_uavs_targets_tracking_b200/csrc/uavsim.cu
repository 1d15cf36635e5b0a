// uavsim.cu -- libuavsim.so: batched UAV/target tracking environment for B200 (sm_100a).
//
// One fused step kernel per block of environments: target motion, UAV kinematics, the all-pairs
// UAV-target / UAV-UAV range tests (positions staged in shared memory), the 12-d weighted-mean
// observation, the three reward terms, the cooperative reward and the coverage count.
// Semantics follow the reference's Environment.step (src/environment.py:120-164) and the UAV/TARGET
// classes (src/agent/uav.py, src/agent/target.py); each section cites the lines it implements.
//
// Numerics: state, distances and every range test are fp64 (the masks must equal the reference's,
// SURVEY.md section 7), compiled with -fmad=false so the parity-critical expressions keep the
// reference's evaluation order.  Range tests compare squared distances against the exact squared
// threshold computed on the host (largest double s with sqrt(s) <= thr), and take sqrt only on hits.
#include <cfloat>
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "step_kernel.cuh"
#include "pmi_kernel.cuh"
#include "pmi_tc_kernel.cuh"
#include "step_fast_kernel.cuh"
#include "step_tile_kernel.cuh"
#include "step_small_kernel.cuh"
#include "aux_kernels.cuh"
#include "replay.cuh"

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// largest double s with sqrt(s) <= thr (strict = false) or sqrt(s) < thr (strict = true); host sqrt and
// device sqrt are both correctly rounded, so `d2 <= s` reproduces `sqrt(d2) <= thr` / `< thr` exactly.
static double exact_sq_threshold(double thr, bool strict) {
  double s = thr * thr;
  auto ok = [&](double v) { double r = sqrt(v); return strict ? (r < thr) : (r <= thr); };
  while (!ok(s)) s = nextafter(s, -INFINITY);
  while (ok(nextafter(s, INFINITY))) s = nextafter(s, INFINITY);
  return s;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is per function and device, not per handle: several handles
// with different shapes may coexist, so only ever raise it.
static int raise_dynamic_smem(const void *fn, int device, size_t bytes) {
  static struct { const void *fn; int device; size_t bytes; } seen[256];
  static int nseen = 0;
  static std::mutex mu;  // handles may be created from several threads
  std::lock_guard<std::mutex> lock(mu);
  int slot = -1;
  for (int k = 0; k < nseen; k++) if (seen[k].fn == fn && seen[k].device == device) slot = k;
  if (slot < 0 && nseen < 256) { slot = nseen++; seen[slot].fn = fn; seen[slot].device = device; seen[slot].bytes = 0; }
  if (slot >= 0 && bytes <= seen[slot].bytes) return 0;
  CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  if (slot >= 0) seen[slot].bytes = bytes;
  return 0;
}

// Guarded fp32 squared threshold for the prefilter.  With coordinates c = fp32(x - centre), |x - centre| <= rmax:
//   coordinate rounding  e_c <= rmax * 2^-24
//   difference           |dx_f - dx| <= 2 e_c + |dx| 2^-24              =: e_d   (for |dx| <= thr)
//   squared distance     |d2_f - d2| <= 2 sqrt(2) thr e_d + 2 e_d^2 + 3 * 2^-24 * thr^2   (products, fma, sum)
// A pair with d2 <= thr^2 therefore has d2_f <= thr^2 + that bound; twice the bound is used, rounded up to fp32.
static float prefilter_threshold(double thr, double rmax) {
  const double u = 1.0 / 16777216.0;
  const double e_c = rmax * u, e_d = 2 * e_c + thr * u;
  const double bound = 2 * 1.4142135623730951 * thr * e_d + 2 * e_d * e_d + 3 * u * thr * thr;
  const double v = thr * thr * (1.0 + 1e-12) + 2 * bound + 1e-6;
  float f = (float)v;
  if ((double)f < v) f = nextafterf(f, INFINITY);
  return nextafterf(f, INFINITY);
}

// Two-sided fp32 guard of the fast step kernel for one radius (same error model as prefilter_threshold, as a
// function of R = largest |coordinate - centre| of an environment):
//   bound(R) = 2 sqrt(2) thr u (2R + thr) + 2 u^2 (2R + thr)^2 + 3 u thr^2,  u = 2^-24
// The kernel evaluates g = c1 R + c0 in fp32 and uses thr^2 rounded up + g / thr^2 rounded down - g; c1 and c0 carry
// twice the bound (as the prefilter always has), the quadratic term at R = rmax, and room for their own rounding.
static GuardK make_guard(double thr, double rmax) {
  const double u = 1.0 / 16777216.0, r2 = 1.4142135623730951;
  const double t2 = thr * thr;
  GuardK g;
  g.t2_up = (float)t2;
  if ((double)g.t2_up < t2) g.t2_up = nextafterf(g.t2_up, INFINITY);
  g.t2_dn = (float)t2;
  if ((double)g.t2_dn > t2) g.t2_dn = nextafterf(g.t2_dn, -INFINITY);
  const double c1 = 4 * r2 * thr * u;
  const double c0 = 2 * r2 * u * t2 + 3 * u * t2 + 2 * u * u * (2 * rmax + thr) * (2 * rmax + thr);
  const double ulp_t2 = (double)nextafterf((float)t2, INFINITY) - (double)(float)t2;
  auto up = [](double v) { float f = (float)v; if ((double)f < v) f = nextafterf(f, INFINITY); return nextafterf(f, INFINITY); };
  g.c1 = up(2 * c1 * (1 + 1e-6));
  g.c0 = up(2 * c0 * (1 + 1e-6) + 4 * ulp_t2 + 1e-6);
  return g;
}

#include "policy.cuh"

extern "C" int uavsim_abi_version(void) { return UAVSIM_ABI_VERSION; }
extern "C" const char *uavsim_last_error(void) { return g_err; }
extern "C" int64_t uavsim_launch_count(const uavsim_t *h) { return h ? h->launches : 0; }
extern "C" int64_t uavsim_step_count(const uavsim_t *h) { return h ? h->t : 0; }

static int uavsim_create_impl(const UavSimParams *p, int64_t n_envs, int64_t env_id_offset, int device, uavsim_t **out);

// Every failure after the handle exists goes through uavsim_destroy (device tables, statistics, streams, events).
extern "C" int uavsim_create(const UavSimParams *p, int64_t n_envs, int64_t env_id_offset, int device,
                             uavsim_t **out) {
  if (!p || !out) { SET_ERR("uavsim_create: NULL argument"); return UAVSIM_ERR_ARG; }
  *out = nullptr;
  const int rc = uavsim_create_impl(p, n_envs, env_id_offset, device, out);
  if (rc && *out) {
    char msg[sizeof(g_err)];
    memcpy(msg, g_err, sizeof(msg));  // keep the first error: destroy may overwrite it
    uavsim_destroy(*out);
    memcpy(g_err, msg, sizeof(msg));
    *out = nullptr;
  }
  return rc;
}

static int uavsim_create_impl(const UavSimParams *p, int64_t n_envs, int64_t env_id_offset, int device, uavsim_t **out) {
  if (n_envs <= 0 || p->n_uav <= 0 || p->m_targets <= 0 || p->na < 2 || p->dp <= 0 || p->dc <= 0) {
    SET_ERR("uavsim_create: need n_envs>0, n_uav>0, m_targets>0, na>=2, dp>0, dc>0");
    return UAVSIM_ERR_ARG;
  }
  if (p->n_uav > UAVSIM_MAX_UAV) {
    SET_ERR("uavsim_create: n_uav=%d exceeds UAVSIM_MAX_UAV=%d", p->n_uav, UAVSIM_MAX_UAV);
    return UAVSIM_ERR_UNSUPPORTED;
  }
  if (env_id_offset < 0 || env_id_offset + n_envs > (int64_t)0xffffffffll) {
    SET_ERR("uavsim_create: global env ids must fit 32 bits");
    return UAVSIM_ERR_UNSUPPORTED;
  }
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { SET_ERR("uavsim_create: device %d of %d", device, ndev); return UAVSIM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(device));
  uavsim *h = (uavsim *)calloc(1, sizeof(uavsim));
  if (!h) { SET_ERR("out of host memory"); return UAVSIM_ERR_ARG; }
  *out = h;  // from here on a failure is cleaned up by the caller through uavsim_destroy
  h->hp = *p;
  h->device = device;
  h->E = n_envs;
  CUDA_TRY(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device));

  KParams &k = h->kp;
  k.n = p->n_uav; k.m = p->m_targets; k.na = p->na; k.num_steps = p->num_steps;
  k.E = n_envs; k.env_id_offset = env_id_offset;
  k.x_max = p->x_max; k.y_max = p->y_max;
  k.dtv_u = p->dt * p->uav_v_max;
  k.dt = p->dt; k.uav_h_max = p->uav_h_max;
  k.dtv_t = p->dt * p->tgt_v_max;
  k.dc = p->dc; k.dp = p->dp; k.two_dp = 2 * p->dp;
  k.tv = p->tgt_v_max; k.uv = p->uav_v_max; k.tv_over_uv = p->tgt_v_max / p->uav_v_max;
  k.s_dp_le = exact_sq_threshold(p->dp, false);
  k.s_dp_lt = exact_sq_threshold(p->dp, true);
  k.s_dc_le = exact_sq_threshold(p->dc, false);
  k.s_2dp_le = exact_sq_threshold(2 * p->dp, false);
  k.alpha = p->alpha; k.beta = p->beta; k.gamma = p->gamma;
  k.tt_hi = (double)(2 * p->m_targets);
  k.dup_lo = -2.718281828459045 / 2 * p->n_uav;
  k.inv_dp = 1.0 / p->dp; k.inv_dc = 1.0 / p->dc; k.inv_na = 1.0 / (double)p->na;
  k.inv_tt_hi = 1.0 / k.tt_hi; k.inv_dup_span = 1.0 / (0.0 - k.dup_lo);
  // fp32 prefilter (step_kernel.cuh): coordinates relative to the map centre, valid while every entity is within
  // rmax of it; the guard band bounds the fp32 error of the squared distance so no true hit is ever dropped
  k.cx = p->x_max / 2; k.cy = p->y_max / 2;
  k.rmax = 32768.0;
  k.f_dp = prefilter_threshold(p->dp, k.rmax);
  {  // one radius for every UAV-UAV test of a step: communication at the partner's new position (dc) or at its old
     // position, bounded through the new one (dc + dt*v), duplicate tracking (2 dp) and the neighbour set (dp).  With
     // the shipped constants dc + dt*v = 520 dominates; a scenario with 2 dp > dc + dt*v needs the larger one.
    double r_uav = p->dc + fabs(k.dtv_u) * (1.0 + 1e-9);
    if (2.0 * p->dp > r_uav) r_uav = 2.0 * p->dp;
    k.f_dcmv = prefilter_threshold(r_uav, k.rmax);
    k.g_pf = make_guard(r_uav, k.rmax);
  }
  k.g_dp = make_guard(p->dp, k.rmax);
  k.g_2dp = make_guard(2 * p->dp, k.rmax);
  k.g_dc = make_guard(p->dc, k.rmax);
  {  // The fast kernel accumulates fp32 offsets between fp32 coordinates; a partner's coordinate rounding, up to
     // R * 2^-24, reaches the observation divided by dp or dc.  Keep that below 2e-6 (the contract is 1e-5); beyond
     // this radius an environment takes the fp64 path.
    const double rmin = p->dp < p->dc ? p->dp : p->dc;
    double rf = 2e-6 * 16777216.0 * rmin;
    if (rf > k.rmax) rf = k.rmax;
    k.r_fast = (float)rf;
    k.r_tile = (float)(rf < 4096.0 ? rf : 4096.0);
    // tile kernel: band centre / half width per radius at two swarm extents (the guard grows with the extent)
    const double cmax = k.cx > k.cy ? k.cx : k.cy;
    const double rr[2] = {1.3 * cmax < k.r_tile ? 1.3 * cmax : (double)k.r_tile, (double)k.r_tile};
    for (int lv = 0; lv < 2; lv++) {
      auto band = [&](const GuardK &G, float &C, float &H) {
        const double gd = ((double)G.c1 * rr[lv] + (double)G.c0) * (1.0 + 1e-6);
        const double hi = (double)G.t2_up + gd, lo = (double)G.t2_dn - gd;
        C = (float)(0.5 * (hi + lo));
        // |fl(s) - C| <= H must hold for every s in [lo, hi]: half the width, the rounding of C and of the subtraction
        const double hw = 0.5 * (hi - lo) + 2.4e-7 * fabs(hi) + fabs((double)C - 0.5 * (hi + lo));
        H = nextafterf((float)hw, INFINITY);
        if ((double)H < hw) H = nextafterf(H, INFINITY);
      };
      k.tb[lv].r = (float)rr[lv];
      if ((double)k.tb[lv].r > rr[lv]) k.tb[lv].r = nextafterf(k.tb[lv].r, 0.f);
      band(k.g_dp, k.tb[lv].Cp, k.tb[lv].Hp);
      band(k.g_2dp, k.tb[lv].Cd, k.tb[lv].Hd);
      band(k.g_dc, k.tb[lv].Cc, k.tb[lv].Hc);
      k.tb[lv].pad = 0.f;
    }
  }
  k.dp_f = (float)p->dp; k.inv_dp_f = (float)k.inv_dp; k.inv_dc_f = (float)k.inv_dc; k.inv_na_f = (float)k.inv_na;
  k.tt_hi_f = (float)k.tt_hi; k.inv_tt_hi_f = (float)k.inv_tt_hi; k.dup_lo_f = (float)k.dup_lo; k.inv_dup_span_f = (float)k.inv_dup_span;
  k.alpha_f = (float)k.alpha; k.beta_f = (float)k.beta; k.gamma_f = (float)k.gamma;
  k.k_ex1_f = (float)(-1.4426950408889634 / k.two_dp); k.tv_over_uv_f = (float)k.tv_over_uv;
  k.cx_f = (float)k.cx; k.cy_f = (float)k.cy;
  k.dtv_u_f = (float)k.dtv_u;
  {
    double tab[FM_TAB_SIZE * 2];
    fm_fill_table(tab);
    CUDA_TRY(cudaMalloc(&h->d_sctab, sizeof(tab)));
    CUDA_TRY(cudaMemcpy(h->d_sctab, tab, sizeof(tab), cudaMemcpyHostToDevice));
    k.sincos_tab = h->d_sctab;
    CUDA_TRY(cudaMalloc(&h->d_fast_ctr, 2 * sizeof(int)));
    CUDA_TRY(cudaMemset(h->d_fast_ctr, 0, 2 * sizeof(int)));
    k.fast_ctr = h->d_fast_ctr;
  }

  // per action: dt * discrete_action(a) (src/agent/uav.py:73-81, :96) in the reference's evaluation order,
  // plus its cosine / sine for the angle-addition update of the observation heading terms
  std::vector<double> dth_v(3 * (size_t)p->na);
  double *dth = dth_v.data();
  for (int a = 0; a < p->na; a++) {
    const int na1 = a + 1;
    const double rate = (double)(2 * na1 - p->na - 1) * p->uav_h_max / (double)(p->na - 1);
    dth[3 * a] = p->dt * rate;
    dth[3 * a + 1] = cos(dth[3 * a]);
    dth[3 * a + 2] = sin(dth[3 * a]);
  }
  CUDA_TRY(cudaMalloc(&h->d_dth, sizeof(double) * 3 * p->na));
  CUDA_TRY(cudaMemcpy(h->d_dth, dth, sizeof(double) * 3 * p->na, cudaMemcpyHostToDevice));
  {  // the same table for the fast kernel: the angle in fp64, its cosine / sine in fp32
    std::vector<ActEntry> tab(p->na);
    for (int a = 0; a < p->na; a++) { tab[a].dth = dth[3 * a]; tab[a].cd = (float)dth[3 * a + 1]; tab[a].sd = (float)dth[3 * a + 2]; }
    CUDA_TRY(cudaMalloc(&h->d_act, sizeof(ActEntry) * p->na));
    CUDA_TRY(cudaMemcpy(h->d_act, tab.data(), sizeof(ActEntry) * p->na, cudaMemcpyHostToDevice));
  }

  // launch geometry of the step kernel: one thread per UAV, nt / n environments per CTA.  Small CTAs keep the
  // phase barriers cheap (the exact pass has data-dependent length); compile-time sizes for the two headline scenarios
  if (k.n == 64 && k.m == 64) { h->nt = UAVSIM_NT64; h->step_fn[0] = uavsim_step_kernel<64, 64, false, UAVSIM_NT64>; h->step_fn[1] = uavsim_step_kernel<64, 64, true, UAVSIM_NT64>; }
  else if (k.n == 10 && k.m == 10) { h->nt = 128; h->step_fn[0] = uavsim_step_kernel<10, 10, false, 128>; h->step_fn[1] = uavsim_step_kernel<10, 10, true, 128>; }
  else { h->nt = 128; h->step_fn[0] = uavsim_step_kernel<0, 0, false, 128>; h->step_fn[1] = uavsim_step_kernel<0, 0, true, 128>; }
  int epb = h->nt / p->n_uav;
  if (epb < 1) epb = 1;
  // the compile-time instances derive nt / n themselves (constant shared-memory offsets); run-time sizes adapt
  const bool fixed_shape = (k.n == 64 && k.m == 64) || (k.n == 10 && k.m == 10);
  if (!fixed_shape) {
    if ((int64_t)epb > n_envs) epb = (int)n_envs;
    while (epb > 1 && step_smem_bytes(k.n, k.m, k.na, epb) > 64 * 1024) epb--;
  }
  h->epb = epb;
  h->smem_step = step_smem_bytes(k.n, k.m, k.na, epb);
  if (h->smem_step > 227 * 1024) {
    SET_ERR("uavsim_create: n_uav=%d m_targets=%d needs %zu B shared memory per CTA", k.n, k.m, h->smem_step);
    return UAVSIM_ERR_UNSUPPORTED;
  }
  for (int v = 0; v < 2; v++) {
    int rc = raise_dynamic_smem((const void *)h->step_fn[v], device, h->smem_step);
    if (rc) return rc;
  }
  int occ = 1;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, h->step_fn[0], h->nt, h->smem_step));
  if (occ < 1) occ = 1;
  h->grid_max = h->sm_count * occ;
  // fast kernel (step_fast_kernel.cuh): 64 x 64 swarms, one environment per 64-thread CTA
  h->has_fast = (k.n == 64 && k.m == 64);
  if (h->has_fast) {
    h->fast_fn[0] = uavsim_step_fast_kernel<64, 64, false>;
    h->fast_fn[1] = uavsim_step_fast_kernel<64, 64, true>;
    h->smem_fast[0] = sizeof(FastSmem<64, 64, false>);
    h->smem_fast[1] = sizeof(FastSmem<64, 64, true>);
    for (int v = 0; v < 2; v++) {
      int rc = raise_dynamic_smem((const void *)h->fast_fn[v], device, h->smem_fast[v]);
      if (rc) return rc;
      int o = 1;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, h->fast_fn[v], FAST_NT, h->smem_fast[v]));
      h->fast_grid_max[v] = h->sm_count * (o < 1 ? 1 : o);
      if (h->fast_grid_max[v] > h->grid_max) h->grid_max = h->fast_grid_max[v];  // statistics slots cover both kernels
    }
    // tile kernel (step_tile_kernel.cuh): the same swarms, one environment per 128-thread CTA
    h->tile_fn[0] = uavsim_step_tile_kernel<false>;
    h->tile_fn[1] = uavsim_step_tile_kernel<true>;
    h->smem_tile[0] = sizeof(TileSmem<false>);
    h->smem_tile[1] = sizeof(TileSmem<true>);
    for (int v = 0; v < 2; v++) {
      int rc = raise_dynamic_smem((const void *)h->tile_fn[v], device, h->smem_tile[v]);
      if (rc) return rc;
      int o = 1;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, h->tile_fn[v], TILE_NT, h->smem_tile[v]));
      h->tile_grid_max[v] = h->sm_count * (o < 1 ? 1 : o);
      if (h->tile_grid_max[v] > h->grid_max) h->grid_max = h->tile_grid_max[v];
    }
  }
  // small-swarm kernel (step_small_kernel.cuh): groups of environments in two-warp CTAs
  h->has_small = (k.n <= SMALL_MAX && k.m <= SMALL_MAX);
  int small_warps = 0;
  if (h->has_small) {
    h->small_fn[0] = uavsim_step_small_kernel<false>;
    h->small_fn[1] = uavsim_step_small_kernel<true>;
    for (int v = 0; v < 2; v++) {
      int o = 1;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, h->small_fn[v], SMALL_NT, 0));
      h->small_grid_max[v] = h->sm_count * (o < 1 ? 1 : o);
      if (h->small_grid_max[v] > small_warps) small_warps = h->small_grid_max[v];
    }
  }
  h->stat_slots = h->grid_max > 4096 ? h->grid_max : 4096;
  if (small_warps > h->stat_slots) h->stat_slots = small_warps;  // one statistics slot per CTA of that kernel too
  CUDA_TRY(cudaMalloc(&h->d_stats, sizeof(long long) * h->stat_slots * STAT_W));
  CUDA_TRY(cudaMalloc(&h->d_stats8, sizeof(double) * 8));
  CUDA_TRY(cudaMallocHost(&h->h_stats8, sizeof(double) * 8));
  CUDA_TRY(cudaMemset(h->d_stats, 0, sizeof(long long) * h->stat_slots * STAT_W));

  CUDA_TRY(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreateWithFlags(&h->ev_user, cudaEventDisableTiming));
  for (int c = 0; c < 16; c++) {
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_in[c], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_comp[c], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_out[c], cudaEventDisableTiming));
  }
  for (int c = 0; c < 2; c++) CUDA_TRY(cudaEventCreateWithFlags(&h->ev_done[c], cudaEventDisableTiming));
  *out = h;
  return 0;
}

extern "C" int uavsim_destroy(uavsim_t *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaFree(h->d_dth); cudaFree(h->d_act); cudaFree(h->d_sctab); cudaFree(h->d_fast_ctr); cudaFree(h->d_stats); cudaFree(h->d_stats8); cudaFreeHost(h->h_stats8);
  cudaFree(h->d_pmi_blob); cudaFree(h->d_tc_tiles);
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_comp) cudaStreamDestroy(h->s_comp);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  if (h->ev_user) cudaEventDestroy(h->ev_user);
  for (int c = 0; c < 16; c++) {
    if (h->ev_in[c]) cudaEventDestroy(h->ev_in[c]);
    if (h->ev_comp[c]) cudaEventDestroy(h->ev_comp[c]);
    if (h->ev_out[c]) cudaEventDestroy(h->ev_out[c]);
  }
  for (int c = 0; c < 2; c++) if (h->ev_done[c]) cudaEventDestroy(h->ev_done[c]);
  free(h);
  return 0;
}

extern "C" int uavsim_bind(uavsim_t *h, const UavSimBuffers *b) {
  if (!h || !b) { SET_ERR("uavsim_bind: NULL argument"); return UAVSIM_ERR_ARG; }
  if (!b->ux || !b->uy || !b->uh || !b->ua || !b->tx || !b->ty || !b->th || !b->actions || !b->obs || !b->rew4 ||
      !b->covered) {
    SET_ERR("uavsim_bind: state, actions, obs, rew4 and covered buffers are required");
    return UAVSIM_ERR_ARG;
  }
  const int nm = (b->obs_mask != 0) + (b->comm_mask != 0) + (b->nbr_mask != 0) + (b->dup_mask != 0) + (b->cover_mask != 0);
  if (nm != 0 && nm != 5) { SET_ERR("uavsim_bind: give all five mask buffers or none"); return UAVSIM_ERR_ARG; }
  if ((reinterpret_cast<uintptr_t>(b->obs) & 15) != 0) { SET_ERR("uavsim_bind: obs must be 16-byte aligned"); return UAVSIM_ERR_ARG; }
  h->buf = *b;
  h->bound = true;
  return 0;
}

extern "C" int uavsim_set_reward_weights(uavsim_t *h, double alpha, double beta, double gamma) {
  if (!h) { SET_ERR("uavsim_set_reward_weights: NULL handle"); return UAVSIM_ERR_ARG; }
  h->hp.alpha = h->kp.alpha = alpha;
  h->hp.beta = h->kp.beta = beta;
  h->hp.gamma = h->kp.gamma = gamma;
  h->kp.alpha_f = (float)alpha; h->kp.beta_f = (float)beta; h->kp.gamma_f = (float)gamma;
  return 0;
}

static int check_bound(uavsim_t *h, const char *who) {
  if (!h) { SET_ERR("%s: NULL handle", who); return UAVSIM_ERR_ARG; }
  if (!h->bound) { SET_ERR("%s: uavsim_bind has not been called", who); return UAVSIM_ERR_UNBOUND; }
  return 0;
}

static int clear_counters(uavsim_t *h, cudaStream_t st) {
  const int count = h->stat_slots * STAT_W;
  uavsim_stats_clear_kernel<<<(count + 255) / 256, 256, 0, st>>>(h->d_stats, count);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  h->t = 0;
  return 0;
}

static int elementwise_grid(uavsim_t *h, int64_t items) {
  int64_t g = (items + 255) / 256;
  const int64_t cap = (int64_t)h->sm_count * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

extern "C" int uavsim_reset(uavsim_t *h, uint64_t seed, void *stream) {
  int rc = check_bound(h, "uavsim_reset");
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t items = h->E * (h->kp.n + h->kp.m);
  uavsim_reset_kernel<<<elementwise_grid(h, items), 256, 0, st>>>(h->kp, h->buf, seed);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return clear_counters(h, st);
}

extern "C" int uavsim_begin_episode(uavsim_t *h, void *stream) {
  int rc = check_bound(h, "uavsim_begin_episode");
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  uavsim_initial_obs_kernel<<<elementwise_grid(h, h->E * h->kp.n), 256, 0, st>>>(h->kp, h->buf);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return clear_counters(h, st);
}

extern "C" int uavsim_random_actions(uavsim_t *h, uint64_t seed, int64_t step, void *stream) {
  int rc = check_bound(h, "uavsim_random_actions");
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  uavsim_random_actions_kernel<<<elementwise_grid(h, h->E * h->kp.n), 256, 0, st>>>(h->kp, h->buf.actions, seed,
                                                                                   (uint32_t)step);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return 0;
}

// PMI launch geometry: G environments per CTA iteration, bounded by threads (G*n <= 256) and by the
// pair buffer (G*n*(n-1) <= pmax)
static int pmi_configure(uavsim_t *h) {
  const int n = h->kp.n, H = h->pmi.H;
  const int TM = (H <= 128) ? 64 : 32;
  int G = PMI_NT / n;
  if (G < 1) G = 1;
  if ((int64_t)G > h->E) G = (int)h->E;
  const int per_env = n * (n - 1) > 0 ? n * (n - 1) : 1;
  while (G > 1 && (int64_t)G * per_env > 8192) G--;
  int pmax = G * per_env;
  size_t smem = pmi_smem_bytes(n, H, G, pmax, TM);
  if (smem > 227 * 1024) {
    SET_ERR("PMI mode: n_uav=%d hidden=%d needs %zu B shared memory per CTA", n, H, smem);
    return UAVSIM_ERR_UNSUPPORTED;
  }
  h->pmi_g = G; h->pmi_pmax = pmax; h->pmi_tm = TM; h->smem_pmi = smem;
  return 0;
}

template <int CPT, int TM>
static int pmi_launch_t(uavsim_t *h, int64_t e0, int64_t cnt, double coop, cudaStream_t st, bool configure_only) {
  auto kern = uavsim_pmi_kernel<CPT, TM>;
  if (configure_only) {
    int rc = raise_dynamic_smem((const void *)kern, h->device, h->smem_pmi);
    if (rc) return rc;
    int occ = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, PMI_NT, h->smem_pmi));
    if (occ < 1) occ = 1;
    h->pmi_grid_max = h->sm_count * occ;
    if (h->pmi_grid_max > h->stat_slots) h->pmi_grid_max = h->stat_slots;
    return 0;
  }
  const int64_t ngroups = (cnt + h->pmi_g - 1) / h->pmi_g;
  const int grid = (int)(ngroups < h->pmi_grid_max ? ngroups : h->pmi_grid_max);
  kern<<<grid, PMI_NT, h->smem_pmi, st>>>(h->kp, h->buf, h->pmi, e0, cnt, h->pmi_g, h->pmi_pmax, coop, h->d_stats);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return 0;
}

// round to TF32 like cvt.rna.tf32.f32 (nearest, ties away from zero): keep 10 mantissa bits
#if !TC_F16
static float host_tf32_rna(float v) {
  uint32_t b;
  memcpy(&b, &v, 4);
  if ((b & 0x7f800000u) != 0x7f800000u) b = (b + 0x1000u) & 0xffffe000u;
  memcpy(&v, &b, 4);
  return v;
}
#endif

// the tensor path can serve this shape and these weights (whatever uavsim_set_pmi_path asked for)
static bool pmi_tensor_available(const uavsim_t *h) {
  const int n = h->kp.n;
  return h->has_tc && n * (n - 1) <= TC_PMAX && n <= TC_AMAX;
}
static bool pmi_use_tensor(const uavsim_t *h) { return h->pmi_path != 1 && pmi_tensor_available(h); }
static const char *pmi_tensor_why_not(const uavsim_t *h) {
  if (h->has_pmi && (h->pmi.H == 64 || h->pmi.H == 128) && !h->tc_range)
    return "these weights exceed the fp16 range of its operands after the per-unit rebalancing (the CUDA-core kernel serves them)";
  return "the tensor-core path needs hidden = 64 or 128 and n_uav*(n_uav-1) <= 16384";
}

static int pmi_tc_launch(uavsim_t *h, int64_t e0, int64_t cnt, double coop, cudaStream_t st) {
  PmiTcDev W;
  W.w0 = h->pmi.w0; W.b0 = h->pmi.b0; W.b1 = h->pmi.b1; W.w2 = h->pmi.w2; W.b2 = h->pmi.b2;
  W.w1_tiles = h->d_tc_tiles;
  W.x_safe = h->tc_x_safe;
  // Group size: the largest that fits (tc_g) fixes the number of waves over the one-CTA-per-SM grid; within that number
  // of waves the groups are made equal, so that every CTA gets the same count (16 384 environments of 10 UAVs: 51 per
  // group would be 322 groups = 2.2 per CTA, i.e. three for some and two for most; 37 per group is 443 = three for all).
  int G = h->tc_g;
  {
    const int64_t g_max = (cnt + G - 1) / G;
    const int64_t waves = (g_max + h->sm_count - 1) / h->sm_count;
    const int64_t slots = waves * h->sm_count;
    const int64_t g_even = (cnt + slots - 1) / slots;
    if (g_even >= 1 && g_even < G) G = (int)g_even;
  }
  const int64_t ngroups = (cnt + G - 1) / G;
  int grid = (int)(ngroups < h->sm_count ? ngroups : h->sm_count);
  if (grid > h->stat_slots) grid = h->stat_slots;
  if (h->pmi.H == 64)
    uavsim_pmi_tc_kernel<64><<<grid, TC_NT, TcSmem::total, st>>>(h->kp, h->buf, W, e0, cnt, G, coop, h->d_stats);
  else
    uavsim_pmi_tc_kernel<128><<<grid, TC_NT, TcSmem::total, st>>>(h->kp, h->buf, W, e0, cnt, G, coop, h->d_stats);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return 0;
}

// Whether a PMI kernel can serve the uploaded weights with the selected path (checked again at every launch: weights
// may be uploaded after the path was chosen).
static int pmi_servable(const uavsim_t *h) {
  if (pmi_use_tensor(h)) return 0;
  if (h->pmi_path == 2) {
    SET_ERR("PMI mode: tensor-core path selected (uavsim_set_pmi_path 2) but unavailable: %s", pmi_tensor_why_not(h));
    return UAVSIM_ERR_UNSUPPORTED;
  }
  if (!h->has_cc) {
    SET_ERR("PMI mode: n_uav=%d is too large for the CUDA-core PMI kernel and the tensor path is %s", h->kp.n,
            h->pmi_path == 1 ? "switched off (uavsim_set_pmi_path 1)" : "unavailable (hidden is neither 64 nor 128)");
    return UAVSIM_ERR_UNSUPPORTED;
  }
  return 0;
}

static int pmi_launch(uavsim_t *h, int64_t e0, int64_t cnt, double coop, cudaStream_t st, bool configure_only) {
  if (!configure_only && pmi_use_tensor(h)) return pmi_tc_launch(h, e0, cnt, coop, st);
  if (!configure_only) {
    const int rc = pmi_servable(h);
    if (rc) return rc;
  }
  switch (h->pmi.H) {
    case 32: return pmi_launch_t<2, 64>(h, e0, cnt, coop, st, configure_only);
    case 64: return pmi_launch_t<4, 64>(h, e0, cnt, coop, st, configure_only);
    case 128: return pmi_launch_t<8, 64>(h, e0, cnt, coop, st, configure_only);
    case 256: return pmi_launch_t<16, 32>(h, e0, cnt, coop, st, configure_only);
  }
  SET_ERR("PMI hidden size %d not supported (32, 64, 128, 256)", h->pmi.H);
  return UAVSIM_ERR_UNSUPPORTED;
}

extern "C" int uavsim_set_pmi_path(uavsim_t *h, int path) {
  if (!h || path < 0 || path > 2) { SET_ERR("uavsim_set_pmi_path: bad argument"); return UAVSIM_ERR_ARG; }
  if (path == 2 && h->has_pmi && !pmi_tensor_available(h)) {
    SET_ERR("uavsim_set_pmi_path: %s", pmi_tensor_why_not(h));
    return UAVSIM_ERR_UNSUPPORTED;
  }
  h->pmi_path = path;
  return 0;
}

extern "C" int uavsim_set_step_path(uavsim_t *h, int path) {
  if (!h || path < 0 || path > 4) { SET_ERR("uavsim_set_step_path: bad argument"); return UAVSIM_ERR_ARG; }
  if ((path == 2 || path == 3) && !h->has_fast) { SET_ERR("uavsim_set_step_path: the fast step kernels serve 64 x 64 swarms only"); return UAVSIM_ERR_UNSUPPORTED; }
  if (path == 4 && !h->has_small) { SET_ERR("uavsim_set_step_path: the small-swarm step kernel serves n_uav, m_targets <= %d", SMALL_MAX); return UAVSIM_ERR_UNSUPPORTED; }
  h->step_path = path;
  return 0;
}

extern "C" int uavsim_set_pmi_weights(uavsim_t *h, const UavSimPmiWeights *w, void *stream) {
  if (!h || !w || !w->w0 || !w->b0 || !w->w1 || !w->b1 || !w->w2) { SET_ERR("uavsim_set_pmi_weights: NULL argument"); return UAVSIM_ERR_ARG; }
  const int H = w->hidden;
  if (H != 32 && H != 64 && H != 128 && H != 256) { SET_ERR("PMI hidden size %d not supported (32, 64, 128, 256)", H); return UAVSIM_ERR_UNSUPPORTED; }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n_w0 = (size_t)3 * H * 5, n_b0 = 3 * H, n_w1 = (size_t)H * 3 * H, n_b1 = H, n_w2 = H;
  const size_t total = n_w0 + n_b0 + n_w1 + n_b1 + n_w2;
  std::vector<float> blob_v(total);  // (kept until the tensor tiles are built from it)
  float *blob = blob_v.data();
  float *q = blob;
  memcpy(q, w->w0, n_w0 * 4); q += n_w0;
  memcpy(q, w->b0, n_b0 * 4); q += n_b0;
  for (int k = 0; k < 3 * H; k++)  // transpose fc1 [H,3H] -> [3H,H]
    for (int o = 0; o < H; o++) q[(size_t)k * H + o] = w->w1[(size_t)o * 3 * H + k];
  q += n_w1;
  memcpy(q, w->b1, n_b1 * 4); q += n_b1;
  memcpy(q, w->w2, n_w2 * 4);
  // Per-unit rebalancing (DESIGN.md section 3.2): ReLU is positively homogeneous, so row u of layer 0 (w0, b0) times
  // 2^s_u and column u of fc1 times 2^-s_u is the same function; with powers of two the fp32 arithmetic of the CUDA-core
  // kernel gives bit-identical results.  s_u brings max(b0_u, 0) + PMI_X_NOM * sum_k |w0_uk| (the activation bound for
  // inputs up to PMI_X_NOM: a negative pre-activation is 0 after the ReLU) to [2^PMI_BAL_T, 2^(PMI_BAL_T+1)), which
  // puts the tensor path's fp16 activations and fc1 halves at the same magnitudes whatever scale the BatchNorm folding
  // gave the unit; it is raised where the fc1 column would otherwise leave fp16's range after the TC_WSCALE pre-scale
  // (that unit's activations then take a smaller input range, see x_safe below).  Both bounds scale with the row, so a
  // network whose BatchNorms are rescaled by 2^k uploads the same blob.
  float *bw0 = blob, *bb0 = blob + n_w0, *bw1 = blob + n_w0 + n_b0;
  for (int u = 0; u < 3 * H; u++) {
    double est = std::max(0.0, (double)bb0[u]), sw = 0, wmax = 0;
    for (int k = 0; k < 5; k++) sw += fabs((double)bw0[u * 5 + k]);
    est += PMI_X_NOM * sw;
    for (int o = 0; o < H; o++) wmax = std::max(wmax, fabs((double)bw1[(size_t)u * H + o]));
    if (!std::isfinite(est) || !std::isfinite(wmax)) continue;  // refused below
    int s = 0, e2;
    if (est > 0) {  // (an all-zero row keeps s = 0)
      frexp(est, &e2);  // est = m * 2^e2, m in [0.5, 1): floor(log2(est)) = e2 - 1
      s = PMI_BAL_T - (e2 - 1);
    }
#if TC_F16
    if (wmax > 0) {  // smallest s with wmax * 2^-s * TC_WSCALE < 65504
      frexp(wmax * TC_WSCALE / 65504.0, &e2);
      s = std::max(s, e2);
    }
#endif
    if (s == 0) continue;
    // only an exact rescaling is applied (no value of the row or the column leaves fp32's normal range)
    auto exact = [](float v, int e) { return ldexpf(ldexpf(v, e), -e) == v; };
    bool ok = exact(bb0[u], s);
    for (int k = 0; k < 5; k++) ok = ok && exact(bw0[u * 5 + k], s);
    for (int o = 0; o < H; o++) ok = ok && exact(bw1[(size_t)u * H + o], -s);
    if (!ok) continue;
    for (int k = 0; k < 5; k++) bw0[u * 5 + k] = ldexpf(bw0[u * 5 + k], s);
    bb0[u] = ldexpf(bb0[u], s);
    for (int o = 0; o < H; o++) bw1[(size_t)u * H + o] = ldexpf(bw1[(size_t)u * H + o], -s);
  }
  // Range of the tensor path (fp16 operands): x_safe is the largest max_k |x_k| of a pair row for which every layer-0
  // activation stays below fp16's largest finite value, with a 2^-8 margin for the fp32 rounding of the pre-activation;
  // the kernel counts rows beyond it.  The tensor path serves the weights when every value is finite, every fc1 half is
  // finite after the TC_WSCALE pre-scale and x_safe covers at least the nominal input bound PMI_X_NOM (in-map
  // observations give pair inputs up to 16); otherwise the CUDA-core kernel does.
  bool finite = std::isfinite(w->b2);
  for (size_t k = 0; k < total; k++) finite = finite && std::isfinite(blob[k]);
  float w1max = 0.f;
  for (size_t k = 0; k < n_w1; k++) w1max = fmaxf(w1max, fabsf(bw1[k]));
  double x_safe = DBL_MAX;
#if TC_F16
  for (int u = 0; u < 3 * H; u++) {
    double sw = 0;
    for (int k = 0; k < 5; k++) sw += fabs((double)bw0[u * 5 + k]);
    if (sw > 0) x_safe = std::min(x_safe, std::max(0.0, 65504.0 * (1.0 - 1.0 / 256) - std::max(0.0, (double)bb0[u])) / sw);
  }
  const bool tc_range = finite && (double)w1max * TC_WSCALE < 65504.0 && x_safe >= PMI_X_NOM;
#else
  const bool tc_range = finite;
#endif
  if (h->d_pmi_blob && h->pmi.H != H) { CUDA_TRY(cudaStreamSynchronize(st)); cudaFree(h->d_pmi_blob); h->d_pmi_blob = nullptr; }
  if (!h->d_pmi_blob) CUDA_TRY(cudaMalloc(&h->d_pmi_blob, total * sizeof(float)));
  CUDA_TRY(cudaMemcpyAsync(h->d_pmi_blob, blob, total * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  h->pmi.H = H;
  h->pmi.w0 = h->d_pmi_blob;
  h->pmi.b0 = h->pmi.w0 + n_w0;
  h->pmi.w1t = h->pmi.b0 + n_b0;
  h->pmi.b1 = h->pmi.w1t + n_w1;
  h->pmi.w2 = h->pmi.b1 + n_b1;
  h->pmi.b2 = w->b2;
  int rc = pmi_configure(h);
  if (!rc) rc = pmi_launch(h, 0, 0, 0.0, st, true);
  h->has_cc = rc == 0;
  const bool tc_shape = (H == 128 || H == 64);
  if (rc && !tc_shape) return rc;  // only the tensor path (hidden 64 / 128) can take over a shape the CUDA-core kernel cannot hold
  h->has_tc = false;
  h->tc_range = tc_range;
  h->has_pmi = true;
  if (tc_shape && !tc_range) {
    if (h->has_cc) return 0;  // the CUDA-core kernel serves these weights (automatic choice; path 2 is refused)
    h->has_pmi = false;
    SET_ERR("uavsim_set_pmi_weights: n_uav=%d needs the tensor-core PMI path, and these weights exceed its fp16 range "
            "(after rebalancing: max |w1'| * %g = %g, pair-row input range %g < %g)", h->kp.n, (double)TC_WSCALE,
            (double)w1max * TC_WSCALE, x_safe, PMI_X_NOM);
    return UAVSIM_ERR_UNSUPPORTED;
  }
  if (tc_shape) {
    // tensor-core path: fc1 (rebalanced, transposed in the blob) split hi/lo and laid out as the K-major UMMA tiles the
    // kernel bulk-copies, chunk c, part {hi, lo}: fp16 (TC_F16, weights pre-scaled by TC_WSCALE): element (unit o, input
    // k) at half (k/8)*(H*8) + o*8 + (k%8); TF32 (H = 128 only): at float (k/4)*512 + o*4 + (k%4)
    const int H3 = 3 * H, nchunk = H3 / TC_KC;
    const size_t tile = (size_t)H * TC_KC * (TC_F16 ? 2 : 4) / 4, total_t = (size_t)nchunk * 2 * tile;
    std::vector<float> tiles_v(total_t);
    float *tiles = tiles_v.data();
    for (int c = 0; c < nchunk; c++)
      for (int o = 0; o < H; o++)
        for (int kk = 0; kk < TC_KC; kk++) {
          const float v = bw1[(size_t)(c * TC_KC + kk) * H + o] * TC_WSCALE;
#if TC_F16
          const __half hi = __float2half_rn(v), lo = __float2half_rn(v - __half2float(hi));
          const size_t e = (size_t)(kk / 8) * ((size_t)H * 8) + (size_t)o * 8 + (kk % 8);
          reinterpret_cast<__half *>(tiles + ((size_t)c * 2 + 0) * tile)[e] = hi;
          reinterpret_cast<__half *>(tiles + ((size_t)c * 2 + 1) * tile)[e] = lo;
#else
          const float hi = host_tf32_rna(v), lo = host_tf32_rna(v - hi);
          const size_t e = (size_t)(kk / 4) * 512 + (size_t)o * 4 + (kk % 4);
          tiles[((size_t)c * 2 + 0) * tile + e] = hi;
          tiles[((size_t)c * 2 + 1) * tile + e] = lo;
#endif
        }
    if (h->d_tc_tiles) { CUDA_TRY(cudaStreamSynchronize(st)); cudaFree(h->d_tc_tiles); h->d_tc_tiles = nullptr; }
    CUDA_TRY(cudaMalloc(&h->d_tc_tiles, total_t * sizeof(float)));
    CUDA_TRY(cudaMemcpyAsync(h->d_tc_tiles, tiles, total_t * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    rc = raise_dynamic_smem(H == 64 ? (const void *)uavsim_pmi_tc_kernel<64> : (const void *)uavsim_pmi_tc_kernel<128>, h->device, TcSmem::total);
    if (rc) return rc;
    const int n = h->kp.n, per_env = n * (n - 1) > 0 ? n * (n - 1) : 1;
    int G = TC_AMAX / n;
    if (G > TC_PMAX / per_env) G = TC_PMAX / per_env;
    if ((int64_t)G > h->E) G = (int)h->E;
    h->tc_g = G < 1 ? 1 : G;
    h->tc_x_safe = (float)std::min(x_safe, (double)FLT_MAX);
    h->has_tc = true;
  }
  return 0;
}

// The fast kernel moves whole arrays with bulk copies: every bound array it touches must be 16-byte aligned.
static bool fast_path_usable(const uavsim_t *h) {
  if (!h->has_fast || h->step_path == 1 || h->step_path == 4) return false;
  const UavSimBuffers &b = h->buf;
  const void *ptrs[] = {b.ux, b.uy, b.uh, b.ua, b.tx, b.ty, b.th, b.actions, b.obs, b.rew4};
  for (const void *q : ptrs)
    if (reinterpret_cast<uintptr_t>(q) & 15) return false;
  return true;
}

// one step over the env range [e0, e0+cnt) on stream st
// `rng`: the small-swarm kernel can draw the random policy's actions in place (seed, step) instead of reading them
// Automatic choice for small swarms: the two-warp kernel while the batch fits ~2.5 waves of its CTAs (there the step is
// bound by the dependency chain of a thread, which that kernel halves), the generic kernel beyond (throughput-bound: one
// thread per UAV issues ~13 % fewer warp instructions; measured at 65 536 environments of 10 x 10: 0.072 vs 0.082 ms).
// In the rollout loop below the FFI (`rollout`: the policy is drawn inside this kernel and the launches overlap through
// programmatic dependent launch, one launch per step instead of two) it stays ahead up to ~10 waves (10 x 10, device loop,
// tools/generic_timing.py: 16 384 envs 0.026 vs 0.042 ms, 49 152 envs 0.065 vs 0.068, 65 536 envs 0.086 vs 0.079).
static bool small_path_in_use(const uavsim_t *h, int64_t cnt, bool rollout = false) {
  if (!h->has_small || (h->step_path != 0 && h->step_path != 4)) return false;
  if (h->step_path == 4) return true;
  const int G = small_group(h->kp.n, h->kp.m);
  const int64_t waves2 = rollout ? 20 : 5;  // twice the number of waves
  return (cnt + G - 1) / G <= (int64_t)h->small_grid_max[0] * waves2 / 2;
}
// `pdl`: a rollout loop below the FFI -- the small-swarm kernel is launched with programmatic dependent launch (the
// other step kernels and the PMI kernels launch plainly).
static int launch_step_range(uavsim_t *h, int mode, double coop, int64_t e0, int64_t cnt, int done_flag, cudaStream_t st,
                             bool pdl = false, int rng_on = 0, uint64_t rng_seed = 0, uint32_t rng_step = 0) {
  if (small_path_in_use(h, cnt, rng_on != 0)) {  // groups of environments in two-warp CTAs
    const int v = (h->buf.obs_mask || h->buf.tracker_cnt) ? 1 : 0;
    const int G = small_group(h->kp.n, h->kp.m);
    const int64_t groups = (cnt + G - 1) / G;
    const int grid = (int)(groups < h->small_grid_max[v] ? groups : h->small_grid_max[v]);
    if (pdl) {  // let this grid be scheduled while the previous kernel drains (it waits before its first load)
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(SMALL_NT); cfg.dynamicSmemBytes = 0; cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      const ActEntry *act_c = h->d_act;
      CUDA_TRY(cudaLaunchKernelEx(&cfg, h->small_fn[v], h->kp, h->buf, act_c, e0, cnt, mode, coop, done_flag, h->d_stats, rng_on, rng_seed, rng_step));
    } else {
      h->small_fn[v]<<<grid, SMALL_NT, 0, st>>>(h->kp, h->buf, h->d_act, e0, cnt, mode, coop, done_flag, h->d_stats, rng_on, rng_seed, rng_step);
    }
  } else if (fast_path_usable(h)) {
    const int v = (h->buf.obs_mask || h->buf.tracker_cnt) ? 1 : 0;
    if (h->step_path != 3) {  // per-UAV candidate walks (the default: faster than the tiles once the swarm has spread)
      const int grid = (int)(cnt < h->fast_grid_max[v] ? cnt : h->fast_grid_max[v]);
      h->fast_fn[v]<<<grid, FAST_NT, h->smem_fast[v], st>>>(h->kp, h->buf, h->d_act, e0, cnt, mode, coop, done_flag, h->d_stats);
    } else {                  // all-pairs tiles on the tensor path
      const int grid = (int)(cnt < h->tile_grid_max[v] ? cnt : h->tile_grid_max[v]);
      h->tile_fn[v]<<<grid, TILE_NT, h->smem_tile[v], st>>>(h->kp, h->buf, h->d_act, e0, cnt, mode, coop, done_flag, h->d_stats);
    }
  } else {
    if (h->step_path >= 2) { SET_ERR("uavsim_step: the selected step kernel cannot serve this shape / these buffers (64 x 64 kernels need 16-byte aligned arrays)"); return UAVSIM_ERR_UNSUPPORTED; }
    const int64_t ngroups = (cnt + h->epb - 1) / h->epb;
    const int grid = (int)(ngroups < h->grid_max ? ngroups : h->grid_max);
    h->step_fn[h->buf.obs_mask ? 1 : 0]<<<grid, h->nt, h->smem_step, st>>>(h->kp, h->buf, h->d_dth, e0, cnt, h->epb, mode, coop, done_flag, h->d_stats);
  }
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  if (mode == UAVSIM_MODE_PMI && coop != 0.0) return pmi_launch(h, e0, cnt, coop, st, false);
  return 0;
}

static int check_step_args(uavsim_t *h, int mode, double coop, const char *who) {
  int rc = check_bound(h, who);
  if (rc) return rc;
  if (mode != UAVSIM_MODE_SELF && mode != UAVSIM_MODE_MEAN && mode != UAVSIM_MODE_PMI) { SET_ERR("%s: bad mode %d", who, mode); return UAVSIM_ERR_ARG; }
  if (mode == UAVSIM_MODE_PMI && coop != 0.0) {
    if (!h->has_pmi) { SET_ERR("%s: mode PMI needs uavsim_set_pmi_weights first", who); return UAVSIM_ERR_NO_PMI; }
    if (!h->buf.raw || !h->buf.nbr_bits) { SET_ERR("%s: mode PMI needs the raw and nbr_bits buffers", who); return UAVSIM_ERR_UNBOUND; }
  }
  return 0;
}

extern "C" int uavsim_step(uavsim_t *h, int mode, double coop, void *stream) {
  int rc = check_step_args(h, mode, coop, "uavsim_step");
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  h->t++;
  const int done = (h->hp.num_steps > 0 && h->t >= h->hp.num_steps) ? 1 : 0;
  return launch_step_range(h, mode, coop, 0, h->E, done, (cudaStream_t)stream);
}

// Random-policy rollout without a host round trip per step (BASELINE configs[1]: "random-policy actions, env step +
// reward only"): nsteps x (action draw, step) queued back to back on `stream`.  At 4 096 small environments a step
// kernel lasts a few microseconds, less than one interpreter-level call, so the loop has to live below the FFI.
extern "C" int uavsim_run_random_policy(uavsim_t *h, int mode, double coop, uint64_t seed, int64_t first_step,
                                        int64_t nsteps, void *stream) {
  int rc = check_step_args(h, mode, coop, "uavsim_run_random_policy");
  if (rc) return rc;
  if (nsteps < 0) { SET_ERR("uavsim_run_random_policy: nsteps < 0"); return UAVSIM_ERR_ARG; }
  for (int64_t k = 0; k < nsteps; k++) {
    if (small_path_in_use(h, h->E, true)) {  // the draw happens inside the step kernel: one launch per step
      CUDA_TRY(cudaSetDevice(h->device));
      h->t++;
      const int done = (h->hp.num_steps > 0 && h->t >= h->hp.num_steps) ? 1 : 0;
      rc = launch_step_range(h, mode, coop, 0, h->E, done, (cudaStream_t)stream, true, 1, seed, (uint32_t)(first_step + k));
      if (rc) return rc;
      continue;
    }
    rc = uavsim_random_actions(h, seed, first_step + k, stream);
    if (rc) return rc;
    rc = uavsim_step(h, mode, coop, stream);
    if (rc) return rc;
  }
  return 0;
}

// Learned-policy rollout below the FFI: nsteps x (policy launch, step) queued back to back.  The handle's bound
// obs / actions / rew4 / covered pointers are pointed at the trajectory slots of each step (the kernels take the buffer
// struct by value, so this costs nothing) and restored before returning.  The step kernel is chosen exactly as
// uavsim_step chooses it -- not with the wider small-kernel range of the random-policy loop, whose draw is fused into
// that kernel -- so every output is bit-identical to the per-step calls.
extern "C" int uavsim_run_policy(uavsim_t *h, int mode, double coop, const UavSimPolicyWeights *w, uint64_t seed,
                                 uint64_t first_counter, int64_t nsteps, const UavSimTrajectory *traj, void *stream) {
  const char *who = "uavsim_run_policy";
  int rc = check_step_args(h, mode, coop, who);
  if (rc) return rc;
  if (nsteps < 0) { SET_ERR("%s: nsteps < 0", who); return UAVSIM_ERR_ARG; }
  rc = policy_check_weights(w, who);
  if (rc) return rc;
  if (w->n_actions != h->kp.na) { SET_ERR("%s: the policy has %d actions, the environment na = %d", who, w->n_actions, h->kp.na); return UAVSIM_ERR_ARG; }
  const UavSimTrajectory tr = traj ? *traj : UavSimTrajectory{nullptr, nullptr, nullptr, nullptr};
  if ((reinterpret_cast<uintptr_t>(tr.obs) & 15) != 0) { SET_ERR("%s: trajectory obs must be 16-byte aligned", who); return UAVSIM_ERR_ARG; }
  const UavSimBuffers home = h->buf;
  const int64_t E = h->E, en = E * h->kp.n;
  auto bind_slot = [&](int64_t k) {
    h->buf.obs = tr.obs ? tr.obs + (k + 1) * en * 12 : home.obs;
    h->buf.actions = tr.actions ? tr.actions + k * en : home.actions;
    h->buf.rew4 = tr.rew4 ? tr.rew4 + k * 4 * en : home.rew4;
    h->buf.covered = tr.covered ? tr.covered + k * E : home.covered;
  };
  if (h->step_path == 2 || h->step_path == 3) {  // the 64 x 64 kernels need every array 16-byte aligned
    bool ok = true;
    for (int64_t k = 0; k < nsteps && k < 4; k++) {  // (slot offsets are multiples of 4 bytes: alignment repeats after 4)
      bind_slot(k);
      ok = ok && fast_path_usable(h);
    }
    h->buf = home;
    if (!ok) {
      SET_ERR("%s: the selected step kernel needs 16-byte aligned trajectory slots (E*n %% 4 == 0 for actions)", who);
      return UAVSIM_ERR_UNSUPPORTED;
    }
  }
  if (mode == UAVSIM_MODE_PMI && coop != 0.0) {
    rc = pmi_servable(h);
    if (rc) return rc;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const PolicyDev W = policy_dev(w);
  PolicyLaunch L;
  rc = policy_plan(en, W, true, h->device, &L);
  if (rc) return rc;

  cudaStream_t st = (cudaStream_t)stream;
  if (tr.obs) CUDA_TRY(cudaMemcpyAsync(tr.obs, home.obs, sizeof(float) * en * 12, cudaMemcpyDeviceToDevice, st));
  for (int64_t k = 0; k < nsteps && rc == 0; k++) {
    const float *obs_k = tr.obs ? tr.obs + k * en * 12 : home.obs;
    bind_slot(k);
    // The first policy launch follows the caller's own work (which may have just written the weights): a plain launch.
    // Later ones follow this loop's step or PMI kernel and may start early.
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)L.blocks); cfg.blockDim = dim3(POLICY_NT); cfg.dynamicSmemBytes = L.smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = k > 0 ? 1 : 0;
    cfg.attrs = at; cfg.numAttrs = 1;
    float *no_probs = nullptr;
    cudaError_t e = cudaLaunchKernelEx(&cfg, L.fn, obs_k, en, W, seed, first_counter + (uint64_t)k, h->buf.actions, no_probs);
    if (e != cudaSuccess) { SET_ERR("%s: policy launch failed: %s", who, cudaGetErrorString(e)); rc = (int)e; break; }
    h->launches++;
    h->t++;
    const int done = (h->hp.num_steps > 0 && h->t >= h->hp.num_steps) ? 1 : 0;
    rc = launch_step_range(h, mode, coop, 0, E, done, st, true);
  }
  h->buf = home;
  if (rc || nsteps == 0) return rc;
  // the bound buffers end as the per-step calls leave them: the last step's outputs and actions
  if (tr.obs) CUDA_TRY(cudaMemcpyAsync(home.obs, tr.obs + nsteps * en * 12, sizeof(float) * en * 12, cudaMemcpyDeviceToDevice, st));
  if (tr.actions) CUDA_TRY(cudaMemcpyAsync(home.actions, tr.actions + (nsteps - 1) * en, sizeof(int32_t) * en, cudaMemcpyDeviceToDevice, st));
  if (tr.rew4) CUDA_TRY(cudaMemcpyAsync(home.rew4, tr.rew4 + (nsteps - 1) * 4 * en, sizeof(float) * 4 * en, cudaMemcpyDeviceToDevice, st));
  if (tr.covered) CUDA_TRY(cudaMemcpyAsync(home.covered, tr.covered + (nsteps - 1) * E, sizeof(int32_t) * E, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// Queues one host-buffer step over `chunks` environment ranges on the three internal streams and returns without
// waiting.  Per chunk: actions up (s_in) -> step kernel (s_comp) -> outputs down (s_out).  Across consecutive calls the
// same chunk of the NEXT step is ordered behind this one's by events: its upload behind this kernel (the kernel reads
// the action array), its kernel behind this download (the kernel overwrites the output arrays), so the download of
// step t -- the link is the bottleneck: 268.7 MB at 64 x 64 x 65 536 -- overlaps upload and kernels of step t+1.
static int step_host_queue(uavsim_t *h, int mode, double coop, const int32_t *h_actions, float *h_obs, float *h_rew4,
                           int32_t *h_covered, int chunks, void *stream, const char *who) {
  int rc = check_step_args(h, mode, coop, who);
  if (rc) return rc;
  if (!h_actions) { SET_ERR("%s: h_actions is NULL", who); return UAVSIM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(h->device));
  if (chunks < 1) chunks = 1;
  if (chunks > 16) chunks = 16;
  if ((int64_t)chunks > h->E) chunks = (int)h->E;
  if (h->host_chunks && h->host_chunks != chunks) {  // other chunk boundaries: the per-chunk events no longer line up
    CUDA_TRY(cudaStreamSynchronize(h->s_out));
    CUDA_TRY(cudaStreamSynchronize(h->s_comp));
  }
  h->host_chunks = chunks;
  const int n = h->kp.n;
  const int64_t E = h->E;
  h->t++;
  const int done = (h->hp.num_steps > 0 && h->t >= h->hp.num_steps) ? 1 : 0;
  // order after whatever the caller queued on its stream
  CUDA_TRY(cudaEventRecord(h->ev_user, (cudaStream_t)stream));
  CUDA_TRY(cudaStreamWaitEvent(h->s_in, h->ev_user, 0));
  CUDA_TRY(cudaStreamWaitEvent(h->s_comp, h->ev_user, 0));
  CUDA_TRY(cudaStreamWaitEvent(h->s_out, h->ev_user, 0));
  for (int c = 0; c < chunks; c++) {
    const int64_t e0 = E * c / chunks, e1 = E * (c + 1) / chunks, cnt = e1 - e0;
    if (h->host_steps_queued) CUDA_TRY(cudaStreamWaitEvent(h->s_in, h->ev_comp[c], 0));   // previous kernel has read its actions
    CUDA_TRY(cudaMemcpyAsync(h->buf.actions + e0 * n, h_actions + e0 * n, sizeof(int32_t) * cnt * n, cudaMemcpyHostToDevice, h->s_in));
    CUDA_TRY(cudaEventRecord(h->ev_in[c], h->s_in));
    CUDA_TRY(cudaStreamWaitEvent(h->s_comp, h->ev_in[c], 0));
    if (h->host_steps_queued) CUDA_TRY(cudaStreamWaitEvent(h->s_comp, h->ev_out[c], 0));  // previous outputs have left the device
    rc = launch_step_range(h, mode, coop, e0, cnt, done, h->s_comp);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(h->ev_comp[c], h->s_comp));
    CUDA_TRY(cudaStreamWaitEvent(h->s_out, h->ev_comp[c], 0));
    if (h_obs)
      CUDA_TRY(cudaMemcpyAsync(h_obs + e0 * n * 12, h->buf.obs + e0 * n * 12, sizeof(float) * cnt * n * 12, cudaMemcpyDeviceToHost, h->s_out));
    if (h_rew4)  // the chunk's rows of the four reward planes [4][E][n]: one strided copy (pitch = one plane)
      CUDA_TRY(cudaMemcpy2DAsync(h_rew4 + e0 * n, sizeof(float) * E * n, h->buf.rew4 + e0 * n, sizeof(float) * E * n,
                                 sizeof(float) * cnt * n, 4, cudaMemcpyDeviceToHost, h->s_out));
    if (h_covered)
      CUDA_TRY(cudaMemcpyAsync(h_covered + e0, h->buf.covered + e0, sizeof(int32_t) * cnt, cudaMemcpyDeviceToHost, h->s_out));
    CUDA_TRY(cudaEventRecord(h->ev_out[c], h->s_out));
  }
  CUDA_TRY(cudaEventRecord(h->ev_done[h->host_steps_queued & 1], h->s_out));
  h->host_steps_queued++;
  return 0;
}

extern "C" int uavsim_step_host(uavsim_t *h, int mode, double coop, const int32_t *h_actions, float *h_obs,
                                float *h_rew4, int32_t *h_covered, int chunks, void *stream) {
  const int rc = step_host_queue(h, mode, coop, h_actions, h_obs, h_rew4, h_covered, chunks, stream, "uavsim_step_host");
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(h->s_out));
  CUDA_TRY(cudaStreamSynchronize(h->s_comp));
  return 0;
}

extern "C" int uavsim_step_host_async(uavsim_t *h, int mode, double coop, const int32_t *h_actions, float *h_obs,
                                      float *h_rew4, int32_t *h_covered, int chunks, void *stream, int64_t *ticket) {
  const int rc = step_host_queue(h, mode, coop, h_actions, h_obs, h_rew4, h_covered, chunks, stream, "uavsim_step_host_async");
  if (rc) return rc;
  if (ticket) *ticket = h->host_steps_queued - 1;
  return 0;
}

extern "C" int uavsim_step_host_wait(uavsim_t *h, int64_t ticket) {
  if (!h) { SET_ERR("uavsim_step_host_wait: NULL handle"); return UAVSIM_ERR_ARG; }
  if (ticket < 0 || ticket >= h->host_steps_queued) { SET_ERR("uavsim_step_host_wait: ticket %lld was never issued", (long long)ticket); return UAVSIM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(h->device));
  // (two event slots: if later steps reused this one, the wait covers them too -- the streams run in order)
  CUDA_TRY(cudaEventSynchronize(h->ev_done[ticket & 1]));
  return 0;
}

extern "C" int uavsim_episode_stats(uavsim_t *h, double out[8], void *stream) {
  if (!h || !out) { SET_ERR("uavsim_episode_stats: NULL argument"); return UAVSIM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  uavsim_stats_reduce_kernel<<<1, 256, 0, st>>>(h->d_stats, h->stat_slots, h->d_stats8);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(h->h_stats8, h->d_stats8, sizeof(double) * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (int k = 0; k < 8; k++) out[k] = h->h_stats8[k];
  return 0;
}

