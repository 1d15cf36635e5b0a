// pmi_tc_kernel.cuh -- PMI reciprocal reward on the 5th-generation tensor cores (tcgen05, sm_100a), H = 128.
//
// Same contract as uavsim_pmi_kernel (pmi_kernel.cuh): for every ordered neighbour pair (i, j) of an environment
// the folded PMINetwork (src/models/PMINet.py:41-62) maps la_i * la_j (12 values) to a logit; a float32 softmax
// over each UAV's neighbours mixes their raw rewards (src/agent/uav.py:262-291).
//
// Mapping.  One CTA per SM, persistent over groups of environments, warp-specialised:
//   warp 0 (one elected lane)  issues every tcgen05.mma (kind::tf32, M = 128, N = 128, K = 8) and the commits.
//   warp 9 (one elected lane)  streams the fc1 weight chunks into a shared-memory ring (cp.async.bulk, TMA engine).
//   warps 1..8 (256 threads)   producers.  A SET is two 128-row tiles; thread (lane quarter w%4, unit half (w-1)/4)
//                              owns row r of BOTH tiles (same TMEM lane, different columns) and half of the units of a
//                              stage: the two rows ride in the two halves of the packed fp32 instructions, so every
//                              layer-0 weight fetched from shared memory serves two rows.  The same threads build the
//                              rows and later do the epilogue.
// The roles meet only through mbarriers (A-ready / B-full / stage-free / accumulators-full / accumulators-free) over
// 4-stage rings with a static schedule; there is no CTA-wide barrier inside a set.
// The 384 -> 128 layer is a [128 x 384] x [384 x 128] GEMM per tile, fp32 accumulators in tensor memory.
// Tensor memory map (512 columns): accumulators of the two tiles in columns 0..255; the A operand lives in TENSOR
// MEMORY too (tcgen05.mma with A from TMEM), columns 256..511 = 4 stages x 2 tiles x {hi k0-7, hi k8-15, lo k0-7,
// lo k8-15}: the producers write their layer-0 activations with tcgen05.st straight from registers.  With A in shared
// memory the three MMAs of a K-slice read 24 KB of operands (A 4 KB + B 4 KB each) and the producers store another
// 8 KB: the shared-memory pipe, not the tensor pipe, was the limit (66 % busy at 57 % tensor activity); now only the
// B operand (12 KB per slice) comes from shared memory.
// Precision: single-pass TF32 (10-bit mantissa) misses the 1e-5 bar (SURVEY.md section 7), so both operands are split
// x = hi + lo (hi = tf32(x), lo = tf32(x - hi)) and every K-slice runs three MMAs hi*hi + lo*hi + hi*lo -- fp32-class
// products, fp32 accumulation.
//   A (activations after layer 0): block-diagonal 12 -> 384, <= 5 FMAs per unit, two units per packed FFMA2; row r of a
//     tile is TMEM lane r, one 32-bit column per K element.
//   B (fc1 weights): pre-split and pre-arranged on the host in the canonical K-major no-swizzle UMMA layout
//     byte(o, k) = (k/4)*2048 + (o/8)*128 + (o%8)*16 + (k%4)*4   (8x16-byte core matrices, LBO 2048, SBO 128),
//     one 16 KB block (hi | lo) per 16-unit chunk = one bulk copy, mbarrier complete_tx.
// Epilogue: tcgen05.ld (32 lanes x 32 columns per warp and instruction) -> bias + ReLU -> dot with fc2, the two
// threads of a row take 64 columns each -> logit in shared memory; then softmax + mix per UAV.
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>

#ifndef TC_WAIT_HINT
#define TC_WAIT_HINT 20000u
#endif
#define TC_SET 2             // tiles per set = accumulators in tensor memory (2 x 128 columns)
#ifndef TC_PARTS
#define TC_PARTS 2           // producer threads per pair row: each takes 16 / TC_PARTS units of a stage and 128 / TC_PARTS accumulator
#endif                       //   columns.  (4 was measured: issue slots 52 % -> 67 % busy, but 27 % more instructions: same time)
#define TC_NP (128 * TC_PARTS)  // producer / epilogue threads (warps 1 .. TC_NP/32): row r of both tiles x one part of the units
#define TC_NT (TC_NP + 64)   // + warp 0 = MMA issue, last warp = fc1 chunk loader (TMA)
#define TC_H 128             // largest hidden size the kernel is instantiated for (64 and 128): sizes the shared-memory layout
#define TC_H3 384
// Operand format of the 384 -> 128 GEMM.  TC_F16 = 1 (default): both operands split into fp16 hi + lo (11 + 11 mantissa bits,
// the same budget as the TF32 split) and multiplied with kind::f16 MMAs, K = 16 per instruction: half the tensor instructions,
// half the shared-memory operand bytes and half the tensor-memory columns of the TF32 variant (TC_F16 = 0, K = 8), for the
// same three products hi*hi + lo*hi + hi*lo.  fc1 is pre-scaled by TC_WSCALE (a power of two, undone in the epilogue) so the
// lo parts of the weights stay out of fp16's subnormal range.
#ifndef TC_F16
#define TC_F16 1
#endif
#if TC_F16
#ifndef TC_KC
#define TC_KC 32             // hidden units per ring stage = two K = 16 MMAs per product (16 was measured: the per-stage
#endif                       //   hand-shake is a quarter of the producers' instructions; 32 halves it)
#define TC_NS (TC_KC == 32 ? 3 : 4)   // stages of the operand rings (an even number of ring turns per set: 12 / 3, 24 / 4)
#define TC_A_BYTES (128 * TC_KC * 2)  // one 128 x TC_KC fp16 weight block (hi or lo)
#define TC_ACOLS (2u * TC_KC)         // TMEM columns per A stage: 2 tiles x (TC_KC/2 hi + TC_KC/2 lo), two fp16 per column
#define TC_MMA_K 16
#define TC_WSCALE 256.0f
#else
#define TC_KC 16             // hidden units per ring stage = two K = 8 MMAs per product
#define TC_NS 4
#define TC_A_BYTES 8192      // one 128 x 16 fp32 weight block (hi or lo)
#define TC_ACOLS 64u         // TMEM columns per A stage: 2 tiles x (16 hi + 16 lo)
#define TC_MMA_K 8
#define TC_WSCALE 1.0f
#endif
#define TC_NCHUNK (TC_H3 / TC_KC)
#define TC_UPT (TC_KC / TC_PARTS)  // units of a stage per producer thread
#if !TC_F16 && TC_PARTS != 2
#error "the TF32 variant keeps two producer threads per row: build it with -DTC_F16=0 -DTC_PARTS=2"
#endif
#define TC_STAGE_BYTES (2 * TC_A_BYTES)  // B_hi + B_lo
// Per-unit rebalancing of the uploaded weights (uavsim_set_pmi_weights): row u of layer 0 is scaled by a power of two so
// that max(b0_u, 0) + PMI_X_NOM * sum_k |w0_uk| lies in [2^PMI_BAL_T, 2^(PMI_BAL_T+1)), column u of fc1 by the inverse.  This puts
// the fp16 activations of inputs up to PMI_X_NOM below 2^(PMI_BAL_T+1) and leaves fc1 times TC_WSCALE room up to 65504:
// with T = 8 and X = 16 the tensor path holds pair-row inputs up to ~2 000 and a folded fc1 weight up to ~1 000 on the
// units of an untrained network (DESIGN.md section 3.2).
#define PMI_BAL_T 8
#define PMI_X_NOM 16.0
#define TC_ACOL0 256u        // first TMEM column of the A ring
#define TC_AMAX 512          // UAVs per environment group
#define TC_PMAX 16384        // neighbour pairs per environment group (logits stay in shared memory until the softmax)

// instruction descriptor: D = F32, A = B = TF32, K-major both, N = 128 (>>3 at bit 17), M = 128 (>>4 at bit 24)
// (kind::f16: A = B = F16 is format 0)
#if TC_F16
#define TC_IDESC_BASE ((1u << 4) | (0u << 7) | (0u << 10) | ((128u >> 4) << 24))
#else
#define TC_IDESC_BASE ((1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 4) << 24))
#endif

struct TcSmem {  // byte offsets inside dynamic shared memory (base is 1024-byte aligned)
  static constexpr uint32_t stage = 0;                                   // TC_NS x TC_STAGE_BYTES (fc1 chunks only)
  static constexpr uint32_t obs = TC_NS * TC_STAGE_BYTES;                   // float [AMAX*12]
  static constexpr uint32_t raw = obs + TC_AMAX * 12 * 4;                // double [AMAX]
  static constexpr uint32_t nbr = raw + TC_AMAX * 8;                     // uint64 [AMAX*2]
  static constexpr uint32_t off = nbr + TC_AMAX * 16;                    // uint32 [AMAX+4]
  static constexpr uint32_t logit = off + (TC_AMAX + 4) * 4;             // float [PMAX]
  static constexpr uint32_t w0 = logit + TC_PMAX * 4;                    // float [192*12]: per unit pair, bias and 5 weights interleaved
  static constexpr uint32_t part = w0 + (TC_H3 / 2) * 12 * 4;          // float [TC_PARTS-1][2][128] fc2 partial dots of the other threads of a row
  static constexpr uint32_t b1 = part + (TC_PARTS - 1) * TC_SET * 128 * 4;   // float [128]
  static constexpr uint32_t w2 = b1 + TC_H * 4;                          // float [128]
  static constexpr uint32_t bar = w2 + TC_H * 4;                         // 3 x TC_NS + 2 mbarriers + tmem pointer
  static constexpr uint32_t total = bar + 128;
};
static_assert(TcSmem::total <= 232448, "tensor PMI kernel: shared memory over the 227 KB per-CTA limit");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded wait: a barrier that never completes (a descriptor bug) traps instead of hanging the GPU.  The suspend-time
// hint lets the hardware park the warp until the phase completes instead of re-polling: spinning producers would
// otherwise take issue slots from the MMA warp and from the producers that still have work.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; spin++) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(TC_WAIT_HINT)
        : "memory");
    if (spin > (1u << 22)) __trap();
  }
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo) {
  // K-major, no swizzle: start address, LBO = 2048 B (between the two 16-byte K halves of an MMA),
  // SBO = 128 B (between 8-row groups), descriptor version 1 (Blackwell)
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(128u >> 4) << 32) |
         (1ull << 46);
}
// The MMA warp and the loader warp run their loops with all 32 lanes converged (warp-uniform control flow and operands,
// so descriptors and addresses live in uniform registers) and predicate the single-thread instructions on an elected lane INSIDE the
// asm: a divergent `if (lane == 0)` around them makes the compiler wrap every tcgen05.mma in an ELECT / R2UR waterfall
// loop, ~16 issue slots per MMA, which made the one issuing thread the bottleneck of the kernel.  TC_ABL_* are
// profiling switches (one MMA per K-slice / no layer-0 work) used for the ablations quoted in DESIGN.md.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand read from tensor memory (lane = row, one column per tf32 element)
__device__ __forceinline__ void umma_tf32_ts_p(uint32_t lead, uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t accumulate, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
#if TC_F16
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
#else
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
#endif

      ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
// registers -> tensor memory: lane l of the warp writes its 8 values to TMEM lane (quarter base + l), columns c .. c+7
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float *v) {
  const uint32_t *u = reinterpret_cast<const uint32_t *>(v);
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st2(uint32_t taddr, const uint32_t *u) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(u[0]), "r"(u[1]) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t *u) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]) : "memory");
}
// ReLU + split of the layer-0 pre-activations of two neighbouring units (u, u') of the thread's two rows:
// acc = {row 0, row 1} of unit u, acc2 = the same of unit u'.  hi is the value truncated to 11 significant bits (one AND), so
// v - hi is exact, has the sign of v, and both conversions are exact up to the final rounding of lo to 11 bits.  The ReLU
// rides on the conversions (.relu: a negative v gives hi = lo = 0); .satfinite keeps an activation beyond fp16's range finite
// (an activation that large comes from a pair row whose inputs exceed PmiTcDev::x_safe; the kernel counts those rows in
// the statistics, pmi_rows_out_of_range, instead of failing).  Outputs: packed {u, u'} per row (lower K index in the low half).
__device__ __forceinline__ void tc_relu_split(uint64_t acc, uint64_t acc2, uint32_t &hi_r0, uint32_t &lo_r0, uint32_t &hi_r1, uint32_t &lo_r1) {
  const uint64_t m = 0xffffe000ffffe000ull;
  const uint64_t h = acc & m, h2 = acc2 & m;
  uint64_t l, l2;
  asm("sub.f32x2 %0, %1, %2;" : "=l"(l) : "l"(acc), "l"(h));
  asm("sub.f32x2 %0, %1, %2;" : "=l"(l2) : "l"(acc2), "l"(h2));
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi_r0) : "f"(__uint_as_float((uint32_t)h2)), "f"(__uint_as_float((uint32_t)h)));
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo_r0) : "f"(__uint_as_float((uint32_t)l2)), "f"(__uint_as_float((uint32_t)l)));
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi_r1) : "f"(__uint_as_float((uint32_t)(h2 >> 32))), "f"(__uint_as_float((uint32_t)(h >> 32))));
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo_r1) : "f"(__uint_as_float((uint32_t)(l2 >> 32))), "f"(__uint_as_float((uint32_t)(l >> 32))));
}
__device__ __forceinline__ void umma_commit_p(uint32_t lead, uint32_t bar) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
               "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar), "r"(lead) : "memory");
}
__device__ __forceinline__ void load_chunk_p(uint32_t lead, uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\t"
               "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %2;\n\t"
               "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "r"(lead) : "memory");
}
// round to TF32 (10 mantissa bits), nearest with ties away from zero like cvt.rna.tf32.f32, for finite inputs: two
// integer instructions (the cvt expands to an inf/nan test plus the same arithmetic)
__device__ __forceinline__ float tf32_rna(float v) {
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ uint64_t tc_pack2(float lo, float hi) {
  return (uint64_t)__float_as_uint(lo) | ((uint64_t)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ uint64_t tc_fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {
  uint32_t *u = reinterpret_cast<uint32_t *>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
        "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
        "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct PmiTcDev {
  const float *w0, *b0, *b1, *w2;  // [384*5] [384] [128] [128] folded fp32
  const float *w1_tiles;           // [24][2][128 x 16] fc1 pre-split (hi | lo) in the UMMA layout
  float b2;
  float x_safe;                    // largest max_k |x_k| of a pair row whose layer-0 activations fit fp16 (host-computed)
};

template <int H>   // hidden size of the PMI network: 128 (src/configs/*.yaml) or 64 (the default of PMINetwork's constructor)
__global__ void __launch_bounds__(TC_NT, 1)
uavsim_pmi_tc_kernel(const KParams P, const UavSimBuffers B, const PmiTcDev W, int64_t env_begin, int64_t env_count,
                     int G, double coop, long long *__restrict__ stats) {
  static_assert(H == 64 || H == 128, "tensor PMI kernel: hidden size 64 or 128");
  constexpr int H3 = 3 * H, NCHUNK = H3 / TC_KC;
  constexpr uint32_t A_BYTES = (uint32_t)H * TC_KC * (TC_F16 ? 2 : 4);   // one H x TC_KC weight block (hi or lo)
  constexpr uint32_t LBO = (uint32_t)H * 16u;                            // bytes between core-matrix columns along K
  constexpr uint32_t IDESC = (TC_IDESC_BASE) | ((uint32_t)(H >> 3) << 17);
  extern __shared__ __align__(1024) unsigned char smem[];
  const int n = P.n, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool producer = warp >= 1 && warp <= TC_NP / 32;   // warp 0 = MMA issue, last warp = weight loader
  // producers: hardware warp w may only touch TMEM lanes 32*(w%4)..+31, so rows follow the warp id
  const int row = 32 * (warp & 3) + lane, half = (warp - 1) >> 2, pt = tid - 32;  // half: which part of the units / columns (0 .. TC_PARTS-1)
  float *s_obs = reinterpret_cast<float *>(smem + TcSmem::obs);
  double *s_raw = reinterpret_cast<double *>(smem + TcSmem::raw);
  uint64_t *s_nbr = reinterpret_cast<uint64_t *>(smem + TcSmem::nbr);
  uint32_t *s_off = reinterpret_cast<uint32_t *>(smem + TcSmem::off);
  float *s_logit = reinterpret_cast<float *>(smem + TcSmem::logit);
  float *s_w0 = reinterpret_cast<float *>(smem + TcSmem::w0);
  float *s_part = reinterpret_cast<float *>(smem + TcSmem::part);
  float *s_b1 = reinterpret_cast<float *>(smem + TcSmem::b1);
  float *s_w2 = reinterpret_cast<float *>(smem + TcSmem::w2);
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(smem + TcSmem::bar + 120);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + TcSmem::bar;
  const uint32_t bar_bfull = bar0, bar_aready = bar0 + 8 * TC_NS, bar_free = bar0 + 16 * TC_NS;  // [TC_NS]: one per stage
  const uint32_t bar_accfull = bar0 + 24 * TC_NS, bar_accfree = bar_accfull + 8;

#pragma unroll 4
  for (int k = tid; k < (H3 / 2) * 12; k += TC_NT) {  // unit pair j: {b, b', w0, w0', .. w4, w4'} -> three 128-bit loads
    const int u = 2 * (k / 12) + (k & 1), e = (k % 12) >> 1;
    s_w0[k] = (e == 0) ? W.b0[u] : W.w0[u * 5 + e - 1];
  }
  for (int k = tid; k < H; k += TC_NT) { s_b1[k] = W.b1[k]; s_w2[k] = W.w2[k]; }
  if (tid == 0) {
    for (int k = 0; k < TC_NS; k++) {
      mbar_init(bar_bfull + 8 * k, 1);              // expect_tx by the loader lane + TMA bytes
      mbar_init(bar_aready + 8 * k, TC_NP / 32);    // one arrive per producer warp
      mbar_init(bar_free + 8 * k, 1);               // tcgen05.commit
    }
    mbar_init(bar_accfull, 1);                      // tcgen05.commit
    mbar_init(bar_accfree, TC_NP / 32);             // one arrive per producer warp
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {  // all of tensor memory: two 128-column fp32 accumulators + the A ring, allocated by one warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *s_tmem;

  // Static ring schedule: a set is TC_NCHUNK = 24 chunks and the rings have TC_NS = 4 stages, so chunk c of every set
  // uses stage c % 4 and it is that stage's (6 * set + c / 4)-th use: the mbarrier phase parity is (c / 4) & 1 in
  // every set, and all shared-memory / tensor-memory addresses are compile-time offsets from the bases.
  static_assert(NCHUNK % (2 * TC_NS) == 0, "ring schedule assumes an even number of ring turns per set");
  uint32_t t = 0;   // sets processed so far by this CTA (phase of the accumulator barriers); same sequence in all roles
  const int64_t ngroups = (env_count + G - 1) / G;
  // Groups beyond the first per CTA come from the launch-wide counter (KParams::fast_ctr, rewound by the last CTA to
  // leave): the pair count of a group follows the swarm's density, so equal group COUNTS are not equal work.  Thread 0
  // draws one group ahead; every role reads the index behind the barrier at the loop top.  The reward sum is a
  // fixed-point count for the same reason as in the step kernels (common.cuh: sf_fx).
  long long fx_r = 0;
  int oor = 0;  // pair rows beyond W.x_safe built by this producer (counted by the threads of unit part 0 only)
  long long *const s_next = reinterpret_cast<long long *>(smem + TcSmem::bar + 112);  // (mbarriers end at +112 at most, the tensor-memory pointer sits at +120)
  long long drawn = 0;
  if (tid == 0 && (int64_t)blockIdx.x < ngroups) drawn = (long long)gridDim.x + (long long)atomicAdd(P.fast_ctr, 1);

  for (int64_t grp = blockIdx.x, grp_next = 0; grp < ngroups; grp = grp_next) {
    const int64_t e0 = env_begin + grp * G;
    const int ne = (int)min((int64_t)G, env_begin + env_count - e0);
    const int A = ne * n;  // UAVs in this group (<= TC_AMAX)
    if (tid == 0) *s_next = drawn;
    __syncthreads();
    grp_next = *s_next;
    if (tid == 0 && grp_next < ngroups) drawn = (long long)gridDim.x + (long long)atomicAdd(P.fast_ctr, 1);
    {  // the group's observations: 48-byte rows, so the block is 16-byte aligned; 128-bit loads, four in flight per
       // thread (a scalar loop waited for every load in turn: 7 % of the kernel at 10 x 10)
      const float4 *src = reinterpret_cast<const float4 *>(B.obs + e0 * n * 12);
      float4 *dst = reinterpret_cast<float4 *>(s_obs);
#pragma unroll 4
      for (int k = tid; k < A * 3; k += TC_NT) dst[k] = __ldg(src + k);
    }
#pragma unroll 2
    for (int a = tid; a < A; a += TC_NT) {
      s_raw[a] = B.raw[e0 * n + a];
      const uint64_t n0 = B.nbr_bits[(e0 * n + a) * 2], n1 = B.nbr_bits[(e0 * n + a) * 2 + 1];
      s_nbr[2 * a] = n0; s_nbr[2 * a + 1] = n1;
      s_off[a + 1] = __popcll(n0) + __popcll(n1);
    }
    __syncthreads();
    if (warp == 1) {  // exclusive scan of the neighbour counts (A <= 512): 16 per lane + warp scan
      const int per = (A + 31) / 32, lo = lane * per;
      uint32_t sum = 0;
      for (int k = 0; k < per; k++) if (lo + k < A) sum += s_off[lo + k + 1];
      uint32_t inc = sum;
      for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
      uint32_t run = inc - sum;
      if (lane == 0) s_off[0] = 0;
      for (int k = 0; k < per; k++) if (lo + k < A) { run += s_off[lo + k + 1]; s_off[lo + k + 1] = run; }
    }
    __syncthreads();
    const int npairs = (int)s_off[A];
    const int ntiles = (npairs + 127) / 128;
    const int nsets = (ntiles + TC_SET - 1) / TC_SET;

    if (warp == 0) {
      // =============================== MMA warp ===============================
      const uint32_t lead = elect_one();
      const int u_nsets = __shfl_sync(0xffffffffu, nsets, 0), u_ntiles = __shfl_sync(0xffffffffu, ntiles, 0);
      const uint32_t u_tmem = __shfl_sync(0xffffffffu, tmem_d, 0);
      for (int set = 0; set < u_nsets; set++, t++) {
        const int nts = min(TC_SET, u_ntiles - set * TC_SET);
        if (t > 0) mbar_wait(bar_accfree, (t - 1) & 1);  // epilogue of the previous set done
#pragma unroll 1
        for (int c4 = 0; c4 < NCHUNK / TC_NS; c4++) {
          const uint32_t par = c4 & 1;
#pragma unroll
          for (int s = 0; s < TC_NS; s++) {
            mbar_wait(bar_aready + 8 * s, par);  // producers have written A (tensor memory)
            mbar_wait(bar_bfull + 8 * s, par);   // weights have landed (shared memory)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // B descriptors differ only in the 14-bit address field: add (byte offset >> 4) to the low word
            const uint64_t dbh0 = umma_desc(sbase + TcSmem::stage + s * TC_STAGE_BYTES, LBO), dbl0 = dbh0 + (A_BYTES >> 4);
#pragma unroll
            for (int q = 0; q < TC_SET; q++) {
              if (q < nts) {
                const uint32_t d_tmem = u_tmem + (uint32_t)H * (uint32_t)q;
                // one MMA consumes K = 16 fp16 (8 TMEM columns of A, two fp16 each) or K = 8 tf32 (8 columns), and two
                // core-matrix columns of B either way
                constexpr int KS = TC_KC / TC_MMA_K;
#pragma unroll
                for (int ks = 0; ks < KS; ks++) {
                  const uint32_t a_hi = u_tmem + TC_ACOL0 + TC_ACOLS * (uint32_t)s + (TC_ACOLS / 2) * (uint32_t)q + 8u * (uint32_t)ks, a_lo = a_hi + TC_ACOLS / 4;
                  const uint64_t dbh = dbh0 + (uint64_t)(ks * 2 * (LBO >> 4)), dbl = dbl0 + (uint64_t)(ks * 2 * (LBO >> 4));
                  umma_tf32_ts_p(lead, d_tmem, a_hi, dbh, (c4 | s | ks) ? 1u : 0u, IDESC);
#ifndef TC_ABL_MMA1
                  umma_tf32_ts_p(lead, d_tmem, a_lo, dbh, 1u, IDESC);
                  umma_tf32_ts_p(lead, d_tmem, a_hi, dbl, 1u, IDESC);
#endif
                }
              }
            }
            umma_commit_p(lead, bar_free + 8 * s);  // both rings' stage s reusable when these MMAs are done
          }
        }
        umma_commit_p(lead, bar_accfull);  // accumulators complete
      }
    } else if (!producer) {
      // =============================== weight loader warp ===============================
      const uint32_t lead = elect_one();
      const int u_nsets = __shfl_sync(0xffffffffu, nsets, 0);
      for (int set = 0; set < u_nsets; set++, t++) {
#pragma unroll 1
        for (int c4 = 0; c4 < NCHUNK / TC_NS; c4++) {
#pragma unroll
          for (int s = 0; s < TC_NS; s++) {
            if (t > 0 || c4 > 0) mbar_wait(bar_free + 8 * s, (c4 & 1) ^ 1);  // the MMAs of the previous use are done
            load_chunk_p(lead, sbase + TcSmem::stage + s * TC_STAGE_BYTES,
                         W.w1_tiles + (size_t)(c4 * TC_NS + s) * (2 * A_BYTES / 4), 2 * A_BYTES, bar_bfull + 8 * s);
          }
        }
      }
    } else {
      // =============================== producers: rows, layer 0, epilogue ===============================
      const uint32_t lane_base = tmem_d + ((uint32_t)((warp & 3) * 32) << 16);
      // this thread's two pair rows of a set (row r of tile 0 and of tile 1): flat pair index -> (UAV a, its k-th
      // neighbour b), x = la_a * la_b (uav.py:280-281); the two rows are packed {row of tile 0, row of tile 1}
      uint64_t xx[12];
      auto build_rows = [&](const int set) {
        float x0[12], x1[12];
        auto build = [&](const int p, float *x) {
          if (p < npairs) {
            int lo = 0, hi = A;  // largest a with off[a] <= p
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_off[mid] <= (uint32_t)p) lo = mid; else hi = mid; }
            const int a = lo;
            int k = p - (int)s_off[a];
            uint64_t w = s_nbr[2 * a];
            int base = (a / n) * n;
            const int c0 = __popcll(w);
            if (k >= c0) { k -= c0; w = s_nbr[2 * a + 1]; base += 64; }
            for (int q = 0; q < k; q++) w &= w - 1;
            const int b = base + __ffsll((long long)w) - 1;
            float mx = 0.f;
#pragma unroll
            for (int q = 0; q < 12; q++) { x[q] = s_obs[a * 12 + q] * s_obs[b * 12 + q]; mx = fmaxf(mx, fabsf(x[q])); }
            oor += (half == 0 && mx > W.x_safe) ? 1 : 0;
          } else {
#pragma unroll
            for (int q = 0; q < 12; q++) x[q] = 0.f;
          }
        };
        build((set * TC_SET) * 128 + row, x0);
        build((set * TC_SET + 1) * 128 + row, x1);
#pragma unroll
        for (int q = 0; q < 12; q++) xx[q] = tc_pack2(x0[q], x1[q]);
      };
      if (nsets > 0) build_rows(0);
      for (int set = 0; set < nsets; set++, t++) {
        const bool live1 = set * TC_SET + 1 < ntiles;  // warp-uniform: the set's second tile exists (the first always does)

        // ---- layer 0 per ring stage of 16 hidden units; this thread computes the 8 units of K-slice `half` for its
        //      two rows and writes them (hi and lo) into the stage's tensor-memory columns.  The three input branches
        //      (communication 5, observation 4, boundary/state 3 inputs; PMINet.py:45-58, BN folded) are unrolled
        //      so the rows stay in registers; each branch covers 8 chunks.
#if !TC_F16
        const uint32_t a_lane = lane_base + TC_ACOL0 + 8u * (uint32_t)half;
#endif
        auto run_chunk = [&](const int c, const uint64_t *xin, const int dim) {
          const uint32_t s = c % TC_NS, c4 = c / TC_NS;
          if (t > 0 || c4 > 0) {  // MMAs that read this stage have completed
            mbar_wait(bar_free + 8 * s, (c4 & 1) ^ 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
#ifdef TC_ABL_NOPROD
          if (c < 0)
#endif
          {
            float h0[TC_UPT], l0[TC_UPT], h1[TC_UPT], l1[TC_UPT];
#pragma unroll
            for (int e = 0; e < TC_UPT; e += 2) {  // unit pair (u, u'): weights interleaved {b b' w0 w0' | w1 w1' w2 w2' | w3 w3' w4 w4'}
              const float4 *wp = reinterpret_cast<const float4 *>(s_w0 + ((c * TC_KC + half * TC_UPT + e) >> 1) * 12);
              const float4 q0 = wp[0], q1 = wp[1];
              uint64_t acc = tc_pack2(q0.x, q0.x), acc2 = tc_pack2(q0.y, q0.y);     // {row 0, row 1} of unit u / u'
              acc = tc_fma2(tc_pack2(q0.z, q0.z), xin[0], acc);   acc2 = tc_fma2(tc_pack2(q0.w, q0.w), xin[0], acc2);
              acc = tc_fma2(tc_pack2(q1.x, q1.x), xin[1], acc);   acc2 = tc_fma2(tc_pack2(q1.y, q1.y), xin[1], acc2);
              acc = tc_fma2(tc_pack2(q1.z, q1.z), xin[2], acc);   acc2 = tc_fma2(tc_pack2(q1.w, q1.w), xin[2], acc2);
              if (dim > 3) {
                const float4 q2 = wp[2];
                acc = tc_fma2(tc_pack2(q2.x, q2.x), xin[3], acc); acc2 = tc_fma2(tc_pack2(q2.y, q2.y), xin[3], acc2);
                if (dim > 4) { acc = tc_fma2(tc_pack2(q2.z, q2.z), xin[4], acc); acc2 = tc_fma2(tc_pack2(q2.w, q2.w), xin[4], acc2); }
              }
#if TC_F16
              // units (u, u') are neighbours along K: one packed fp16 pair per tile
              tc_relu_split(acc, acc2, reinterpret_cast<uint32_t *>(h0)[e >> 1], reinterpret_cast<uint32_t *>(l0)[e >> 1],
                            reinterpret_cast<uint32_t *>(h1)[e >> 1], reinterpret_cast<uint32_t *>(l1)[e >> 1]);
            }
            {  // this thread's TC_UPT units = TC_UPT / 2 columns of the stage: hi | lo of tile 0, hi | lo of tile 1
              const uint32_t a4 = lane_base + TC_ACOL0 + (uint32_t)(TC_UPT / 2) * (uint32_t)half + TC_ACOLS * s;
              auto st = [](uint32_t addr, const float *v) {
                const uint32_t *u = reinterpret_cast<const uint32_t *>(v);
                if (TC_UPT == 16) tmem_st8(addr, v);
                else if (TC_UPT == 8) tmem_st4(addr, u);
                else tmem_st2(addr, u);
              };
              st(a4, h0);
              st(a4 + TC_ACOLS / 4, l0);
              if (live1) {
                st(a4 + TC_ACOLS / 2, h1);
                st(a4 + 3 * TC_ACOLS / 4, l1);
              }
            }
#else
              const float a00 = fmaxf(__uint_as_float((uint32_t)acc), 0.f), a01 = fmaxf(__uint_as_float((uint32_t)(acc >> 32)), 0.f);
              const float a10 = fmaxf(__uint_as_float((uint32_t)acc2), 0.f), a11 = fmaxf(__uint_as_float((uint32_t)(acc2 >> 32)), 0.f);
              h0[e] = tf32_rna(a00); l0[e] = tf32_rna(a00 - h0[e]);              // unit u,  tile 0
              h1[e] = tf32_rna(a01); l1[e] = tf32_rna(a01 - h1[e]);              // unit u,  tile 1
              h0[e + 1] = tf32_rna(a10); l0[e + 1] = tf32_rna(a10 - h0[e + 1]);  // unit u', tile 0
              h1[e + 1] = tf32_rna(a11); l1[e + 1] = tf32_rna(a11 - h1[e + 1]);  // unit u', tile 1
            }
            tmem_st8(a_lane + TC_ACOLS * s, h0);
            tmem_st8(a_lane + TC_ACOLS * s + 16u, l0);
            if (live1) {
              tmem_st8(a_lane + TC_ACOLS * s + 32u, h1);
              tmem_st8(a_lane + TC_ACOLS * s + 48u, l1);
            }
#endif
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_aready + 8 * s);
        };
#pragma unroll 1
        for (int cc = 0; cc < NCHUNK / 3; cc++) run_chunk(cc, xx, 5);
#pragma unroll 1
        for (int cc = NCHUNK / 3; cc < 2 * NCHUNK / 3; cc++) run_chunk(cc, xx + 5, 4);
#pragma unroll 1
        for (int cc = 2 * NCHUNK / 3; cc < NCHUNK; cc++) run_chunk(cc, xx + 9, 3);

        // the rows of the next set are built while the tensor pipe drains the last stages of this one
        if (set + 1 < nsets) build_rows(set + 1);

        // ---- epilogue: bias + ReLU + fc2 (PMINet.py:59-62); the two threads of a row take 64 accumulator columns each
        mbar_wait(bar_accfull, t & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float part[TC_SET] = {0.f, 0.f};
#pragma unroll
        for (int q = 0; q < TC_SET; q++) {
          if (q == 0 || live1) {
#pragma unroll 1
            for (int cb = half * (H / TC_PARTS); cb < (half + 1) * (H / TC_PARTS); cb += 32) {
              float v[32];
              tmem_ld32(lane_base + (uint32_t)H * (uint32_t)q + (uint32_t)cb, v);
              float acc = part[q];
#pragma unroll
              for (int k = 0; k < 32; k++) acc = fmaf(s_w2[cb + k], fmaxf(fmaf(v[k], 1.0f / TC_WSCALE, s_b1[cb + k]), 0.f), acc);
              part[q] = acc;
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_accfree);  // this warp's rows have left tensor memory
        // combine the two halves of each row (producer-only named barrier: warps 0 and 9 are elsewhere)
        if (half) { s_part[(half - 1) * 256 + row] = part[0]; s_part[(half - 1) * 256 + 128 + row] = part[1]; }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_NP) : "memory");
        if (!half) {
#pragma unroll
          for (int q = 0; q < TC_SET; q++) {
            const int p = (set * TC_SET + q) * 128 + row;
            float sum = part[q];
#pragma unroll
            for (int h2 = 0; h2 < TC_PARTS - 1; h2++) sum += s_part[h2 * 256 + q * 128 + row];
            if (p < npairs) s_logit[p] = sum + W.b2;
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_NP) : "memory");
      }
    }
    __syncthreads();

    // ---- softmax over each UAV's neighbours (scipy.special.softmax on float32) and the mix (uav.py:284-290)
    if (producer) {
      for (int a = pt; a < A; a += TC_NP) {
        const uint32_t lo = s_off[a], hi = s_off[a + 1];
        const double raw = s_raw[a];
        double r;
        if (hi > lo) {
          float mx = s_logit[lo];
          for (uint32_t q = lo + 1; q < hi; q++) mx = fmaxf(mx, s_logit[q]);
          float ssum = 0.f;
          for (uint32_t q = lo; q < hi; q++) ssum += expf(s_logit[q] - mx);
          double acc = 0;
          uint32_t q = lo;
          const int base = (a / n) * n;
          for (int hh = 0; hh < 2; hh++) {
            uint64_t w = s_nbr[2 * a + hh];
            while (w) {
              const int j = __ffsll((long long)w) - 1;
              w &= w - 1;
              const float wgt = expf(s_logit[q] - mx) / ssum;
              acc += s_raw[base + 64 * hh + j] * (double)wgt;
              q++;
            }
          }
          r = (1 - coop) * raw + coop * acc;
        } else {
          r = (1 - coop) * raw;
        }
        r = fmin(fmax(r, -1.0), 1.0);
        B.rew4[e0 * n + a] = (float)r;
        fx_r += sf_fx((float)r);
      }
    }
  }
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(512u) : "memory");
  work_counter_leave(P.fast_ctr);
  stats_commit(stats + (size_t)blockIdx.x * STAT_W, fx_r, 0, 0, 0, 0, 0, 0, oor);
}
