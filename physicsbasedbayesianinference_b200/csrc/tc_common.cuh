// PTX wrappers shared by the tcgen05 kernels (k_dense_tc3, k_logistic_tc, k_logistic_tc3): mbarriers, TMA bulk
// copies, tensor-memory allocation / loads / stores, UMMA descriptors and the MMA issue forms used here.
// sm_100a only.
#pragma once

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"

namespace ehmc {

constexpr int TC_M = 128;  // particle rows of one UMMA tile = TMEM lanes

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar_addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(bar_addr), "r"(parity)
      : "memory");
  return ok != 0;
}
// The *_a forms take a precomputed 32-bit shared address: inside a serial evaluation chain the generic -> shared
// conversion (with its S2UR CgaCtaId) would otherwise be re-materialised every time.
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity) {
  while (!mbar_try_wait_a(bar_addr, parity)) {
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_a(smem_u32(bar), parity); }
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  return mbar_try_wait_a(smem_u32(bar), parity);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// one elected lane of a converged warp (lets the compiler keep tcgen05 operands in uniform registers)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// pin() makes a value opaque to the compiler: computed once, kept in a register
__device__ __forceinline__ void pin(uint32_t& x) { asm volatile("" : "+r"(x)); }
__device__ __forceinline__ void pin(uint64_t& x) { asm volatile("" : "+l"(x)); }
__device__ __forceinline__ void pin(float& x) { asm volatile("" : "+f"(x)); }

// ---- tensor memory ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// Loads are issue-only; the matching tmem_wait_ld* takes the loaded registers as read-write operands, so every
// later use of them depends on the wait and the compiler cannot hoist arithmetic above it.
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&u)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_issue2(uint32_t taddr, uint32_t (&u)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_issue(uint32_t taddr, uint32_t (&u)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&u)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]),
                 "+r"(u[8]), "+r"(u[9]), "+r"(u[10]), "+r"(u[11]), "+r"(u[12]), "+r"(u[13]), "+r"(u[14]), "+r"(u[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld8(uint32_t (&u)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld4(uint32_t (&u)[4]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]) : : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&u)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16};" ::"r"(taddr),
      "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
      "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&u)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(u[0]),
               "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&u)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(u[0]), "r"(u[1]),
               "r"(u[2]), "r"(u[3])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// generic N-column wrappers (N = 16, 8 or 4)
template <int N>
__device__ __forceinline__ void tm_ld(uint32_t taddr, uint32_t* u) {
  if constexpr (N == 16) tmem_ld16_issue(taddr, *reinterpret_cast<uint32_t(*)[16]>(u));
  else if constexpr (N == 8) tmem_ld8_issue2(taddr, *reinterpret_cast<uint32_t(*)[8]>(u));
  else tmem_ld4_issue(taddr, *reinterpret_cast<uint32_t(*)[4]>(u));
}
template <int N>
__device__ __forceinline__ void tm_wait(uint32_t* u) {
  if constexpr (N == 16) tmem_wait_ld16(*reinterpret_cast<uint32_t(*)[16]>(u));
  else if constexpr (N == 8) tmem_wait_ld8(*reinterpret_cast<uint32_t(*)[8]>(u));
  else tmem_wait_ld4(*reinterpret_cast<uint32_t(*)[4]>(u));
}
template <int N>
__device__ __forceinline__ void tm_st(uint32_t taddr, const uint32_t* u) {
  if constexpr (N == 16) tmem_st16(taddr, *reinterpret_cast<const uint32_t(*)[16]>(u));
  else if constexpr (N == 8) tmem_st8(taddr, *reinterpret_cast<const uint32_t(*)[8]>(u));
  else tmem_st4(taddr, *reinterpret_cast<const uint32_t(*)[4]>(u));
}

// ---- UMMA descriptors ---------------------------------------------------------------------------
// No-swizzle shared-memory matrix descriptor; lbo / sbo in bytes.  Operands are stored in the canonical layout
// [K/8 (16-byte chunks)][rows][8 x 16-bit]: core matrices (8 rows x 16 B) are contiguous along the rows.
//   K-major use : lbo = rows * 16 (next K chunk), sbo = 128 (next 8 rows)
//   MN-major use: lbo = 128, sbo = rows * 16
__device__ __forceinline__ uint64_t umma_desc2(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (sm_100); layout_type = 0 (no swizzle), base_offset = 0
  return d;
}
// K-major operand of `rows` rows
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t rows) { return umma_desc2(saddr, rows * 16u, 128u); }

// instruction descriptors, kind::f16: D = F32, A / B = F16 (0) or BF16 (1), B optionally MN-major
__host__ __device__ constexpr uint32_t umma_idesc_16(int M, int N, int bf16, int b_mn_major) {
  return (1u << 4)                                                    // D format F32
         | ((uint32_t)bf16 << 7) | ((uint32_t)bf16 << 10)            // A, B format
         | ((uint32_t)b_mn_major << 16)                              // B major: 0 = K, 1 = MN
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);  // N / 8, M / 16
}
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) { return umma_idesc_16(M, N, 0, 0); }
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int b_mn_major) {
  return umma_idesc_16(M, N, 1, b_mn_major);
}

// D[tmem] (+)= A[tmem] * B[smem], 16-bit inputs (format from idesc), fp32 accumulate; one thread issues
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with A in shared memory
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar_addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) { umma_commit_a(smem_u32(bar)); }

// ---- fp16 pairs ---------------------------------------------------------------------------------
__device__ __forceinline__ float2 h2_unpack(uint32_t w) {
  return __half22float2(*reinterpret_cast<const __half2*>(&w));
}
__device__ __forceinline__ uint32_t h2_pack(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
// same, saturating to +-65504 instead of +-inf (cvt.rn.satfinite): an overflowing operand stays finite, so that
// hi - lo never forms inf - inf = NaN; a non-finite input becomes NaN / max and is caught by the caller's checks
__device__ __forceinline__ uint32_t h2_pack_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// sm_100 mixed-precision FADD / FFMA (SASS FHADD / FHFMA): an fp16 operand is widened inside the
// instruction, so "float + half" and "float - half" cost one issue slot instead of two.
__device__ __forceinline__ float add_h(unsigned short a, float c) {
  float d;
  asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(d) : "h"(a), "f"(c));
  return d;
}
__device__ __forceinline__ float sub_h(float c, unsigned short a) {  // c - a
  float d;
  const unsigned short m1 = 0xBC00;  // -1.0
  asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(d) : "h"(a), "h"(m1), "f"(c));
  return d;
}
__device__ __forceinline__ unsigned short h_lo(uint32_t w) { return (unsigned short)(w & 0xffffu); }
__device__ __forceinline__ unsigned short h_hi(uint32_t w) { return (unsigned short)(w >> 16); }
// (hi, lo) fp16 pair words of two consecutive values: hi = rn16(x), lo = rn16(x - hi)  ->  |x - hi - lo| <= 2^-24 |x|
__device__ __forceinline__ void split16(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = h2_pack(x0, x1);
  lo = h2_pack(sub_h(x0, h_lo(hi)), sub_h(x1, h_hi(hi)));
}

// Saturating form: an operand past +-65504 becomes +-65504 instead of +-inf (hi = inf, lo = x - inf = -inf would
// turn the whole row into NaN); h16_saturated() recognises it afterwards.
__device__ __forceinline__ void split16_sat(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = h2_pack_sat(x0, x1);
  lo = h2_pack_sat(sub_h(x0, h_lo(hi)), sub_h(x1, h_hi(hi)));
}
// nonzero iff either half of the pair word is +-65504 (0x7BFF) or beyond (inf / NaN)
__device__ __forceinline__ uint32_t h16_saturated(uint32_t w) {
  const uint32_t a = w & 0x7fff7fffu;
  return (uint32_t)((a & 0xffffu) >= 0x7bffu) | (uint32_t)((a >> 16) >= 0x7bffu);
}

// ---- host: fp16 (hi, lo) split of a constant operand (Lambda of k_dense_tc3, X of k_logistic_tcs) ----------------
// One power-of-two scale serves the whole matrix: max |v| (v rounded to float32) lands in [2^(target-1), 2^target).
struct Fp16Split {
  double amax = 0.0;  // max |float32(v)|
  int shift = 0;      // scale = 2^shift, clamped to [2^-100, 2^100]
  double scale = 1.0;
  Fp16Split(const std::vector<double>& v, int target) {
    for (double e : v) amax = std::max(amax, std::fabs((double)(float)e));
    int ex = 0;
    if (amax > 0 && std::isfinite(amax)) std::frexp(amax, &ex);  // amax = f * 2^ex, f in [0.5, 1)
    shift = std::max(-100, std::min(100, target - ex));
    scale = std::ldexp(1.0, shift);
  }
  // x = float32(float32(v) * scale) as hi = rn16(x), lo = rn16(x - hi); returns x, *rem = x - hi - lo (exact)
  float operator()(double v, __half* hi, __half* lo, double* rem) const {
    const float x = (float)((double)(float)v * scale);
    *hi = __float2half_rn(x);
    *lo = __float2half_rn(x - __half2float(*hi));
    *rem = (double)x - (double)__half2float(*hi) - (double)__half2float(*lo);
    return x;
  }
};

}  // namespace ehmc
