// rx_common.cuh -- shared definitions of the sm_100a Gen2 receive path:
// derived configuration, the numerical contract (how each libm/libgcc call the
// reference makes is evaluated on the device), mbarrier / TMA-bulk PTX wrappers.
//
// Numerical contract (SURVEY.md Appendix A.5; every item is exercised by the
// parity tests against the compiled reference):
//   * no FMA contraction anywhere: this translation unit is built with
//     -fmad=false and all arithmetic that must round like the reference uses
//     the explicit _rn intrinsics;
//   * std::abs(complex<float>) = glibc cabsf = (float)sqrt((double)re*re + (double)im*im)
//     (gate_impl.cc:130);
//   * z / complex<float>(N,0) = one IEEE float division per component
//     (libgcc __divsc3 with a zero imaginary divisor; gate_impl.cc:141, tag_decoder_impl.cc:103);
//   * std::norm = re*re + im*im with three roundings (libstdc++ 13);
//   * complex * complex = (ac - bd, ad + bc) with separately rounded products.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rfid_b200.h"

namespace rfid_b200 {

// ---- protocol constants: include/rfid/global_vars.h:72-143 of the reference ----
constexpr int kT1_D = 240;                // us
constexpr int kPW_D = 12;                 // us
constexpr int kT2_D = 480, kCW_D = 250, kP_DOWN_D = 2000, kDELIM_D = 12, kTRCAL_D = 200;  // us, reader TX (global_vars.h:88-97)
constexpr int kNumPulsesCommand = 5;
constexpr int kTagPreambleBits = 6;
constexpr int kRN16Bits = 17;
constexpr int kEPCBits = 129;
constexpr int kWinSizeD = 250;            // us
constexpr int kDcSizeD = 120;             // us
constexpr int kReaderFreq = 40000;        // BLF
constexpr float kThreshFraction = 0.75f;
constexpr unsigned kPreambleMask = 0xC4B; // TAG_PREAMBLE {1,1,0,1,0,0,1,0,0,0,1,1}: bit j = P[j]

// Derived sample counts (gate_impl.cc:48-53,115,121; tag_decoder_impl.cc:60), computed on the
// host with the reference's own double/float expression order.
struct RxConfig {
  int adc_rate, decim, ntaps;
  int fs_dec;
  int n_T1, n_PW, n_tag_bit_i;
  float n_tag_bit_f;
  int win_length, dc_length;
  int len_rn16, len_epc;
  int fixed_q, max_queries, max_tags;
  int mf_q, mf_rem;        // ntaps / decim, ntaps % decim
  int sync_range;          // number of i with i < 1.5 * n_tag_bit_f   (tag_decoder_impl.cc:85)
  float t_min, t_max;      // EPC period search bounds (tag_decoder_impl.cc:151-152)
  // division by the two ring lengths: reciprocal + "fast" flag when the multiply-correct sequence of
  // f_div_const has been verified exhaustively for this divisor (tools/micro/verify_constdiv.c)
  float win_recip, dc_recip;
  int win_div_fast, dc_div_fast;
};

// ---------------------------------------------------------------- arithmetic primitives
__device__ __forceinline__ float f_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float f_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float f_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float f_div(float a, float b) { return __fdiv_rn(a, b); }

// IEEE-exact x / d for a constant d whose reciprocal c = RN(1/d) passed the exhaustive check: q = RN(x*c),
// r = x - q*d (exact, fused), result = RN(q + r*c).  Three instructions instead of the ~10 of div.rn.  Only
// applied where no intermediate can underflow / overflow; everything else takes the general division.
__device__ __noinline__ float f_div_general(float x, float d) { return __fdiv_rn(x, d); }

// branch-free halves of f_div_const, so that several divisions can be in flight together:
// the multiply-correct quotient, and whether x is inside the range for which it is verified
__device__ __forceinline__ float f_div_fast(float x, float d, float c)
{
  const float q = __fmul_rn(x, c);
  return __fmaf_rn(__fmaf_rn(-q, d, x), c, q);
}
constexpr float kDivFastMin = 7.9e-31f, kDivFastMax = 1.2e30f;  // verified dividend range of f_div_fast
__device__ __forceinline__ bool f_div_fast_ok(float x)
{
  const float ax = fabsf(x);
  return ax >= kDivFastMin && ax <= kDivFastMax;
}

__device__ __forceinline__ float f_div_const(float x, float d, float c, int fast)
{
  const float ax = fabsf(x);
  if (fast && ax >= 7.9e-31f && ax <= 1.2e30f) {
    const float q = __fmul_rn(x, c);
    const float r = __fmaf_rn(-q, d, x);
    return __fmaf_rn(r, c, q);
  }
  return f_div_general(x, d);  // rare: out of the verified range, or an unverified divisor
}

// glibc cabsf(re + i*im): products are exact in double, one rounding for the sum, correctly
// rounded double sqrt, one rounding to float.
__device__ __forceinline__ float cabsf_ref(float re, float im)
{
  double dr = (double)re, di = (double)im;
  double s = __fma_rn(di, di, __dmul_rn(dr, dr));  // dr*dr exact (48 bits) => fma == round(dr*dr + di*di)
  return __double2float_rn(__dsqrt_rn(s));
}

// rare paths kept out of the callers' instruction stream (the capture kernels are instruction-cache sensitive)
__device__ __noinline__ float cabsf_ref_call(float re, float im) { return cabsf_ref(re, im); }
__device__ __noinline__ float f_div_const_call(float x, float d, float c, int fast) { return f_div_const(x, d, c, fast); }

// The same value without the branches of __dsqrt_rn, so that several evaluations interleave: s as above, one Newton step
// on rsqrt.approx.f64 (relative error after the step < 2^-40), rounded to float.  That equals
// (float)sqrt_rn(s) whenever the approximation is farther than its own error bound from every float rounding boundary
// (the mid-points between adjacent floats, 29 bits below the double's leading bit); `risky` reports the rest -- values
// within 2^-38 of a boundary (one sample in 2^13), zero, and magnitudes where the float result would be subnormal or
// infinite -- for which the caller evaluates cabsf_ref.  tools/micro/cabs_check.cu compares the pair against cabsf_ref.
__device__ __forceinline__ float cabsf_quick(float re, float im, bool& risky)
{
  const double dr = (double)re, di = (double)im;
  const double s = __fma_rn(di, di, __dmul_rn(dr, dr));
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(s));
  double g = __dmul_rn(s, y);
  const double h = __dmul_rn(0.5, y);
  const double r = __fma_rn(-g, h, 0.5);
  g = __fma_rn(g, r, g);
  const unsigned long long bits = (unsigned long long)__double_as_longlong(g);
  const unsigned low = (unsigned)bits & 0x1FFFFFFFu;                 // the 29 bits a float does not keep
  const unsigned hi = (unsigned)(bits >> 32);
  const bool near_mid = (unsigned)(low - 0x10000000u + 0x8000u) < 0x10000u;   // |low - mid| < 2^15  (2^-38 relative)
  const bool range_ok = hi > 0x38200000u && hi < 0x47E00000u;       // 2^-125 < g < 2^127: normal float, finite, not NaN
  risky = near_mid || !range_ok;
  return __double2float_rn(g);
}

__device__ __forceinline__ float2 c_add(float2 a, float2 b) { return make_float2(f_add(a.x, b.x), f_add(a.y, b.y)); }
// complex add as ONE packed instruction (sm_100 add.rn.f32x2: two independent IEEE round-to-nearest adds)
__device__ __forceinline__ float2 c_add2(float2 a, float2 b)
{
  unsigned long long ua, ub, ud;
  ua = ((unsigned long long)__float_as_uint(a.y) << 32) | __float_as_uint(a.x);
  ub = ((unsigned long long)__float_as_uint(b.y) << 32) | __float_as_uint(b.x);
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(ud) : "l"(ua), "l"(ub));
  return make_float2(__uint_as_float((unsigned)ud), __uint_as_float((unsigned)(ud >> 32)));
}
__device__ __forceinline__ float2 c_sub(float2 a, float2 b) { return make_float2(f_sub(a.x, b.x), f_sub(a.y, b.y)); }
__device__ __forceinline__ float c_norm(float2 a) { return f_add(f_mul(a.x, a.x), f_mul(a.y, a.y)); }
// std::real((a - b) * std::conj(h)): (x+iy)(c+id) with d = -h.y, real = x*c - y*d
__device__ __forceinline__ float c_proj(float2 a, float2 b, float2 h)
{
  float x = f_sub(a.x, b.x), y = f_sub(a.y, b.y);
  return f_sub(f_mul(x, h.x), f_mul(y, -h.y));
}

// ---------------------------------------------------------------- mbarrier / TMA (sm_90+ PTX)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
// arrive without release semantics (the default .release.cta makes the arriving thread's earlier writes visible first)
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar)
{
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.relaxed.cta.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking test (try_wait may park the thread for a system-dependent time when the phase is not complete): for a
// warp that watches more than one barrier
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// spin a few times (the phase is usually complete or about to be), then back off so that a waiting warp
// does not take issue slots away from the latency-critical warps of the co-resident CTAs
#ifndef RFID_B200_MBAR_BACKOFF_NS
#define RFID_B200_MBAR_BACKOFF_NS 200
#endif
#ifndef RFID_B200_MBAR_SPINS
#define RFID_B200_MBAR_SPINS 4
#endif
constexpr unsigned kMbarBackoffNs = RFID_B200_MBAR_BACKOFF_NS;
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
  for (int i = 0; i < RFID_B200_MBAR_SPINS; i++)
    if (mbar_try_wait(bar, parity)) return;
  while (!mbar_try_wait(bar, parity)) __nanosleep(kMbarBackoffNs);
}
// wait for a phase that is not on this warp's critical path: let the hardware park the warp
// (suspend-time hint, ns) instead of burning issue slots that the sequencer warps need
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity, uint32_t hint_ns = 20000)
{
  uint32_t ok = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
        : "memory");
  } while (!ok);
}
// wait of a warp that has nothing else to do: test, sleep, test ... (the suspend-time hint of try_wait returns after a few
// dozen cycles on this part, so a hinted loop spins; an explicit sleep keeps an idle warp out of the issue slots)
__device__ __forceinline__ void mbar_wait_idle(uint64_t* bar, uint32_t parity, unsigned sleep_ns)
{
  while (!mbar_try_wait(bar, parity)) __nanosleep(sleep_ns);
}
// one try_wait with a suspend-time hint: true when the phase of parity `parity` has completed; false after (about) hint_ns
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t hint_ns)
{
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
      : "memory");
  return ok != 0;
}
// 1-D bulk copy global -> shared through the TMA engine; completion is signalled on `bar`
// (SASS: UBLKCP).  dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// same, with an L2 eviction hint for data that is read exactly once (the raw capture): evict-first keeps the streaming
// input from displacing the kernel's L2-resident scratch
__device__ __forceinline__ unsigned long long l2_policy_evict_first()
{
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_1d_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, unsigned long long pol)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- programmatic dependent launch.  A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may be
// scheduled while the kernel before it on the stream still runs, as soon as every CTA of that kernel has executed
// pdl_launch_dependents (or exited).  pdl_wait returns once that kernel has completed and its stores are visible.  In a
// launch without the attribute both are no-ops.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- launch timing (rfid_b200_kernel_time).  A launch gets one slot {earliest CTA start, latest CTA end} in %globaltimer
// ns, reset by the host to {~0, 0}; nullptr = timing off.  Every warp calls stamp_warp_end once, after its last global
// store; the CTA's last warp stamps the end.  warps_done is a shared counter zeroed before any warp can get there.
__device__ __forceinline__ unsigned long long global_ns()
{
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void stamp_cta_start(unsigned long long* slot)
{
  if (slot && threadIdx.x == 0) atomicMin(slot, global_ns());
}
__device__ __forceinline__ void stamp_warp_end(unsigned long long* slot, unsigned* warps_done)
{
  if (!slot) return;
  __syncwarp();
  if ((threadIdx.x & 31) == 0 && atomicAdd(warps_done, 1u) == blockDim.x / 32 - 1) atomicMax(slot + 1, global_ns());
}

}  // namespace rfid_b200
