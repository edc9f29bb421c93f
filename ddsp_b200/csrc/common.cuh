// Shared helpers for libddsp_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ddsp_b200.h"

namespace ddsp {

// ---- error reporting (thread-local string, no global mutable state) --------
void set_error(const char* fmt, ...);
void count_launch();

#define DDSP_REQUIRE(cond, code, ...)  \
  do {                                 \
    if (!(cond)) {                     \
      ::ddsp::set_error(__VA_ARGS__);  \
      return (code);                   \
    }                                  \
  } while (0)

#define DDSP_CHECK_LAUNCH(name)                                         \
  do {                                                                  \
    ::ddsp::count_launch();                                             \
    cudaError_t e__ = cudaGetLastError();                               \
    if (e__ != cudaSuccess) {                                           \
      ::ddsp::set_error("%s: CUDA error: %s", name,                     \
                        cudaGetErrorString(e__));                       \
      return DDSP_B200_E_CUDA;                                          \
    }                                                                   \
  } while (0)

constexpr int kNumSMs = 148;  // B200

// ---- fixed-point phase ------------------------------------------------------
// Phase is kept in *turns* as a 64-bit fixed-point fraction (2^64 == 1 turn).
// Wrapping integer addition is exact modular arithmetic, so the phase of the
// k-th harmonic is the wrapping product k * phase - no accumulation error, no
// large-argument sin.  This is the intent of core.angular_cumsum
// (core.py:799-866) carried out exactly.
__device__ __forceinline__ unsigned long long turns_to_fix64(double turns) {
  double fr = turns - rint(turns);  // [-0.5, 0.5]
  return (unsigned long long)__double2ll_rn(fr * 18446744073709551616.0);
}

// core.exp_sigmoid (core.py:386-404): 2 * sigmoid(x)^ln(10) + 1e-7, evaluated
// as 2 * 2^(-ln10 * log2(1 + e^-x)) + 1e-7 on the SFU (3 MUFU ops): both limits
// are exact (x -> -inf: 1e-7, x -> +inf: 2 + 1e-7) and nothing overflows to NaN.
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float exp_sigmoid_f(float x) {
  const float kLog2e = 1.4426950408889634f;
  const float kLn10 = 2.302585092994046f;
  const float t = ex2_approx(-x * kLog2e);          // e^-x  (inf for x << 0)
  float l;                                           // log2(1 + e^-x), arg >= 1
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(1.0f + t));
  return fmaf(2.0f, ex2_approx(-kLn10 * l), 1e-7f);
}

// tf.nn.sigmoid (ModDelay's default phase_scale_fn, effects.py:331-344):
// 1 / (1 + e^-x) with e^-x on the SFU and a correctly rounded reciprocal; both
// limits are exact (x -> -inf: 0, x -> +inf: 1).
__device__ __forceinline__ float sigmoid_f(float x) {
  return __frcp_rn(1.0f + ex2_approx(-x * 1.4426950408889634f));
}

// ---- Philox4x32-10 (Salmon et al., SC'11) ----------------------------------
struct Philox4 {
  uint32_t x, y, z, w;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1,
                                                 uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

// 23 mantissa bits -> [1, 2) -> 2x - 3 in [-1, 1).
__device__ __forceinline__ float u32_to_pm1(uint32_t r) {
  return 2.0f * __uint_as_float((r >> 9) | 0x3F800000u) - 3.0f;
}

// Four consecutive noise samples (index 4*q .. 4*q+3) of batch item b.
__device__ __forceinline__ float4 noise4(uint32_t q, uint32_t b, uint64_t seed,
                                         uint64_t offset) {
  Philox4 r = philox4x32_10(q, b, (uint32_t)offset, (uint32_t)(offset >> 32),
                            (uint32_t)seed, (uint32_t)(seed >> 32));
  return make_float4(u32_to_pm1(r.x), u32_to_pm1(r.y), u32_to_pm1(r.z),
                     u32_to_pm1(r.w));
}

// --- mbarrier / TMA bulk copy (PTX) -----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(void* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src,
                                             uint32_t bytes, void* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// DDSP_MBAR_HINT_NS > 0: pass a suspend-time hint to try_wait, so that a waiting
// warp sleeps in hardware (and is woken by the phase flip) instead of coming back
// to the issue stage every few hundred cycles.
#ifndef DDSP_MBAR_HINT_NS
#define DDSP_MBAR_HINT_NS 0
#endif
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t phase) {
#if DDSP_MBAR_HINT_NS > 0
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(phase), "r"((uint32_t)DDSP_MBAR_HINT_NS)
      : "memory");
#else
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
#endif
}

__device__ __forceinline__ void mbar_arrive(void* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// Named barrier over a subset of the CTA (ids 1..15; 0 is __syncthreads).
__device__ __forceinline__ void named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ddsp
