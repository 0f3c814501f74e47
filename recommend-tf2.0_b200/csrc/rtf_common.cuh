// Shared device helpers for librtf_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rtf_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "librtf_b200 is written for sm_100a (B200) only"
#endif

#define RTF_CHECK_LAUNCH()                         \
  do {                                             \
    cudaError_t e__ = cudaGetLastError();          \
    if (e__ != cudaSuccess) return (int)e__;       \
  } while (0)

namespace rtf {

constexpr int kNumSMs = 148;  // B200

// Padding constant the reference masks logits with: -2**32 + 1, which rounds to
// -4294967296.0f in fp32 (src/ctr/layers/modules.py:161, src/match/layers/modules.py:90).
constexpr float kPadLogit = -4294967296.0f;

__device__ __forceinline__ float4 ldg_nc_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_cs_f4(float* p, const float4& v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ float4 f4_add(const float4& a, const float4& b) {
  // explicit round-to-nearest adds: never contracted, so sums are reproducible
  return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z),
                     __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float4 f4_scale(const float4& a, float s) {
  return make_float4(__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s),
                     __fmul_rn(a.w, s));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) ------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- fp32 -> three bf16 planes (the dense GEMM's operand split) -------------------
// The transform of CUTLASS's emulated FastF32 mainloop, restated bit for bit, for a pair of
// values (a, b) -> bf16x2 words {lo = a, hi = b}:
//   x0 = RN_satfinite(x);  r = (x - x0) * 2^S;  x1 = RN_satfinite(r);  x2 = RN_satfinite((r - x1) * 2^S)
// S = kPlaneScale is the mainloop's ScalingFactor (8 for bf16).
constexpr int kPlaneScale = 8;
__device__ __forceinline__ uint32_t cvt_bf16x2_satfinite(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void split_bf16x3(float a, float b, uint32_t& p0, uint32_t& p1,
                                             uint32_t& p2) {
  const float s = (float)(1 << kPlaneScale);
  p0 = cvt_bf16x2_satfinite(a, b);
  a = __fmul_rn(__fsub_rn(a, __uint_as_float(p0 << 16)), s);
  b = __fmul_rn(__fsub_rn(b, __uint_as_float(p0 & 0xffff0000u)), s);
  p1 = cvt_bf16x2_satfinite(a, b);
  a = __fmul_rn(__fsub_rn(a, __uint_as_float(p1 << 16)), s);
  b = __fmul_rn(__fsub_rn(b, __uint_as_float(p1 & 0xffff0000u)), s);
  p2 = cvt_bf16x2_satfinite(a, b);
}

// id load with bounds check; returns -1 for an out-of-range id
template <typename IdT>
__device__ __forceinline__ long long load_id(const IdT* ids, long long idx, long long rows,
                                             int32_t* err) {
  long long id = (long long)__ldg(ids + idx);
  if (id < 0 || id >= rows) {
    if (err) atomicOr(err, 1);
    return -1;
  }
  return id;
}

}  // namespace rtf
