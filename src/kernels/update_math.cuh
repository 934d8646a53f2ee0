/**
 * \file update_math.cuh
 * \brief Device helpers shared by the dense (update_kernels.cu) and row-sparse
 *        (update_rows_kernels.cu) optimizer kernels: vector loads and stores, bf16 / fp8-block
 *        decode, and the per-element AdamW / SGD step. Both kernels must round alike, so the
 *        optimizer math lives here once.
 */
#ifndef PS_KERNELS_UPDATE_MATH_CUH_
#define PS_KERNELS_UPDATE_MATH_CUH_
#include <cuda_bf16.h>
#include <cuda_fp8.h>

#include <cstdint>

#include "kernels/ps_kernels.h"

namespace {

__device__ __forceinline__ int4 ldg16(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg8(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];"
               : "=r"(r.x), "=r"(r.y)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ldf4(const float* p) {
  float4 r;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stf4(float* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void st16(void* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ float2 bf2(uint32_t u) {
  __nv_bfloat162 t = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(t);
}
__device__ __forceinline__ uint32_t pk(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float e8m0(uint32_t biased) {
  const int be = max(1, min(254, static_cast<int>(biased)));
  return __uint_as_float(static_cast<uint32_t>(be) << 23);
}
__device__ __forceinline__ void fp8x4_to_f32(uint32_t q, float s, float* out) {
  const __half2_raw lo = __nv_cvt_fp8x2_to_halfraw2(static_cast<__nv_fp8x2_storage_t>(q & 0xffffu),
                                                    __NV_E4M3);
  const __half2_raw hi = __nv_cvt_fp8x2_to_halfraw2(static_cast<__nv_fp8x2_storage_t>(q >> 16),
                                                    __NV_E4M3);
  const float2 a = __half22float2(__half2(lo)), b = __half22float2(__half2(hi));
  out[0] = a.x * s; out[1] = a.y * s; out[2] = b.x * s; out[3] = b.y * s;
}

/*! single-instruction MUFU.SQRT (<= 1 ulp-ish); the IEEE sqrtf expands to ~10 instructions */
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

/*!
 * o.bias_corr1 / o.bias_corr2 hold the RECIPROCALS 1/(1-beta^t) here (the launchers invert them
 * on the host) so the per-element math is FMA + one MUFU.SQRT + one MUFU.RCP:
 * the kernel must stay memory-bound, and the IEEE div/sqrt sequences cost ~170 issue slots
 * per element, right at the instruction roofline for 28 B/element at 6.5 TB/s.
 */
template <int OPT>
__device__ __forceinline__ void step(float& p, float& m, float& v, float g,
                                     const ps_opt_params& o) {
  if (OPT == PS_OPT_ADAMW) {
    m = fmaf(o.beta1, m, (1.f - o.beta1) * g);
    v = fmaf(o.beta2, v, (1.f - o.beta2) * g * g);
    const float denom = fast_sqrt(v * o.bias_corr2) + o.eps;
    const float upd = __fdividef(m * o.bias_corr1, denom);
    p = p - o.lr * fmaf(o.weight_decay, p, upd);
  } else {
    g += o.weight_decay * p;
    m = o.beta1 * m + g;
    p = p - o.lr * m;
  }
}

}  // namespace
#endif  // PS_KERNELS_UPDATE_MATH_CUH_
