// Storage / MMA-operand element type of activations and weights.
//
// Default fp16 (CDC_ACT_FP16=1).  BASELINE.json's north_star names bf16 *and* a 1e-2 max-abs per-step
// tolerance against the fp32 oracle; tools/precision_study.py (CPU emulation of every storage point)
// and the first B200 run agree that bf16 operands put the pinned network at 0.024-0.031 max-abs
// (8 mantissa bits, ~55 roundings deep), while fp16 -- same 16-bit width, same tcgen05 kind::f16
// throughput, 11 mantissa bits -- lands at ~0.0035.  Accumulation, GroupNorm statistics, FiLM, the
// sampler state x_t and x0_hat are fp32 either way.  Build with -DCDC_ACT_FP16=0 for the bf16 variant.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#ifndef CDC_ACT_FP16
#define CDC_ACT_FP16 1
#endif

namespace cdc {

#if CDC_ACT_FP16
typedef __half act_t;
constexpr uint32_t kUmmaFormat = 0;  // tcgen05 kind::f16 a_format / b_format: 0 = F16
#define CDC_TMA_DTYPE CU_TENSOR_MAP_DATA_TYPE_FLOAT16
constexpr float kActMax = 65504.0f;  // values beyond it are stored saturated (and counted: ConvParams::sat)
__device__ __forceinline__ uint32_t pack_act2(float lo, float hi) {  // saturating: never stores inf
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_act2_nosat(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float act_lo(uint32_t u) { return __half2float(__ushort_as_half(static_cast<unsigned short>(u & 0xFFFFu))); }
__device__ __forceinline__ float act_hi(uint32_t u) { return __half2float(__ushort_as_half(static_cast<unsigned short>(u >> 16))); }
// Saturation diagnostics on PACKED outputs: running per-half max of |x| (one or two instructions per word), and the test
// "a half holds the largest finite magnitude", i.e. pack_act2 clamped it.
__device__ __forceinline__ uint32_t act2_absmax(uint32_t m, uint32_t u) {
    const __half2 r = __hmax2(*reinterpret_cast<const __half2*>(&m), __habs2(*reinterpret_cast<const __half2*>(&u)));
    return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t act2_absmax(uint32_t m, const uint4& v) {
    return act2_absmax(act2_absmax(act2_absmax(act2_absmax(m, v.x), v.y), v.z), v.w);
}
__device__ __forceinline__ bool act2_is_sat(uint32_t m) { return (m & 0xFFFFu) == 0x7BFFu || (m >> 16) == 0x7BFFu; }
// one value, saturating like pack_act2 (+-inf and finite values beyond the range -> +-65504) and keeping NaN a NaN
__device__ __forceinline__ act_t to_act(float v) {
    unsigned short r;
    asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(v));
    return __ushort_as_half(r);
}
__device__ __forceinline__ float from_act(act_t v) { return __half2float(v); }
#else
typedef __nv_bfloat16 act_t;
constexpr uint32_t kUmmaFormat = 1;  // 1 = BF16
constexpr float kActMax = 3.3895313892515355e38f;  // bf16 maximum
#define CDC_TMA_DTYPE CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
__device__ __forceinline__ uint32_t pack_act2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_act2_nosat(float lo, float hi) { return pack_act2(lo, hi); }
__device__ __forceinline__ float act_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float act_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t act2_absmax(uint32_t m, uint32_t) { return m; }  // bf16 has fp32's range: nothing to count
__device__ __forceinline__ uint32_t act2_absmax(uint32_t m, const uint4&) { return m; }
__device__ __forceinline__ bool act2_is_sat(uint32_t) { return false; }
__device__ __forceinline__ act_t to_act(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ float from_act(act_t v) { return __bfloat162float(v); }
#endif

}  // namespace cdc
