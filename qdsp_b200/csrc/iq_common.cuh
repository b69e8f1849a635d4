// qdsp_b200/csrc/iq_common.cuh — the one conversion rule of the library for integer IQ (include/qdsp_b200.h,
// qdsp_iq_convert_process), on the device: iq_convert_kernel (k_pointwise.cu) and the spectrum frames kernel
// (k_spectrum.cu) both read integer samples through these functions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "internal.cuh"

namespace qdsp {

// y = (float(x) + offset) * scale, each step rounded to float32 (numpy:
// (x.astype(np.float32) + np.float32(offset)) * np.float32(scale)). float(x) is formed exactly on the ALU and FMA pipes
// instead of I2F: the component, made unsigned (x + 2^15 / x + 2^7 for the signed formats), is placed in the low mantissa
// bits of 2^23 by one PRMT, and 2^23 plus the bias is subtracted (exact below 2^24).
template <int FMT>
__device__ __forceinline__ float2 iq_finish(uint32_t m0, uint32_t m1, IqConv c) {
    const float M = FMT == QDSP_CS16 ? 8421376.0f : FMT == QDSP_CS8 ? 8388736.0f : 8388608.0f;   // 2^23 + bias
    const float2 x = __fadd2_rn(make_float2(__uint_as_float(m0), __uint_as_float(m1)), make_float2(-M, -M));
    return __fmul2_rn(__fadd2_rn(x, make_float2(c.offset, c.offset)), make_float2(c.scale, c.scale));
}
// one cs16 sample from its 32-bit word
__device__ __forceinline__ float2 iq_cs16(uint32_t w, IqConv c) {
    const uint32_t u = w ^ 0x80008000u;
    return iq_finish<QDSP_CS16>(__byte_perm(u, 0x4B000000u, 0x7410), __byte_perm(u, 0x4B000000u, 0x7432), c);
}
// two 8-bit samples from their 32-bit word (the low half only is meaningful for a single sample)
template <int FMT>
__device__ __forceinline__ float4 iq_b8x2(uint32_t w, IqConv c) {
    const uint32_t u = FMT == QDSP_CS8 ? (w ^ 0x80808080u) : w;
    const float2 s0 = iq_finish<FMT>(__byte_perm(u, 0x4B000000u, 0x7440), __byte_perm(u, 0x4B000000u, 0x7441), c);
    const float2 s1 = iq_finish<FMT>(__byte_perm(u, 0x4B000000u, 0x7442), __byte_perm(u, 0x4B000000u, 0x7443), c);
    return make_float4(s0.x, s0.y, s1.x, s1.y);
}
template <int FMT>
__device__ __forceinline__ float2 iq_one(const void* in, long long i, IqConv c) {
    if (FMT == QDSP_CS16) return iq_cs16(reinterpret_cast<const uint32_t*>(in)[i], c);
    const float4 v = iq_b8x2<FMT>(reinterpret_cast<const uint16_t*>(in)[i], c);
    return make_float2(v.x, v.y);
}

}  // namespace qdsp
