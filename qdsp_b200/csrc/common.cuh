// qdsp_b200/csrc/common.cuh — shared device helpers for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define QDSP_FL_M_PI 3.1415926535f  // reference src/dsp/types.h:4 (the reference's float "pi")

namespace qdsp {

// ---- error plumbing (host) ---------------------------------------------------------------
void set_last_error(const char* fmt, ...);
#define QDSP_CUDA_OK(expr)                                                                   \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            qdsp::set_last_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr,                \
                                 cudaGetErrorString(_e));                                    \
            return -1;                                                                       \
        }                                                                                    \
    } while (0)

// ---- complex helpers (device) ------------------------------------------------------------
// Fast-mode complex multiply: FMA contraction allowed (differs from the x86 no-FMA reference by
// <= 1 ulp per component; within the 1e-5 rel-L2 parity budget).
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -(a.y * b.y)), fmaf(a.x, b.y, a.y * b.x));
}
// Reference-exact complex multiply: (ac - bd, ad + bc) with every product and sum rounded
// separately, exactly like std::complex<float> operator* on x86-64 without FMA.
__device__ __forceinline__ float2 cmul_exact(float2 a, float2 b) {
    return make_float2(__fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)),
                       __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
}

// acc += x * t (complex sample times real tap) in one packed FFMA2 (Blackwell f32x2 pipe).
__device__ __forceinline__ float2 cmac(float2 x, float t, float2 acc) {
    return __ffma2_rn(x, make_float2(t, t), acc);
}

// NCO phase: 64-bit fixed-point "turns" (1 turn = 2^64). phase(n) = phase0 + n * f, exact modulo
// 2^64, so the closed-form oscillator never loses precision however long the stream runs.
__device__ __forceinline__ float2 phasor_from_turns(uint64_t turns) {
    // Exact quadrant reduction in integers: turns = q * 2^62 + r, r in [-2^61, 2^61), so the
    // float angle handed to sincosf is within +-pi/4 (quantisation <= 5e-8 rad) and the
    // quadrant rotation is a swap/negate.
    const uint64_t t = turns + (1ull << 61);
    const unsigned q = (unsigned)(t >> 62);
    const int64_t r = (int64_t)(t & ((1ull << 62) - 1)) - (1ll << 61);
    const float ang = (float)(int32_t)(r >> 30) * (6.283185307179586f / 17179869184.0f);  // 2*pi / 2^34
    float s, c;
    sincosf(ang, &s, &c);
    switch (q) {
        case 0: return make_float2(c, s);
        case 1: return make_float2(-s, c);
        case 2: return make_float2(-c, -s);
        default: return make_float2(s, -c);
    }
}
__device__ __forceinline__ float2 phasor_from_turns_f64(uint64_t turns) {
    const double ang = (double)(int64_t)turns * (6.283185307179586476925286766559 / 18446744073709551616.0);
    double s, c;
    sincos(ang, &s, &c);
    return make_float2((float)c, (float)s);
}

// fast_arctan2 exactly as the reference evaluates it (src/dsp/demodulator.h:11-30): IEEE
// divisions, no FMA contraction, the macro-expanded constant expressions.
__device__ __forceinline__ float fast_arctan2_ref(float y, float x) {
    const float c1 = QDSP_FL_M_PI / 4.0f;           // FAST_ATAN2_COEF1
    const float c2 = 3.0f * QDSP_FL_M_PI / 4.0f;    // FAST_ATAN2_COEF2 (macro-expanded order)
    const float abs_y = fabsf(y);
    if (x == 0.0f && y == 0.0f) return 0.0f;
    // branch-free selection of the reference's two cases; the arithmetic per case is unchanged
    const bool pos = x >= 0.0f;
    const float num = pos ? __fsub_rn(x, abs_y) : __fadd_rn(x, abs_y);
    const float den = pos ? __fadd_rn(x, abs_y) : __fsub_rn(abs_y, x);
    const float r = __fdiv_rn(num, den);
    const float angle = __fsub_rn(pos ? c1 : c2, __fmul_rn(c1, r));
    return (y < 0.0f) ? -angle : angle;
}
// One FloatFMDemod step (src/dsp/demodulator.h:88-92) given current and previous phase.
__device__ __forceinline__ float fm_step_ref(float cur, float prev, float phasorSpeed) {
    float diff = __fsub_rn(cur, prev);
    if (diff > 3.1415926535f) diff = __fsub_rn(diff, 2 * 3.1415926535f);
    else if (diff <= -3.1415926535f) diff = __fadd_rn(diff, 2 * 3.1415926535f);
    return __fdiv_rn(diff, phasorSpeed);
}

// streaming 128-bit global load that does not pollute L1 (input IQ is read once per tile)
__device__ __forceinline__ float4 ldg_stream128(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ldg_stream64(const float2* p) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
// the same for one integer IQ pair: a 32-bit (cs16) or 16-bit (cs8 / cu8) word, zero-extended
__device__ __forceinline__ uint32_t ldg_stream32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ldg_stream16(const uint16_t* p) {
    uint16_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return v;
}

}  // namespace qdsp
