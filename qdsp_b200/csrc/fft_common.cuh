// qdsp_b200/csrc/fft_common.cuh — small power-of-two DFTs in registers, shared by the FFT kernels (k_chanfft.cu: the
// channelizer's 256-point FFTs; k_spectrum.cu: the power spectrum's 64..16384-point FFTs).
#pragma once
#include <cuda_runtime.h>

namespace qdsp {

// a * e^{-j 2 pi P / 16}, P a compile-time constant after unrolling
__device__ __forceinline__ float2 mul_w16(float2 a, int P) {
    constexpr float C1 = 0.9238795325112867f, S1 = 0.3826834323650898f, H = 0.7071067811865476f;
    switch (P) {
        case 0: return a;
        case 1: return make_float2(fmaf(a.x, C1, a.y * S1), fmaf(a.y, C1, -a.x * S1));
        case 2: return make_float2(H * (a.x + a.y), H * (a.y - a.x));
        case 3: return make_float2(fmaf(a.x, S1, a.y * C1), fmaf(a.y, S1, -a.x * C1));
        case 4: return make_float2(a.y, -a.x);
        case 5: return make_float2(fmaf(a.y, C1, -a.x * S1), -fmaf(a.y, S1, a.x * C1));
        case 6: return make_float2(H * (a.y - a.x), -H * (a.x + a.y));
        default: return make_float2(fmaf(a.y, S1, -a.x * C1), -fmaf(a.y, C1, a.x * S1));
    }
}
__host__ __device__ constexpr int bitrev4(int i) { return ((i & 1) << 3) | ((i & 2) << 1) | ((i & 4) >> 1) | ((i & 8) >> 3); }
// bit reversal of i in log2(R) bits, R in {2, 4, 8, 16}
template <int R>
__host__ __device__ constexpr int bitrev(int i) {
    return R == 16 ? bitrev4(i) : R == 8 ? (bitrev4(i) >> 1) : R == 4 ? (bitrev4(i) >> 2) : (bitrev4(i) >> 3);
}
// R-point forward DFT in registers (radix-2 decimation in frequency), R in {2, 4, 8, 16}; X[k] is left in a[bitrev<R>(k)].
// The twiddle of a radix-2 stage of span `half` is W_{2 half}^{i mod half} = e^{-j 2 pi ((i mod half) 8 / half) / 16}
// whatever R is, so every R takes its twiddles from mul_w16.
template <int R>
__device__ __forceinline__ void fft_radix(float2 (&a)[R]) {
#pragma unroll
    for (int half = R / 2; half >= 1; half >>= 1) {
#pragma unroll
        for (int i = 0; i < R; i++) {
            if ((i & half) == 0) {
                const int j = i + half;
                const float2 t = make_float2(a[i].x - a[j].x, a[i].y - a[j].y);
                a[i] = make_float2(a[i].x + a[j].x, a[i].y + a[j].y);
                a[j] = mul_w16(t, (i & (half - 1)) * (8 / half));
            }
        }
    }
}
// 16-point forward DFT in registers; X[k] is left in a[bitrev4(k)]
__device__ __forceinline__ void fft16(float2 (&a)[16]) { fft_radix<16>(a); }

}  // namespace qdsp
