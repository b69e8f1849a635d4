// qdsp_b200/csrc/k_clock.cu — MMClockRecovery<float | complex_t>::run (reference src/dsp/clock_recovery.h:127-215):
// Mueller & Mueller symbol-timing recovery with an 8-tap, 129-phase interpolator table.
//
// The recurrence is data dependent in its INDEX (which input sample the next symbol is interpolated at depends on the
// phase error of the previous symbol), so this first implementation keeps the reference's order exactly: one warp per
// stream stages windows of the input in shared memory with coalesced loads, lane 0 walks the symbols. Every float
// operation is rounded where the x86 reference rounds it (sequential dot product, no contraction): outputs, per-block
// output counts and the carried state are bit-identical to the reference. Throughput is latency bound (about one
// symbol per 150-200 cycles); independent streams scale across CTAs (one per stream). A chunk-speculative walk of a
// single long stream was measured and removed: on a locked signal almost every chunk had to be re-walked (DESIGN.md).
#include "internal.cuh"
#include "kernels.cuh"

namespace qdsp {

constexpr int kMmWin = 4096;     // samples staged per window
constexpr int kMmHalo = 8;       // an output at sample i reads x[i-7 .. i]

__device__ __forceinline__ float mm_step(float v) { return v > 0.0f ? 1.0f : -1.0f; }   // DSP_STEP, utils/macros.h:6

// state layout == oracle/port.c: [0] mu [1] dynOmega [2] lastOutput [3..8] p0 p1 p2 [9..14] c0 c1 c2 [15] nextOffset
// [16..29] delay[0..6] as (re, im) pairs (float streams use the re slots)
template <bool CPLX>
__global__ void __launch_bounds__(32) mm_kernel(const float* __restrict__ in, PartitionDev part, const float* __restrict__ taps_g,
                                                float omega, float gainOmega, float muGain, float omegaMin, float omegaMax,
                                                float* __restrict__ state, float* __restrict__ out, int* __restrict__ out_counts,
                                                long long* __restrict__ total_out) {
    constexpr int ES = CPLX ? 2 : 1;
    __shared__ float s_taps[129 * 8];
    __shared__ float s_x[(kMmWin + kMmHalo) * ES];
    const int lane = threadIdx.x;
    for (int k = lane; k < 129 * 8; k += 32) s_taps[k] = taps_g[k];

    float mu = state[0], dynOmega = state[1], lastOutput = state[2];
    float2 p0 = make_float2(state[3], state[4]), p1 = make_float2(state[5], state[6]), p2 = make_float2(state[7], state[8]);
    float2 c0 = make_float2(state[9], state[10]), c1 = make_float2(state[11], state[12]), c2 = make_float2(state[13], state[14]);
    int nextOffset = (int)state[15];
    long long total = 0;

    for (int b = 0; b < part.nblocks; b++) {
        const BlkInfo bi = part.get(b);
        const int count = bi.count;
        const long long S = bi.in_start;
        const int maxOut = (int)__fmul_rn(__fmul_rn(2.0f, omega), (float)count);   // clock_recovery.h:135
        int outCount = 0;
        int i = nextOffset < 0 ? 0 : nextOffset;   // negative only after the maxOut cap fired (the reference then reads delay[i < 0])
        // windows of the block: samples [w0 - 7, w0 + kMmWin) of the block-relative stream; what lies before the call's
        // first sample comes from the carried delay[] (the previous call's last 7 samples)
        for (int w0 = i / kMmWin * kMmWin; w0 < count; w0 += kMmWin) {
            __syncwarp();
            // 8 loads per lane in flight together (a load-store loop would expose the DRAM latency 128 times per window)
            for (int e0 = lane; e0 < kMmWin + kMmHalo - 1; e0 += 8 * 32) {
                float2 v[8];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int e = e0 + 32 * j;
                    const long long g = S + w0 - 7 + e;             // call-relative sample index
                    v[j] = make_float2(0.f, 0.f);
                    if (e < kMmWin + kMmHalo - 1) {
                        if (g >= 0) {
                            if (g < part.total) {
                                if (CPLX) v[j] = reinterpret_cast<const float2*>(in)[g];
                                else v[j].x = in[g];
                            }
                        } else {
                            v[j] = make_float2(state[16 + 2 * (int)(g + 7)], state[17 + 2 * (int)(g + 7)]);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int e = e0 + 32 * j;
                    if (e < kMmWin + kMmHalo - 1) {
                        if (CPLX) reinterpret_cast<float2*>(s_x)[e] = v[j];
                        else s_x[e] = v[j].x;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) {
                const int wend = w0 + kMmWin < count ? w0 + kMmWin : count;
                while (i < wend && outCount < maxOut) {
                    const float* t8 = s_taps + 8 * (int)roundf(__fmul_rn(mu, 128.0f));
                    const float* src = s_x + (i - w0) * ES;        // x[i-7 .. i]
                    float phaseError;
                    if (!CPLX) {
                        float outVal = 0.0f;
#pragma unroll
                        for (int k = 0; k < 8; k++) outVal = __fadd_rn(outVal, __fmul_rn(src[k], t8[k]));
                        out[total + outCount] = outVal;
                        outCount++;
                        phaseError = __fsub_rn(__fmul_rn(mm_step(lastOutput), outVal), __fmul_rn(lastOutput, mm_step(outVal)));
                        lastOutput = outVal;
                    } else {
                        p2 = p1;
                        p1 = p0;
                        c2 = c1;
                        c1 = c0;
                        float re = 0.0f, im = 0.0f;
#pragma unroll
                        for (int k = 0; k < 8; k++) {
                            re = __fadd_rn(re, __fmul_rn(src[2 * k], t8[k]));
                            im = __fadd_rn(im, __fmul_rn(src[2 * k + 1], t8[k]));
                        }
                        p0 = make_float2(re, im);
                        reinterpret_cast<float2*>(out)[total + outCount] = p0;
                        outCount++;
                        c0 = make_float2(mm_step(p0.x), mm_step(p0.y));
                        // (((p0 - p2) * conj(c1)) - ((c0 - c2) * conj(p1))).re, clock_recovery.h:181 with types.h:17-27
                        const float ar = __fsub_rn(p0.x, p2.x), ai = __fsub_rn(p0.y, p2.y);
                        const float dr = __fsub_rn(c0.x, c2.x), di = __fsub_rn(c0.y, c2.y);
                        const float ab = __fsub_rn(__fmul_rn(ar, c1.x), __fmul_rn(ai, -c1.y));
                        const float de = __fsub_rn(__fmul_rn(dr, p1.x), __fmul_rn(di, -p1.y));
                        phaseError = __fsub_rn(ab, de);
                    }
                    if (phaseError > 1.0f) phaseError = 1.0f;
                    if (phaseError < -1.0f) phaseError = -1.0f;
                    dynOmega = __fadd_rn(dynOmega, __fmul_rn(gainOmega, phaseError));
                    if (dynOmega > omegaMax) dynOmega = omegaMax;
                    else if (dynOmega < omegaMin) dynOmega = omegaMin;
                    mu = __fadd_rn(__fadd_rn(mu, dynOmega), __fmul_rn(muGain, phaseError));
                    const float roundedStep = floorf(mu);
                    i += (int)roundedStep;
                    if (i < 0) i = 0;
                    mu = __fsub_rn(mu, roundedStep);
                }
            }
            i = __shfl_sync(0xffffffffu, i, 0);
            outCount = __shfl_sync(0xffffffffu, outCount, 0);
            if (outCount >= maxOut) break;
            if (i >= w0 + 2 * kMmWin) w0 = i / kMmWin * kMmWin - kMmWin;   // a step longer than a window (huge omega)
        }
        nextOffset = i - count;                                    // clock_recovery.h:208
        if (lane == 0 && out_counts) out_counts[b] = outCount;
        total += outCount;
    }
    __syncwarp();
    // the call's last 7 samples become delay[0..6] (clock_recovery.h:211); shorter calls shift the old tail
    if (lane < 7) {
        const long long g = part.total - 7 + lane;
        float2 v;
        if (g >= 0) {
            if (CPLX) v = reinterpret_cast<const float2*>(in)[g];
            else v = make_float2(in[g], 0.f);
        } else {
            v = make_float2(state[16 + 2 * (int)(g + 7)], state[17 + 2 * (int)(g + 7)]);
        }
        __syncwarp(0x7f);
        state[16 + 2 * lane] = v.x;
        state[17 + 2 * lane] = v.y;
    }
    if (lane == 0) {
        state[0] = mu;
        state[1] = dynOmega;
        state[2] = lastOutput;
        state[3] = p0.x; state[4] = p0.y; state[5] = p1.x; state[6] = p1.y; state[7] = p2.x; state[8] = p2.y;
        state[9] = c0.x; state[10] = c0.y; state[11] = c1.x; state[12] = c1.y; state[13] = c2.x; state[14] = c2.y;
        state[15] = (float)nextOffset;
        *total_out = total;
    }
}

int launch_mm(int cplx, const void* in, const Partition& part, const float* taps_dev, float omega, float gainOmega,
              float muGain, float omegaMin, float omegaMax, float* state, void* out, int* out_counts_dev,
              long long* total_dev, cudaStream_t s) {
    if (cplx)
        mm_kernel<true><<<1, 32, 0, s>>>((const float*)in, part.view, taps_dev, omega, gainOmega, muGain, omegaMin, omegaMax,
                                         state, (float*)out, out_counts_dev, total_dev);
    else
        mm_kernel<false><<<1, 32, 0, s>>>((const float*)in, part.view, taps_dev, omega, gainOmega, muGain, omegaMin, omegaMax,
                                          state, (float*)out, out_counts_dev, total_dev);
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
