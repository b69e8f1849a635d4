// qdsp_b200/csrc/k_pointwise.cu — the reference's element-wise, layout and per-block-statistic blocks
// ("next" rows of the scope table): math.h Add/Substract/Multiply, audio.h, convertion.h, processing.h
// Volume / DelayImag / Squelch / Threshold, demodulator.h AMDemod / SSBDemod.
// All are HBM-bound streaming passes: 128-bit accesses where the layout allows, grid-stride over a grid
// sized in multiples of the SM count. Arithmetic uses the reference's operation order with every
// product and sum rounded separately (the x86-64 reference has no FMA), so the results are bit-exact
// except where a block reduces over a whole run() call (AMDemod / Squelch mean: summed in double here,
// sequentially in float by the reference).
#include "internal.cuh"
#include "kernels.cuh"

namespace qdsp {

static int pw_sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}
static int pw_grid(long long work_items, int threads, int ctas_per_sm) {
    long long g = (work_items + threads - 1) / threads;
    const long long cap = (long long)pw_sm_count() * ctas_per_sm;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---- math.h: Add / Substract / Multiply (reference math.h:21-43, 68-90, 115-137) ---------------------
// op 0/1/2 = a+b / a-b / a*b over n floats; op 3 = complex multiply over n complex samples
// (volk_32fc_x2_multiply_32fc: (ar*br - ai*bi, ar*bi + ai*br)).
template <int OP>
__device__ __forceinline__ float math_op(float a, float b) {
    return OP == 0 ? __fadd_rn(a, b) : (OP == 1 ? __fsub_rn(a, b) : __fmul_rn(a, b));
}
template <int OP>
__global__ void __launch_bounds__(256) math_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                   float* __restrict__ out, long long n, int vec) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nq = vec ? (n >> 2) : 0;
    for (long long q = tid; q < nq; q += stride) {
        const float4 x = ldg_stream128(reinterpret_cast<const float4*>(a) + q);
        const float4 y = ldg_stream128(reinterpret_cast<const float4*>(b) + q);
        float4 r;
        if (OP == 3) {
            const float2 r0 = cmul_exact(make_float2(x.x, x.y), make_float2(y.x, y.y));
            const float2 r1 = cmul_exact(make_float2(x.z, x.w), make_float2(y.z, y.w));
            r = make_float4(r0.x, r0.y, r1.x, r1.y);
        } else {
            r = make_float4(math_op<OP>(x.x, y.x), math_op<OP>(x.y, y.y), math_op<OP>(x.z, y.z), math_op<OP>(x.w, y.w));
        }
        reinterpret_cast<float4*>(out)[q] = r;
    }
    // scalar tail (and the whole range when a pointer is not 16-byte aligned)
    if (OP == 3) {
        for (long long i = (nq << 1) + tid; i < (n >> 1); i += stride) {
            const float2 r = cmul_exact(reinterpret_cast<const float2*>(a)[i], reinterpret_cast<const float2*>(b)[i]);
            reinterpret_cast<float2*>(out)[i] = r;
        }
    } else {
        for (long long i = (nq << 2) + tid; i < n; i += stride) out[i] = math_op<OP>(a[i], b[i]);
    }
}
int launch_math(int op, int complex_mul, const float* a, const float* b, float* out, long long nfloats, cudaStream_t s) {
    if (nfloats <= 0) return 0;
    const int vec = aligned16(a) && aligned16(b) && aligned16(out);
    const int g = pw_grid(nfloats / 4 + 1, 256, 8);
    if (op == 2 && complex_mul) math_kernel<3><<<g, 256, 0, s>>>(a, b, out, nfloats, vec);
    else if (op == 0) math_kernel<0><<<g, 256, 0, s>>>(a, b, out, nfloats, vec);
    else if (op == 1) math_kernel<1><<<g, 256, 0, s>>>(a, b, out, nfloats, vec);
    else if (op == 2) math_kernel<2><<<g, 256, 0, s>>>(a, b, out, nfloats, vec);
    else {
        set_last_error("math: unknown op %d", op);
        return -1;
    }
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- audio.h / convertion.h layout shuffles ----------------------------------------------------------
// mode 0: out0[i] = {in0[i], in1 ? in1[i] : fill}   (MonoToStereo: in1 == in0; ChannelsToStereo; RealToComplex: fill 0)
// mode 1: out0[i] = (in0[i].l + in0[i].r) * 0.5f    (StereoToMono, audio.h:129-131)
// mode 2: out0[i] = in0[i].re, out1[i] = in0[i].im  (StereoToChannels / ComplexToReal / ComplexToImag: either may be null)
__global__ void __launch_bounds__(256) layout_kernel(int mode, const float* __restrict__ in0, const float* __restrict__ in1,
                                                     float* __restrict__ out0, float* __restrict__ out1, long long count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += stride) {
        if (mode == 0) {
            reinterpret_cast<float2*>(out0)[i] = make_float2(in0[i], in1 ? in1[i] : 0.0f);
        } else if (mode == 1) {
            const float2 v = reinterpret_cast<const float2*>(in0)[i];
            out0[i] = __fmul_rn(__fadd_rn(v.x, v.y), 0.5f);
        } else {
            const float2 v = reinterpret_cast<const float2*>(in0)[i];
            if (out0) out0[i] = v.x;
            if (out1) out1[i] = v.y;
        }
    }
}
int launch_layout(int mode, const float* in0, const float* in1, float* out0, float* out1, long long count, cudaStream_t s) {
    if (count <= 0) return 0;
    layout_kernel<<<pw_grid(count, 256, 8), 256, 0, s>>>(mode, in0, in1, out0, out1, count);
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- Volume<T>::run (processing.h:388-411): out = in * level, or zeros when muted ----------------------
__global__ void __launch_bounds__(256) scale_kernel(const float* __restrict__ in, float* __restrict__ out, long long n,
                                                    float level, int vec) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nq = vec ? (n >> 2) : 0;
    for (long long q = tid; q < nq; q += stride) {
        const float4 x = ldg_stream128(reinterpret_cast<const float4*>(in) + q);
        reinterpret_cast<float4*>(out)[q] =
            make_float4(__fmul_rn(x.x, level), __fmul_rn(x.y, level), __fmul_rn(x.z, level), __fmul_rn(x.w, level));
    }
    for (long long i = (nq << 2) + tid; i < n; i += stride) out[i] = __fmul_rn(in[i], level);
}
int launch_scale(const float* in, float* out, long long nfloats, float level, cudaStream_t s) {
    if (nfloats <= 0) return 0;
    scale_kernel<<<pw_grid(nfloats / 4 + 1, 256, 8), 256, 0, s>>>(in, out, nfloats, level, aligned16(in) && aligned16(out));
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- Threshold::run (processing.h:593-595): out[i] = in[i] > 0.0f, uint8 --------------------------------
__global__ void __launch_bounds__(256) threshold_kernel(const float* __restrict__ in, unsigned char* __restrict__ out,
                                                        long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) out[i] = in[i] > 0.0f ? 1 : 0;
}
int launch_threshold(const float* in, unsigned char* out, long long n, cudaStream_t s) {
    if (n <= 0) return 0;
    threshold_kernel<<<pw_grid(n, 256, 8), 256, 0, s>>>(in, out, n);
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- DelayImag::run (processing.h:325-330): out[i] = {in[i].re, in[i-1].im}, carried lastIm -------------
__global__ void __launch_bounds__(256) delay_imag_kernel(const float2* __restrict__ in, float2* __restrict__ out,
                                                         long long count, const float* __restrict__ state_in,
                                                         float* __restrict__ state_out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += stride) {
        const float2 v = in[i];
        const float im = i > 0 ? in[i - 1].y : *state_in;
        out[i] = make_float2(v.x, im);
        if (i == count - 1) *state_out = v.y;
    }
}
int launch_delay_imag(const float2* in, float2* out, long long count, const float* state_in, float* state_out,
                      cudaStream_t s) {
    if (count <= 0) return 0;
    delay_imag_kernel<<<pw_grid(count, 256, 8), 256, 0, s>>>(in, out, count, state_in, state_out);
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- per-run()-block mean magnitude (AMDemod demodulator.h:359-371, Squelch processing.h:465-468) -------
// volk_32fc_magnitude_32f: sqrtf(re*re + im*im), products and sum rounded separately.
__device__ __forceinline__ float mag_ref(float2 v) {
    return __fsqrt_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)));
}
constexpr int kMagPartsMax = 128;   // partial sums per run() block (a fixed function of the partition: deterministic order)

// pass 1: partial sums of the magnitudes of block b0 + blockIdx.y, part blockIdx.x (double accumulation); optionally
// writes the magnitudes
__global__ void __launch_bounds__(256) mag_partial_kernel(const float2* __restrict__ in, PartitionDev part, int b0, int parts,
                                                          float* __restrict__ mag_out, double* __restrict__ partial) {
    const int b = b0 + blockIdx.y;
    const BlkInfo bi = part.get(b);
    const float2* x = in + bi.in_start;
    float* m = mag_out ? mag_out + bi.in_start : nullptr;
    double acc = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < bi.count; i += gridDim.x * blockDim.x) {
        const float v = mag_ref(x[i]);
        if (m) m[i] = v;
        acc += (double)v;
    }
    __shared__ double s_w[8];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += s_w[w];
        partial[(size_t)b * parts + blockIdx.x] = t;
    }
}
__device__ __forceinline__ float block_mean(const double* __restrict__ partial, int b, int parts, int count) {
    double t = 0.0;
    for (int p = 0; p < parts; p++) t += partial[(size_t)b * parts + p];
    return __fdiv_rn((float)t, (float)count);   // avg /= (float)count, demodulator.h:366 / processing.h:468
}
// AMDemod pass 2: out[i] = mag[i] - mean(block) (in place on the magnitudes pass 1 wrote)
__global__ void __launch_bounds__(256) am_finish_kernel(float* __restrict__ out, PartitionDev part, int b0, int parts,
                                                        const double* __restrict__ partial) {
    const int b = b0 + blockIdx.y;
    const BlkInfo bi = part.get(b);
    const float avg = block_mean(partial, b, parts, bi.count);
    float* y = out + bi.in_start;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < bi.count; i += gridDim.x * blockDim.x)
        y[i] = __fsub_rn(y[i], avg);
}
// Squelch pass 2: copy the block if 10*log10f(mean) >= level, zeros otherwise
__global__ void __launch_bounds__(256) squelch_finish_kernel(const float2* __restrict__ in, float2* __restrict__ out,
                                                             PartitionDev part, int b0, int parts,
                                                             const double* __restrict__ partial, float level) {
    const int b = b0 + blockIdx.y;
    const BlkInfo bi = part.get(b);
    const float mean = block_mean(partial, b, parts, bi.count);
    const bool open = __fmul_rn(10.0f, log10f(mean)) >= level;
    const float2* x = in + bi.in_start;
    float2* y = out + bi.in_start;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < bi.count; i += gridDim.x * blockDim.x)
        y[i] = open ? x[i] : make_float2(0.0f, 0.0f);
}
size_t mag_scratch_bytes(int nblocks) { return sizeof(double) * kMagPartsMax * (size_t)(nblocks > 0 ? nblocks : 1); }

// The two passes run over groups of run() blocks (grid.y <= 65535 blocks, `budget_samples` samples per group).
// Measured on B200 (2^26 samples, run() blocks of 1e6): L2-sized groups (5-6 Mi samples, so that pass 2 re-reads from
// the 126 MB L2) take 0.64-0.73 ms against 0.33 ms for one group -- 22 short dependent launches lose more to
// ramp-up/tail than the saved DRAM pass gains -- so the budget is unlimited.
static long long blk_start(const Partition& p, int b) {
    if (b >= p.view.nblocks) return p.view.total;
    return p.view.table ? p.host[b].in_start : (long long)b * p.view.block_size;
}
template <class P1, class P2>
static int for_block_groups(const Partition& part, long long budget_samples, P1 pass1, P2 pass2) {
    const int nb = part.view.nblocks;
    // 32 partial sums per run() block and 256 CTAs per block in pass 2 measured best for 1e6-sample blocks (202 / 200 GS/s
    // for AMDemod / Squelch; 128 parts and 512 CTAs: 139 / 142); short blocks get fewer parts
    int parts = (part.max_count + 8191) / 8192;
    parts = parts < 1 ? 1 : (parts > 32 ? 32 : parts);
    int gx = (part.max_count + 255) / 256;
    gx = gx < 1 ? 1 : (gx > 256 ? 256 : gx);
    for (int b0 = 0; b0 < nb;) {
        int b1 = b0 + 1;
        while (b1 < nb && b1 - b0 < 65535 && blk_start(part, b1 + 1) - blk_start(part, b0) <= budget_samples) b1++;
        if (pass1(b0, b1 - b0, parts) != 0) return -1;
        if (pass2(b0, b1 - b0, parts, gx) != 0) return -1;
        b0 = b1;
    }
    return 0;
}
int launch_amdemod(const float2* in, float* out, const Partition& part, double* partial, cudaStream_t s) {
    if (part.view.nblocks <= 0) return 0;
    return for_block_groups(
        part, 1ll << 62,
        [&](int b0, int n, int parts) {
            mag_partial_kernel<<<dim3(parts, n), 256, 0, s>>>(in, part.view, b0, parts, out, partial);
            QDSP_LAUNCH_OK();
            return 0;
        },
        [&](int b0, int n, int parts, int gx) {
            am_finish_kernel<<<dim3(gx, n), 256, 0, s>>>(out, part.view, b0, parts, partial);
            QDSP_LAUNCH_OK();
            return 0;
        });
}
int launch_squelch(const float2* in, float2* out, const Partition& part, double* partial, float level, cudaStream_t s) {
    if (part.view.nblocks <= 0) return 0;
    return for_block_groups(
        part, 1ll << 62,
        [&](int b0, int n, int parts) {
            mag_partial_kernel<<<dim3(parts, n), 256, 0, s>>>(in, part.view, b0, parts, nullptr, partial);
            QDSP_LAUNCH_OK();
            return 0;
        },
        [&](int b0, int n, int parts, int gx) {
            squelch_finish_kernel<<<dim3(gx, n), 256, 0, s>>>(in, out, part.view, b0, parts, partial, level);
            QDSP_LAUNCH_OK();
            return 0;
        });
}

// ---- SSBDemod::run (demodulator.h:479-482): VOLK rotator, then the real part ----------------------------
// Same closed-form NCO as the translator; only re(in * phase) is formed and stored (12 B per sample).
__global__ void __launch_bounds__(256) ssb_kernel(const float2* __restrict__ in, float* __restrict__ out, long long count,
                                                  uint64_t phase0, uint64_t step, float2 inc1, float2 inc2, float2 inc3) {
    const long long nquad = count >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < nquad; q += stride) {
        const long long n = q << 2;
        const float4 a = ldg_stream128(reinterpret_cast<const float4*>(in + n));
        const float4 b = ldg_stream128(reinterpret_cast<const float4*>(in + n + 2));
        const float2 p0 = phasor_from_turns(phase0 + step * (uint64_t)n);
        const float2 p1 = cmul(p0, inc1), p2 = cmul(p0, inc2), p3 = cmul(p0, inc3);
        float4 y;
        y.x = __fsub_rn(__fmul_rn(a.x, p0.x), __fmul_rn(a.y, p0.y));
        y.y = __fsub_rn(__fmul_rn(a.z, p1.x), __fmul_rn(a.w, p1.y));
        y.z = __fsub_rn(__fmul_rn(b.x, p2.x), __fmul_rn(b.y, p2.y));
        y.w = __fsub_rn(__fmul_rn(b.z, p3.x), __fmul_rn(b.w, p3.y));
        reinterpret_cast<float4*>(out)[q] = y;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (long long n = nquad << 2; n < count; n++) {
            const float2 p = phasor_from_turns(phase0 + step * (uint64_t)n);
            out[n] = __fsub_rn(__fmul_rn(in[n].x, p.x), __fmul_rn(in[n].y, p.y));
        }
    }
}
int launch_ssb(const float2* in, float* out, long long count, uint64_t phase0, uint64_t step, float2 inc1, float2 inc2,
               float2 inc3, cudaStream_t s) {
    if (count <= 0) return 0;
    if (!aligned16(in) || !aligned16(out)) {
        set_last_error("ssbdemod: buffers must be 16-byte aligned");
        return -1;
    }
    ssb_kernel<<<pw_grid(count / 4 + 1, 256, 8), 256, 0, s>>>(in, out, count, phase0, step, inc1, inc2, inc3);
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- SineSource::run (source.h:56): VOLK rotator over a buffer of ones == the NCO phasor itself -----------
__global__ void __launch_bounds__(256) sine_kernel(float2* __restrict__ out, long long count, uint64_t phase0, uint64_t step,
                                                   float2 inc1, float2 inc2, float2 inc3) {
    const long long nquad = (count + 3) >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < nquad; q += stride) {
        const long long n = q << 2;
        const float2 p0 = phasor_from_turns(phase0 + step * (uint64_t)n);
        const float2 p[4] = {p0, cmul(p0, inc1), cmul(p0, inc2), cmul(p0, inc3)};
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (n + j < count) out[n + j] = p[j];
    }
}
int launch_sine(float2* out, long long count, uint64_t phase0, uint64_t step, float2 inc1, float2 inc2, float2 inc3,
                cudaStream_t s) {
    if (count <= 0) return 0;
    sine_kernel<<<pw_grid(count / 4 + 1, 256, 8), 256, 0, s>>>(out, count, phase0, step, inc1, inc2, inc3);
    QDSP_LAUNCH_OK();
    return 0;
}

// ---- integer IQ -> cf32 (qdsp_iq_convert_process) ----------------------------------------------------------------------
// The one conversion rule of the library: y = (float(x) + offset) * scale, each step rounded to float32 (numpy:
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
// Two samples per thread: one 8-byte (cs16) or 4-byte (8-bit) load and one 16-byte store, so a warp's loads and stores
// each cover one contiguous range. That needs the pair of samples aligned in the input and 16-byte aligned in the
// output from sample `head` (0 or 1) on; the head, the odd tail, and everything when the two alignments disagree, go
// one sample per thread (still contiguous across the warp).
template <int FMT>
__global__ void __launch_bounds__(256) iq_convert_kernel(const void* __restrict__ in, float2* __restrict__ out, long long count,
                                                         long long head, long long npairs, IqConv c) {
    constexpr int E = FMT == QDSP_CS16 ? 4 : 2;   // input bytes per sample
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const char* in2 = reinterpret_cast<const char*>(in) + head * E;
    float4* out2 = reinterpret_cast<float4*>(out + head);
    for (long long p = tid; p < npairs; p += stride) {
        float4 v;
        if (FMT == QDSP_CS16) {
            const uint2 w = __ldcs(reinterpret_cast<const uint2*>(in2) + p);
            const float2 s0 = iq_cs16(w.x, c), s1 = iq_cs16(w.y, c);
            v = make_float4(s0.x, s0.y, s1.x, s1.y);
        } else {
            v = iq_b8x2<FMT>(__ldcs(reinterpret_cast<const unsigned int*>(in2) + p), c);
        }
        out2[p] = v;
    }
    const long long tail0 = head + 2 * npairs;
    for (long long i = tid; i < head + (count - tail0); i += stride) {
        const long long j = i < head ? i : tail0 + (i - head);
        out[j] = iq_one<FMT>(in, j, c);
    }
}
int launch_iq_convert(int fmt, IqConv c, const void* in, float2* out, long long count, cudaStream_t s) {
    if (count <= 0) return 0;
    const int E = iq_pair_bytes(fmt);
    const long long head = (reinterpret_cast<uintptr_t>(in) % (2 * E)) ? 1 : 0;
    long long npairs = count > head ? (count - head) / 2 : 0;
    if (!aligned16(out + head)) npairs = 0;
    const int g = pw_grid(npairs > 0 ? npairs : count, 256, 8);
    if (fmt == QDSP_CS16) iq_convert_kernel<QDSP_CS16><<<g, 256, 0, s>>>(in, out, count, head, npairs, c);
    else if (fmt == QDSP_CS8) iq_convert_kernel<QDSP_CS8><<<g, 256, 0, s>>>(in, out, count, head, npairs, c);
    else iq_convert_kernel<QDSP_CU8><<<g, 256, 0, s>>>(in, out, count, head, npairs, c);
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
