// qdsp_b200/csrc/k_spectrum.cu — Welch power spectrum of a cf32 stream for sm_100a: windowed N-point FFT frames
// (N = 64 .. 16384, hop apart), |X|^2, the mean of `average` consecutive frames per output row, FFT-shifted.
//
// Rows are a pure function of the stream, whatever the split into calls. The frames of a row are cut into slices of S
// frames (S from N and A only, spectrum_slice_len); a slice is summed in frame order, a row sums its slice sums in slice
// order. A CTA that runs G frames side by side (small N) gives frame k of a slice to lane k mod G, each lane sums its
// frames in order, and the slice sum adds the G lane sums in lane order. Every sum is sequential and continues from a
// carried value, so a call that ends mid-slice or mid-row stores the lane sums of the open slice and the running sum of
// the open row's finished slices, and the next call continues them to the same bits.
//
// spectrum_frames_kernel: one CTA per slice (or the part of it this call completes). Thread (lane g, column j) loads
// samples j + r N / 16 (r < 16) of its frame straight from global memory (coalesced across j), in the input format FMT
// (cf32, or cs16 / cs8 / cu8 words converted by the rule of iq_common.cuh), windows them and runs the first
// radix-16 pass in registers; the remaining passes are Stockham radix-16 passes (and one radix-2/4/8 pass for log2 N
// mod 4) through a padded shared-memory frame, twiddles from a float64-designed table. The last pass leaves 16 bins per
// thread, always the same ones, so the frame-order power sums stay in registers across the frames. Up to 512 threads a
// CTA, the next wave's samples are loaded while the current wave's passes run.
// spectrum_rows_kernel: sums the slice sums of each row in slice order, divides by A, stores FFT-shifted.
#include <math.h>
#include <new>
#include <vector>
#include "fft_common.cuh"
#include "iq_common.cuh"
#include "kernels.cuh"

namespace qdsp {

struct SpectrumPlan {
    int N = 0, logN = 0, hop = 0, A = 0, S = 0, spr = 0, G = 0;
    long long umax = 0;                 // slices per launch (scratch rows)
    float* window = nullptr;            // [N]
    float2* tw = nullptr;               // [N] e^{-j 2 pi k / N}
    float* open[2] = {nullptr, nullptr};    // [G][N] lane sums of the open slice (ping-pong)
    float* rowp[2] = {nullptr, nullptr};    // [N] running sum of the open row's finished slices (ping-pong)
    float2* tail[2] = {nullptr, nullptr};   // [2N] samples from the first incomplete frame on, as cf32 (ping-pong; the
                                            // second N: the head of an integer call, launch_spectrum)
    float* slices = nullptr;            // [umax][N] finished slice sums of one launch
    int cur = 0, tcur = 0;
    long long pos = 0;                  // samples seen
    long long frames_done = 0;          // frames summed
    long long tail0 = 0;                // stream position of tail[tcur][0]
};

struct SpecArgs {
    const void* in;                     // cf32, or integer pairs (the frames kernel's FMT)
    const float2* tail;
    long long pos, tail0;               // stream positions of in[0] and tail[0]
    long long fa, fb;                   // frames [fa, fb) of this launch
    long long s_a;                      // first slice of this launch
    int hop, A, S, spr;
    const float* window;
    const float2* tw;
    const float* open_in;
    float* open_out;
    float* slices;
    IqConv conv;                        // integer input
};

template <int LOGN>
struct SpGeom {
    static constexpr int N = 1 << LOGN;
    static constexpr int TPF = N / 16;                         // threads per frame
    static constexpr int G = TPF >= 128 ? 1 : 128 / TPF;       // frames side by side: at least 128 threads a CTA
    static constexpr int THREADS = TPF * G;
    static constexpr int MINB = THREADS >= 512 ? 1 : 512 / THREADS;   // at least 512 threads an SM: <= 128 registers
    static constexpr int RL = LOGN % 4 ? 1 << (LOGN % 4) : 16; // radix of the last pass
    static constexpr int P16 = LOGN / 4;                       // radix-16 passes, the first one included
    static constexpr int PADN = N + N / 16;                    // frame in shared memory, one pad word per 16
};
__device__ __forceinline__ int sp_pad(int p) { return p + (p >> 4); }

__host__ __device__ inline long long sp_slice_start(long long s, int A, int S, int spr) { return (s / spr) * A + (s % spr) * S; }
__host__ __device__ inline long long sp_slice_end(long long s, int A, int S, int spr) {
    const long long j = s % spr;
    return (s / spr) * A + ((j + 1) * S < A ? (j + 1) * S : A);
}
__host__ __device__ inline long long sp_slice_of(long long f, int A, int S, int spr) { return (f / A) * spr + (f % A) / S; }

// integer pair i of this call's input as its raw word (FMT QDSP_CS16: 32 bits; QDSP_CS8 / QDSP_CU8: 16), and a raw word
// converted by the rule of iq_common.cuh
template <int FMT>
__device__ __forceinline__ uint32_t sp_word(const void* in, long long i) {
    if (FMT == QDSP_CS16) return ldg_stream32(reinterpret_cast<const uint32_t*>(in) + i);
    return ldg_stream16(reinterpret_cast<const uint16_t*>(in) + i);
}
template <int FMT>
__device__ __forceinline__ float2 sp_convert(uint32_t w, IqConv c) {
    if (FMT == QDSP_CS16) return iq_cs16(w, c);
    const float4 v = iq_b8x2<FMT>(w, c);
    return make_float2(v.x, v.y);
}
// sample i of this call's input, as cf32: FMT is QDSP_CF32, QDSP_CS16, QDSP_CS8 or QDSP_CU8
template <int FMT>
__device__ __forceinline__ float2 sp_sample(const void* in, long long i, IqConv c) {
    if (FMT == QDSP_CF32) return ldg_stream64(reinterpret_cast<const float2*>(in) + i);
    return sp_convert<FMT>(sp_word<FMT>(in, i), c);
}

// the bin of accumulator e of column j after the last pass
template <int LOGN>
__device__ __forceinline__ int sp_bin(int j, int e) {
    using Gm = SpGeom<LOGN>;
    constexpr int RL = Gm::RL;
    return j + (e / RL) * Gm::TPF + (e % RL) * (Gm::N / RL);
}

template <int LOGN, int FMT>
__global__ void __launch_bounds__(SpGeom<LOGN>::THREADS, SpGeom<LOGN>::MINB) spectrum_frames_kernel(const SpecArgs a) {
    using Gm = SpGeom<LOGN>;
    constexpr int N = Gm::N, TPF = Gm::TPF, G = Gm::G, RL = Gm::RL;
    extern __shared__ __align__(16) unsigned char smem_sp[];
    const int t = threadIdx.x, g = t / TPF, j = t - g * TPF;
    float2* sm = reinterpret_cast<float2*>(smem_sp) + g * Gm::PADN;
    const long long s = a.s_a + blockIdx.x;
    const long long base = sp_slice_start(s, a.A, a.S, a.spr), send = sp_slice_end(s, a.A, a.S, a.spr);
    const long long ua = base > a.fa ? base : a.fa, ub = send < a.fb ? send : a.fb;
    // 1024 threads a CTA leave 64 registers a thread: there the power sums live in shared memory, after the frame
    constexpr bool SACC = Gm::THREADS > 512;
    float racc[SACC ? 1 : 16];
    float* sacc = reinterpret_cast<float*>(smem_sp + (size_t)G * Gm::PADN * sizeof(float2));
    auto acc = [&](int e) -> float& { return SACC ? sacc[e * Gm::THREADS + t] : racc[SACC ? 0 : e]; };
    const bool cont = ua > base;         // the slice was opened by an earlier launch: continue its lane sums
#pragma unroll
    for (int e = 0; e < 16; e++) acc(e) = cont ? a.open_in[g * N + sp_bin<LOGN>(j, e)] : 0.0f;
    const long long w0 = (ua - base) / G, w1 = (ub - 1 - base) / G;
    // samples j + r TPF of this lane's frame in wave wv (zeros for a lane without a frame in that wave)
    auto fetch = [&](long long wv, float2 (&x)[16]) {
        const long long f = base + wv * G + g;
        const bool live = f >= ua && f < ub;
        const long long q0 = f * a.hop + j;
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const long long q = q0 + r * TPF;
            x[r] = make_float2(0.f, 0.f);
            if (live) x[r] = q >= a.pos ? sp_sample<FMT>(a.in, q - a.pos, a.conv) : __ldg(a.tail + (q - a.tail0));
        }
    };
    // up to 512 threads a CTA: the next wave's samples are loaded while this wave's passes run (32 more registers; at
    // 1024 threads, 64 registers a thread, there is no room for them)
    constexpr bool PF = Gm::THREADS <= 512;
    // Integer input: the prefetch holds the raw words (16 registers instead of 32), converted when the wave is taken, so
    // the loads are in flight during the previous wave's passes (converted as they arrive, they would be waited for
    // before those passes). The integer kernels never take a frame that starts in the carried tail (launch_spectrum).
    constexpr bool RAW = PF && FMT != QDSP_CF32;
    auto fetch_raw = [&](long long wv, uint32_t (&w)[16]) {
        const long long f = base + wv * G + g;
        const bool live = f >= ua && f < ub;
        const long long i0 = f * a.hop + j - a.pos;
#pragma unroll
        for (int r = 0; r < 16; r++) {
            w[r] = 0;
            if (live) w[r] = sp_word<FMT>(a.in, i0 + r * TPF);
        }
    };
    float2 nx[RAW ? 1 : 16];
    uint32_t nw[RAW ? 16 : 1];
    if constexpr (RAW) fetch_raw(w0, nw);
    else if (PF) fetch(w0, nx);
#pragma unroll 1
    for (long long wv = w0; wv <= w1; wv++) {
        const long long f = base + wv * G + g;
        const bool live = f >= ua && f < ub;
        float2 v[16];
        if constexpr (RAW) {
#pragma unroll
            for (int r = 0; r < 16; r++) v[r] = sp_convert<FMT>(nw[r], a.conv);
            if (wv < w1) fetch_raw(wv + 1, nw);
        } else if (PF) {
#pragma unroll
            for (int r = 0; r < 16; r++) v[r] = nx[r];
            if (wv < w1) fetch(wv + 1, nx);
        } else {
            fetch(wv, v);
        }
        // pass 0 (Ns = 1): samples j + r TPF of the frame, windowed, one radix-16 DFT
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const float wr = __ldg(a.window + j + r * TPF);
            v[r] = make_float2(v[r].x * wr, v[r].y * wr);
        }
        fft16(v);
        __syncthreads();                 // the previous frame's last pass has read the shared frame
#pragma unroll
        for (int k = 0; k < 16; k++) sm[sp_pad(j * 16 + k)] = v[bitrev4(k)];
        // radix-16 Stockham passes: Ns = 16, 256, ...
        int Ns = 16;
#pragma unroll
        for (int p = 0; p < Gm::P16 - 1; p++) {
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 16; r++) v[r] = sm[sp_pad(j + r * TPF)];
            const int jm = j & (Ns - 1), step = N / (Ns * 16);
#pragma unroll
            for (int r = 1; r < 16; r++) v[r] = cmul(v[r], __ldg(a.tw + jm * r * step));
            fft16(v);
            const bool last = RL == 16 && p == Gm::P16 - 2;
            if (!last) {
                __syncthreads();
                const int d = (j - jm) * 16 + jm;
#pragma unroll
                for (int k = 0; k < 16; k++) sm[sp_pad(d + k * Ns)] = v[bitrev4(k)];
            }
            Ns *= 16;
        }
        if (RL == 16) {
            // the last radix-16 pass (Ns = N / 16 = TPF, so jm = j) left bin j + k TPF in v[bitrev4(k)]
            if (live) {
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const float2 X = v[bitrev4(k)];
                    acc(k) += fmaf(X.x, X.x, X.y * X.y);
                }
            }
        } else {
            // last pass, radix RL (Ns = N / RL): butterflies jj = j + qq TPF, bins jj + k N / RL
            __syncthreads();
#pragma unroll
            for (int qq = 0; qq < 16 / RL; qq++) {
                const int jj = j + qq * TPF;
                float2 u[RL];
#pragma unroll
                for (int r = 0; r < RL; r++) u[r] = sm[sp_pad(jj + r * (N / RL))];
#pragma unroll
                for (int r = 1; r < RL; r++) u[r] = cmul(u[r], __ldg(a.tw + jj * r));
                fft_radix<RL>(u);
                if (live) {
#pragma unroll
                    for (int k = 0; k < RL; k++) {
                        const float2 X = u[bitrev<RL>(k)];
                        acc(qq * RL + k) += fmaf(X.x, X.x, X.y * X.y);
                    }
                }
            }
        }
    }
    if (ub == send) {
        // the slice is complete: its sum is the lane sums added in lane order
        float* dst = a.slices + (size_t)blockIdx.x * N;
        if (G == 1) {
#pragma unroll
            for (int e = 0; e < 16; e++) dst[sp_bin<LOGN>(j, e)] = acc(e);
        } else {
            float* lanes = reinterpret_cast<float*>(smem_sp);    // [G][N]
            __syncthreads();
#pragma unroll
            for (int e = 0; e < 16; e++) lanes[g * N + sp_bin<LOGN>(j, e)] = acc(e);
            __syncthreads();
            for (int b = t; b < N; b += Gm::THREADS) {
                float sum = lanes[b];
#pragma unroll 1
                for (int l = 1; l < G; l++) sum += lanes[l * N + b];
                dst[b] = sum;
            }
        }
    } else {
#pragma unroll
        for (int e = 0; e < 16; e++) a.open_out[g * N + sp_bin<LOGN>(j, e)] = acc(e);
    }
}

struct SpecRowArgs {
    const float* slices;
    const float* row_in;
    float* row_out;
    float* out;
    long long s_a, s_done;              // first slice of the launch, one past its last finished slice
    long long r_a, r_out0;              // first row of the launch, first row of this call's output
    int N, A, spr;
};

// thread = (row, bin): the row's finished slice sums of this launch in slice order, after the carried ones
__global__ void __launch_bounds__(256) spectrum_rows_kernel(const SpecRowArgs a) {
    const int b = blockIdx.y * 256 + threadIdx.x;
    if (b >= a.N) return;
    const long long r = a.r_a + blockIdx.x;
    const long long s0 = r * a.spr, s1 = s0 + a.spr;           // the row's slices [s0, s1)
    const long long sb = s0 > a.s_a ? s0 : a.s_a, se = s1 < a.s_done ? s1 : a.s_done;
    float acc = a.s_a > s0 ? a.row_in[b] : 0.0f;
#pragma unroll 1
    for (long long s = sb; s < se; s++) acc += a.slices[(size_t)(s - a.s_a) * a.N + b];
    if (se == s1) a.out[(size_t)(r - a.r_out0) * a.N + ((b + (a.N >> 1)) & (a.N - 1))] = acc / (float)a.A;
    else a.row_out[b] = acc;
}

// ---- host side -------------------------------------------------------------------------------------
// Frames per slice: about 64 K samples of frames per slice whatever N is (enough CTAs for one long row at N = 16384,
// few slice sums to add at small N); a function of N and A only, never of the device or the call.
static int spectrum_slice_len(int N, int A) {
    const int s = 65536 / N;
    return A < s ? A : s;
}

// Integer input is read by the frames kernel itself, except where that kernel has no prefetch (N = 16384: 1024 threads at
// 64 registers, where even 16 raw words spill) and reads every sample (hop <= N). There the kernel is bound by its
// instructions, the conversion's instructions take as long as a conversion pass over the whole call, and the native read
// measured 0.2-0.3 % slower than that pass on cs8 / cu8 (DESIGN.md §6.0e): the handle converts first.
bool spectrum_native_integer(const SpectrumPlan* p) { return p->N / 16 <= 512 || p->hop > p->N; }

static long long sp_frames_complete(const SpectrumPlan* p, long long P) { return P >= p->N ? (P - p->N) / p->hop + 1 : 0; }

long long spectrum_out_rows(const SpectrumPlan* p, long long count) {
    if (count < 0) return -1;
    return sp_frames_complete(p, p->pos + count) / p->A - p->frames_done / p->A;
}

void spectrum_plan_destroy(SpectrumPlan* p) {
    if (!p) return;
    cudaFree(p->window);
    cudaFree(p->tw);
    for (int i = 0; i < 2; i++) {
        cudaFree(p->open[i]);
        cudaFree(p->rowp[i]);
        cudaFree(p->tail[i]);
    }
    cudaFree(p->slices);
    delete p;
}

SpectrumPlan* spectrum_plan_create(int N, const float* window, int hop, int A) {
    SpectrumPlan* p = new (std::nothrow) SpectrumPlan();
    if (!p) return nullptr;
    p->N = N;
    while ((1 << p->logN) < N) p->logN++;
    p->hop = hop;
    p->A = A;
    p->S = spectrum_slice_len(N, A);
    p->spr = (A + p->S - 1) / p->S;
    p->G = N / 16 >= 128 ? 1 : 128 / (N / 16);
    p->umax = ((long long)8 << 20) / N;   // 32 MB of slice sums per launch: stays in L2 for the row kernel
    std::vector<float> w(N, 1.0f);
    if (window)
        for (int i = 0; i < N; i++) w[i] = window[i];
    std::vector<float2> tw(N);
    for (int k = 0; k < N; k++) {
        const double ang = -6.283185307179586476925286766559 * (double)k / (double)N;
        tw[k] = make_float2((float)cos(ang), (float)sin(ang));
    }
    bool ok = cudaMalloc(&p->window, N * sizeof(float)) == cudaSuccess &&
              cudaMemcpy(p->window, w.data(), N * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc(&p->tw, N * sizeof(float2)) == cudaSuccess &&
              cudaMemcpy(p->tw, tw.data(), N * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc(&p->slices, (size_t)p->umax * N * sizeof(float)) == cudaSuccess;
    for (int i = 0; ok && i < 2; i++)
        ok = cudaMalloc(&p->open[i], (size_t)p->G * N * sizeof(float)) == cudaSuccess &&
             cudaMalloc(&p->rowp[i], N * sizeof(float)) == cudaSuccess && cudaMalloc(&p->tail[i], 2 * N * sizeof(float2)) == cudaSuccess;
    if (!ok) {
        set_last_error("spectrum_create: device allocation failed");
        spectrum_plan_destroy(p);
        return nullptr;
    }
    return p;
}

void spectrum_plan_reset(SpectrumPlan* p) {
    p->cur = p->tcur = 0;
    p->pos = p->frames_done = p->tail0 = 0;
}

template <int LOGN, int FMT>
static int sp_launch_frames(const SpecArgs& a, long long units, cudaStream_t s) {
    using Gm = SpGeom<LOGN>;
    const size_t smem = (size_t)Gm::G * Gm::PADN * sizeof(float2) + (Gm::THREADS > 512 ? (size_t)Gm::THREADS * 16 * sizeof(float) : 0);
    static bool attr_dev[64] = {};      // opt-in shared memory is a per-device function attribute
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_dev[dev & 63]) {
        QDSP_CUDA_OK(cudaFuncSetAttribute(spectrum_frames_kernel<LOGN, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_dev[dev & 63] = true;
    }
    spectrum_frames_kernel<LOGN, FMT><<<(unsigned)units, Gm::THREADS, smem, s>>>(a);
    QDSP_LAUNCH_OK();
    return 0;
}

template <int LOGN>
static int sp_launch_frames(int fmt, const SpecArgs& a, long long units, cudaStream_t s) {
    switch (fmt) {
        case QDSP_CF32: return sp_launch_frames<LOGN, QDSP_CF32>(a, units, s);
        case QDSP_CS16: return sp_launch_frames<LOGN, QDSP_CS16>(a, units, s);
        case QDSP_CS8: return sp_launch_frames<LOGN, QDSP_CS8>(a, units, s);
        case QDSP_CU8: return sp_launch_frames<LOGN, QDSP_CU8>(a, units, s);
    }
    return -1;
}

long long launch_spectrum(SpectrumPlan* p, const void* in, int fmt, IqConv conv, float* rows_out, long long count,
                          cudaStream_t s) {
    const int N = p->N;
    const long long pos_end = p->pos + count;
    const long long f_end = sp_frames_complete(p, pos_end);
    const long long r_out0 = p->frames_done / p->A;
    // Integer input: the frames [frames_done, f1) start in the carried tail (before this call's first sample) and end
    // before sample pos + min(count, N). They are taken by the cf32 kernel from the tail followed by this call's first
    // min(count, N) samples converted to cf32, the same cut as a call boundary; the integer kernels read this call's
    // input only, and need no registers for the tail.
    long long f1 = p->frames_done;
    const float2* head = nullptr;
    if (fmt != QDSP_CF32) {
        f1 = (p->pos + p->hop - 1) / p->hop;
        if (f1 > f_end) f1 = f_end;
        if (f1 > p->frames_done) {
            float2* h = p->tail[p->tcur] + (p->pos - p->tail0);   // pos - tail0 < N: the tail holds an incomplete frame
            if (launch_iq_convert(fmt, conv, in, h, count < N ? count : N, s) != 0) return -1;
            head = h;
        }
    }
    for (long long fa = p->frames_done; fa < f_end;) {
        const long long s_a = sp_slice_of(fa, p->A, p->S, p->spr);
        long long fb = sp_slice_start(s_a + p->umax, p->A, p->S, p->spr);
        if (fb > f_end) fb = f_end;
        const bool in_head = fa < f1;
        if (in_head && fb > f1) fb = f1;
        const long long s_b = sp_slice_of(fb - 1, p->A, p->S, p->spr);
        const long long s_done = sp_slice_end(s_b, p->A, p->S, p->spr) == fb ? s_b + 1 : s_b;
        SpecArgs a{};
        a.in = in_head ? head : in;
        a.tail = p->tail[p->tcur];
        a.pos = p->pos;
        a.tail0 = p->tail0;
        a.fa = fa;
        a.fb = fb;
        a.s_a = s_a;
        a.hop = p->hop;
        a.A = p->A;
        a.S = p->S;
        a.spr = p->spr;
        a.window = p->window;
        a.tw = p->tw;
        a.open_in = p->open[p->cur];
        a.open_out = p->open[p->cur ^ 1];
        a.slices = p->slices;
        a.conv = conv;
        const long long units = s_b - s_a + 1;
        const int kfmt = in_head ? QDSP_CF32 : fmt;
        int rc = -1;
        switch (p->logN) {
            case 6: rc = sp_launch_frames<6>(kfmt, a, units, s); break;
            case 7: rc = sp_launch_frames<7>(kfmt, a, units, s); break;
            case 8: rc = sp_launch_frames<8>(kfmt, a, units, s); break;
            case 9: rc = sp_launch_frames<9>(kfmt, a, units, s); break;
            case 10: rc = sp_launch_frames<10>(kfmt, a, units, s); break;
            case 11: rc = sp_launch_frames<11>(kfmt, a, units, s); break;
            case 12: rc = sp_launch_frames<12>(kfmt, a, units, s); break;
            case 13: rc = sp_launch_frames<13>(kfmt, a, units, s); break;
            case 14: rc = sp_launch_frames<14>(kfmt, a, units, s); break;
        }
        if (rc != 0) return -1;
        SpecRowArgs ra{};
        ra.slices = p->slices;
        ra.row_in = p->rowp[p->cur];
        ra.row_out = p->rowp[p->cur ^ 1];
        ra.out = rows_out;
        ra.s_a = s_a;
        ra.s_done = s_done;
        ra.r_a = s_a / p->spr;
        ra.r_out0 = r_out0;
        ra.N = N;
        ra.A = p->A;
        ra.spr = p->spr;
        const long long nrows = s_b / p->spr - ra.r_a + 1;
        spectrum_rows_kernel<<<dim3((unsigned)nrows, (N + 255) / 256), 256, 0, s>>>(ra);
        QDSP_LAUNCH_OK();
        p->cur ^= 1;
        fa = fb;
    }
    // carry the samples from the first incomplete frame on (fewer than N), converted to cf32: the format may change with
    // the next call
    const long long t0 = f_end * p->hop;
    if (t0 < pos_end) {
        float2* dst = p->tail[p->tcur ^ 1];
        long long off = 0;
        if (t0 < p->pos) {
            off = p->pos - t0;
            QDSP_CUDA_OK(cudaMemcpyAsync(dst, p->tail[p->tcur] + (t0 - p->tail0), off * sizeof(float2), cudaMemcpyDeviceToDevice, s));
        }
        const long long from = t0 > p->pos ? t0 - p->pos : 0;
        if (fmt == QDSP_CF32) {
            QDSP_CUDA_OK(cudaMemcpyAsync(dst + off, static_cast<const float2*>(in) + from, (count - from) * sizeof(float2),
                                         cudaMemcpyDeviceToDevice, s));
        } else if (launch_iq_convert(fmt, conv, static_cast<const char*>(in) + from * iq_pair_bytes(fmt), dst + off,
                                     count - from, s) != 0) {
            return -1;
        }
        p->tcur ^= 1;
    }
    p->tail0 = t0;
    p->pos = pos_end;
    const long long rows = f_end / p->A - r_out0;
    p->frames_done = f_end;
    return rows;
}

}  // namespace qdsp
