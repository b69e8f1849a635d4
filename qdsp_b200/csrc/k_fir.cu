// qdsp_b200/csrc/k_fir.cu — dense complex FIR for sm_100a (FIR<complex_t>::run, reference
// src/dsp/filter.h:51-74): y[n] = sum_j taps[j] * x[n - (T-1) + j], cf32 samples, real taps.
//
// Three kernels, all FP32-bound (4*T flop per sample) and built around the packed FFMA2 pipe:
//   fir_cplx_kernel<T, K>   T = 63 / 127 / 255 (config 1a): taps in the constant bank, tap loop fully unrolled
//   fir_longcplx_kernel     256 ... 4095 taps (config 3): taps in the constant bank, groups of 36 at a uniform offset
//       both: packed operand = the sample (re, im) as it lies in the raw TMA window, tap = scalar uniform-register
//       operand, nine-sample sliding register window (see the comments at the kernels, and DESIGN.md 6.2)
//   fir_dense_kernel        any other case (longer filters, input not 16-byte aligned); also the engine of the
//       small-decimation variant fir_decim_kernel. Its scheme:
//   * samples are staged in shared memory as quads (re[2m], re[2m+1], im[2m], im[2m+1]); taps as pairs
//     (h[2u], h[2u+1]). One FFMA2 then performs two real MACs of the SAME output,
//         accRe += (re[2m], re[2m+1]) * (h[2u], h[2u+1])     (lanes summed once at the end)
//     so no register holds a duplicated tap and every FFMA2 does two useful MACs.
//   * outputs whose window starts on an odd sample use a second tap table shifted by one
//     (h[2u-1], h[2u]); a warp works on one parity, so tap loads are warp-uniform broadcasts.
//   * each thread owns R = 9 outputs (stride 2) and slides a 9-quad register window over the taps:
//     one 128-bit shared load + one broadcast tap load per 18 FFMA2. R odd makes the lane stride
//     9*16 B, which is conflict-free for 128-bit shared loads.
//   * the whole input window of a tile stays resident (NOUT + T - 1 samples), so the tap loop runs
//     without any block-level barrier; two CTAs per SM overlap one tile's staging with the other's math.
#include <stdlib.h>
#include <mutex>
#include <new>
#include <vector>
#include "decim_common.cuh"

namespace qdsp {

constexpr int kFirR = 9;                        // outputs per thread
constexpr int kFirWarps = 8;                    // 4 even-parity + 4 odd-parity warps
constexpr int kFirThreads = kFirWarps * 32;
constexpr int kFirNout = (kFirWarps / 2) * 64 * kFirR;   // 2304 outputs per tile

struct FirPlan {
    int T = 0;
    int U = 0;                  // tap pairs per parity table
    float2* taps_dev = nullptr; // [2][U]: even table (h[2u], h[2u+1]); odd table (h[2u-1], h[2u])
    float taps_host[256] = {};  // T <= 255: the taps again, for the constant-bank kernel (fir_cplx_kernel)
    std::vector<float> taps_long;   // 255 < T <= 4095: the same for fir_longcplx_kernel
};

FirPlan* fir_plan_create(const float* taps, int T) {
    if (T < 2) return nullptr;
    FirPlan* p = new (std::nothrow) FirPlan();
    if (!p) return nullptr;
    p->T = T;
    if (T <= 255)
        for (int j = 0; j < T; j++) p->taps_host[j] = taps[j];
    else if (T <= 4095)
        p->taps_long.assign(taps, taps + T);
    int U = (T + 2) / 2;                        // enough pairs for the odd table's extra leading zero
    const int Upad = ((U + kFirR - 1) / kFirR) * kFirR;
    if ((Upad - U) * 33 <= U) U = Upad;         // long filters: round up to whole groups of R (< 3 % more work, leaner kernel);
    p->U = U;                                   // short ones end inside the last group (127 taps: 64 pairs, not 72)
    // shared memory: quads for NOUT/2 + U pairs (+ slack) and both tap tables
    const size_t smem = ((size_t)kFirNout / 2 + U + 8) * 16 + (size_t)2 * U * 8;
    if (smem > 110 * 1024) {                    // keep two CTAs per SM; longer filters use the generic kernel
        delete p;
        return nullptr;
    }
    std::vector<float2> tab((size_t)2 * U, make_float2(0.f, 0.f));
    auto h = [&](int j) { return (j >= 0 && j < T) ? taps[j] : 0.0f; };
    for (int u = 0; u < U; u++) {
        tab[u] = make_float2(h(2 * u), h(2 * u + 1));
        tab[(size_t)U + u] = make_float2(h(2 * u - 1), h(2 * u));
    }
    if (cudaMalloc(&p->taps_dev, tab.size() * sizeof(float2)) != cudaSuccess ||
        cudaMemcpy(p->taps_dev, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("fir_plan_create: tap upload failed");
        delete p;
        return nullptr;
    }
    return p;
}
void fir_plan_destroy(FirPlan* p) {
    if (!p) return;
    if (p->taps_dev) cudaFree(p->taps_dev);
    delete p;
}

// a tile of kFirNout outputs parked in shared memory -> global, 128-bit stores when the destination allows
template <int NT = kFirThreads, int NOUT = kFirNout>
__device__ __forceinline__ void store_tile(const float2* so, float2* __restrict__ out, long long first, long long limit) {
    const int t = threadIdx.x;
    const long long left = limit - first;
    const int nvalid = left < NOUT ? (int)left : NOUT;
    float2* dst = out + first;
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        const int nq = nvalid >> 1;
        for (int q = t; q < nq; q += NT)
            reinterpret_cast<float4*>(dst)[q] = reinterpret_cast<const float4*>(so)[q];
        if (t == 0 && (nvalid & 1)) dst[nvalid - 1] = so[nvalid - 1];
    } else {
        for (int i = t; i < nvalid; i += NT) dst[i] = so[i];
    }
}

template <int NW, bool TAIL>
__global__ void __launch_bounds__(NW * 32, NW == 8 ? 2 : 4)
fir_dense_kernel(VStream<float2> xs, long long count, const float2* __restrict__ taps, int T, int U,
                 float2* __restrict__ out) {
    constexpr int R = kFirR;
    constexpr int NT = NW * 32, NOUT = (NW / 2) * 64 * kFirR;   // threads, outputs per tile
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int npairs = NOUT / 2 + U + 8;
    float4* sq = reinterpret_cast<float4*>(smem_raw);                 // [npairs] sample quads
    float2* st = reinterpret_cast<float2*>(smem_raw + (size_t)npairs * 16);  // [2][U] tap pairs
    const int t = threadIdx.x;
    const long long n_t = (long long)blockIdx.x * NOUT;           // first output of the tile
    const long long B = n_t - (T - 1);                                // sample index of quad 0, element 0

    // ---- staging: taps, then the tile's window as (re, re, im, im) quads --------------------------
    // interior tiles whose window starts on an even sample: ONE TMA bulk copy drops the raw interleaved window
    // (re0, im0, re1, im1 per 16 bytes) into the quad array -- the whole tile in flight at once, no staging registers --
    // and every thread then swaps the two middle floats of its quads in place
    __shared__ uint64_t s_mbar;
    const bool tma_tile = (B & 1) == 0 && (reinterpret_cast<uintptr_t>(xs.in) & 15) == 0 && B >= 0 &&
                          B + 2 * (long long)npairs <= count;
    if (tma_tile) {
        if (t == 0) {
            mbar_init(&s_mbar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (t == 0) {
            mbar_arrive_expect_tx(&s_mbar, (uint32_t)npairs * 16u);
            tma_bulk_g2s(sq, xs.in + B, (uint32_t)npairs * 16u, &s_mbar);
        }
    }
    for (int i = t; i < 2 * U; i += NT) st[i] = taps[i];
    if (tma_tile) {
        mbar_wait(&s_mbar, 0);
        for (int q = t; q < npairs; q += NT) {
            const float4 a = sq[q];
            sq[q] = make_float4(a.x, a.z, a.y, a.w);
        }
    } else if ((B & 1) == 0 && (reinterpret_cast<uintptr_t>(xs.in) & 15) == 0) {
        // the window starts on an even sample (odd tap counts): one 128-bit load -> one quad, 4 in flight per thread
        for (int q0 = t; q0 < npairs; q0 += 4 * NT) {
            float4 a[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int q = q0 + j * NT;
                const long long i0 = B + 2 * (long long)q;
                if (q < npairs && i0 >= 0 && i0 + 2 <= count) {
                    a[j] = ldg_stream128(reinterpret_cast<const float4*>(xs.in + i0));
                } else {
                    const float2 v0 = (q < npairs && i0 < count) ? xs.at(i0) : make_float2(0.f, 0.f);
                    const float2 v1 = (q < npairs && i0 + 1 < count) ? xs.at(i0 + 1) : make_float2(0.f, 0.f);
                    a[j] = make_float4(v0.x, v0.y, v1.x, v1.y);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int q = q0 + j * NT;
                if (q < npairs) sq[q] = make_float4(a[j].x, a[j].z, a[j].y, a[j].w);
            }
        }
    } else {
        float* sf = reinterpret_cast<float*>(sq);
        const int nsamp = 2 * npairs;
        // batches of 8 loads per thread in flight together (a one-at-a-time loop exposes the DRAM latency 8x)
        for (int e0 = t; e0 < nsamp; e0 += 8 * NT) {
            float2 v[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                const long long i = B + e;
                v[j] = (e < nsamp && i < count) ? xs.at(i) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                if (e < nsamp) {
                    const int q = e >> 1, h = e & 1;
                    sf[4 * q + h] = v[j].x;
                    sf[4 * q + 2 + h] = v[j].y;
                }
            }
        }
    }
    __syncthreads();

    // ---- roles: warp w: parity = w & 1, warp-pair wp = w >> 1 covers 64*R consecutive outputs ----------
    const int w = t >> 5, lane = t & 31;
    const int parity = w & 1, wp = w >> 1;
    const int j0 = wp * 32 * R + lane * R;        // first pair index of this thread's window (u = 0)
    const float2* tt = st + parity * U;
    const float4* win = sq + j0;

    float2 accRe[R], accIm[R];
    float4 W[R];
#pragma unroll
    for (int i = 0; i < R; i++) {
        accRe[i] = make_float2(0.f, 0.f);
        accIm[i] = make_float2(0.f, 0.f);
        W[i] = win[i];
    }
    // output i accumulates H_u (.) S_{j0 + i + u}; window register W[(u + i) % R] holds S_{j0 + i + u}
    const int Ufull = (U / R) * R;
#pragma unroll 1
    for (int u0 = 0; u0 < Ufull; u0 += R) {
#pragma unroll
        for (int k = 0; k < R; k++) {
            const float2 hh = tt[u0 + k];
#pragma unroll
            for (int i = 0; i < R; i++) {
                const float4 s = W[(k + i) % R];
                accRe[i] = __ffma2_rn(make_float2(s.x, s.y), hh, accRe[i]);
                accIm[i] = __ffma2_rn(make_float2(s.z, s.w), hh, accIm[i]);
            }
            W[k] = win[u0 + k + R];               // S_{j0 + (u0+k+1) + (R-1)} replaces S_{j0 + u0 + k}
        }
    }
    // the last, partial group of R (TAIL: U is not a multiple of R -- 127 taps are 64 pairs, not 72)
#pragma unroll
    for (int k = 0; k < R - 1; k++) {
        if (TAIL && Ufull + k < U) {
            const float2 hh = tt[Ufull + k];
#pragma unroll
            for (int i = 0; i < R; i++) {
                const float4 s = W[(k + i) % R];
                accRe[i] = __ffma2_rn(make_float2(s.x, s.y), hh, accRe[i]);
                accIm[i] = __ffma2_rn(make_float2(s.z, s.w), hh, accIm[i]);
            }
            W[k] = win[Ufull + k + R];
        }
    }
    // ---- store: outputs n = n_t + 2*(j0 + i) + parity. A thread's outputs are 16 bytes apart and the lanes 144:
    // exchange them through the (now dead) sample window so that the tile leaves as coalesced 128-bit stores ----
    __syncthreads();
    float2* so = reinterpret_cast<float2*>(smem_raw);                 // [NOUT], 18 KB <= the window's footprint
#pragma unroll
    for (int i = 0; i < R; i++)
        so[2 * (j0 + i) + parity] = make_float2(accRe[i].x + accRe[i].y, accIm[i].x + accIm[i].y);
    __syncthreads();
    store_tile<NT, NOUT>(so, out, n_t, count);
}

// =================================================================================================
// Decimating variant (PolyphaseResampler with interp = 1 and a small decimation D, e.g. config 1b: D = 4,
// 127 taps): y[k] = sum_t h[t] * x[D*k + t - T]  (reference src/dsp/resampling.h:121-125 with I = 1).
// The input is split into its D polyphase sub-streams x_r[m] = x[base + D*m + r] while it is staged, each
// sub-stream is a dense FIR with taps h_r[q] = h[D*q + r], and all D sub-filters accumulate into the same
// 9 register-blocked outputs per thread -- the inner loop is the dense kernel's (one 128-bit shared load
// + one broadcast tap load per 18 FFMA2, conflict-free lane stride).
// =================================================================================================
struct FirDecimPlan {
    int T = 0, D = 0;
    int U = 0;                   // tap pairs per (sub-stream, parity) table, multiple of kFirR
    float2* taps_dev = nullptr;  // [2 pads][D][2][U]
};

FirDecimPlan* fir_decim_plan_create(const float* taps, int T, int D) {
    if (T < 2 || D < 2 || D > 8) return nullptr;
    const int tq = (T + 1 + D - 1) / D;          // taps of the longest sub-filter (one more tap slot for pad = 1)
    int U = (tq + 2) / 2;
    U = ((U + kFirR - 1) / kFirR) * kFirR;
    const size_t smem = (size_t)D * (kFirNout / 2 + U + 8) * 16 + (size_t)D * 2 * U * 8;
    if (smem > 110 * 1024) return nullptr;       // keep two CTAs per SM
    FirDecimPlan* p = new (std::nothrow) FirDecimPlan();
    if (!p) return nullptr;
    p->T = T;
    p->D = D;
    p->U = U;
    // [pad][D][2][U]: the tile's first staged sample is moved back by pad = 0 / 1 so that it sits on an even sample
    // index (128-bit global loads); the taps move with it: g[t] = h[t - pad]
    std::vector<float2> tab((size_t)2 * D * 2 * U, make_float2(0.f, 0.f));
    for (int pad = 0; pad < 2; pad++)
        for (int r = 0; r < D; r++) {
            auto h = [&](int q) {
                const int t = D * q + r - pad;
                return (q >= 0 && t >= 0 && t < T) ? taps[t] : 0.0f;
            };
            for (int u = 0; u < U; u++) {
                tab[(((size_t)pad * D + r) * 2 + 0) * U + u] = make_float2(h(2 * u), h(2 * u + 1));
                tab[(((size_t)pad * D + r) * 2 + 1) * U + u] = make_float2(h(2 * u - 1), h(2 * u));
            }
        }
    if (cudaMalloc(&p->taps_dev, tab.size() * sizeof(float2)) != cudaSuccess ||
        cudaMemcpy(p->taps_dev, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("fir_decim_plan_create: tap upload failed");
        delete p;
        return nullptr;
    }
    return p;
}
void fir_decim_plan_destroy(FirDecimPlan* p) {
    if (!p) return;
    if (p->taps_dev) cudaFree(p->taps_dev);
    delete p;
}

// DT > 0: compile-time decimation with vectorised staging (one thread moves 2*D consecutive samples = D 128-bit
// global loads into D sample quads = D 128-bit shared stores); DT == 0: run-time D, scalar staging.
template <int DT, int NW>
__global__ void __launch_bounds__(NW * 32, NW == 8 ? 2 : 4)
fir_decim_kernel(VStream<float2> xs, long long count, long long n_out, const float2* __restrict__ taps, int T, int Drt,
                 int U, float2* __restrict__ out) {
    constexpr int R = kFirR;
    constexpr int NT = NW * 32, NOUT = (NW / 2) * 64 * kFirR;   // threads, outputs per tile
    const int D = DT ? DT : Drt;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int npairs = NOUT / 2 + U + 8;                         // per sub-stream
    float4* sq = reinterpret_cast<float4*>(smem_raw);                 // [D][npairs] sample quads
    float2* st = reinterpret_cast<float2*>(smem_raw + (size_t)D * npairs * 16);  // [D][2][U]
    const int t = threadIdx.x;
    const long long k_t = (long long)blockIdx.x * NOUT;           // first output of the tile
    // with DT the staged window starts on an even sample index (pad = 0 / 1 samples earlier; the tap tables of that pad
    // are shifted by the same amount)
    const int pad = DT ? (int)(((long long)D * k_t - T) & 1) : 0;
    const long long B = (long long)D * k_t - T - pad;                 // sample index of sub-stream 0, element 0

    {
        const float2* tsrc = taps + (size_t)pad * D * 2 * U;
        for (int i = t; i < D * 2 * U; i += NT) st[i] = tsrc[i];
    }
    if (DT) {
        const bool in_aligned = (reinterpret_cast<uintptr_t>(xs.in) & 15) == 0;
        // two units (2 x 2*D samples) per thread in flight together: the tile's ~5 units per thread otherwise expose the
        // DRAM latency one after the other
        for (int g0 = t; g0 < npairs; g0 += 2 * NT) {
            float2 v[2][2 * (DT ? DT : 1)];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int g = g0 + h * NT;
                const long long i0 = B + (long long)2 * DT * g;      // even
                if (g < npairs && in_aligned && i0 >= 0 && i0 + 2 * DT <= count) {
                    const float4* src = reinterpret_cast<const float4*>(xs.in + i0);
#pragma unroll
                    for (int j = 0; j < DT; j++) {
                        const float4 a = ldg_stream128(src + j);
                        v[h][2 * j] = make_float2(a.x, a.y);
                        v[h][2 * j + 1] = make_float2(a.z, a.w);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 2 * DT; j++)
                        v[h][j] = (g < npairs && i0 + j < count) ? xs.at(i0 + j) : make_float2(0.f, 0.f);
                }
            }
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int g = g0 + h * NT;
                if (g < npairs) {
#pragma unroll
                    for (int r = 0; r < DT; r++)   // sub-stream r: elements 2g and 2g+1 are the unit's samples r and D + r
                        sq[(size_t)r * npairs + g] = make_float4(v[h][r].x, v[h][DT + r].x, v[h][r].y, v[h][DT + r].y);
                }
            }
        }
    } else {
        float* sf = reinterpret_cast<float*>(sq);
        const int nsamp = 2 * npairs * D;                             // consecutive input samples of the tile
        for (int e0 = t; e0 < nsamp; e0 += 8 * NT) {
            float2 v[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                const long long i = B + e;
                v[j] = (e < nsamp && i < count) ? xs.at(i) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                if (e < nsamp) {
                    const int r = e % D, m = e / D;                   // sub-stream, index within it
                    const int q = m >> 1, h = m & 1;
                    sf[((size_t)r * npairs + q) * 4 + h] = v[j].x;
                    sf[((size_t)r * npairs + q) * 4 + 2 + h] = v[j].y;
                }
            }
        }
    }
    __syncthreads();

    const int w = t >> 5, lane = t & 31;
    const int parity = w & 1, wp = w >> 1;
    const int j0 = wp * 32 * R + lane * R;
    float2 accRe[R], accIm[R];
#pragma unroll
    for (int i = 0; i < R; i++) {
        accRe[i] = make_float2(0.f, 0.f);
        accIm[i] = make_float2(0.f, 0.f);
    }
#pragma unroll 1
    for (int r = 0; r < D; r++) {
        const float2* tt = st + ((size_t)r * 2 + parity) * U;
        const float4* win = sq + (size_t)r * npairs + j0;
        float4 W[R];
#pragma unroll
        for (int i = 0; i < R; i++) W[i] = win[i];
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += R) {
#pragma unroll
            for (int k = 0; k < R; k++) {
                const float2 hh = tt[u0 + k];
#pragma unroll
                for (int i = 0; i < R; i++) {
                    const float4 s = W[(k + i) % R];
                    accRe[i] = __ffma2_rn(make_float2(s.x, s.y), hh, accRe[i]);
                    accIm[i] = __ffma2_rn(make_float2(s.z, s.w), hh, accIm[i]);
                }
                W[k] = win[u0 + k + R];
            }
        }
    }
    __syncthreads();
    float2* so = reinterpret_cast<float2*>(smem_raw);                 // [NOUT] outputs, then coalesced stores
#pragma unroll
    for (int i = 0; i < R; i++)
        so[2 * (j0 + i) + parity] = make_float2(accRe[i].x + accRe[i].y, accIm[i].x + accIm[i].y);
    __syncthreads();
    store_tile<NT, NOUT>(so, out, k_t, n_out);
}

// count input samples (one regular partition: every run() block a multiple of D, so the output grid is uniform)
int launch_fir_decim(FirDecimPlan* plan, const float2* hist, int H, const float2* in, long long count,
                     long long n_out, float2* out, cudaStream_t s) {
    if (n_out <= 0) return 0;
    VStream<float2> xs{hist, in, H};
    // short sub-filters (config 1b: 32 taps per sub-stream): 128-thread CTAs with 1152-output tiles, 4-5 per SM, overlap one
    // CTA's staging with the others' math better than 2 x 256 threads; long ones keep the big tile (less halo per output)
    const int NW = plan->U <= 36 ? 4 : 8;
    const int nout = (NW / 2) * 64 * kFirR;
    const size_t smem = (size_t)plan->D * (nout / 2 + plan->U + 8) * 16 + (size_t)plan->D * 2 * plan->U * 8;
    const long long tiles = (n_out + nout - 1) / nout;
#define QDSP_FIR_DECIM_LAUNCH(DT, NWT)                                                                             \
    {                                                                                                              \
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_decim_kernel<DT, NWT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024)); \
        fir_decim_kernel<DT, NWT><<<(unsigned)tiles, NWT * 32, smem, s>>>(xs, count, n_out, plan->taps_dev, plan->T, plan->D, \
                                                                          plan->U, out);                           \
    }
    if (plan->D == 2 && NW == 4) QDSP_FIR_DECIM_LAUNCH(2, 4)
    else if (plan->D == 2) QDSP_FIR_DECIM_LAUNCH(2, 8)
    else if (plan->D == 4 && NW == 4) QDSP_FIR_DECIM_LAUNCH(4, 4)
    else if (plan->D == 4) QDSP_FIR_DECIM_LAUNCH(4, 8)
    else if (plan->D == 8 && NW == 4) QDSP_FIR_DECIM_LAUNCH(8, 4)
    else if (plan->D == 8) QDSP_FIR_DECIM_LAUNCH(8, 8)
    else QDSP_FIR_DECIM_LAUNCH(0, 8)
#undef QDSP_FIR_DECIM_LAUNCH
    QDSP_LAUNCH_OK();
    return 0;
}

// =================================================================================================
// Short dense FIR (config 1a: 127 taps) with the taps in the constant bank -- the dense sibling of k_firrow.cu's
// complex-pair form. A CTA is ONE warp with its own tile: K steps of 32 lanes x R = 9 consecutive outputs; the tile's raw
// interleaved window (K*288 + T - 1 samples) arrives by ONE TMA bulk copy and is used as it lies: the packed FFMA2 operand
// is the sample (re, im), the tap enters both halves as a scalar uniform-register operand (`FFMA2 R, R, UR.F32, R`), the
// tap loop is fully unrolled (T is a template parameter), a lane slides a 9-sample register window: per tap ONE 64-bit
// shared load (lane stride 72 bytes: conflict-free) and nine FFMA2. Against fir_dense_kernel for this length: no quad
// re-layout pass, no parity tables, no horizontal adds, no shared-memory output exchange, no CTA barrier.
// =================================================================================================
struct FirCplxArgs {
    const float2* hist;
    const float2* in;
    int H;
    long long count;
    float2* out;
    float2* hist_next;        // when non-null: CTA 0 writes the advanced history tail here (filter.h:71)
    alignas(16) float g[256];
};
template <int T, int K>
__global__ void __launch_bounds__(32) fir_cplx_kernel(const __grid_constant__ FirCplxArgs fa) {
    constexpr int R = 9, STEP = 32 * R, NOUT = K * STEP, NS = NOUT + T - 1;
    static_assert((NS * 8) % 16 == 0 && ((T - 1) % 2) == 0, "the window is a whole number of 16-byte units and starts on an even sample");
    __shared__ __align__(128) float2 win[NS];
    __shared__ uint64_t s_mbar;
    const int lane = threadIdx.x;
    const long long n_t = (long long)blockIdx.x * NOUT;               // first output of the tile
    const long long B = n_t - (T - 1);                                // sample index of win[0]
    // overlapped consecutive calls (decim_common.cuh): CTA 0 folds the history, a tile whose window starts before sample 0
    // reads it
    if (blockIdx.x == 0 || B < 0) pdl_wait();
    if (blockIdx.x == 0 && fa.hist_next != nullptr) fold_history(fa.hist, fa.in, +fa.H, +fa.count, fa.hist_next, lane, 32);
    if (B >= 0 && B + NS <= fa.count) {
        if (lane == 0) {
            mbar_init(&s_mbar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_arrive_expect_tx(&s_mbar, (uint32_t)NS * 8u);
            tma_bulk_g2s(win, fa.in + B, (uint32_t)NS * 8u, &s_mbar);
        }
        pdl_launch_dependents();
        __syncwarp();
        mbar_wait(&s_mbar, 0);
    } else {   // history before sample 0 / ragged end: guarded fill
        pdl_launch_dependents();
        VStream<float2> xs{fa.hist, fa.in, fa.H};
        for (int e = lane; e < NS; e += 32) {
            const long long idx = B + e;
            win[e] = idx < fa.count ? xs.at(idx) : make_float2(0.f, 0.f);
        }
        __syncwarp();
    }
#pragma unroll 1
    for (int k = 0; k < K; k++) {
        const f32x2_t* base = reinterpret_cast<const f32x2_t*>(win) + k * STEP + R * lane;
        f32x2_t W[R], acc[R];
#pragma unroll
        for (int i = 0; i < R; i++) W[i] = base[i];
#pragma unroll
        for (int j = 0; j < T; j++) {
            const f32x2_t g = pk2(fa.g[j], fa.g[j]);
#pragma unroll
            for (int r = 0; r < R; r++) {
                if (j == 0) acc[r] = fmul2x(W[(r + j) % R], g);
                else acc[r] = ffma2x(W[(r + j) % R], g, acc[r]);
            }
            if (j + R <= T - 1 + R - 1) W[j % R] = base[j + R];       // element j is dead, element j + R enters
        }
        const long long n0 = n_t + k * STEP + R * lane;
#pragma unroll
        for (int r = 0; r < R; r++)
            if (n0 + r < fa.count) fa.out[n0 + r] = unpk2(acc[r]);
    }
}

// =================================================================================================
// Long dense FIR (config 3: 4095 taps) in the same form: the sample (re, im) is the packed operand, the tap a scalar
// uniform-register operand from the constant bank (the whole filter travels as a kernel parameter, <= 4105 floats), a lane
// slides a nine-sample register window (one conflict-free 64-bit shared load per tap). The tap loop cannot be unrolled
// over 4095 taps: it runs in groups of 36 (the window rotation is static inside a group: 36 = 4 x 9) whose constant-bank
// offset is a uniform register. A CTA of 8 warps shares ONE raw window (2304 + Tp - 1 samples, one TMA bulk copy, used as
// it lies -- no quad re-layout, no parity tables); the filter is padded in FRONT with zeros to Tp = 36 m + 1 taps (the
// window must start on an even sample, so Tp is odd: one leading tap, then m groups).
// =================================================================================================
constexpr int kFlG = 36;                    // taps per group
constexpr int kFlMaxTp = 36 * 114 + 1;      // 4105: room for 4095 taps
struct FirLongArgs {
    const float2* hist;
    const float2* in;
    int H;
    int Tp;                   // padded tap count, 36 m + 1
    long long count;
    float2* out;
    float2* hist_next;        // when non-null: CTA 0 writes the advanced history tail here (filter.h:71)
    alignas(16) float g[kFlMaxTp + 3];
};
__global__ void __launch_bounds__(256, 3) fir_longcplx_kernel(const __grid_constant__ FirLongArgs fa) {
    constexpr int R = 9, NWARP = 8, NT = NWARP * 32, NOUT = NT * R;       // 2304 outputs per tile
    extern __shared__ __align__(128) unsigned char fl_smem[];
    float2* win = reinterpret_cast<float2*>(fl_smem);
    __shared__ uint64_t s_mbar;
    const int t = threadIdx.x;
    const int Tp = fa.Tp;
    const int NS = NOUT + Tp - 1;                                         // even: NOUT even, Tp odd
    const long long n_t = (long long)blockIdx.x * NOUT;                   // first output of the tile
    const long long B = n_t - (Tp - 1);                                   // sample index of win[0] (even)
    // overlapped consecutive calls: as in fir_cplx_kernel (with 4095 taps, tiles after the first may start before sample 0)
    if (blockIdx.x == 0 || B < 0) pdl_wait();
    if (blockIdx.x == 0 && fa.hist_next != nullptr) fold_history(fa.hist, fa.in, +fa.H, +fa.count, fa.hist_next, t, NT);
    pdl_launch_dependents();
    if (B >= 0 && B + NS <= fa.count) {
        if (t == 0) {
            mbar_init(&s_mbar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (t == 0) {
            mbar_arrive_expect_tx(&s_mbar, (uint32_t)NS * 8u);
            tma_bulk_g2s(win, fa.in + B, (uint32_t)NS * 8u, &s_mbar);
        }
        mbar_wait(&s_mbar, 0);
    } else {   // history before sample 0 / ragged end: guarded fill, 8 loads per thread in flight
        VStream<float2> xs{fa.hist, fa.in, fa.H};
        for (int e0 = t; e0 < NS; e0 += 8 * NT) {
            float2 v[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                const long long idx = B + e;
                v[j] = (e < NS && idx < fa.count) ? xs.at(idx) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int e = e0 + j * NT;
                if (e < NS) win[e] = v[j];
            }
        }
        __syncthreads();
    }
    const f32x2_t* base = reinterpret_cast<const f32x2_t*>(win) + R * t;  // element e of this thread = win[9 t + e]
    f32x2_t W[R], acc[R];
#pragma unroll
    for (int i = 0; i < R; i++) W[i] = base[i];
    {   // the leading tap (j = 0): elements 0 .. 8, then element 9 replaces element 0
        const f32x2_t g = pk2(fa.g[0], fa.g[0]);
#pragma unroll
        for (int r = 0; r < R; r++) acc[r] = fmul2x(W[r], g);
        W[0] = base[R];
    }
    const int ngroups = (Tp - 1) / kFlG;
#pragma unroll 1
    for (int gi = 0; gi < ngroups; gi++) {
        const int j0 = 1 + gi * kFlG;                                     // first tap of the group; j0 % 9 == 1
        const float* gt = fa.g + j0;
        const f32x2_t* bj = base + j0;
#pragma unroll
        for (int jj = 0; jj < kFlG; jj++) {
            const f32x2_t g = pk2(gt[jj], gt[jj]);
#pragma unroll
            for (int r = 0; r < R; r++) acc[r] = ffma2x(W[(r + 1 + jj) % R], g, acc[r]);
            W[(1 + jj) % R] = bj[jj + R];                                 // element j is dead, element j + 9 enters
        }
    }
    const long long n0 = n_t + (long long)R * t;
#pragma unroll
    for (int r = 0; r < R; r++)
        if (n0 + r < fa.count) fa.out[n0 + r] = unpk2(acc[r]);
}

// hist_next / overlap_prev / advanced: when the constant-bank kernels take the call and `hist_next` is given, the kernel's
// first CTA writes the advanced history tail there (*advanced = true: the caller flips its double buffer instead of
// launching the advance kernel); overlap_prev lets the grid start while the previous call of the same handle drains
int launch_fir_dense(FirPlan* plan, const float2* hist, int H, const float2* in, long long count, int lead,
                     float2* out, cudaStream_t s, float2* hist_next, bool overlap_prev, bool* advanced) {
    if (advanced) *advanced = false;
    if (count <= 0) return 0;
    if (lead != 1) {
        set_last_error("fir_dense: only the FIR alignment (lead = 1) is implemented");
        return -1;
    }
    // constant-bank kernel: instantiated for 63 / 127 / 255 taps; a filter of T taps runs as the next instantiated length TT
    // with TT - T leading zero taps (y[n] = sum_j g[j] x[n - (TT-1) + j], g[j] = h[j - (TT - T)]) when that costs < 1/3 more work
    const int TT = plan->T <= 63 ? 63 : (plan->T <= 127 ? 127 : 255);
    if (plan->T <= 255 && 4 * plan->T > 3 * TT && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
        constexpr int K = 4;
        static FirCplxArgs fa;
        static std::mutex mtx;
        std::lock_guard<std::mutex> lk(mtx);
        fa.hist = hist;
        fa.in = in;
        fa.H = H;
        fa.count = count;
        fa.out = out;
        fa.hist_next = hist_next;
        const int z = TT - plan->T;
        for (int j = 0; j < 256; j++) fa.g[j] = (j >= z && j < TT) ? plan->taps_host[j - z] : 0.0f;
        const long long tiles = (count + K * 288 - 1) / (K * 288);
        const void* kern = TT == 63 ? (const void*)fir_cplx_kernel<63, K>
                                    : (TT == 127 ? (const void*)fir_cplx_kernel<127, K> : (const void*)fir_cplx_kernel<255, K>);
        QDSP_CUDA_OK(launch_ex(kern, dim3((unsigned)tiles), dim3(32), 0, s, overlap_prev, &fa));
        QDSP_LAUNCH_OK();
        if (advanced && hist_next) *advanced = true;
        return 0;
    }
    if (plan->T > 255 && plan->T <= 4095 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
        !plan->taps_long.empty()) {
        static FirLongArgs la;
        static std::mutex mtx;
        std::lock_guard<std::mutex> lk(mtx);
        const int m = (plan->T - 1 + kFlG - 1) / kFlG;            // groups after the leading tap
        const int Tp = m * kFlG + 1, z = Tp - plan->T;
        la.hist = hist;
        la.in = in;
        la.H = H;
        la.Tp = Tp;
        la.count = count;
        la.out = out;
        la.hist_next = hist_next;
        for (int j = 0; j < kFlMaxTp + 3; j++) la.g[j] = (j >= z && j < Tp) ? plan->taps_long[j - z] : 0.0f;
        const size_t smem = ((size_t)2304 + Tp + 8) * 8;
        // per device (the attribute belongs to the current context), so set on every call: it is a cheap driver lookup
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_longcplx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(((size_t)2304 + kFlMaxTp + 8) * 8)));
        const long long tiles = (count + 2304 - 1) / 2304;
        QDSP_CUDA_OK(launch_ex((const void*)fir_longcplx_kernel, dim3((unsigned)tiles), dim3(256), smem, s, overlap_prev, &la));
        QDSP_LAUNCH_OK();
        if (advanced && hist_next) *advanced = true;
        return 0;
    }
    VStream<float2> xs{hist, in, H};
    // short filters (config 1a: 127 taps): 128-thread CTAs with 1152-output tiles, 5 per SM; long ones keep the 2304-output
    // tile (the window's T-1 halo is staged once per tile)
    const int NW = plan->U <= 144 ? 4 : 8;
    const int nout = (NW / 2) * 64 * kFirR;
    const size_t smem = ((size_t)nout / 2 + plan->U + 8) * 16 + (size_t)2 * plan->U * 8;
    const long long tiles = (count + nout - 1) / nout;
    if (NW == 4) {
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_dense_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_dense_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        if (plan->U % kFirR)
            fir_dense_kernel<4, true><<<(unsigned)tiles, 128, smem, s>>>(xs, count, plan->taps_dev, plan->T, plan->U, out);
        else
            fir_dense_kernel<4, false><<<(unsigned)tiles, 128, smem, s>>>(xs, count, plan->taps_dev, plan->T, plan->U, out);
    } else {
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_dense_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        QDSP_CUDA_OK(cudaFuncSetAttribute(fir_dense_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        if (plan->U % kFirR)
            fir_dense_kernel<8, true><<<(unsigned)tiles, 256, smem, s>>>(xs, count, plan->taps_dev, plan->T, plan->U, out);
        else
            fir_dense_kernel<8, false><<<(unsigned)tiles, 256, smem, s>>>(xs, count, plan->taps_dev, plan->T, plan->U, out);
    }
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
