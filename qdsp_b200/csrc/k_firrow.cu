// qdsp_b200/csrc/k_firrow.cu — row-per-lane decimating FIR for SMALL decimations (PolyphaseResampler<complex_t> with
// interp = 1, D = 4: BASELINE config 1b, reference resampling.h:99-132), the small-D sibling of k_rowlane.cu.
//
// The stream is cut into rows of DROW = 28 samples = NPH = DROW / D = 7 outputs. Output k = NPH*r + j (row r, phase j) is
//     y[k] = sum_q S_{j,q}(r + q),   S_{j,q}(row) = sum_{c < DROW} g_j[q*DROW + c] * x[row, c],   g_j[u] = h[u - j*D - pad]
// i.e. NPH decimate-by-DROW filters whose taps are shifted copies of h (Q = 6 tap rows cover the 127 + 24 + 1 window).
// Lane l of a step owns row 32*i + l and computes all NPH x Q row partials of its 28 samples. The packed FFMA2 operand is
// the sample as it lies in shared memory, (re, im), and the tap enters both halves: acc(re, im) += x(re, im) * (g, g). The
// taps are compile-time offsets into the kernel-parameter constant bank -> scalar uniform-register operands (one 128-bit
// constant load per 4 FFMA2), dead (zero) tap pairs are skipped at compile time (T is a template parameter): 32.0 FFMA2
// per input sample against the algorithmic 31.75. A form that re-paired the samples as (re, re) / (im, im) spent 3.9
// FMUL2-by-one packs and 2.9 FADD per sample besides and ran slower (314 against 323 GS/s, DESIGN.md 6.0c); it was
// removed. Output (r, j) then gathers its Q partials from lanes r .. r+Q-1 with shuffles; lanes whose window runs past
// lane 31 finish one step later (as in k_rowlane.cu). No shared-memory exchange, no CTA barrier; a CTA is one warp with
// its own TMA ring, one bulk copy of 32 contiguous rows per stage. The 224-byte row pitch makes the per-lane 128-bit loads
// 2-way bank conflicted (irrelevant); 16-sample rows (128-byte pitch) would need one padded copy per row, and ncu showed
// the per-copy issue sequence eating 20 % of the instruction slots.
#include <math.h>
#include <mutex>
#include <new>
#include "decim_common.cuh"

namespace qdsp {

template <int NPH, int Q, int DROW>
struct FirRowArgs {
    const float2* hist;
    const float2* in;
    int H;
    long long count;          // input samples of this call
    long long n_out;          // outputs of this call
    int T, pad;
    int nstep;                // steps (of 32 rows) per tile
    float2* out;
    float2* hist_next;        // when non-null: CTA 0 writes the advanced history tail here (resampling.h:129)
    alignas(16) float g[NPH][Q * DROW];   // g[j][u] = h[u - j*D - pad], zero outside
};

// is the tap pair (columns 2c, 2c+1 of tap row q) of phase j live for T taps?
__host__ __device__ constexpr bool firrow_live(int j, int q, int c, int D, int DROW, int pad, int T) {
    const int u0 = q * DROW + 2 * c, lo = j * D + pad, hi = j * D + pad + T;
    return u0 + 2 > lo && u0 < hi;
}
__host__ __device__ constexpr int firrow_first(int j, int q, int D, int DROW, int pad, int T) {
    for (int c = 0; c < DROW / 2; c++)
        if (firrow_live(j, q, c, D, DROW, pad, T)) return c;
    return -1;
}

template <int D, int DROW, int Q, int T, int PAD, int NSTG>
__global__ void __launch_bounds__(32) fir_rowcplx_kernel(const __grid_constant__ FirRowArgs<DROW / D, Q, DROW> fa) {
    constexpr int NPH = DROW / D;
    constexpr int PITCH = DROW * 8;
    constexpr uint32_t STAGE_BYTES = 32u * PITCH;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const int rows_per_tile = 32 * fa.nstep - (Q - 1);
    const long long row_t0 = (long long)blockIdx.x * rows_per_tile;
    const long long nrows_total = (fa.n_out + NPH - 1) / NPH;
    // overlapped consecutive calls (decim_common.cuh): CTA 0 alone waits -- it folds the history, and only tile 0's window
    // starts before sample 0
    if (blockIdx.x == 0) pdl_wait();
    if (fa.hist_next != nullptr && blockIdx.x == 0) fold_history(fa.hist, fa.in, fa.H, fa.count, fa.hist_next, lane, 32);
    if (row_t0 >= nrows_total) return;
    const long long left = nrows_total - row_t0;
    const int nrows_emit = left < rows_per_tile ? (int)left : rows_per_tile;
    const int nsteps = (nrows_emit + (Q - 1) + 31) / 32;
    const long long base = -(long long)fa.T - PAD + row_t0 * DROW;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + NSTG * STAGE_BYTES);
    if (lane == 0) {
        for (int s = 0; s < NSTG; s++) mbar_init(&mbar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    auto issue = [&](int i) {
        if (i >= nsteps) return;
        const int slot = i % NSTG;
        unsigned char* dst = smem_raw + slot * STAGE_BYTES;
        const long long s0 = base + (long long)i * (32 * DROW);
        if (s0 >= 0 && s0 + 32 * DROW <= fa.count) {
            if (lane == 0) {
                mbar_arrive_expect_tx(&mbar[slot], STAGE_BYTES);
                tma_bulk_g2s(dst, fa.in + s0, STAGE_BYTES, &mbar[slot]);
            }
        } else {
            VStream<float2> xs{fa.hist, fa.in, fa.H};
            for (int e = lane; e < 32 * DROW; e += 32) {
                const int rr = e / DROW, cc = e - rr * DROW;
                const long long idx = s0 + e;
                reinterpret_cast<float2*>(dst + rr * PITCH)[cc] = idx < fa.count ? xs.at(idx) : make_float2(0.f, 0.f);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&mbar[slot]);
        }
    };
    for (int i = 0; i < NSTG; i++) issue(i);
    pdl_launch_dependents();
    float2 old[NPH];
#pragma unroll
    for (int j = 0; j < NPH; j++) old[j] = make_float2(0.f, 0.f);
    const bool tail_lane = lane >= 32 - (Q - 1);
#pragma unroll 1
    for (int i = 0; i < nsteps; i++) {
        const int slot = i % NSTG;
        mbar_wait(&mbar[slot], (uint32_t)((i / NSTG) & 1));
        const ulonglong2* xrow = reinterpret_cast<const ulonglong2*>(smem_raw + slot * STAGE_BYTES + lane * PITCH);
        f32x2_t X[DROW];                                 // (re, im) of the row's samples, as loaded
#pragma unroll
        for (int c = 0; c < DROW / 2; c++) {
            const ulonglong2 v = xrow[c];
            X[2 * c] = v.x;
            X[2 * c + 1] = v.y;
        }
        __syncwarp();
        issue(i + NSTG);
        float2 yv[NPH];
#pragma unroll
        for (int j0 = 0; j0 < NPH; j0 += 2) {
            constexpr int NJ = 2;
            f32x2_t acc[NJ][Q];
#pragma unroll
            for (int c4 = 0; c4 < DROW / 4; c4++) {      // four columns per 128-bit constant-bank tap load
#pragma unroll
                for (int jj = 0; jj < NJ; jj++) {
                    if (j0 + jj >= NPH) continue;
#pragma unroll
                    for (int q = 0; q < Q; q++) {
                        const bool l0 = firrow_live(j0 + jj, q, 2 * c4, D, DROW, PAD, T);
                        const bool l1 = firrow_live(j0 + jj, q, 2 * c4 + 1, D, DROW, PAD, T);
                        if (l0 || l1) {
                            const float4 g4 = *reinterpret_cast<const float4*>(&fa.g[j0 + jj][q * DROW + 4 * c4]);
                            const float gg[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
                            for (int hh = 0; hh < 4; hh++) {
                                const int col = 4 * c4 + hh;
                                if ((hh < 2) ? l0 : l1) {
                                    const f32x2_t g = pk2(gg[hh], gg[hh]);
                                    if (col == 2 * firrow_first(j0 + jj, q, D, DROW, PAD, T)) acc[jj][q] = fmul2x(X[col], g);
                                    else acc[jj][q] = ffma2x(X[col], g, acc[jj][q]);
                                }
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int jj = 0; jj < NJ; jj++) {
                const int j = j0 + jj;
                if (j >= NPH) continue;
                float2 cur = make_float2(0.f, 0.f);
#pragma unroll
                for (int q = 0; q < Q; q++) {
                    if (firrow_first(j, q, D, DROW, PAD, T) >= 0) {
                        const float2 sv = unpk2(acc[jj][q]);
                        if (q == 0) {
                            cur = sv;
                        } else {
                            float2 p;
                            p.x = __shfl_sync(0xffffffffu, sv.x, (lane + q) & 31);
                            p.y = __shfl_sync(0xffffffffu, sv.y, (lane + q) & 31);
                            if (lane + q < 32) cur = __fadd2_rn(cur, p);
                            else old[j] = __fadd2_rn(old[j], p);
                        }
                    }
                }
                yv[j] = tail_lane ? old[j] : cur;
                if (tail_lane) old[j] = cur;
            }
        }
        const int rrel = 32 * i + lane - (tail_lane ? 32 : 0);
        if (rrel >= 0 && rrel < nrows_emit) {
            const long long k = (row_t0 + rrel) * NPH;
            float2* o = fa.out + k;
#pragma unroll
            for (int j = 0; j < NPH; j++)
                if (k + j < fa.n_out) o[j] = yv[j];
        }
    }
}

// ---- sliding-window variant -------------------------------------------------------------------------------------
// The decimating sibling of k_fir.cu's fir_cplx_kernel: a CTA is one warp with its own tile (32 lanes x R = 9 consecutive
// OUTPUTS = 36 consecutive input samples per lane), the tile's raw window arrives by one TMA bulk copy, the
// sample (re, im) is the packed FFMA2 operand and the tap enters as a scalar uniform-register operand from the constant
// bank. Output k0 + r at tap u reads window element 4 r + u (elements count from sample 4 k0 - T - 1: one pad sample keeps
// the window 16-byte aligned, tap u = h[u - 1], u = 1..T): the lane keeps the 33 live elements in a statically rotated
// register file of 36 and loads ONE pair (128 bits; lane stride 288 bytes: 2-way bank conflict, i.e. the wavefronts of a
// conflict-free 64-bit load per element) every second tap: nine FFMA2 per tap, nothing else on the FMA pipe -- no row
// partials to gather across lanes, no shuffles, no packs.
struct FirSlideArgs {
    const float2* hist;
    const float2* in;
    int H;
    long long count;          // input samples of this call
    long long n_out;          // outputs of this call
    float2* out;
    float2* hist_next;        // when non-null: CTA 0 writes the advanced history tail here (resampling.h:129)
    alignas(16) float g[128]; // g[u] = h[u - 1], g[0] = 0
};
template <int T>
__global__ void __launch_bounds__(32) fir_slide4_kernel(const __grid_constant__ FirSlideArgs fa) {
    constexpr int D = 4, R = 9, LSTEP = D * R, NOUT = 32 * R;
    constexpr int EMAX = D * (R - 1) + T;                    // last window element a lane touches (159)
    constexpr int NS = D * NOUT - LSTEP + EMAX + 1;          // samples of the tile's window (last lane)
    constexpr int NW = 36;                                   // register file: >= D*(R-1) + 1 live elements + the pair in flight
    static_assert((T & 1) == 1 && (NS & 1) == 0 && NW % 2 == 0 && NW >= D * (R - 1) + 3, "geometry");
    __shared__ __align__(128) float2 win[NS];
    __shared__ uint64_t s_mbar;
    const int lane = threadIdx.x;
    // overlapped consecutive calls (decim_common.cuh): CTA 0 alone waits -- it folds the history, and only tile 0's window
    // starts before sample 0
    if (blockIdx.x == 0) pdl_wait();
    if (fa.hist_next != nullptr && blockIdx.x == 0) fold_history(fa.hist, fa.in, fa.H, fa.count, fa.hist_next, lane, 32);
    const long long k_t = (long long)blockIdx.x * NOUT;               // first output of the tile
    if (k_t >= fa.n_out) return;
    const long long B = D * k_t - T - 1;                              // sample index of win[0]
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
    const ulonglong2* base = reinterpret_cast<const ulonglong2*>(win + LSTEP * lane);   // element pairs
    f32x2_t W[NW], acc[R];
#pragma unroll
    for (int m = 0; m < (D * (R - 1) + 2) / 2; m++) {          // elements 0 .. 33
        const ulonglong2 v = base[m];
        W[2 * m] = v.x;
        W[2 * m + 1] = v.y;
    }
#pragma unroll
    for (int u = 1; u <= T; u++) {
        const f32x2_t g = pk2(fa.g[u], fa.g[u]);
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (u == 1) acc[r] = fmul2x(W[(D * r + u) % NW], g);
            else acc[r] = ffma2x(W[(D * r + u) % NW], g, acc[r]);
        }
        // elements <= u are dead; tap u + 1 needs element u + 1 + D (R - 1): pairs (u + 33, u + 34) enter on odd u
        if ((u & 1) && u + D * (R - 1) + 1 <= EMAX) {
            const ulonglong2 v = base[(u + D * (R - 1) + 1) / 2];
            W[(u + D * (R - 1) + 1) % NW] = v.x;
            W[(u + D * (R - 1) + 2) % NW] = v.y;
        }
    }
    const long long k0 = k_t + R * lane;
#pragma unroll
    for (int r = 0; r < R; r++)
        if (k0 + r < fa.n_out) fa.out[k0 + r] = unpk2(acc[r]);
}

// ---- host side -------------------------------------------------------------------------------------
bool firrow_supported(int T, int D) { return D == 4 && T == 127; }

int launch_firrow(const float* taps_host, int T, int D, const float2* hist, float2* hist_next, int H, const float2* in,
                  long long count, long long n_out, float2* out, cudaStream_t s, bool overlap_prev) {
    if (n_out <= 0) return 0;
    constexpr int DROW = 28, Q = 6, NPH = 7;
    if (!firrow_supported(T, D) || (reinterpret_cast<uintptr_t>(in) & 15) != 0) {
        set_last_error("firrow: unsupported geometry");
        return -1;
    }
    static FirRowArgs<NPH, Q, DROW> fa;
    static FirSlideArgs sa;
    static std::mutex mtx;
    std::lock_guard<std::mutex> lk(mtx);
    // the sliding-window kernel wins away from BASELINE's 2^24-sample call (size sweep in DESIGN.md 6.0c): calls of >= 2^25
    // samples take it
    if (count >= (1ll << 25)) {
        sa.hist = hist;
        sa.in = in;
        sa.H = H;
        sa.count = count;
        sa.n_out = n_out;
        sa.out = out;
        sa.hist_next = hist_next;
        sa.g[0] = 0.0f;
        for (int u = 1; u < 128; u++) sa.g[u] = taps_host[u - 1];
        const dim3 grid((unsigned)((n_out + 288 - 1) / 288));
        QDSP_CUDA_OK(launch_ex((const void*)fir_slide4_kernel<127>, grid, dim3(32), 0, s, overlap_prev, &sa));
    } else {
        constexpr int PAD = 1;                   // T odd: the window starts one sample early so that rows are 16-byte aligned
        fa.hist = hist;
        fa.in = in;
        fa.H = H;
        fa.count = count;
        fa.n_out = n_out;
        fa.T = T;
        fa.pad = PAD;
        // steps (of 32 rows) per one-warp tile: with consecutive calls overlapped the drain no longer favours the shortest
        // tile (G samples/s at 2^24 per call, two boxes: 2: 346, 3: 348 / 359, 4: 347, 6: 355 / 368, 8: 357, 10: 332,
        // 12: 273)
        fa.nstep = 6;
        fa.out = out;
        fa.hist_next = hist_next;
        for (int j = 0; j < NPH; j++)
            for (int u = 0; u < Q * DROW; u++) {
                const int t = u - j * D - PAD;
                fa.g[j][u] = (t >= 0 && t < T) ? taps_host[t] : 0.0f;
            }
        const long long nrows = (n_out + NPH - 1) / NPH;
        const int rows_per_tile = 32 * fa.nstep - (Q - 1);
        const long long tiles = (nrows + rows_per_tile - 1) / rows_per_tile;
        constexpr int NSTG = 2;                  // 2 slots: 15 warps per SM (315 GS/s); 3 slots: 10 (310)
        constexpr size_t smem = NSTG * 32 * (DROW * 8) + NSTG * 8 + 16;
        auto kern = fir_rowcplx_kernel<4, DROW, Q, 127, PAD, NSTG>;
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        QDSP_CUDA_OK(launch_ex((const void*)kern, dim3((unsigned)tiles), dim3(32), smem, s, overlap_prev, &fa));
    }
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
