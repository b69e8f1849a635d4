// qdsp_b200/csrc/decim_common.cuh — pieces shared by the FIR kernel families (k_decim.cu: column-pair kernels;
// k_rowlane.cu, k_firrow.cu: row-per-lane kernels; k_fir.cu: dense FIR): plan / argument structs, mbarrier + TMA
// bulk-copy PTX wrappers, the overlapped-call helpers (programmatic dependent launch, folded history advance), and
// the brute-force single output used for a block's leading FM-demod angle.
#pragma once
#include <stdlib.h>
#include <vector>
#include "internal.cuh"
#include "kernels.cuh"

namespace qdsp {

// packed f32x2 values as opaque 64-bit registers: built once per column pair, never re-materialised from their halves
// (with float2 temporaries ptxas re-packs the (re, re) pairs in front of nearly every FFMA2: 880 MOVs per 512 FFMA2)
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pk2(float a, float b) {
    f32x2_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    asm volatile("" : "+l"(r));
    return r;
}
__device__ __forceinline__ float2 unpk2(f32x2_t v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ f32x2_t ffma2x(f32x2_t a, f32x2_t b, f32x2_t c) {
    f32x2_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2_t fmul2x(f32x2_t a, f32x2_t b) {
    f32x2_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}


struct DecimPlan {
    int T = 0, D = 0, Q = 0, P = 0;
    int NSEG = 0, R = 0, NSTAGE = 0, NSUP = 0, NT = 0;
    // wide rows are cut into column slices of `D` samples each (DS = full decimation = global row stride); every
    // slice is an independent CTA stream producing partial outputs that finish_kernel sums (and demodulates)
    int DS = 0, nslices = 1;
    float2* taps_dev = nullptr;  // [nslices][2][Q][P] tap pairs for pad = 0 / 1 (g[t] = h[t - pad])
    float2* ypart = nullptr;     // [nch * nslices][ypart_stride] partial outputs (sliced plans only)
    size_t ypart_cap = 0;
};

struct DecimArgs {
    const float2* hist;
    const float2* in;
    int H;
    long long n_in;
    const float2* taps;  // [2][Q][P]
    PartitionDev part;
    int T, D, P, NSEG, R, NSTAGE, NSUP, L;
    int DS, nslices;     // global row stride (full decimation) and column slices per row (1 = unsliced)
    int plane_fast;      // grid = (planes, tiles, blocks) instead of (tiles, blocks, planes): see launch_decim
    const NcoDev* nco;
    long long abs0;
    float phasor_speed;
    const float* demod_in;
    float* demod_out;
    float2* out_iq;
    float* audio;
    long long out_stride;
};

// ---- PTX wrappers: mbarrier + TMA bulk copy (SASS: SYNCS / UBLKCP) -----------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- overlapped consecutive calls (DESIGN.md §6.0f) ---------------------------------------------------------------
// The kernels of k_fir.cu (fir_cplx_kernel, fir_longcplx_kernel), k_firrow.cu (fir_rowcplx_kernel, fir_slide4_kernel)
// and k_rowlane.cu (decim_rowlane_kernel) fold the history advance into their launch: a CTA writes the advanced tail to
// `hist_next` (fold_history), the other half of the handle's double buffer, and the next call reads it as `hist`. The
// next call of the same handle may then be launched with programmatic dependent launch (launch_ex, overlap) and start
// while this grid drains. Ordering rests on one rule: whatever the previous grid also touches -- `hist`, which it wrote,
// `hist_next`, which it read as its `hist`, and the fused chain's demodulator phase and audio -- a CTA touches only after
// pdl_wait(), which returns once the previous grid has completed and its writes are visible. Every other access reads
// this call's `in` and writes this call's `out`; the launcher overlaps a call only when those do not touch the previous
// call's buffers (api.cu, CallChain). A grid that has waited completes after its predecessor, so the order holds down
// a whole chain of calls. pdl_launch_dependents() only lets the next grid be scheduled early; where a kernel calls it does
// not change what it computes. Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

// folded history advance (filter.h:71 / resampling.h:129): hist_next[j] = (hist ++ in)[count - H + j], the CTA's threads
// t, t + nt, ... sharing the H elements. The kernels pass fields of their __grid_constant__ parameter; taken by reference,
// a field is read where the loop reads it. A caller that wants H and count loaded once before the loop passes values
// (k_fir.cu: +fa.H).
__device__ __forceinline__ void fold_history(const float2* const& hist, const float2* const& in, const int& H, const long long& count,
                                             float2* const& hist_next, int t, int nt) {
    for (int j = t; j < H; j += nt) {
        const long long v = count - H + j;
        hist_next[j] = v >= 0 ? in[v] : hist[H + v];
    }
}

// single output by brute force (warp-cooperative): used for the one "previous output" a block's first
// tile needs when the previous run() block did not end on the decimation grid.
template <bool ROT>
__device__ float2 direct_output_warp(const DecimArgs& a, long long win_start, uint64_t ph0, uint64_t step) {
    // y = sum_t h[t] * x'[win_start + t]; taps table pad=0 holds h at [q][p] pairs == flat h[t]
    const float* h = reinterpret_cast<const float*>(a.taps);
    const int lane = threadIdx.x & 31;
    VStream<float2> xs{a.hist, a.in, a.H};
    float2 acc = make_float2(0.f, 0.f);
    for (int t = lane; t < a.T; t += 32) {
        const long long i = win_start + t;
        float2 v = (i < a.n_in) ? xs.at(i) : make_float2(0.f, 0.f);
        if (ROT) v = cmul(v, phasor_from_turns(ph0 + step * (uint64_t)i));
        acc.x = fmaf(v.x, h[t], acc.x);
        acc.y = fmaf(v.y, h[t], acc.y);
    }
    for (int o = 16; o > 0; o >>= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
    }
    return acc;
}

}  // namespace qdsp
