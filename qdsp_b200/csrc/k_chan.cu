// qdsp_b200/csrc/k_chan.cu — channel-per-lane decimating FIR for sm_100a: the multi-channel fused
// xlate -> resample (-> demod) pass of N VFOs fed by one Splitter (reference routing.h:47-57, vfo.h:19-36,
// resampling.h:99-132, processing.h:55-70), for WIDE rows (config 4: 61.44 MS/s -> 48 kS/s, D = 1280, 10 241 taps).
//
// Every channel applies the same taps to the same wideband samples; only the NCO differs. So a warp's 32 LANES ARE 32
// CHANNELS: a staged input sample is loaded once (a broadcast shared-memory load) and consumed by all of them -- the
// wideband stream is read from HBM once per GPU, not once per channel -- and the tap pairs are warp-uniform, so they
// come from the kernel-parameter constant bank as uniform-register FFMA2 operands (no tap registers, no tap loads).
// Rows (D samples) are cut into column slices of DC samples (grid.z); the taps live in __constant__ memory and are
// addressed with a uniform (per-CTA) slice offset plus compile-time offsets; a single-warp CTA walks a segment of rows
// of one slice for one group of 32 channels:
//     per column pair: 1 broadcast LDS.128, the per-lane NCO rotation of the two samples, 8 x 2 FFMA2 (tap rows q = 0..7)
//     per row: the row's partials S_q join the 9 outputs in flight (O[q] = O[q-1] + S_q), output row-8 leaves as a
//              partial sum of this slice.
// The per-slice partial outputs are summed (and FM-demodulated, demodulator.h:87-94) by decim_finish_kernel.
// The lane's phasor runs down the row by recurrence (two interleaved phasors, packed), re-seeded exactly (closed form)
// at the start of every row slice.
#include <math.h>
#include <mutex>
#include <new>
#include "decim_common.cuh"

namespace qdsp {

// taps of the plan that currently owns the constant bank: g[q*DS + col] = h[q*DS + col - pad], q < 8 (float4 = 2 column pairs)
__constant__ float4 c_chan_taps[8 * 1280 / 4];

struct ChanArgs {
    DecimArgs a;              // hist, in, H, n_in, part, T, DS, nco, abs0; out_iq = partial planes, out_stride = plane pitch
    int nslices;
    int seg_rows;             // outputs per segment (CTA)
    int pad;                  // tap-table alignment pad (uniform over the batch)
    int nch, groups;
    float g8[2];              // tap row 8, columns 0..1 of slice 0 (the stray taps of T = 8*DS + 1)
    const float* taps_dev;    // [8][DS] taps in global memory (shared-memory tap variant)
};

// SLICE is a template parameter so that every constant-bank tap address is an immediate: ptxas then feeds the FFMA2s
// from uniform registers (LDCU.128 c[3][imm]); with a run-time slice offset it falls back to per-thread LDC loads.
// SLICE < 0: run-time slice (blockIdx.z), the slice's 8 x DC taps are staged in shared memory and read with broadcast
// loads -- one body for every slice, used when few channel groups run per GPU (the immediate-tap bodies of different
// slices would otherwise be resident together and thrash the instruction cache: ncu `no_instructions` stalls).
template <int DS, int DC, bool ROT, int SLICE, int NR = 1>
__device__ __forceinline__ void chan_body(const ChanArgs& ca) {
    constexpr int PAIRS = DC / 2;
    constexpr int RS = 4;                       // rows per ring stage (a multiple of NR)
    static_assert(RS % NR == 0, "rows per step");
    constexpr int NSTG = 4;                     // ring depth
    constexpr uint32_t ROW_BYTES = DC * 8u;
    constexpr uint32_t STAGE_BYTES = RS * ROW_BYTES;
    static_assert(DC % 4 == 0 && DS % DC == 0, "slice geometry");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const DecimArgs& a = ca.a;
    const int lane = threadIdx.x;
    const int seg = blockIdx.x;
    const int slice = SLICE >= 0 ? SLICE : (int)blockIdx.z;
    const int b = blockIdx.y / ca.groups, group = blockIdx.y - b * ca.groups;
    const BlkInfo bi = a.part.get(b);
    const int k0 = seg * ca.seg_rows;
    // shared-memory carve-up: [staged taps (shared-memory-tap variant)][TMA ring | mbarriers]
    constexpr uint32_t TAPS_BYTES = SLICE < 0 ? 8u * DC * 4u : 0u;
    unsigned char* smem_cta = smem_raw;
    unsigned char* smem_warp = smem_raw + TAPS_BYTES;
    const int nout = bi.out_count - k0 < ca.seg_rows ? bi.out_count - k0 : ca.seg_rows;
    const int nrows = nout + 8;                                   // rows k0 .. k0 + nout - 1 + 8
    const int nstages = (nrows + RS - 1) / RS;
    // row r of the segment, this slice: samples [row0 + r*DS, + DC)
    const long long row0 = bi.in_start + (long long)k0 * DS - a.T - ca.pad + (long long)slice * DC;
    const int ch = group * 32 + lane;
    const bool ch_ok = ch < ca.nch;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_warp + NSTG * STAGE_BYTES);
    // taps of this slice: constant bank at immediate offsets, or shared memory [pair][q] (8 tap pairs = 64 bytes per pair)
    const float4* gt = c_chan_taps + (SLICE >= 0 ? SLICE : 0) * (DC / 4);
    float4* gs = reinterpret_cast<float4*>(smem_cta);
    if (SLICE < 0) {
        float2* gs2 = reinterpret_cast<float2*>(gs);
        const float* gsrc = ca.taps_dev;                      // [8][DS] floats (pad applied)
        for (int e = lane; e < PAIRS * 8; e += 32) {
            const int c = e >> 3, q = e & 7;
            const float* src = gsrc + (size_t)q * DS + (size_t)slice * DC + 2 * c;
            gs2[e] = make_float2(src[0], src[1]);
        }
    }
    __syncwarp();
    if (k0 >= bi.out_count) return;

    uint64_t nco_step = 0, nco_ph0 = 0;
    if (ROT) {
        const NcoDev nd = a.nco[ch_ok ? ch : 0];
        nco_step = nd.step;
        nco_ph0 = nd.init + nco_step * (uint64_t)a.abs0;
    }
    if (lane == 0) {
        for (int s = 0; s < NSTG; s++) mbar_init(&mbar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    auto issue = [&](int st) {
        if (st >= nstages) return;
        const int slot = st % NSTG;
        unsigned char* dst = smem_warp + slot * STAGE_BYTES;
        const long long s0 = row0 + (long long)st * RS * DS;                    // first sample of the stage's first row
        const long long last_end = s0 + (long long)(RS - 1) * DS + DC;
        if (s0 >= 0 && last_end <= a.n_in) {
            if (lane == 0) mbar_arrive_expect_tx(&mbar[slot], STAGE_BYTES);
            __syncwarp();
            if (lane < RS) tma_bulk_g2s(dst + lane * ROW_BYTES, a.in + s0 + (long long)lane * DS, ROW_BYTES, &mbar[slot]);
        } else {   // history before sample 0 / ragged end of the caller's buffer: guarded fill
            VStream<float2> xs{a.hist, a.in, a.H};
            float2* d2 = reinterpret_cast<float2*>(dst);
            for (int e = lane; e < RS * DC; e += 32) {
                const int rr = e / DC;
                const long long idx = s0 + (long long)rr * DS + (e - rr * DC);
                d2[e] = idx < a.n_in ? xs.at(idx) : make_float2(0.f, 0.f);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&mbar[slot]);
        }
    };
    for (int st = 0; st < NSTG; st++) issue(st);

    // per-lane NCO constants: every row slice starts from an exact (closed-form) seed; along the row two interleaved
    // phasors (columns c, c+1) advance by w^2
    float2 w1 = make_float2(1.f, 0.f), w2 = make_float2(1.f, 0.f);
    if (ROT) {
        w1 = phasor_from_turns(nco_step);
        w2 = phasor_from_turns(nco_step * 2ull);
    }
    const float2 wr2 = make_float2(w2.x, w2.x), wi2 = make_float2(w2.y, w2.y), nwi2 = make_float2(-w2.y, -w2.y);
    const float2 g8 = slice == 0 ? make_float2(ca.g8[0], ca.g8[1]) : make_float2(0.f, 0.f);

    float2 O[8];                 // outputs in flight: O[q] = partial of output (row - q)
#pragma unroll
    for (int q = 0; q < 8; q++) O[q] = make_float2(0.f, 0.f);
    float2* plane = a.out_iq + ((size_t)(ch_ok ? ch : 0) * ca.nslices + slice) * (size_t)a.out_stride + bi.out_start + k0;

#pragma unroll 1
    for (int st = 0; st < nstages; st++) {
        const int slot = st % NSTG;
        mbar_wait(&mbar[slot], (uint32_t)((st / NSTG) & 1));
#pragma unroll 1
        for (int rr = 0; rr < RS; rr += NR) {
            const int r = st * RS + rr;
            if (r >= nrows) break;
            // NR rows per step: one set of tap loads feeds the FFMA2s of NR rows (halves the tap traffic for NR = 2)
            const float4* xrow[NR];
            float2 PR[NR], PI[NR];
#pragma unroll
            for (int j = 0; j < NR; j++) {
                xrow[j] = reinterpret_cast<const float4*>(smem_warp + slot * STAGE_BYTES + (rr + j) * ROW_BYTES);
                PR[j] = make_float2(1.f, 1.f);
                PI[j] = make_float2(0.f, 0.f);
                if (ROT) {
                    const long long n0 = row0 + (long long)(r + j) * DS;
                    const float2 p0 = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)n0);
                    const float2 p1 = cmul(p0, w1);
                    PR[j] = make_float2(p0.x, p1.x);
                    PI[j] = make_float2(p0.y, p1.y);
                }
            }
            float2 aRe[NR][8], aIm[NR][8];
            float2 sRe[NR], sIm[NR];
#pragma unroll
            for (int c = 0; c < PAIRS; c++) {
                float2 RE[NR], IM[NR];
#pragma unroll
#pragma unroll
                for (int j = 0; j < NR; j++) {
                    const float4 v = xrow[j][c];
                    if (ROT) {
                        RE[j].x = fmaf(v.x, PR[j].x, -(v.y * PI[j].x));
                        IM[j].x = fmaf(v.x, PI[j].x, v.y * PR[j].x);
                        RE[j].y = fmaf(v.z, PR[j].y, -(v.w * PI[j].y));
                        IM[j].y = fmaf(v.z, PI[j].y, v.w * PR[j].y);
                        const float2 nPR = __ffma2_rn(PI[j], nwi2, __fmul2_rn(PR[j], wr2));
                        PI[j] = __ffma2_rn(PI[j], wr2, __fmul2_rn(PR[j], wi2));
                        PR[j] = nPR;
                    } else {
                        RE[j] = make_float2(v.x, v.z);
                        IM[j] = make_float2(v.y, v.w);
                    }
                }
                float4 gq[4];
                if (SLICE < 0) {
#pragma unroll
                    for (int j = 0; j < 4; j++) gq[j] = gs[c * 4 + j];
                }
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    float2 g;
                    if (SLICE >= 0) {
                        const float4 g4 = gt[q * (DS / 4) + c / 2];
                        g = (c & 1) ? make_float2(g4.z, g4.w) : make_float2(g4.x, g4.y);
                    } else {
                        g = (q & 1) ? make_float2(gq[q >> 1].z, gq[q >> 1].w) : make_float2(gq[q >> 1].x, gq[q >> 1].y);
                    }
#pragma unroll
                    for (int j = 0; j < NR; j++) {
                        if (c == 0) {
                            aRe[j][q] = __fmul2_rn(RE[j], g);
                            aIm[j][q] = __fmul2_rn(IM[j], g);
                        } else {
                            aRe[j][q] = __ffma2_rn(RE[j], g, aRe[j][q]);
                            aIm[j][q] = __ffma2_rn(IM[j], g, aIm[j][q]);
                        }
                    }
                }
                if (c == 0) {
#pragma unroll
                    for (int j = 0; j < NR; j++) {
                        sRe[j] = __fmul2_rn(RE[j], g8);
                        sIm[j] = __fmul2_rn(IM[j], g8);
                    }
                }
            }
            // outputs in flight: output (row - q) takes that row's S_q
#pragma unroll
            for (int j = 0; j < NR; j++) {
                auto fin = [&](float2 re2, float2 im2) { return make_float2(re2.x + re2.y, im2.x + im2.y); };
                const float2 s8 = fin(sRe[j], sIm[j]);
                const float2 y = __fadd2_rn(O[7], s8);                 // output row - 8 is complete
#pragma unroll
                for (int q = 7; q >= 1; q--) O[q] = __fadd2_rn(O[q - 1], fin(aRe[j][q], aIm[j][q]));
                O[0] = fin(aRe[j][0], aIm[j][0]);
                const int k = r + j - 8;
                if (k >= 0 && k < nout && ch_ok) plane[k] = y;
            }
        }
        __syncwarp();
        issue(st + NSTG);
    }
}

template <int DS, int DC, bool ROT, int S0>
__device__ __forceinline__ void chan_dispatch(int slice, const ChanArgs& ca) {
    if constexpr (S0 < DS / DC) {
        if (slice == S0) chan_body<DS, DC, ROT, S0>(ca);
        else chan_dispatch<DS, DC, ROT, S0 + 1>(slice, ca);
    }
}
// grid = (segments, run() blocks x channel groups, slices): the CTAs resident together belong to one or two slices, so the
// instruction working set is one or two of the DS/DC bodies
template <int DS, int DC, bool ROT>
__global__ void __launch_bounds__(32) chan_kernel(const __grid_constant__ ChanArgs ca) {
    chan_dispatch<DS, DC, ROT, 0>((int)blockIdx.z, ca);
}
// NR = 2: one set of shared-memory tap loads feeds two rows
template <int DS, int DC, bool ROT>
__global__ void __launch_bounds__(32) chan_smemtaps_kernel(const __grid_constant__ ChanArgs ca) {
    chan_body<DS, DC, ROT, -1, 2>(ca);
}

// ---- host side -------------------------------------------------------------------------------------
bool chan_supported(const DecimPlan* plan) {
    // wide rows of a geometry instantiated below, 8 full tap rows + at most the two stray taps of row 8
    return (plan->DS == 1280 || plan->DS == 128) && plan->T + 1 <= 8 * plan->DS + 2 && plan->T > 4 * plan->DS;
}

// The constant bank holds ONE plan's taps at a time. Uploads are enqueued on the launching stream (stream-ordered with
// the kernels that read them); switching to another plan or stream first waits for the device to drain.
static std::mutex g_chan_mtx;
static const void* g_chan_owner = nullptr;
static int g_chan_owner_pad = -1;
static cudaStream_t g_chan_owner_stream = nullptr;
static float* g_chan_taps_dev = nullptr;

template <int DS, int DC>
static int launch_chan_t(DecimPlan* plan, const float* taps_host, const float2* hist, int H, const float2* in,
                         const Partition& part, bool rot, const NcoDev* nco_dev, long long abs0, int nch, float2* ypart,
                         long long ystride, int pad, cudaStream_t s) {
    std::lock_guard<std::mutex> lk(g_chan_mtx);
    const int T = plan->T;
    auto h = [&](long long t) { return (t >= 0 && t < T) ? taps_host[t] : 0.0f; };
    if (g_chan_owner != plan || g_chan_owner_pad != pad || g_chan_owner_stream != s) {
        if (g_chan_owner != nullptr) QDSP_CUDA_OK(cudaDeviceSynchronize());
        static std::vector<float> tab;
        tab.assign(8 * 1280, 0.0f);
        for (int q = 0; q < 8; q++)
            for (int c = 0; c < DS; c++) tab[(size_t)q * DS + c] = h((long long)q * DS + c - pad);
        QDSP_CUDA_OK(cudaMemcpyToSymbolAsync(c_chan_taps, tab.data(), sizeof(float) * 8 * DS, 0, cudaMemcpyHostToDevice, s));
        if (!g_chan_taps_dev) QDSP_CUDA_OK(cudaMalloc(&g_chan_taps_dev, sizeof(float) * 8 * 1280));
        QDSP_CUDA_OK(cudaMemcpyAsync(g_chan_taps_dev, tab.data(), sizeof(float) * 8 * DS, cudaMemcpyHostToDevice, s));
        QDSP_CUDA_OK(cudaStreamSynchronize(s));   // `tab` is reused by the next upload
        g_chan_owner = plan;
        g_chan_owner_pad = pad;
        g_chan_owner_stream = s;
    }
    ChanArgs ca{};
    DecimArgs& a = ca.a;
    a.hist = hist;
    a.in = in;
    a.H = H;
    a.n_in = part.view.total;
    a.part = part.view;
    a.T = T;
    a.DS = DS;
    a.D = DC;
    a.nco = nco_dev;
    a.abs0 = abs0;
    a.out_iq = ypart;
    a.out_stride = ystride;
    ca.nslices = DS / DC;
    ca.pad = pad;
    ca.nch = nch;
    ca.groups = (nch + 31) / 32;
    ca.g8[0] = h(8ll * DS - pad);
    ca.g8[1] = h(8ll * DS + 1 - pad);
    ca.taps_dev = g_chan_taps_dev;
    // outputs per segment (CTA): enough single-warp CTAs to fill the machine several times over; the halo is 8 rows
    // B200, 2^26 samples (GS/s wideband): 32 ch (1 group): 80: 27.0, 128: 31.0, 160: 29.3, 320: 29.5; 256 ch: 128: 4.41, 160: 4.44, 320: 3.69
    ca.seg_rows = ca.groups < 4 ? 128 : 160;
    dim3 grid((part.max_out + ca.seg_rows - 1) / ca.seg_rows, part.view.nblocks * ca.groups, ca.nslices);
    if (grid.y > 65535) {
        set_last_error("chan: too many run() blocks x channel groups (%u)", grid.y);
        return -1;
    }
    // few channel groups: the slice bodies with immediate taps would be resident side by side (instruction-cache thrash);
    // use the one-body variant with taps in shared memory
    const bool smemtaps = ca.groups < 4;
    constexpr size_t smem = 4 * 4 * DC * 8 + 64 + 8 * DC * 4 + 64;
    if (rot && smemtaps) {
        auto kern = chan_smemtaps_kernel<DS, DC, true>;
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 32, smem, s>>>(ca);
    } else if (rot) {
        auto kern = chan_kernel<DS, DC, true>;
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 32, smem, s>>>(ca);
    } else {
        auto kern = chan_kernel<DS, DC, false>;
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 32, smem, s>>>(ca);
    }
    QDSP_LAUNCH_OK();
    return 0;
}

void chan_plan_released(const DecimPlan* plan) {
    std::lock_guard<std::mutex> lk(g_chan_mtx);
    if (g_chan_owner == plan) g_chan_owner = nullptr;     // a new plan may be allocated at the same address
}

// mode: 0 = resampled IQ out, 1 = fused NCO + FM demod (audio [+ iq])
int launch_chan(DecimPlan* plan, const float* taps_host, const float2* hist, int H, const float2* in, const Partition& part,
                int mode, const NcoDev* nco_dev, long long abs0, int nch, float phasor_speed, const float* demod_in,
                float* demod_out, float2* out_iq, float* audio, long long out_stride, int pad, cudaStream_t s) {
    if (part.view.nblocks == 0 || part.max_out == 0) return 0;
    constexpr int DC = 64;
    const int nslices = plan->DS / DC;
    const size_t ystride = (size_t)((part.total_out + 63) / 64) * 64;
    const size_t need = (size_t)nch * nslices * ystride;
    if (need > plan->ypart_cap) {
        if (plan->ypart) cudaFree(plan->ypart);
        plan->ypart = nullptr;
        plan->ypart_cap = 0;
        QDSP_CUDA_OK(cudaMalloc(&plan->ypart, need * sizeof(float2)));
        plan->ypart_cap = need;
    }
    int rc;
    if (plan->DS == 1280)
        rc = launch_chan_t<1280, DC>(plan, taps_host, hist, H, in, part, mode == 1, nco_dev, abs0, nch, plan->ypart, (long long)ystride, pad, s);
    else
        rc = launch_chan_t<128, DC>(plan, taps_host, hist, H, in, part, mode == 1, nco_dev, abs0, nch, plan->ypart, (long long)ystride, pad, s);
    if (rc != 0) return rc;
    return launch_decim_finish(plan->ypart, (long long)ystride, nslices, part.total_out, mode == 1 ? 1 : 0, phasor_speed, demod_in,
                               demod_out, out_iq, audio, out_stride, nch, s);
}

}  // namespace qdsp
