// qdsp_b200/csrc/k_rowlane.cu — row-per-lane decimating FIR for sm_100a (interp = 1, narrow rows), with the NCO
// prologue and FM-demod epilogue of the fused xlate -> resample -> demod pass (reference vfo.h:19-36,
// resampling.h:99-132, processing.h:55-70, demodulator.h:81-99).
//
// Formulation. Rows of D samples, taps zero-padded to Q*D (g[q*D + c]); with W_c = e^{j*theta*c} and
// P_r = e^{j*theta*n(r, 0)} (n = absolute sample index of the row's first column)
//     y[k] = sum_{q<Q} P_{k+q} * S_q(k+q),      S_q(r) = sum_{c<D} g[q*D + c] * (x[r, c] * W_c)
// A WARP owns a run of consecutive rows; lane j of step i owns row 32*i + j and computes the Q row partials S_q of
// its row for all columns: 2*Q accumulators (column-pair packed, one FFMA2 = two MACs), the tap pairs and W_c come
// from the kernel-parameter constant bank as UNIFORM register operands (FFMA2 R, R, UR, R: no tap registers, no tap
// loads through the LSU), the row's samples from shared memory with one conflict-free 128-bit load per 2*Q FFMA2
// (lane stride = row pitch = D*8 bytes, (D/2) odd). Output k then needs Q values that live in the Q lanes
// k .. k+Q-1: Q-1 shuffles per step, lanes whose window runs past lane 31 finish one step later. Nothing is
// exchanged through shared memory and there is no CTA barrier: a CTA is ONE warp with its own TMA ring
// (one cp.async.bulk of 32 contiguous rows per stage, completion on an mbarrier), 8 CTAs per SM.
// Tiles overlap by Q-1 rows (+1 for the demodulator's leading angle): 3.6 % re-read at the default 8 steps per tile.
// The last history_advance of the batch (filter.h:71 / resampling.h:129) is done by CTA (0,0): no extra launch.
#include <math.h>
#include <mutex>
#include <new>
#include "decim_common.cuh"

namespace qdsp {

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <int Q, int D>
struct RowArgs {
    DecimArgs a;
    float2* hist_next;        // when non-null: CTA (0,0) writes the advanced history tail here
    unsigned long long* tstamp;   // when non-null (timing ring slot, %globaltimer ns): [0] min CTA start, [1] max CTA end
    int nstep;                // steps (of 32 rows) per full tile
    int pad;                  // tap-table alignment pad (uniform over the batch)
    float g[Q * D];           // g[q*D + c] = h[q*D + c - pad], zero outside [0, T)
    float2 w[D];              // W_c
};

template <int Q, int D, int JLIVE, int NSTG, bool ROT, bool DEMOD>
__global__ void __launch_bounds__(32) decim_rowlane_kernel(const __grid_constant__ RowArgs<Q, D> ra) {
    constexpr int LEAD = DEMOD ? 1 : 0;
    constexpr int P = D / 2;
    constexpr uint32_t STAGE_BYTES = 32u * D * 8u;
    static_assert((P & 1) == 1, "row pitch must be an odd number of 16-byte units (conflict-free 128-bit loads)");
    static_assert(Q >= 2 && Q <= 24, "Q");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const DecimArgs& a = ra.a;
    const int lane = threadIdx.x;
    const int tile = blockIdx.x, b = blockIdx.y;
    const BlkInfo bi = a.part.get(b);
    const int LT = 32 * ra.nstep - (Q - 1) - LEAD;     // outputs per full tile
    const int k0 = tile * LT;
    if (ra.tstamp != nullptr && tile == 0 && b == 0 && lane == 0) atomicMin(&ra.tstamp[0], globaltimer_ns());

    // Overlapped consecutive calls (decim_common.cuh). A CTA waits at its start when it folds the history (CTA (0,0)), when
    // its rows or its leading-angle window reach before sample 0, or when it takes its leading angle from `demod_in`.
    // Every fused CTA waits again before it stores its held audio and `demod_out`, so write-after-write on them stays ordered
    // whatever buffers the caller passes; the launcher only refuses an input that overlaps the previous call's audio.
    if (ra.hist_next != nullptr && tile == 0 && b == 0) {
        pdl_wait();
        fold_history(a.hist, a.in, a.H, a.n_in, ra.hist_next, lane, 32);
    }
    if (k0 >= bi.out_count) return;

    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + NSTG * STAGE_BYTES);
    const int pad = ra.pad;
    const int nout = bi.out_count - k0 < LT ? bi.out_count - k0 : LT;      // outputs this tile emits
    const int nsteps = (nout + LEAD + Q - 1 + 31) / 32;                    // rows needed / 32
    // row r of the tile (r = 32*i + lane) starts at sample row0 + r*D (relative to this call's input)
    const long long row0 = bi.in_start + (long long)(k0 - LEAD) * D - a.T - pad;

    uint64_t nco_step = 0, nco_ph0 = 0;
    if (ROT) {
        nco_step = a.nco[0].step;
        nco_ph0 = a.nco[0].init + nco_step * (uint64_t)a.abs0;
    }
    if (lane == 0) {
        for (int s = 0; s < NSTG; s++) mbar_init(&mbar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // leading angle of the block's very first output
    bool use_override = false;
    float override_ang = 0.f;
    int pb = b - 1;
    BlkInfo pbi{};
    long long ovr_win = 0;     // first sample of the window of the previous block's last output (off-grid hand-over)
    if (DEMOD && tile == 0) {
        while (pb >= 0) {
            pbi = a.part.get(pb);
            if (pbi.out_count > 0) break;
            pb--;
        }
        if (pb < 0) {
            use_override = true;
        } else if (pb != b - 1 || pbi.in_start + (long long)pbi.out_count * D != bi.in_start) {
            use_override = true;  // previous block's last output is off this block's row grid
            ovr_win = pbi.in_start + (long long)(pbi.out_count - 1) * D - a.T;
        }
    }
    if (row0 < 0 || (use_override && (pb < 0 || ovr_win < 0))) pdl_wait();
    if (use_override) {
        if (pb < 0) {
            override_ang = a.demod_in[0];
        } else {
            const float2 y = direct_output_warp<ROT>(a, ovr_win, nco_ph0, nco_step);
            override_ang = fast_arctan2_ref(y.y, y.x);
        }
    }
    __syncwarp();

    // ---- producer: stage i = rows [32 i, 32 i + 32) = one contiguous run of 32*D samples ------------------
    auto issue = [&](int i) {
        if (i >= nsteps) return;
        const int slot = i % NSTG;
        unsigned char* dst = smem_raw + slot * STAGE_BYTES;
        const long long s0 = row0 + (long long)i * (32 * D);
        if (s0 >= 0 && s0 + 32 * D <= a.n_in) {
            if (lane == 0) {
                mbar_arrive_expect_tx(&mbar[slot], STAGE_BYTES);
                tma_bulk_g2s(dst, a.in + s0, STAGE_BYTES, &mbar[slot]);
            }
        } else {   // history before sample 0 / ragged end of the caller's buffer: guarded fill
            VStream<float2> xs{a.hist, a.in, a.H};
            float2* d2 = reinterpret_cast<float2*>(dst);
            for (int e = lane; e < 32 * D; e += 32) {
                const long long idx = s0 + e;
                d2[e] = idx < a.n_in ? xs.at(idx) : make_float2(0.f, 0.f);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&mbar[slot]);
        }
    };
    for (int i = 0; i < NSTG; i++) issue(i);
    pdl_launch_dependents();

    // ---- per-lane state -------------------------------------------------------------------------------
    float2 Pr = make_float2(1.f, 0.f);        // row phasor of this lane's current row
    float2 old = make_float2(0.f, 0.f);       // partial output of (previous step, this lane), lanes >= 32-(Q-1)
    float ang_saved = 0.f;
    const bool tail_lane = lane >= 32 - (Q - 1);
    const long long obase = a.out_stride * 0 + bi.out_start + k0 - LEAD;   // output index of tile-relative output 0
    // the tile's audio, indexed by tile-relative output (32 per step), stored after the wait for the previous grid
    float* hold = reinterpret_cast<float*>(smem_raw + NSTG * STAGE_BYTES + NSTG * 8 + 16);
    bool last_here = false;                   // this lane computes the call's last output: its angle is `demod_out`
    float last_ang = 0.f;

#pragma unroll 1
    for (int i = 0; i < nsteps; i++) {
        const int slot = i % NSTG;
        if (ROT) {
            // the row phasor is a pure function of the row's absolute sample index (closed form, no recurrence down the
            // rows): an output's value does not depend on which tile / step / lane computes it, so any batching of the
            // stream into process() calls (and the chunking of process_host) gives bit-identical audio
            const long long n0 = row0 + (long long)(32 * i + lane) * D;
            Pr = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)n0);
        }
        mbar_wait(&mbar[slot], (uint32_t)((i / NSTG) & 1));
        const float4* xrow = reinterpret_cast<const float4*>(smem_raw + slot * STAGE_BYTES + lane * (D * 8));
        float2 aRe[Q], aIm[Q];
#pragma unroll
        for (int c = 0; c < P; c++) {
            const float4 v = xrow[c];
            float2 RE, IM;
            if (ROT) {
                const float2 w0 = ra.w[2 * c], w1 = ra.w[2 * c + 1];
                RE.x = fmaf(v.x, w0.x, -(v.y * w0.y));
                IM.x = fmaf(v.x, w0.y, v.y * w0.x);
                RE.y = fmaf(v.z, w1.x, -(v.w * w1.y));
                IM.y = fmaf(v.z, w1.y, v.w * w1.x);
            } else {
                RE = make_float2(v.x, v.z);
                IM = make_float2(v.y, v.w);
            }
#pragma unroll
            for (int q = 0; q < Q; q++) {
                if (q * D + 2 * c < JLIVE) {
                    const float2 g = make_float2(ra.g[q * D + 2 * c], ra.g[q * D + 2 * c + 1]);
                    if (c == 0) {
                        aRe[q] = __fmul2_rn(RE, g);
                        aIm[q] = __fmul2_rn(IM, g);
                    } else {
                        aRe[q] = __ffma2_rn(RE, g, aRe[q]);
                        aIm[q] = __ffma2_rn(IM, g, aIm[q]);
                    }
                }
            }
        }
        __syncwarp();              // every lane is done with the slot
        issue(i + NSTG);           // refill it

        // ---- row partials -> outputs: V_q = P_r * S_q; output of row r takes V_q from lane (r + q) --------
        float2 cur = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < Q; q++) {
            float2 s = make_float2(aRe[q].x + aRe[q].y, aIm[q].x + aIm[q].y);
            if (ROT) s = cmul(s, Pr);
            if (q == 0) {
                cur = s;
            } else {
                float2 p;
                p.x = __shfl_sync(0xffffffffu, s.x, (lane + q) & 31);
                p.y = __shfl_sync(0xffffffffu, s.y, (lane + q) & 31);
                if (lane + q < 32) cur = __fadd2_rn(cur, p);
                else old = __fadd2_rn(old, p);      // row of THIS step, output of the previous step's lane
            }
        }
        // lanes < 32-(Q-1): output of this step's row is complete; tail lanes: the previous step's output is
        const float2 y = tail_lane ? old : cur;
        if (tail_lane) old = cur;
        const int orel = 32 * i + lane - (tail_lane ? 32 : 0);     // tile-relative output (0 = the leading one)
        const bool live = orel >= LEAD && orel < nout + LEAD;
        const long long oidx = obase + orel;
        if (DEMOD) {
            const float ang = fast_arctan2_ref(y.y, y.x);
            float prev = __shfl_sync(0xffffffffu, ang, (lane + 31) & 31);
            const float prev_tail = __shfl_sync(0xffffffffu, ang_saved, 32 - Q);   // lane 32-(Q-1)-1 of the previous step
            if (lane == 32 - (Q - 1)) prev = prev_tail;
            if (use_override && orel == 1) prev = override_ang;
            ang_saved = ang;
            if (live) {
                hold[orel] = fm_step_ref(ang, prev, a.phasor_speed);
                if (oidx == a.part.total_out - 1) {
                    last_here = true;
                    last_ang = ang;
                }
                if (a.out_iq) a.out_iq[oidx] = y;    // calls that want IQ are never overlapped (launch_decim_rowlane)
            }
        } else {
            if (live) a.out_iq[oidx] = y;
        }
    }
    if (DEMOD) {
        pdl_wait();
        __syncwarp();
        for (int e = LEAD + lane; e < nout + LEAD; e += 32) a.audio[obase + e] = hold[e];
        if (last_here) a.demod_out[0] = last_ang;
    }
    if (ra.tstamp != nullptr) {
        __syncwarp();
        if (lane == 0) atomicMax(&ra.tstamp[1], globaltimer_ns());
    }
}

// ---- host side -------------------------------------------------------------------------------------
bool rowlane_supported(const DecimPlan* plan) {
    return plan->nslices == 1 && plan->DS == 50 && plan->Q == 9 && plan->T + 1 > 8 * 50;
}

// the tap-table alignment pad must be the same for every run() block of the batch: -1 if it is not
int rowlane_uniform_pad(const Partition& part, int T) {
    if (part.view.nblocks <= 0) return -1;
    if (part.view.table == nullptr) {
        if (part.view.nblocks > 1 && (part.view.block_size & 1)) return -1;
        return T & 1;
    }
    const int pad = (int)((part.host[0].in_start - T) & 1);
    for (int b = 1; b < part.view.nblocks; b++)
        if ((int)((part.host[b].in_start - T) & 1) != pad) return -1;
    return pad;
}

int launch_decim_rowlane(DecimPlan* plan, const float* taps_host, const float2* hist, float2* hist_next, int H,
                         const float2* in, const Partition& part, int mode, const NcoDev* nco_dev, const NcoDev* nco_host,
                         long long abs0, float phasor_speed, const float* demod_in, float* demod_out, float2* out_iq,
                         float* audio, int pad, cudaStream_t s, bool overlap_prev, unsigned long long* tstamp) {
    constexpr int Q = 9, D = 50, NSTG = 2;
    static RowArgs<Q, D> ra;     // large (4 KB): built in place; launches copy it at enqueue time
    static std::mutex mtx;
    std::lock_guard<std::mutex> lk(mtx);
    DecimArgs& a = ra.a;
    a = DecimArgs{};
    a.hist = hist;
    a.in = in;
    a.H = H;
    a.n_in = part.view.total;
    a.taps = plan->taps_dev;   // pad-0 table == flat h[t] (direct_output_warp)
    a.part = part.view;
    a.T = plan->T;
    a.D = D;
    a.DS = D;
    a.nslices = 1;
    a.nco = nco_dev;
    a.abs0 = abs0;
    a.phasor_speed = phasor_speed;
    a.demod_in = demod_in;
    a.demod_out = demod_out;
    a.out_iq = out_iq;
    a.audio = audio;
    a.out_stride = 0;
    ra.hist_next = hist_next;
    ra.tstamp = tstamp;
    // B200 sweeps (GS/s), DESIGN.md 6.0. Isolated launches: 4: 811, 6: 823, 8: 824, 9: 787, 10: 802, 12: 792, 16: 808,
    // 20: 806, 24: 793, 32: 773. Consecutive calls overlapped, bench.py's 100-call burst: 8: 878, 16: 866; under the power
    // cap (2 s loop) 16 steps win instead (797 vs 775): less tile re-read, fewer instructions per sample.
    ra.nstep = 8;
    ra.pad = pad;
    for (int j = 0; j < Q * D; j++) {
        const int t = j - pad;
        ra.g[j] = (t >= 0 && t < plan->T) ? taps_host[t] : 0.0f;
    }
    const bool fused = mode == 1;
    if (fused) {
        const double th = (double)(int64_t)nco_host[0].step * (6.283185307179586476925286766559 / 18446744073709551616.0);
        for (int c = 0; c < D; c++) ra.w[c] = make_float2((float)cos(th * c), (float)sin(th * c));
    } else {
        for (int c = 0; c < D; c++) ra.w[c] = make_float2(1.f, 0.f);
    }
    const int lead = fused ? 1 : 0;
    const int LT = 32 * ra.nstep - (Q - 1) - lead;
    dim3 grid((part.max_out + LT - 1) / LT, part.view.nblocks, 1);
    if (grid.x < 1) grid.x = 1;
    // TMA ring + mbarriers, then (fused) the tile's held audio: one float per lane per step
    const size_t smem = NSTG * 32 * D * 8 + NSTG * 8 + 16 + (fused ? (size_t)ra.nstep * 32 * sizeof(float) : 0);
    const bool overlap = overlap_prev && fused && out_iq == nullptr;
#define QDSP_ROW_LAUNCH(JL, ROTV, DEMV)                                                                   \
    {                                                                                                     \
        auto kern = decim_rowlane_kernel<Q, D, JL, NSTG, ROTV, DEMV>;                                     \
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        QDSP_CUDA_OK(launch_ex((const void*)kern, grid, dim3(32), smem, s, overlap, &ra));                \
    }
    // T <= 401: the last tap row (q = 8) has live taps in its first column pair only
    if (plan->T + 1 <= 402) {
        if (fused) QDSP_ROW_LAUNCH(402, true, true) else QDSP_ROW_LAUNCH(402, false, false)
    } else {
        if (fused) QDSP_ROW_LAUNCH(Q * D, true, true) else QDSP_ROW_LAUNCH(Q * D, false, false)
    }
#undef QDSP_ROW_LAUNCH
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
