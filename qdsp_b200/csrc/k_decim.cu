// qdsp_b200/csrc/k_decim.cu — column-parallel decimating FIR for sm_100a (interp = 1, even decim D),
// with an optional NCO prologue and FM-demod epilogue: the fused xlate -> resample -> demod pass of
// the reference's VFO + FloatFMDemod chain (vfo.h:19-36, resampling.h:99-132, demodulator.h:81-99).
//
// Formulation. View the stream as a matrix with rows of D samples. With taps zero-padded to Q*D,
//     y[k] = sum_{r<D} sum_{q<Q} g[q*D + r] * x'[base + (k+q)*D + r]
// so column r is a Q-tap FIR over the column's own sub-stream. A thread owns a PAIR of adjacent
// columns and keeps their Q tap pairs in registers; it walks down the rows with Q partial outputs in
// flight (static register rotation: the row loop is unrolled by Q). One FFMA2 (packed f32x2) does
// the two columns' MACs for re, another for im: (re[r], re[r+1]) * (g[r], g[r+1]) — no duplicated
// tap registers, one 128-bit shared-memory load per 2 samples per 2*Q FFMA2.
//
// Data movement. A CTA covers NSEG row segments of L outputs each; every segment streams its rows
// through a ring of NSTAGE shared-memory stages filled by TMA bulk copies (cp.async.bulk, completion
// on an mbarrier) — R rows per stage per segment. Segments whose chunk would cross the ends of the
// caller's buffer (history before sample 0, ragged tail) are filled by guarded loads instead.
// Column partial sums are exchanged through a small double-buffered shared array and reduced by
// 8-lane groups; the epilogue applies fast_arctan2 + phase difference on chip, so neither the
// translated nor the resampled IQ ever reaches HBM (unless the caller asks for the IQ).
#include <stdlib.h>
#include <new>
#include <vector>
#include "decim_common.cuh"

namespace qdsp {

// shared-memory pitches (used by the kernel and by the launcher's size computation)
__host__ __device__ inline int decim_seg_pad(int D) {
    // chunk = R*D samples; pad (in samples, even) so that pitch*8 == D*8 (mod 128)
    const int want = (D * 8) % 128, have = (3 * D * 8) % 128;
    const int pad_bytes = ((want - have) % 128 + 128) % 128;
    return pad_bytes / 8;   // D even => both residues are multiples of 16: pad is an even sample count
}
__host__ __device__ inline int decim_ppad_sup(int P) {
    int p = P;
    while ((p & 3) != 2) p++;
    return p;
}

// packed f32x2 helpers for the two-column phasor recurrence
__device__ __forceinline__ float2 neg2(float2 v) { return make_float2(-v.x, -v.y); }

template <int Q, bool ROT, bool DEMOD, bool SUPRED, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) decim_kernel(const DecimArgs a) {
    constexpr int R = 3;            // rows per stage per segment
    constexpr int NS = Q / R;       // stages per super-iteration == ring depth: slot index is static
    constexpr int LEAD = DEMOD ? 1 : 0;
    static_assert(Q % R == 0 && NS >= 2, "Q must be a multiple of 3, at least 6");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int D = a.D;
    const int NSEG = a.NSEG;
    const int P = D / 2, L = a.L;
    const int t = threadIdx.x;
    const int tile_x = a.plane_fast ? blockIdx.y : blockIdx.x;
    const int b = a.plane_fast ? blockIdx.z : blockIdx.y;
    const int plane = a.plane_fast ? blockIdx.x : blockIdx.z;   // output plane: channel, or (channel, slice) for sliced rows
    const int ch = plane / a.nslices, slice = plane - ch * a.nslices;
    const int DSg = a.DS;                        // global row stride; == D unless the rows are sliced
    const long long col_off = (long long)slice * D;
    const BlkInfo bi = a.part.get(b);
    const int k0 = tile_x * (NSEG * L);
    if (k0 >= bi.out_count) return;

    // ---- shared memory carve-up (byte offsets from the dynamic base) ---------------------------
    const int chunk_elems = R * D;                                   // per segment per stage
    const long long chunk_span = (long long)R * a.DS;                // global samples one stage advances
    const long long chunk_tail = (long long)(R - 1) * a.DS + D;      // samples from a chunk's first to past its last
    const uint32_t chunk_bytes = (uint32_t)chunk_elems * 8u;
    // segment pitch in a ring slot: padded so that a warp whose lanes straddle two segments keeps walking
    // consecutive 16-byte bank groups (pitch == row bytes mod 128)
    const int seg_pitch = chunk_elems + decim_seg_pad(D);
    const uint32_t stage_bytes = (uint32_t)NSEG * (uint32_t)seg_pitch * 8u;
    // partial-buffer row pitch: odd for the 8-lane per-stage reduce; == 2 (mod 4) for the 2-lane SUPRED reduce
    // (lane pairs read 16 contiguous bytes, 16 rows land on 8 distinct 16-byte bank groups: 2 wavefronts)
    const int Ppad = SUPRED ? decim_ppad_sup(P) : (P | 1);
    // SUPRED (narrow rows): partials of a whole super-iteration (Q rows) are kept and reduced once per
    // super-iteration by 2 lanes per output; otherwise per stage (R rows) by 8 lanes per output
    constexpr int PROWS = SUPRED ? Q : R;
    const uint32_t pbuf_half = (uint32_t)(NSEG * PROWS * Ppad) * 8u; // one parity of the partial buffer
    constexpr int RY = 4 * Q;                                        // SUPRED: parked outputs live in a ring
    const int LL = SUPRED ? RY : L + LEAD;                           // outputs kept per segment
    const int LOUT = L + LEAD;                                       // outputs produced per segment
    float2* X = reinterpret_cast<float2*>(smem_raw);
    float2* Pbuf = reinterpret_cast<float2*>(smem_raw + NS * stage_bytes);                   // [2][NSEG*R][Ppad]
    float2* ybuf = reinterpret_cast<float2*>(smem_raw + NS * stage_bytes + 2 * pbuf_half);   // [NSEG][LL]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(ybuf + NSEG * LL);                          // [NS]
    float* s_misc = reinterpret_cast<float*>(mbar + NS);                                     // [0]=override angle
    // wide rows (more than 64 column pairs): the partial reduce runs in two levels, P -> 64 -> 1
    const bool two_level = P > 64;
    float2* P2 = reinterpret_cast<float2*>(s_misc + 4);                                      // [2][NSEG*R][64]

    // ---- thread roles ------------------------------------------------------------------------
    const int seg = t / P;
    const int pair = t - seg * P;
    const bool in_grid = seg < NSEG;
    const int pad = (int)((bi.in_start - a.T) & 1);
    const int ks = k0 + seg * L - LEAD;  // first output (the leading one when DEMOD) of this segment
    const long long seg_base = bi.in_start + (long long)ks * DSg - a.T - pad + col_off;
    const bool seg_active = in_grid && (k0 + seg * L < bi.out_count);
    // rows this CTA really needs: its fullest segment (segment 0) has min(L, out_count - k0) outputs
    const int need = (bi.out_count - k0 < L ? bi.out_count - k0 : L) + LEAD + Q - 1;
    const int nsup = (need + Q - 1) / Q < a.NSUP ? (need + Q - 1) / Q : a.NSUP;
    const int nst = nsup * NS;
    // producer bookkeeping: stages [fast_lo, fast_hi) of this segment are plain TMA bulk copies; stages
    // outside (history before sample 0, ragged end of the caller's buffer) are filled by guarded loads
    int fast_lo = 0, fast_hi = 0, live_hi = 0;
    if (seg_active) {
        live_hi = nst;
        const long long lo = seg_base >= 0 ? 0 : (-seg_base + chunk_span - 1) / chunk_span;
        const long long room = a.n_in - seg_base - chunk_tail;    // chunks that end inside the buffer
        const long long hi = room < 0 ? 0 : room / chunk_span + 1;
        fast_lo = (int)(lo < nst ? lo : nst);
        fast_hi = (int)(hi < nst ? hi : nst);
    }

    uint64_t nco_step = 0, nco_ph0 = 0;
    if (ROT) {
        nco_step = a.nco[ch].step;
        nco_ph0 = a.nco[ch].init + nco_step * (uint64_t)a.abs0;
    }

    if (t == 0) {
        for (int s = 0; s < NS; s++) mbar_init(&mbar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // leading-angle override of the block's very first output (warp 0)
    bool use_override = false;
    if (DEMOD && tile_x == 0) {
        int pb = b - 1;
        BlkInfo pbi{};
        while (pb >= 0) {
            pbi = a.part.get(pb);
            if (pbi.out_count > 0) break;
            pb--;
        }
        if (pb < 0) {
            use_override = true;
            if (t == 0) s_misc[0] = a.demod_in[ch];
        } else if (pb != b - 1 || pbi.in_start + (long long)pbi.out_count * DSg != bi.in_start) {
            use_override = true;  // previous block's last output is off this block's row grid
            if (t < 32) {
                const float2 y = direct_output_warp<ROT>(
                    a, pbi.in_start + (long long)(pbi.out_count - 1) * DSg - a.T, nco_ph0, nco_step);
                if (t == 0) s_misc[0] = fast_arctan2_ref(y.y, y.x);
            }
        }
    }
    __syncthreads();

    // ---- producer: warp 0, lane l issues segment l's TMA bulk copy; one mbarrier arrival per stage ----
    // (edge tiles -- history before sample 0 or the ragged end of the buffer -- also run the guarded fill)
    float2* xseg = X + (size_t)seg * seg_pitch;
    const int nactive = (bi.out_count - k0 + L - 1) / L < NSEG ? (bi.out_count - k0 + L - 1) / L : NSEG;
    const long long tile_first = bi.in_start + (long long)(k0 - LEAD) * DSg - a.T - pad + col_off;
    const long long tile_last = tile_first + (long long)(nactive - 1) * L * DSg + (long long)(nst - 1) * chunk_span + chunk_tail;
    const bool edge_tile = tile_first < 0 || tile_last > a.n_in;
    const float2* p_gsrc = nullptr;     // producer lane's segment
    int p_lo = 0, p_hi = 0;
    unsigned char* p_dst = nullptr;
    if (t < 32 && t < nactive) {
        const long long pbase = tile_first + (long long)t * L * DSg;
        const long long lo = pbase >= 0 ? 0 : (-pbase + chunk_span - 1) / chunk_span;
        const long long room = a.n_in - pbase - chunk_tail;
        const long long hi = room < 0 ? 0 : room / chunk_span + 1;
        p_lo = (int)(lo < nst ? lo : nst);
        p_hi = (int)(hi < nst ? hi : nst);
        p_gsrc = a.in + pbase;
        p_dst = reinterpret_cast<unsigned char*>(X + (size_t)t * seg_pitch);
    }
    auto issue = [&](int it, int slot) {
        if (t < 32) {
            const bool fast = it >= p_lo && it < p_hi;
            const unsigned m = __ballot_sync(0xffffffffu, fast);
            if (t == 0) mbar_arrive_expect_tx(&mbar[slot], (uint32_t)__popc(m) * chunk_bytes);
            __syncwarp();
            if (fast) {
                if (DSg == D) {
                    tma_bulk_g2s(p_dst + slot * stage_bytes, p_gsrc + (size_t)it * chunk_elems, chunk_bytes, &mbar[slot]);
                } else {   // sliced rows: one bulk copy per row (row stride DSg in memory, D contiguous samples)
                    for (int rr = 0; rr < R; rr++)
                        tma_bulk_g2s(p_dst + slot * stage_bytes + (size_t)rr * D * 8, p_gsrc + ((size_t)it * R + rr) * DSg,
                                     (uint32_t)D * 8u, &mbar[slot]);
                }
            }
        }
        if (edge_tile && in_grid) {
            const bool fast = it >= fast_lo && it < fast_hi;
            if (!fast && it < live_hi) {
                VStream<float2> xs{a.hist, a.in, a.H};
                float2* dst = reinterpret_cast<float2*>(reinterpret_cast<unsigned char*>(xseg) + slot * stage_bytes);
                const long long start = seg_base + (long long)it * chunk_span;
                for (int e = pair; e < chunk_elems; e += P) {
                    const int rr = e / D;
                    const long long i = start + (long long)rr * DSg + (e - rr * D);
                    dst[e] = (i < a.n_in) ? xs.at(i) : make_float2(0.f, 0.f);
                }
            }
        }
    };

    // ---- per-thread constants: tap pairs, phasors -------------------------------------------------
    float2 tp[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) tp[q] = make_float2(0.f, 0.f);
    if (in_grid) {
        const float2* tt = a.taps + ((size_t)slice * 2 + pad) * Q * P;
#pragma unroll
        for (int q = 0; q < Q; q++) tp[q] = tt[q * P + pair];
    }
    // phasors of the pair's two columns, packed (re, re) / (im, im) so one FFMA2 advances both
    float2 PR = make_float2(1.f, 1.f), PI = make_float2(0.f, 0.f);
    float2 wr2 = make_float2(1.f, 1.f), wi2 = make_float2(0.f, 0.f);
    const long long col0 = seg_base + 2 * pair;  // sample index of (row 0, first column of the pair)
    if (ROT) {
        const float2 w = phasor_from_turns(nco_step * (uint64_t)DSg);
        wr2 = make_float2(w.x, w.x);
        wi2 = make_float2(w.y, w.y);
    }

    float2 accRe[Q], accIm[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) accRe[q] = accIm[q] = make_float2(0.f, 0.f);

    // my float4 (two adjacent samples) in slot 0, row 0; my partial slot in parity 0, row 0
    const unsigned char* xme = reinterpret_cast<const unsigned char*>(reinterpret_cast<const float4*>(xseg) + pair);
    unsigned char* pme = reinterpret_cast<unsigned char*>(Pbuf + (seg * PROWS) * Ppad + pair);
    const uint32_t row_bytes = (uint32_t)D * 8u;
    const uint32_t prow_bytes = (uint32_t)Ppad * 8u;

    // ---- reduction role: 8 lanes sum one output's P column partials, lane 0 parks y in ybuf ------------
    const int u = t & 7, o = t >> 3;
    const bool ovalid = o < NSEG * R;
    const int so = o / R, ro = o - so * R;
    const unsigned char* pbr = reinterpret_cast<const unsigned char*>(Pbuf + o * Ppad + u);
    float2* yrow = ybuf + so * LL + (ro - (Q - 1));  // + it*R = this lane's output slot at stage it
    const bool ylane = ovalid && u == 0 && (k0 + so * L < bi.out_count);

    for (int s = 0; s < NS; s++) issue(s, s);
    __syncthreads();

    // level 2 of the wide-row reduce (also the whole reduce of narrow rows): 8 lanes per output
    auto finish_output = [&](int it, float2 sacc) {
#pragma unroll
        for (int sh = 4; sh > 0; sh >>= 1) {
            sacc.x += __shfl_xor_sync(0xffffffffu, sacc.x, sh);
            sacc.y += __shfl_xor_sync(0xffffffffu, sacc.y, sh);
        }
        const int j = it * R + ro - (Q - 1);
        if (ylane && j >= 0 && j < LOUT) yrow[it * R] = sacc;
    };
    auto reduce_stage = [&](int it, int par) {
        if (two_level) {
            // level 1, stage `it`: 64 lanes per output fold P partials into 64
            const int NO = NSEG * R;
            for (int idx = t; idx < NO * 64; idx += blockDim.x) {
                const int o1 = idx >> 6, l1 = idx & 63;
                const float2* pb = reinterpret_cast<const float2*>(reinterpret_cast<const unsigned char*>(Pbuf) + par * pbuf_half) + o1 * Ppad;
                float2 s1 = make_float2(0.f, 0.f);
                for (int pp = l1; pp < P; pp += 64) {
                    const float2 v = pb[pp];
                    s1.x += v.x;
                    s1.y += v.y;
                }
                P2[(par * NO + o1) * 64 + l1] = s1;
            }
            // level 2, stage `it - 1` (its level-1 sums became visible at this stage's barrier)
            if (it >= 1) {
                float2 sacc = make_float2(0.f, 0.f);
                if (ovalid) {
                    const float2* p2 = P2 + (((par ^ 1) * NO + o) * 64);
#pragma unroll
                    for (int i8 = 0; i8 < 8; i8++) {
                        const float2 v = p2[u + 8 * i8];
                        sacc.x += v.x;
                        sacc.y += v.y;
                    }
                }
                finish_output(it - 1, sacc);
            }
            return;
        }
        float2 sacc = make_float2(0.f, 0.f);
        if (ovalid) {
            const float2* pb = reinterpret_cast<const float2*>(pbr + par * pbuf_half);
            for (int pp = u; pp < P; pp += 8) {
                const float2 v = pb[pp - u];
                sacc.x += v.x;
                sacc.y += v.y;
            }
        }
        finish_output(it, sacc);
    };

    // SUPRED: all NSEG*Q outputs of super-iteration `sup`, 2 lanes per output (packed adds), parked in the ring
    auto reduce_super = [&](int sup) {
        const int o2 = t >> 1, u2 = t & 1;
        float2 sacc = make_float2(0.f, 0.f);
        const bool v2 = o2 < NSEG * Q;
        const int s2 = o2 / Q, i2 = o2 - s2 * Q;
        if (v2) {
            const float2* pb = reinterpret_cast<const float2*>(reinterpret_cast<const unsigned char*>(Pbuf) + (sup & 1) * pbuf_half) + o2 * Ppad;
            for (int pp = u2; pp < P; pp += 2) sacc = __fadd2_rn(sacc, pb[pp]);
        }
        sacc.x += __shfl_xor_sync(0xffffffffu, sacc.x, 1);
        sacc.y += __shfl_xor_sync(0xffffffffu, sacc.y, 1);
        const int j = sup * Q + i2 - (Q - 1);
        if (v2 && u2 == 0 && j >= 0 && j < LOUT && (k0 + s2 * L < bi.out_count)) ybuf[s2 * RY + (j % RY)] = sacc;
    };

    // ---- epilogue of one finished super-iteration: Q outputs per segment, one thread per output --------
    auto epilogue = [&](int sup) {
        if (t >= NSEG * Q) return;
        const int es = t / Q, er = t - es * Q;
        const int j = sup * Q + er - (Q - 1);           // 0 = the segment's leading output
        const int k = k0 + es * L - LEAD + j;           // output index within the block
        if (j < LEAD || j >= LOUT || k >= bi.out_count) return;
        const float2 y = ybuf[es * LL + (SUPRED ? j % RY : j)];
        const long long oidx = plane * a.out_stride + bi.out_start + k;
        if (DEMOD) {
            const float cur = fast_arctan2_ref(y.y, y.x);
            float prev;
            if (use_override && es == 0 && j == 1) prev = s_misc[0];
            else {
                const float2 yp = ybuf[es * LL + (SUPRED ? (j - 1) % RY : j - 1)];
                prev = fast_arctan2_ref(yp.y, yp.x);
            }
            a.audio[oidx] = fm_step_ref(cur, prev, a.phasor_speed);
            if (bi.out_start + k == a.part.total_out - 1) a.demod_out[ch] = cur;
            if (a.out_iq) a.out_iq[oidx] = y;
        } else {
            a.out_iq[oidx] = y;
        }
    };

    // ---- main loop: nsup super-iterations of Q rows (= NS stages, one ring slot each) ----------------
#pragma unroll 1
    for (int sup = 0; sup < nsup; sup++) {
        if (ROT && (sup & 7) == 0 && seg_active) {
            // exact phasor re-seed (closed form) every 8*Q rows bounds the recurrence's rounding walk
            const long long i0 = col0 + (long long)sup * Q * DSg;
            const float2 p0 = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)i0);
            const float2 p1 = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)(i0 + 1));
            PR = make_float2(p0.x, p1.x);
            PI = make_float2(p0.y, p1.y);
        }
        const uint32_t parity = (uint32_t)(sup & 1);
#pragma unroll
        for (int slot = 0; slot < NS; slot++) {
            const int par = SUPRED ? (sup & 1) : ((sup * NS + slot) & 1);  // partial-buffer parity of this stage
            mbar_wait(&mbar[slot], parity);
            if (seg_active) {
                const unsigned char* xs_ = xme + slot * stage_bytes;
                unsigned char* ps_ = pme + par * pbuf_half + (SUPRED ? slot * R * prow_bytes : 0u);
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int i = slot * R + r;     // row within the super-iteration: compile-time
                    const float4 v = *reinterpret_cast<const float4*>(xs_ + r * row_bytes);
                    float2 RE, IM;
                    if (ROT) {
                        // x' = x * p for both columns; results land directly in the packed (col r, col r+1) pairs
                        RE.x = fmaf(v.x, PR.x, -(v.y * PI.x));
                        IM.x = fmaf(v.x, PI.x, v.y * PR.x);
                        RE.y = fmaf(v.z, PR.y, -(v.w * PI.y));
                        IM.y = fmaf(v.z, PI.y, v.w * PR.y);
                        // p *= w for both columns in 4 packed ops
                        const float2 nPR = __ffma2_rn(PI, neg2(wi2), __fmul2_rn(PR, wr2));
                        PI = __ffma2_rn(PI, wr2, __fmul2_rn(PR, wi2));
                        PR = nPR;
                    } else {
                        RE = make_float2(v.x, v.z);
                        IM = make_float2(v.y, v.w);
                    }
#pragma unroll
                    for (int q = 0; q < Q; q++) {
                        const int sl = (i - q + Q) % Q;
                        if (q == 0) {
                            accRe[sl] = __fmul2_rn(RE, tp[0]);
                            accIm[sl] = __fmul2_rn(IM, tp[0]);
                        } else {
                            accRe[sl] = __ffma2_rn(RE, tp[q], accRe[sl]);
                            accIm[sl] = __ffma2_rn(IM, tp[q], accIm[sl]);
                        }
                    }
                    const int e = (i + 1) % Q;  // the output whose last tap (q = Q-1) was just applied
                    *reinterpret_cast<float2*>(ps_ + r * prow_bytes) =
                        make_float2(accRe[e].x + accRe[e].y, accIm[e].x + accIm[e].y);
                }
            }
            __syncthreads();                       // stage consumed, partials visible
            issue((sup + 1) * NS + slot, slot);    // refill the slot just drained
            if (SUPRED) {
                if (slot == NS - 1) reduce_super(sup);
            } else {
                reduce_stage(sup * NS + slot, par);
            }
            // all of the previous super-iteration's outputs were parked before this barrier (the two-level
            // reduce of wide rows finishes them one stage later)
            if (slot == (two_level ? 1 : 0) && sup > 0) epilogue(sup - 1);
        }
    }
    __syncthreads();
    if (two_level) {
        // flush level 2 of the last stage
        float2 sacc = make_float2(0.f, 0.f);
        const int lastit = nsup * NS - 1, NO = NSEG * R;
        if (ovalid) {
            const float2* p2 = P2 + (((lastit & 1) * NO + o) * 64);
#pragma unroll
            for (int i8 = 0; i8 < 8; i8++) {
                const float2 v = p2[u + 8 * i8];
                sacc.x += v.x;
                sacc.y += v.y;
            }
        }
        finish_output(lastit, sacc);
        __syncthreads();
    }
    epilogue(nsup - 1);
}

// ---- v2: one stage per super-iteration, dedicated producer/finisher warp ---------------------------
// Same column-pair formulation as decim_kernel above, restructured around what its profiles showed:
//  * a ring slot holds a whole super-iteration (Q rows per segment): ONE CTA barrier per Q rows publishes the
//    column partials and releases the slot (v1 needs one per 3 rows), and the 9 row loads of a stage are scheduled
//    ahead of the FFMA2 stream;
//  * warps 0-3 only run the FIR main body; a fifth warp owns everything with a long dependent chain: it arms the
//    mbarriers and issues the TMA bulk copies (double-buffered ring: one stage in flight while one is consumed), and
//    it finishes the NSEG*Q outputs of super-iteration s while the compute warps are already in s+1 -- one lane per
//    output: sum the P column partials (128-bit shared loads), fast_arctan2, previous angle from the neighbouring
//    lane, fm step, store. Nothing of that sits between a compute warp and its next row any more.
// Measured alternatives (config 2, same box, GS/s): finishing pass on two of the four compute warps 608; this
// layout 640; the same with mbarrier hand-overs instead of the CTA barrier 618; two aux warps at 80 registers 601;
// a 6-slot ring of 3-row stages (more bytes in flight, but a wait in front of every third row) 465; a 3-slot ring at
// 3 CTAs/SM 585. Without the finishing pass the kernel runs at 725 (the data-movement ceiling of this layout is
// 715-745), i.e. what is left is the aux warp's latency chain and one stage of prefetch depth.
// Compile-time geometry only (D, NSEG); 160-thread CTAs, 4 per SM.
template <int Q, int D, int NSEG>
struct SupGeom {
    static constexpr int P = D / 2;
    static constexpr int NSLOT = 2;
    static constexpr int chunk_elems = Q * D;
    static constexpr uint32_t chunk_bytes = (uint32_t)chunk_elems * 8u;
    static constexpr int seg_pad = ((((D * 8) % 128) - (int)(chunk_bytes % 128u)) % 128 + 128) % 128 / 8;
    static constexpr int seg_pitch = chunk_elems + seg_pad;
    static constexpr uint32_t stage_bytes = (uint32_t)NSEG * (uint32_t)seg_pitch * 8u;
    static constexpr int Ppad = P + ((2 - (P & 3)) & 3);          // even (16-byte rows), == 2 (mod 4)
    static constexpr uint32_t pbuf_half = (uint32_t)(NSEG * Q * Ppad) * 8u;
    static constexpr int SA = 32 / Q;                             // segments the finisher covers per pass
    static constexpr int NPASS = (NSEG + SA - 1) / SA;
    static constexpr size_t off_pbuf = (size_t)NSLOT * stage_bytes;
    static constexpr size_t off_mbar = (off_pbuf + 2 * (size_t)pbuf_half + 7) / 8 * 8;
    static constexpr size_t off_misc = off_mbar + NSLOT * 8;      // [0] override angle
    static constexpr size_t smem_bytes = off_misc + 16;
    static_assert(off_pbuf % 16 == 0 && (Ppad * 8) % 16 == 0 && pbuf_half % 16 == 0, "128-bit partial loads");
};

__device__ __forceinline__ void cta_sync() { asm volatile("bar.sync 0;" ::: "memory"); }

template <int Q, int D, int NSEG, bool ROT, bool DEMOD>
__global__ void __launch_bounds__(160, 4) decim_sup_kernel(const DecimArgs a) {
    using G = SupGeom<Q, D, NSEG>;
    constexpr int P = G::P;
    constexpr int LEAD = DEMOD ? 1 : 0;
    constexpr int NSLOT = G::NSLOT;
    static_assert(NSEG * P <= 128 && NSEG <= 32, "CTA geometry");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int L = a.L;
    const int t = threadIdx.x;
    const int warp = t >> 5, lane = t & 31;
    const int tile_x = a.plane_fast ? blockIdx.y : blockIdx.x;
    const int b = a.plane_fast ? blockIdx.z : blockIdx.y;
    const int plane = a.plane_fast ? blockIdx.x : blockIdx.z;
    const int ch = plane / a.nslices, slice = plane - ch * a.nslices;
    const int DSg = a.DS;
    const long long col_off = (long long)slice * D;
    const BlkInfo bi = a.part.get(b);
    const int k0 = tile_x * (NSEG * L);
    if (k0 >= bi.out_count) return;

    const long long chunk_span = (long long)Q * DSg;               // global samples one stage advances
    const long long chunk_tail = (long long)(Q - 1) * DSg + D;     // from a chunk's first sample to past its last
    const int LOUT = L + LEAD;
    float2* X = reinterpret_cast<float2*>(smem_raw);
    float2* Pbuf = reinterpret_cast<float2*>(smem_raw + G::off_pbuf);   // [2][NSEG*Q][Ppad]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + G::off_mbar);
    float* s_misc = reinterpret_cast<float*>(smem_raw + G::off_misc);

    const int pad = (int)((bi.in_start - a.T) & 1);
    const int need = (bi.out_count - k0 < L ? bi.out_count - k0 : L) + LEAD + Q - 1;
    const int nsup = (need + Q - 1) / Q < a.NSUP ? (need + Q - 1) / Q : a.NSUP;
    const int nactive = (bi.out_count - k0 + L - 1) / L < NSEG ? (bi.out_count - k0 + L - 1) / L : NSEG;

    uint64_t nco_step = 0, nco_ph0 = 0;
    if (ROT) {
        nco_step = a.nco[ch].step;
        nco_ph0 = a.nco[ch].init + nco_step * (uint64_t)a.abs0;
    }
    if (t == 0) {
        for (int s = 0; s < NSLOT; s++) mbar_init(&mbar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    bool use_override = false;
    if (DEMOD && tile_x == 0) {
        int pb = b - 1;
        BlkInfo pbi{};
        while (pb >= 0) {
            pbi = a.part.get(pb);
            if (pbi.out_count > 0) break;
            pb--;
        }
        if (pb < 0) {
            use_override = true;
            if (t == 0) s_misc[0] = a.demod_in[ch];
        } else if (pb != b - 1 || pbi.in_start + (long long)pbi.out_count * DSg != bi.in_start) {
            use_override = true;
            if (t < 32) {
                const float2 y = direct_output_warp<ROT>(
                    a, pbi.in_start + (long long)(pbi.out_count - 1) * DSg - a.T, nco_ph0, nco_step);
                if (t == 0) s_misc[0] = fast_arctan2_ref(y.y, y.x);
            }
        }
    }
    cta_sync();

    if (warp >= 4) {
        const int ap = warp - 4;   // aux warp: 0 = producer + finisher (160-thread CTAs have no other)
        // ================= producer + finisher warp =====================================================
        const long long tile_first = bi.in_start + (long long)(k0 - LEAD) * DSg - a.T - pad + col_off;
        const long long tile_last = tile_first + (long long)(nactive - 1) * L * DSg + (long long)(nsup - 1) * chunk_span + chunk_tail;
        const bool edge_tile = tile_first < 0 || tile_last > a.n_in;
        // lane l copies segment l: stages [p_lo, p_hi) lie inside the caller's buffer (all of them on interior
        // tiles); the rest (history before sample 0, ragged end) is filled by guarded loads
        const bool is_prod = lane < nactive;
        const long long pbase = tile_first + (long long)lane * L * DSg;
        int p_lo = 0, p_hi = 0;
        if (is_prod) {
            const long long lo = pbase >= 0 ? 0 : (-pbase + chunk_span - 1) / chunk_span;
            const long long room = a.n_in - pbase - chunk_tail;
            const long long hi = room < 0 ? 0 : room / chunk_span + 1;
            p_lo = (int)(lo < nsup ? lo : nsup);
            p_hi = (int)(hi < nsup ? hi : nsup);
        }
        const float2* p_gsrc = a.in + pbase;
        unsigned char* p_dst = reinterpret_cast<unsigned char*>(X + (size_t)lane * G::seg_pitch);
        auto issue = [&](int it, int slot) {
            if (it >= nsup) return;
            const bool fast = is_prod && it >= p_lo && it < p_hi;
            const unsigned m = __ballot_sync(0xffffffffu, fast);
            if (lane == 0) mbar_arrive_expect_tx(&mbar[slot], (uint32_t)__popc(m) * G::chunk_bytes);
            __syncwarp();
            if (fast) {
                if (DSg == D) {
                    tma_bulk_g2s(p_dst + slot * G::stage_bytes, p_gsrc + (size_t)it * G::chunk_elems, G::chunk_bytes, &mbar[slot]);
                } else {   // sliced rows: one bulk copy per row
#pragma unroll 1
                    for (int rr = 0; rr < Q; rr++)
                        tma_bulk_g2s(p_dst + slot * G::stage_bytes + (size_t)rr * D * 8, p_gsrc + ((size_t)it * Q + rr) * DSg,
                                     (uint32_t)D * 8u, &mbar[slot]);
                }
            }
            if (edge_tile) {
                VStream<float2> xs{a.hist, a.in, a.H};
                for (int sg = 0; sg < nactive; sg++) {
                    const int lo = __shfl_sync(0xffffffffu, p_lo, sg), hi = __shfl_sync(0xffffffffu, p_hi, sg);
                    if (it >= lo && it < hi) continue;
                    float2* dst = reinterpret_cast<float2*>(reinterpret_cast<unsigned char*>(X + (size_t)sg * G::seg_pitch) + slot * G::stage_bytes);
                    const long long start = tile_first + (long long)sg * L * DSg + (long long)it * chunk_span;
                    for (int e = lane; e < G::chunk_elems; e += 32) {
                        const int rr = e / D;
                        const long long i = start + (long long)rr * DSg + (e - rr * D);
                        dst[e] = (i < a.n_in) ? xs.at(i) : make_float2(0.f, 0.f);
                    }
                }
            }
        };
        // finisher roles: pass p covers segments [p*SA, (p+1)*SA), lane = local segment * Q + row
        const int fls = lane / Q, fi = lane - fls * Q;
        float lastcur[G::NPASS];
#pragma unroll
        for (int p = 0; p < G::NPASS; p++) lastcur[p] = 0.f;
        auto finish = [&](int sup, int par) {
#pragma unroll
            for (int p = 0; p < G::NPASS; p++) {
                const int fs = p * G::SA + fls;
                const bool fvalid = fls < G::SA && fs < NSEG;
                const float4* pb = reinterpret_cast<const float4*>(
                    reinterpret_cast<const unsigned char*>(Pbuf + (fvalid ? (fs * Q + fi) : 0) * G::Ppad) + par * G::pbuf_half);
                float2 s0 = make_float2(0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
#pragma unroll
                for (int m = 0; m < P / 2; m++) {
                    const float4 v = pb[m];
                    if (m & 1) {
                        s2 = __fadd2_rn(s2, make_float2(v.x, v.y));
                        s3 = __fadd2_rn(s3, make_float2(v.z, v.w));
                    } else {
                        s0 = __fadd2_rn(s0, make_float2(v.x, v.y));
                        s1 = __fadd2_rn(s1, make_float2(v.z, v.w));
                    }
                }
                if (P & 1) s0 = __fadd2_rn(s0, *reinterpret_cast<const float2*>(pb + P / 2));
                const float2 y = __fadd2_rn(__fadd2_rn(s0, s1), __fadd2_rn(s2, s3));
                const int j = sup * Q + fi - (Q - 1);                  // 0 = the segment's leading output (DEMOD)
                const int k = k0 + fs * L - LEAD + j;                  // output index within the block
                const bool live = fvalid && (k0 + fs * L < bi.out_count) && j >= LEAD && j < LOUT && k < bi.out_count;
                const long long oidx = plane * a.out_stride + bi.out_start + k;
                if (DEMOD) {
                    const float cur = fast_arctan2_ref(y.y, y.x);
                    float prev = __shfl_up_sync(0xffffffffu, cur, 1);
                    // row 0 continues from the segment's last output of the previous super-iteration (row Q-1)
                    const float carry = __shfl_sync(0xffffffffu, lastcur[p], (lane + Q - 1) & 31);
                    if (fi == 0) prev = carry;
                    if (use_override && fs == 0 && j == 1) prev = s_misc[0];
                    lastcur[p] = cur;
                    if (live) {
                        a.audio[oidx] = fm_step_ref(cur, prev, a.phasor_speed);
                        if (bi.out_start + k == a.part.total_out - 1) a.demod_out[ch] = cur;
                        if (a.out_iq) a.out_iq[oidx] = y;
                    }
                } else {
                    if (live) a.out_iq[oidx] = y;
                }
            }
        };
#pragma unroll 1
        if (ap == 0) {
            for (int s = 0; s < NSLOT; s++) issue(s, s);
        }
        cta_sync();
        int slot = 0;
#pragma unroll 1
        for (int sup = 0; sup < nsup; sup++) {
            cta_sync();                  // compute warps are done with slot `slot`; partials of `sup` visible
            if (ap == 0) issue(sup + NSLOT, slot);
            finish(sup, sup & 1);
            slot = slot == NSLOT - 1 ? 0 : slot + 1;
        }
        return;
    }

    // ================= compute warps: FIR main body ======================================================
    const int seg = t / P;
    const int pair = t - seg * P;
    const bool in_grid = seg < NSEG;
    const int ks = k0 + seg * L - LEAD;
    const long long seg_base = bi.in_start + (long long)ks * DSg - a.T - pad + col_off;
    const bool seg_active = in_grid && (k0 + seg * L < bi.out_count);
    float2 tp[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) tp[q] = make_float2(0.f, 0.f);
    if (in_grid) {
        const float2* tt = a.taps + ((size_t)slice * 2 + pad) * Q * P;
#pragma unroll
        for (int q = 0; q < Q; q++) tp[q] = tt[q * P + pair];
    }
    float2 PR = make_float2(1.f, 1.f), PI = make_float2(0.f, 0.f);
    float2 wr2 = make_float2(1.f, 1.f), wi2 = make_float2(0.f, 0.f);
    const long long col0 = seg_base + 2 * pair;
    if (ROT) {
        const float2 w = phasor_from_turns(nco_step * (uint64_t)DSg);
        wr2 = make_float2(w.x, w.x);
        wi2 = make_float2(w.y, w.y);
    }
    float2 accRe[Q], accIm[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) accRe[q] = accIm[q] = make_float2(0.f, 0.f);

    const unsigned char* xme = reinterpret_cast<const unsigned char*>(reinterpret_cast<const float4*>(X + (size_t)seg * G::seg_pitch) + pair);
    unsigned char* pme = reinterpret_cast<unsigned char*>(Pbuf + (seg * Q) * G::Ppad + pair);
    constexpr uint32_t row_bytes = (uint32_t)D * 8u;
    constexpr uint32_t prow_bytes = (uint32_t)G::Ppad * 8u;

    cta_sync();                          // pairs with the producer's prologue barrier
    int slot = 0;
    uint32_t parity = 0;
#pragma unroll 1
    for (int sup = 0; sup < nsup; sup++) {
        if (ROT && (sup & 7) == 0 && seg_active) {
            // exact phasor re-seed (closed form) every 8*Q rows bounds the recurrence's rounding walk
            const long long i0 = col0 + (long long)sup * Q * DSg;
            const float2 p0 = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)i0);
            const float2 p1 = phasor_from_turns(nco_ph0 + nco_step * (uint64_t)(i0 + 1));
            PR = make_float2(p0.x, p1.x);
            PI = make_float2(p0.y, p1.y);
        }
        mbar_wait(&mbar[slot], parity);
        if (seg_active) {
            const unsigned char* xs_ = xme + slot * G::stage_bytes;
            unsigned char* ps_ = pme + (sup & 1) * G::pbuf_half;
#pragma unroll
            for (int i = 0; i < Q; i++) {
                const float4 v = *reinterpret_cast<const float4*>(xs_ + i * row_bytes);
                float2 RE, IM;
                if (ROT) {
                    // x' = x * p for both columns; results land directly in the packed (col r, col r+1) pairs
                    RE.x = fmaf(v.x, PR.x, -(v.y * PI.x));
                    IM.x = fmaf(v.x, PI.x, v.y * PR.x);
                    RE.y = fmaf(v.z, PR.y, -(v.w * PI.y));
                    IM.y = fmaf(v.z, PI.y, v.w * PR.y);
                    // p *= w for both columns in 4 packed ops
                    const float2 nPR = __ffma2_rn(PI, neg2(wi2), __fmul2_rn(PR, wr2));
                    PI = __ffma2_rn(PI, wr2, __fmul2_rn(PR, wi2));
                    PR = nPR;
                } else {
                    RE = make_float2(v.x, v.z);
                    IM = make_float2(v.y, v.w);
                }
#pragma unroll
                for (int q = 0; q < Q; q++) {
                    const int sl = (i - q + Q) % Q;
                    if (q == 0) {
                        accRe[sl] = __fmul2_rn(RE, tp[0]);
                        accIm[sl] = __fmul2_rn(IM, tp[0]);
                    } else {
                        accRe[sl] = __ffma2_rn(RE, tp[q], accRe[sl]);
                        accIm[sl] = __ffma2_rn(IM, tp[q], accIm[sl]);
                    }
                }
                const int e = (i + 1) % Q;    // the output whose last tap (q = Q-1) was just applied
                *reinterpret_cast<float2*>(ps_ + i * prow_bytes) =
                    make_float2(accRe[e].x + accRe[e].y, accIm[e].x + accIm[e].y);
            }
        }
        cta_sync();                      // slot consumed, this super-iteration's partials visible
        if (slot == NSLOT - 1) {
            slot = 0;
            parity ^= 1u;
        } else {
            slot++;
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------
bool decim_plan_supported(int T, int interp, int decim) {
    if (interp != 1 || (decim & 1) || decim < 8) return false;
    const int Q = (T + 1 + decim - 1) / decim;
    if (Q > 9 || Q < 2) return false;       // instantiated: Q in {6, 9} (padded up)
    if (decim / 2 > 640) return false;
    return true;
}
static int round_q(int Q) { return Q <= 6 ? 6 : 9; }

DecimPlan* decim_plan_create(const float* taps, int T, int D) {
    if (!decim_plan_supported(T, 1, D)) return nullptr;
    DecimPlan* p = new (std::nothrow) DecimPlan();
    if (!p) return nullptr;
    p->T = T;
    p->DS = D;
    p->nslices = 1;
    // wide rows (config 4: D = 1280) are cut into 128-column slices: each slice is a narrow-row stream of its own
    // (128-thread CTAs, 2-lane partial reduce) whose partial outputs finish_kernel sums
    if (D > 128 && D % 128 == 0) p->nslices = D / 128;
    const int Dc = D / p->nslices;
    p->D = Dc;
    p->P = Dc / 2;
    p->Q = round_q((T + 1 + D - 1) / D);
    p->R = 3;
    p->NSTAGE = p->Q / 3;
    // segments per CTA: ~320 threads (two CTAs per SM with up to 96 registers per thread: no spills); the
    // reduction role needs 8 lanes per output of a stage, i.e. NT >= 24 * NSEG
    // measured on B200 (config 2): 128-thread CTAs x 5 per SM beat 320 x 2 (445 vs 374 GS/s): the per-stage
    // CTA barrier then only couples 4 warps while four other CTAs keep the SM busy
    int nseg = 128 / p->P >= 1 ? 128 / p->P : 320 / p->P;
    if (nseg > 13) nseg = 13;
    if (nseg < 1) nseg = 1;
    p->NSEG = nseg;
    int nt = nseg * p->P > nseg * 24 ? nseg * p->P : nseg * 24;   // 24 >= Q: also enough epilogue threads
    p->NT = ((nt + 31) / 32) * 32;
    if (p->NT < 64) p->NT = 64;
    // super-iterations per CTA, measured on B200: config 2: 15: 639, 19: 644, 20: 665, 22: 659,
    // 24: 665, 26: 640, 29: 636, 44: 646 GS/s; config 4 (wideband): 12: 17.7, 16: 18.4, 20: 19.4, 29: 17.4, 36: 17.9 GS/s
    p->NSUP = 20;
    std::vector<float2> tab((size_t)p->nslices * 2 * p->Q * p->P, make_float2(0.f, 0.f));
    for (int sl = 0; sl < p->nslices; sl++)
        for (int pad = 0; pad < 2; pad++)
            for (int q = 0; q < p->Q; q++)
                for (int c = 0; c < p->P; c++) {
                    const int t0 = q * D + sl * Dc + 2 * c - pad, t1 = t0 + 1;
                    float2 v;
                    v.x = (t0 >= 0 && t0 < T) ? taps[t0] : 0.0f;
                    v.y = (t1 >= 0 && t1 < T) ? taps[t1] : 0.0f;
                    tab[(((size_t)sl * 2 + pad) * p->Q + q) * p->P + c] = v;
                }
    if (cudaMalloc(&p->taps_dev, tab.size() * sizeof(float2)) != cudaSuccess ||
        cudaMemcpy(p->taps_dev, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("decim_plan_create: tap upload failed");
        delete p;
        return nullptr;
    }
    return p;
}
void decim_plan_destroy(DecimPlan* p) {
    if (!p) return;
    chan_plan_released(p);
    if (p->taps_dev) cudaFree(p->taps_dev);
    if (p->ypart) cudaFree(p->ypart);
    delete p;
}

// sliced rows: sum the per-slice partial outputs; optionally apply the FM-demod epilogue (demodulator.h:87-94)
__global__ void __launch_bounds__(256) decim_finish_kernel(const float2* __restrict__ ypart, long long ypart_stride,
                                                          int nslices, long long total_out, int demod,
                                                          float phasor_speed, const float* __restrict__ demod_in,
                                                          float* __restrict__ demod_out, float2* __restrict__ out_iq,
                                                          float* __restrict__ audio, long long out_stride) {
    const int ch = blockIdx.y;
    const long long stride = (long long)gridDim.x * blockDim.x;
    auto total = [&](long long o) {
        float2 y = make_float2(0.f, 0.f);
        for (int sl = 0; sl < nslices; sl++) {
            const float2 v = ypart[((size_t)ch * nslices + sl) * ypart_stride + o];
            y.x += v.x;
            y.y += v.y;
        }
        return y;
    };
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < total_out; o += stride) {
        const float2 y = total(o);
        if (out_iq) out_iq[ch * out_stride + o] = y;
        if (demod) {
            const float cur = fast_arctan2_ref(y.y, y.x);
            float prev;
            if (o > 0) {
                const float2 yp = total(o - 1);
                prev = fast_arctan2_ref(yp.y, yp.x);
            } else {
                prev = demod_in[ch];
            }
            audio[ch * out_stride + o] = fm_step_ref(cur, prev, phasor_speed);
            if (o == total_out - 1) demod_out[ch] = cur;
        }
    }
}

int launch_decim_finish(const float2* ypart, long long ypart_stride, int nslices, long long total_out, int demod,
                        float phasor_speed, const float* demod_in, float* demod_out, float2* out_iq, float* audio,
                        long long out_stride, int nch, cudaStream_t s) {
    if (total_out <= 0) return 0;
    long long gx = (total_out + 255) / 256;
    if (gx > 1024) gx = 1024;
    decim_finish_kernel<<<dim3((unsigned)gx, nch), 256, 0, s>>>(ypart, ypart_stride, nslices, total_out, demod, phasor_speed,
                                                                 demod_in, demod_out, out_iq, audio, out_stride);
    QDSP_LAUNCH_OK();
    return 0;
}

template <int Q, bool ROT, bool DEMOD, bool SUPRED>
static int launch_decim_t(const DecimArgs& a, dim3 grid, int NT, size_t smem, cudaStream_t s) {
    // launch bounds pick the CTAs/SM that 96 registers per thread allow (640 threads per SM)
#define QDSP_DECIM_LAUNCH(MAXT, MINB)                                                                          \
    {                                                                                                          \
        auto kern = decim_kernel<Q, ROT, DEMOD, SUPRED, MAXT, MINB>;                                                  \
        QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));     \
        kern<<<grid, NT, smem, s>>>(a);                                                                        \
    }
    if (NT <= 128) QDSP_DECIM_LAUNCH(128, 5)
    else if (NT <= 160) QDSP_DECIM_LAUNCH(160, 4)
    else if (NT <= 320) QDSP_DECIM_LAUNCH(320, 2)
    else QDSP_DECIM_LAUNCH(640, 1)
#undef QDSP_DECIM_LAUNCH
    QDSP_LAUNCH_OK();
    return 0;
}

template <int Q, int D, int NSEG, bool ROT, bool DEMOD>
static int launch_decim_sup_t(const DecimArgs& a, dim3 grid, cudaStream_t s) {
    auto kern = decim_sup_kernel<Q, D, NSEG, ROT, DEMOD>;
    constexpr size_t smem = SupGeom<Q, D, NSEG>::smem_bytes;
    QDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 160, smem, s>>>(a);
    QDSP_LAUNCH_OK();
    return 0;
}

int launch_decim(DecimPlan* plan, const float2* hist, int H, const float2* in, const Partition& part, int mode,
                 const NcoDev* nco, long long abs0, int nch, float phasor_speed, const float* demod_in,
                 float* demod_out, float2* out_iq, float* audio, long long out_stride, cudaStream_t s) {
    if (part.view.nblocks == 0 || part.max_out == 0) return 0;
    if ((reinterpret_cast<uintptr_t>(in) & 15) != 0) {
        set_last_error("decim: input pointer must be 16-byte aligned for TMA bulk copies");
        return -1;
    }
    const int lead = mode == 1 ? 1 : 0;
    DecimArgs a{};
    a.hist = hist;
    a.in = in;
    a.H = H;
    a.n_in = part.view.total;
    a.taps = plan->taps_dev;
    a.part = part.view;
    a.T = plan->T;
    a.D = plan->D;
    a.DS = plan->DS;
    a.nslices = plan->nslices;
    a.P = plan->P;
    a.NSEG = plan->NSEG;
    a.R = plan->R;
    a.NSTAGE = plan->NSTAGE;
    a.NSUP = plan->NSUP;
    const bool sliced = plan->nslices > 1;
    a.L = plan->NSUP * plan->Q - (plan->Q - 1) - (sliced ? 0 : lead);
    a.nco = nco;
    a.abs0 = abs0;
    a.phasor_speed = phasor_speed;
    a.demod_in = demod_in;
    a.demod_out = demod_out;
    a.out_iq = out_iq;
    a.audio = audio;
    a.out_stride = out_stride;
    const int per_tile = a.NSEG * a.L;
    dim3 grid((part.max_out + per_tile - 1) / per_tile, part.view.nblocks, nch * plan->nslices);
    // several planes (channels x column slices) read the same input: make the plane the fastest grid dimension so that
    // the CTAs resident together are the planes of the same few input tiles -- the tile is fetched from DRAM once and the
    // other planes hit L2 (config 4, 32 channels: 3.98 GB -> see DESIGN.md of DRAM reads per 134 MB of input)
    a.plane_fast = nch * plan->nslices > 1 && grid.x <= 65535 && grid.y <= 65535;
    if (a.plane_fast) grid = dim3(nch * plan->nslices, grid.x, grid.y);
    const size_t stage_bytes = (size_t)a.NSEG * (a.R * a.D + decim_seg_pad(a.D)) * sizeof(float2);
    const size_t smem_stage = (size_t)a.NSTAGE * stage_bytes + (size_t)2 * a.NSEG * a.R * (a.P | 1) * sizeof(float2) +
                              (size_t)a.NSEG * (a.L + 1) * sizeof(float2) + 16 + a.NSTAGE * 8 + 64 +
                              (a.P > 64 ? (size_t)2 * a.NSEG * a.R * 64 * sizeof(float2) : 0);
    const size_t smem_sup = (size_t)a.NSTAGE * stage_bytes + (size_t)2 * a.NSEG * plan->Q * decim_ppad_sup(a.P) * sizeof(float2) +
                            (size_t)a.NSEG * 4 * plan->Q * sizeof(float2) + 16 + a.NSTAGE * 8 + 64;
    if (smem_stage > 227 * 1024) {
        set_last_error("decim: tile does not fit shared memory (%zu bytes)", smem_stage);
        return -1;
    }
    const bool fused = mode == 1;
    if (sliced) {
        // partial outputs per (channel, slice) -> scratch, then the finish kernel sums them and demodulates
        const size_t ystride = (size_t)((part.total_out + 63) / 64) * 64;
        const size_t need = (size_t)nch * plan->nslices * ystride;
        if (need > plan->ypart_cap) {
            if (plan->ypart) cudaFree(plan->ypart);
            plan->ypart = nullptr;
            plan->ypart_cap = 0;
            QDSP_CUDA_OK(cudaMalloc(&plan->ypart, need * sizeof(float2)));
            plan->ypart_cap = need;
        }
        a.out_iq = plan->ypart;
        a.audio = nullptr;
        a.out_stride = (long long)ystride;
        const bool sup = plan->NT >= 2 * plan->NSEG * plan->Q;
        const size_t sm = sup ? smem_sup : smem_stage;
        int rc;
        // 128-column slices: P = 64, NSEG = 2, NT = 128, so Q = 9 always takes the super-iteration kernel (config 4)
        if (plan->Q == 9 && plan->D == 128 && plan->NSEG == 2 && sup && plan->NT == 128)
            rc = fused ? launch_decim_sup_t<9, 128, 2, true, false>(a, grid, s) : launch_decim_sup_t<9, 128, 2, false, false>(a, grid, s);
        else if (plan->Q == 9)
            rc = fused ? (sup ? launch_decim_t<9, true, false, true>(a, grid, plan->NT, sm, s) : launch_decim_t<9, true, false, false>(a, grid, plan->NT, sm, s))
                       : (sup ? launch_decim_t<9, false, false, true>(a, grid, plan->NT, sm, s) : launch_decim_t<9, false, false, false>(a, grid, plan->NT, sm, s));
        else
            rc = fused ? (sup ? launch_decim_t<6, true, false, true>(a, grid, plan->NT, sm, s) : launch_decim_t<6, true, false, false>(a, grid, plan->NT, sm, s))
                       : (sup ? launch_decim_t<6, false, false, true>(a, grid, plan->NT, sm, s) : launch_decim_t<6, false, false, false>(a, grid, plan->NT, sm, s));
        if (rc != 0) return rc;
        long long gx = (part.total_out + 255) / 256;
        if (gx > 1024) gx = 1024;
        if (gx < 1) gx = 1;
        decim_finish_kernel<<<dim3((unsigned)gx, nch), 256, 0, s>>>(plan->ypart, (long long)ystride, plan->nslices,
                                                                     part.total_out, fused ? 1 : 0, phasor_speed, demod_in,
                                                                     demod_out, out_iq, audio, out_stride);
        QDSP_LAUNCH_OK();
        return 0;
    }
    const bool supred = plan->P <= 64 && plan->NT >= 2 * plan->NSEG * plan->Q;
    const size_t smem = supred ? smem_sup : smem_stage;
    // D = 50: P = 25, NSEG = 5, NT = 128, so Q = 9 always takes the super-iteration kernel (config 2)
    if (plan->Q == 9 && plan->D == 50 && plan->NSEG == 5 && supred && plan->NT == 128)
        return fused ? launch_decim_sup_t<9, 50, 5, true, true>(a, grid, s) : launch_decim_sup_t<9, 50, 5, false, false>(a, grid, s);
    if (plan->Q == 9)
        return fused ? (supred ? launch_decim_t<9, true, true, true>(a, grid, plan->NT, smem, s) : launch_decim_t<9, true, true, false>(a, grid, plan->NT, smem, s))
                     : (supred ? launch_decim_t<9, false, false, true>(a, grid, plan->NT, smem, s) : launch_decim_t<9, false, false, false>(a, grid, plan->NT, smem, s));
    if (plan->Q == 6)
        return fused ? (supred ? launch_decim_t<6, true, true, true>(a, grid, plan->NT, smem, s) : launch_decim_t<6, true, true, false>(a, grid, plan->NT, smem, s))
                     : (supred ? launch_decim_t<6, false, false, true>(a, grid, plan->NT, smem, s) : launch_decim_t<6, false, false, false>(a, grid, plan->NT, smem, s));
    set_last_error("decim: unsupported Q=%d", plan->Q);
    return -1;
}

}  // namespace qdsp
