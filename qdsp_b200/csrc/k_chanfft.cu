// qdsp_b200/csrc/k_chanfft.cu — FFT polyphase channelizer for sm_100a: the ALGORITHMIC alternative (SURVEY.md §8 f4) to the
// direct-form channelizer (k_chan.cu) for the case BASELINE config 4 actually is: M channels spaced fs / M apart, decimation a
// multiple of M. The reference computes every channel as its own VFO (routing.h:47-57 -> vfo.h:19-36 -> resampling.h:99-132)
// + FloatFMDemod (demodulator.h:81-99): M x 10 241 MACs per output row. With theta_k = beta - 2 pi k / M + delta_k (beta =
// channel 0's NCO step, delta_k = what float32 rounding of the reference's phaseDelta leaves, |delta_k| < 2e-7 rad/sample):
//
//   y_k[m] = sum_t h[t] x[N] e^{j theta_k N},  N = N_s(m) + t
//          = e^{-j 2 pi k (N_s mod M) / M} e^{j delta_k N_c} * sum_{r<M} e^{-j 2 pi k r / M} ( u_m[r] + j delta_k v_m[r] ) + O((delta T / 2)^2)
//   u_m[r] = sum_j h[r + M j] x'[N_s + r + M j],   v_m[r] = sum_j (r + M j - t_c) h[r + M j] x'[...],   x'[N] = x[N] e^{j beta N}
//
// i.e. ONE pass of M column filters (J = 41 taps each) over the pre-rotated stream and two M-point FFTs per output row give
// all M channels: 2 x 10 241 MACs + 2 FFTs instead of M x 10 241 MACs (about 100x fewer flops for M = 256). The first-order
// term in delta_k is what keeps parity with the reference's float32 NCO frequencies (delta T / 2 ~ 1e-3 rad would not pass
// the 1e-4 audio bar; the second-order residue is ~5e-7).
//
// When channel 0 is itself on the bin grid (config 4: offsets (k - 128) fs / 256) beta is a bin shift and x' = x: no
// pre-rotation at all, channel k is bin (k - b) mod M, and channel 0's own rounding goes into delta_0.
//
// Kernel A (chanfft_poly_kernel): thread = column r, walks down the rows (M samples each) of a segment with its J packed
// (g, g') taps in registers (g' = (t - T/2) g); 9 outputs in flight (static slot rotation: 9 group bodies of 5 rows); per
// sample and output two FFMA2: (Re u, Re v) += (g, g') Re x' and the same for Im. Rows arrive by TMA bulk copy (5 contiguous
// rows per stage). Writes U, V per (row, column).
// Kernel B (chanfft_fft_kernel): 15 output rows (+ the predecessor of the first, for the FM difference) per CTA; the two
// 256-point FFTs of a row as 16 x 16 with both 16-point passes in registers and ONE shared-memory transpose; per-channel
// phase (64-bit turn arithmetic, MUFU sin/cos), first-order correction, fast_arctan2 + FM step, transposed store of the
// audio and / or of the channel samples themselves (the complex baseband, qdsp_channelizer_process_iq).
#include <math.h>
#include <new>
#include <vector>
#include "decim_common.cuh"
#include "fft_common.cuh"

namespace qdsp {

constexpr int kCfM = 256;      // channels = FFT size
constexpr int kCfDR = 5;       // rows (of M samples) per output: decimation = 5 * 256 = 1280
constexpr int kCfJ = 41;       // taps per column: 41 * 256 >= 10 241 + 1
constexpr int kCfSlots = 9;    // outputs in flight: ceil(41 / 5)
constexpr int kCfStages = 8;    // ring depth of the column-filter kernel (stage = 5 rows x 256 columns = 10 KB)
constexpr int kCfRB = 16;      // rows per CTA of the FFT kernel: the predecessor of the first + 15 new ones
constexpr int kCfNew = kCfRB - 1;
constexpr int kCfLd = 17;      // padded leading dimension of the 16 x 16 transpose tiles

struct ChanFftPlan {
    int T = 0, D = 0, nch = 0;
    int twob = 0;                       // channel k sits on half-bin (twob - 2 k) mod 2 M of the raw stream (rotate: twob = 0)
    bool rotate = false;                // pre-rotate the stream by channel 0's NCO (comb neither on the bin nor the half-bin grid)
    float2* gpair_dev = nullptr;        // [J * M] (g, (t' - pad - T/2) g), g[t'] = h[t' - pad]
    long long* dturn_dev = nullptr;     // [M] delta_k in turns * 2^64 (signed)
    long long* dt0_dev = nullptr;       // [M] round(delta_k * T / 2) + (phase_k - phase_0) in the same unit
    float* delta_dev = nullptr;         // [M] delta_k in rad / sample
    float2* uv = nullptr;               // [2][rows][M] scratch: U then V
    size_t uv_cap = 0;
    double max_delta = 0.0;
};

struct ChanFftArgs {
    const float2* hist;
    const float2* in;
    int H;
    long long n_in;
    PartitionDev part;
    int T, pad, seg_rows;
    int twist;                          // not pre-rotated, comb on the half-bin grid: column twist e^{j pi r / M}
    long long abs0;
    uint64_t beta_step, beta_ph0;
    const float2* gpair;                // [J * M]
    float2* U;
    float2* V;
};

// one group = the 5 rows (of 256 samples) between two output starts; this thread's column of them. Accumulators are packed
// (u, v) pairs -- aR = (Re u, Re v), aI = (Im u, Im v) -- so one FFMA2 with the packed (g, g') tap advances both sums.
template <int S, bool ROT>
__device__ __forceinline__ void chanfft_group(const float2* __restrict__ tile, int r /* lane */, const f32x2_t (&gp)[kCfJ], f32x2_t (&aR)[kCfSlots],
                                              f32x2_t (&aI)[kCfSlots], float2& p, const float2 w256, f32x2_t& fR, f32x2_t& fI) {
    aR[S] = 0ull;                          // a new output starts in this group
    aI[S] = 0ull;
    float2 x[kCfDR];
#pragma unroll
    for (int ir = 0; ir < kCfDR; ir++) x[ir] = tile[ir * kCfM + r];
#pragma unroll
    for (int ir = 0; ir < kCfDR; ir++) {
        float2 z = x[ir];
        if (ROT) {
            z = cmul(z, p);
            p = cmul(p, w256);
        }
        const f32x2_t zr = pk2(z.x, z.x), zi = pk2(z.y, z.y);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int slot = (S - i + kCfSlots) % kCfSlots;
            aR[slot] = ffma2x(gp[5 * i + ir], zr, aR[slot]);
            aI[slot] = ffma2x(gp[5 * i + ir], zi, aI[slot]);
        }
        if (ir == 0) {                     // tap row 40: the output that started 8 groups ago completes
            const int slot = (S + 1) % kCfSlots;
            aR[slot] = ffma2x(gp[40], zr, aR[slot]);
            aI[slot] = ffma2x(gp[40], zi, aI[slot]);
            fR = aR[slot];
            fI = aI[slot];
        }
    }
}

// Producer / consumer: warp 8 feeds a ring of CTA-wide stages (5 contiguous rows = ONE 10 KB bulk copy per stage; the edge
// stages, which reach into the history or past the end, it writes itself), warps 0..7 own 32 columns each and drift freely
// up to the ring depth: full / empty mbarriers per stage, no CTA-wide barrier. The 9 group bodies run in sequence inside one
// loop (static accumulator slots, no indirect branch, no register shuffles at a join).
constexpr int kCfConsumers = kCfM / 32;
constexpr int kCfPolyThreads = kCfM + 32;

template <int S, bool ROT>
__device__ __forceinline__ void chanfft_step(const ChanFftArgs& a, int gi, int nout, long long row0, int r, int lane, const unsigned char* smem_raw,
                                             uint64_t* full, uint64_t* empty, const f32x2_t (&gp)[kCfJ], f32x2_t (&aR)[kCfSlots],
                                             f32x2_t (&aI)[kCfSlots], float2& p, const float2 w256, const float2 cr, float2* Uo, float2* Vo) {
    constexpr uint32_t STAGE_BYTES = kCfDR * kCfM * 8u;
    const int slot = gi % kCfStages;
    if (ROT && (S % 3) == 0) {     // exact phasor re-seed every 3 groups (15 rows): x'[N] = x[N] e^{j beta N}, N absolute
        const long long N = a.abs0 + row0 + (long long)gi * (kCfDR * kCfM) + r;
        p = phasor_from_turns(a.beta_ph0 + a.beta_step * (uint64_t)N);
    }
    mbar_wait(&full[slot], (uint32_t)((gi / kCfStages) & 1));
    const float2* tile = reinterpret_cast<const float2*>(smem_raw + slot * STAGE_BYTES) + (r - lane);
    f32x2_t fR = 0ull, fI = 0ull;
    chanfft_group<S, ROT>(tile, lane, gp, aR, aI, p, w256, fR, fI);
    __syncwarp();                  // every lane is done with the slot
    if (lane == 0) mbar_arrive(&empty[slot]);
    const int m = gi - 8;          // the output completed by this group's first row
    if (m >= 0 && m < nout) {
        const float2 re = unpk2(fR), im = unpk2(fI);
        float2 uu = make_float2(re.x, im.x), vv = make_float2(re.y, im.y);
        if (!ROT) {
            uu = cmul(uu, cr);
            vv = cmul(vv, cr);
        }
        Uo[(size_t)m * kCfM] = uu;
        Vo[(size_t)m * kCfM] = vv;
    }
}

template <bool ROT>
__global__ void __launch_bounds__(kCfPolyThreads, 1) chanfft_poly_kernel(const ChanFftArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr uint32_t STAGE_BYTES = kCfDR * kCfM * 8u;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kCfStages * STAGE_BYTES);
    uint64_t* empty = full + kCfStages;
    const int r = threadIdx.x, warp = r >> 5, lane = r & 31;
    const int seg = blockIdx.x, b = blockIdx.y;
    const BlkInfo bi = a.part.get(b);
    const int k0 = seg * a.seg_rows;
    if (k0 >= bi.out_count) return;
    const int nout = bi.out_count - k0 < a.seg_rows ? bi.out_count - k0 : a.seg_rows;
    const int ngroups = nout + 8;
    // group gi of the segment = rows 5 (k0 + gi) .. +4; row rho starts at sample row0 + 256 rho (relative to this call's input)
    const long long row0 = bi.in_start - a.T - a.pad + (long long)k0 * (kCfDR * kCfM);
    if (r == 0) {
        for (int s = 0; s < kCfStages; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kCfConsumers);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp == kCfConsumers) {
        // ---- producer warp
#pragma unroll 1
        for (int gi = 0; gi < ngroups; gi++) {
            const int slot = gi % kCfStages;
            if (gi >= kCfStages) mbar_wait(&empty[slot], (uint32_t)(((gi / kCfStages) - 1) & 1));
            float2* dst = reinterpret_cast<float2*>(smem_raw + slot * STAGE_BYTES);
            const long long s0 = row0 + (long long)gi * (kCfDR * kCfM);
            if (s0 >= 0 && s0 + kCfDR * kCfM <= a.n_in) {
                if (lane == 0) {
                    mbar_arrive_expect_tx(&full[slot], STAGE_BYTES);
                    tma_bulk_g2s(dst, a.in + s0, STAGE_BYTES, &full[slot]);
                }
            } else {
                // 40 independent (predicated, branch-free) loads in flight per lane: this path is the one CTA-serial stretch
                float2 v[kCfDR * kCfM / 32];
#pragma unroll
                for (int e = 0; e < kCfDR * kCfM / 32; e++) {
                    const long long idx = s0 + e * 32 + lane;
                    const float2* src = idx >= 0 ? a.in + idx : a.hist + (a.H + idx);
                    v[e] = make_float2(0.f, 0.f);
                    if (idx < a.n_in && idx >= -(long long)a.H) v[e] = __ldg(src);
                }
#pragma unroll
                for (int e = 0; e < kCfDR * kCfM / 32; e++) dst[e * 32 + lane] = v[e];
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[slot]);
            }
        }
        return;
    }
    // ---- consumer warps: column r
    f32x2_t gp[kCfJ];
#pragma unroll
    for (int j = 0; j < kCfJ; j++) {
        const float2 g = a.gpair[j * kCfM + r];
        gp[j] = pk2(g.x, g.y);
    }
    f32x2_t aR[kCfSlots], aI[kCfSlots];
#pragma unroll
    for (int s = 0; s < kCfSlots; s++) aR[s] = aI[s] = 0ull;
    const float2 w256 = ROT ? phasor_from_turns(a.beta_step * (uint64_t)kCfM) : make_float2(1.f, 0.f);
    float2 p = make_float2(1.f, 0.f);
    // not pre-rotated: the column's constant twist e^{j pi twist r / M} (half-bin combs; 1 for combs on the bin grid)
    float2 cr = make_float2(1.f, 0.f);
    if (!ROT && a.twist) {
        float sn, cs;
        sincospif((float)r / (float)kCfM, &sn, &cs);
        cr = make_float2(cs, sn);
    }
    float2* Uo = a.U + (size_t)(bi.out_start + k0) * kCfM + r;
    float2* Vo = a.V + (size_t)(bi.out_start + k0) * kCfM + r;
    int gi = 0;
#define QDSP_CF_STEP(S)                                                                                              \
    if (gi >= ngroups) break;                                                                                        \
    chanfft_step<S, ROT>(a, gi, nout, row0, r, lane, smem_raw, full, empty, gp, aR, aI, p, w256, cr, Uo, Vo);        \
    gi++;
#pragma unroll 1
    for (;;) {
        QDSP_CF_STEP(0) QDSP_CF_STEP(1) QDSP_CF_STEP(2) QDSP_CF_STEP(3) QDSP_CF_STEP(4)
        QDSP_CF_STEP(5) QDSP_CF_STEP(6) QDSP_CF_STEP(7) QDSP_CF_STEP(8)
    }
#undef QDSP_CF_STEP
}

struct ChanFftBArgs {
    const float2* U;
    const float2* V;
    long long total_out;
    long long abs0;                 // absolute index of this call's first input sample
    int T, pad, D, twob;            // twob: channel 0 sits on half-bin twob of the raw stream (0 when pre-rotated)
    uint64_t ph0;                   // channel 0's NCO phase constant when the stream is not pre-rotated (the rest: dt0)
    const long long* dturn;         // [M]
    const long long* dt0;           // [M]
    const float* delta;             // [M]
    const float* demod_in;
    float* demod_out;
    float* audio;
    long long out_stride;
    float inv_speed;                // 1 / phasorSpeed (demodulator.h:91)
    float2* iq;                     // [M][out_stride] channel baseband (IQ instantiations)
};

// The reference's fast_arctan2 (demodulator.h:11-30) with the quotient from the reciprocal unit (<= 2 ulp: 2e-7 rad) and a
// multiply by 1 / phasorSpeed in the FM step: this path's outputs are not bit-images of the reference's anyway (the FFT
// reorders every sum), its budget is the 1e-4 audio tolerance.
__device__ __forceinline__ float fast_arctan2_rcp(float y, float x) {
    const float c1 = QDSP_FL_M_PI / 4.0f, c2 = 3.0f * QDSP_FL_M_PI / 4.0f;
    const float abs_y = fabsf(y);
    const bool pos = x >= 0.0f;
    const float num = pos ? x - abs_y : x + abs_y;
    const float den = pos ? x + abs_y : abs_y - x;
    const float r = __fdividef(num, den);
    float angle = fmaf(-c1, r, pos ? c1 : c2);
    if (den == 0.0f) angle = 0.0f;                  // x == y == 0
    return (y < 0.0f) ? -angle : angle;
}
__device__ __forceinline__ float fm_step_mul(float cur, float prev, float inv_speed) {
    float diff = cur - prev;
    if (diff > 3.1415926535f) diff -= 2 * 3.1415926535f;
    else if (diff <= -3.1415926535f) diff += 2 * 3.1415926535f;
    return diff * inv_speed;
}
// e^{j 2 pi turns / 2^64} from the special-function unit (absolute error ~4e-7: the epilogue's budget is 1e-4)
__device__ __forceinline__ float2 phasor_mufu(uint64_t turns) {
    const float ang = (float)(int32_t)(turns >> 32) * (6.283185307179586f / 4294967296.0f);
    float s, c;
    __sincosf(ang, &s, &c);
    return make_float2(c, s);
}

// 256-point FFTs as 16 x 16 (four-step) with both 16-point passes in registers: thread (f, c) = (row of the CTA, column).
// Pass 1: column n2 = c of row f, over n1 (input index 16 n1 + n2), twiddle W256^{n2 k1}; transpose through shared memory;
// pass 2: k1 = c, over n2: bins k1 + 16 k2. U and V of a row share the thread (and the twiddles).
// AUDIO: FM audio into `audio`; IQ: the channel samples y themselves into `iq`, staged in the (by then free) transpose tiles
// and stored transposed like the audio. Without AUDIO the angle is taken only where the carried state needs it: the last row.
template <bool AUDIO, bool IQ>
__global__ void __launch_bounds__(kCfM, 2) chanfft_fft_kernel(const ChanFftBArgs a) {
    extern __shared__ __align__(16) unsigned char smem_b[];
    float2* sU = reinterpret_cast<float2*>(smem_b);
    float2* sV = sU + kCfRB * 16 * kCfLd;
    float2* tw = sV + kCfRB * 16 * kCfLd;
    float* s_ang = reinterpret_cast<float*>(tw + kCfM);            // [kCfRB][M + 1]
    float2* s_y = sU;                                                // [kCfRB][M + 1] (IQ): over the transpose tiles
    const int t = threadIdx.x, f = t >> 4, c = t & 15;
    const long long m0 = (long long)blockIdx.x * kCfNew;
    const long long m = m0 - 1 + f;
    const long long mm = m < 0 ? 0 : (m >= a.total_out ? a.total_out - 1 : m);
    {
        float sn, cs;
        sincospif(-(float)(f * c) / 128.0f, &sn, &cs);             // tw[k1][n2] = W256^{n2 k1}: lanes read consecutive entries
        tw[t] = make_float2(cs, sn);
    }
    float2 u[16], v[16];
    const float2* Ur = a.U + (size_t)mm * kCfM + c;
    const float2* Vr = a.V + (size_t)mm * kCfM + c;
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        u[n1] = Ur[16 * n1];
        v[n1] = Vr[16 * n1];
    }
    fft16(u);
    fft16(v);
    __syncthreads();
    float2* su = sU + f * (16 * kCfLd);
    float2* sv = sV + f * (16 * kCfLd);
#pragma unroll
    for (int k1 = 0; k1 < 16; k1++) {
        const float2 w = tw[k1 * 16 + c];
        su[k1 * kCfLd + c] = cmul(u[bitrev4(k1)], w);
        sv[k1 * kCfLd + c] = cmul(v[bitrev4(k1)], w);
    }
    __syncthreads();
#pragma unroll
    for (int n2 = 0; n2 < 16; n2++) {
        u[n2] = su[c * kCfLd + n2];
        v[n2] = sv[c * kCfLd + n2];
    }
    fft16(u);
    fft16(v);
    if (IQ) __syncthreads();               // every row is done with the transpose tiles: s_y overwrites them
    // epilogue: bins c + 16 k2 of row m
    const long long Ns = a.abs0 + m * (long long)a.D - a.T;
    const unsigned A9 = (unsigned)((Ns - a.pad) & (2 * kCfM - 1));
    float* ang_row = s_ang + f * (kCfM + 1);
    const bool carried = (m < 0);          // the row before this call's first: its angle is the carried demodulator state
    const bool last = (m == a.total_out - 1);
#pragma unroll
    for (int k2 = 0; k2 < 16; k2++) {
        const int bin = c + 16 * k2;
        const int k = (bin + (a.twob >> 1)) & (kCfM - 1);
        const float2 Uf = u[bitrev4(k2)], Vf = v[bitrev4(k2)];
        const float delta = __ldg(a.delta + k);
        const float2 Y = make_float2(fmaf(-delta, Vf.y, Uf.x), fmaf(delta, Vf.x, Uf.y));    // Uf + j delta Vf
        // channel phase: phi0 + delta_k (N_s + T/2) + 2 pi (twob - 2 k) (N_s - pad) / (2 M), modular 64-bit turn arithmetic
        const unsigned hb = (unsigned)(a.twob - 2 * k) & (2 * kCfM - 1);
        const unsigned long long turns = a.ph0 + (unsigned long long)__ldg(a.dturn + k) * (unsigned long long)Ns +
                                         (unsigned long long)__ldg(a.dt0 + k) + ((unsigned long long)(hb * A9) << 55);
        const float2 y = cmul(Y, phasor_mufu(turns));
        if (AUDIO) ang_row[k] = fast_arctan2_rcp(y.y, y.x);
        if (IQ) s_y[f * (kCfM + 1) + k] = y;
    }
    if (carried || last) {
#pragma unroll 1
        for (int k2 = 0; k2 < 16; k2++) {
            const int k = (c + 16 * k2 + (a.twob >> 1)) & (kCfM - 1);
            if (!AUDIO) {
                // the thread's own s_y entries: the last row's angle is the carried state
                if (last) a.demod_out[k] = fast_arctan2_rcp(s_y[f * (kCfM + 1) + k].y, s_y[f * (kCfM + 1) + k].x);
            } else if (carried) ang_row[k] = a.demod_in[k];
            else a.demod_out[k] = ang_row[k];
        }
    }
    __syncthreads();
    // transposed store: consecutive threads write consecutive rows of one channel (nothing for the carried row)
    for (int idx = t; idx < kCfNew * kCfM; idx += kCfM) {
        const int k = idx / kCfNew, mr = idx - k * kCfNew;
        if (m0 + mr < a.total_out) {
            if (AUDIO)
                a.audio[(size_t)k * a.out_stride + m0 + mr] = fm_step_mul(s_ang[(mr + 1) * (kCfM + 1) + k], s_ang[mr * (kCfM + 1) + k], a.inv_speed);
            if (IQ) a.iq[(size_t)k * a.out_stride + m0 + mr] = s_y[(mr + 1) * (kCfM + 1) + k];
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------
ChanFftPlan* chanfft_plan_create(const float* taps, int T, int interp, int decim, int nch, const uint64_t* nco_steps,
                                 const uint64_t* nco_phases, bool* failed) {
    if (failed) *failed = false;
    if (interp != 1 || nch != kCfM || decim != kCfDR * kCfM || T + 1 > kCfJ * kCfM) return nullptr;
    const double to_rad = 6.283185307179586476925286766559 / 18446744073709551616.0;
    // is channel 0 on the half-bin grid of the M-point FFT (theta_0 = 2 pi hb / (2 M) within rounding)? then no pre-rotation
    // is needed: e^{j theta_0 (A + r + M j)} = [row phase] x [bin shift hb / 2] x [column twist e^{j pi r / M} if hb is odd] x
    // [(-1)^j if hb is odd: folded into the taps]. Otherwise rotate the stream by channel 0's NCO first (hb = 0).
    const uint64_t hb_near = (nco_steps[0] + (1ull << 54)) >> 55;
    const long long res0 = (long long)(nco_steps[0] - (hb_near << 55));
    const bool rotate = fabs((double)res0 * to_rad) > 2e-6;
    const uint64_t base = rotate ? nco_steps[0] : (hb_near << 55);
    const int twob = rotate ? 0 : (int)(hb_near & (2 * kCfM - 1));
    // channel k must sit on the bin grid: theta_k = base - 2 pi k / M + delta_k with a tiny delta_k
    std::vector<long long> dturn(kCfM), dt0(kCfM);
    std::vector<float> delta(kCfM);
    double maxd = 0.0;
    for (int k = 0; k < kCfM; k++) {
        const uint64_t ideal = base - ((uint64_t)k << 56);               // 2^64 / 256 = 2^56 per bin
        const long long d = (long long)(nco_steps[k] - ideal);
        const double rad = (double)d * to_rad;
        if (fabs(rad) > 2e-6) return nullptr;                            // not a uniform comb: direct form
        dturn[k] = d;
        // channel k's phase constant enters its epilogue turn count as a difference to channel 0's: launch_chanfft adds
        // channel 0's (the common ph0, or the pre-rotation's beta_ph0), and y_k carries e^{j phase_k} as a whole-row factor
        const uint64_t dph = nco_phases ? nco_phases[k] - nco_phases[0] : 0ull;
        dt0[k] = (long long)((uint64_t)llrint((double)d * 0.5 * (double)T) + dph);
        delta[k] = (float)rad;
        if (fabs(rad) > maxd) maxd = fabs(rad);
    }
    ChanFftPlan* p = new (std::nothrow) ChanFftPlan();
    if (!p) {
        set_last_error("chanfft_plan_create: out of host memory");
        if (failed) *failed = true;
        return nullptr;
    }
    p->T = T;
    p->D = decim;
    p->nch = nch;
    p->rotate = rotate;
    p->twob = twob;
    p->max_delta = maxd;
    const int pad = T & 1;
    const double tc = 0.5 * (double)T;
    std::vector<float2> g((size_t)kCfJ * kCfM);
    for (int tp = 0; tp < kCfJ * kCfM; tp++) {
        const int t = tp - pad;
        float h = (t >= 0 && t < T) ? taps[t] : 0.0f;
        if ((twob & 1) && ((tp / kCfM) & 1)) h = -h;          // half-bin comb: e^{j theta_0 M j} = (-1)^j
        g[tp] = make_float2(h, (float)(((double)t - tc) * (double)h));
    }
    if (cudaMalloc(&p->gpair_dev, g.size() * sizeof(float2)) != cudaSuccess ||
        cudaMemcpy(p->gpair_dev, g.data(), g.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMalloc(&p->dturn_dev, kCfM * sizeof(long long)) != cudaSuccess ||
        cudaMemcpy(p->dturn_dev, dturn.data(), kCfM * sizeof(long long), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMalloc(&p->dt0_dev, kCfM * sizeof(long long)) != cudaSuccess ||
        cudaMemcpy(p->dt0_dev, dt0.data(), kCfM * sizeof(long long), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMalloc(&p->delta_dev, kCfM * sizeof(float)) != cudaSuccess ||
        cudaMemcpy(p->delta_dev, delta.data(), kCfM * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("chanfft_plan_create: device allocation failed");
        if (failed) *failed = true;
        chanfft_plan_destroy(p);
        return nullptr;
    }
    return p;
}
void chanfft_plan_destroy(ChanFftPlan* p) {
    if (!p) return;
    if (p->gpair_dev) cudaFree(p->gpair_dev);
    if (p->dturn_dev) cudaFree(p->dturn_dev);
    if (p->dt0_dev) cudaFree(p->dt0_dev);
    if (p->delta_dev) cudaFree(p->delta_dev);
    if (p->uv) cudaFree(p->uv);
    delete p;
}
void chanfft_plan_take_scratch(ChanFftPlan* to, ChanFftPlan* from) {
    if (!to || !from || to->uv) return;
    to->uv = from->uv;
    to->uv_cap = from->uv_cap;
    from->uv = nullptr;
    from->uv_cap = 0;
}
// usable for this batch? uniform run() partition on the decimation grid, 16-byte aligned input
bool chanfft_usable(const ChanFftPlan* p, const Partition& part, const void* in) {
    if (!p || part.view.table != nullptr || part.total_out <= 0) return false;
    if (part.view.nblocks > 1 && (part.view.block_size % p->D) != 0) return false;
    return (reinterpret_cast<uintptr_t>(in) & 15) == 0;
}

// Segment length (output rows per CTA of the column-filter kernel): every segment pays 8 lead-in groups, and the grid runs
// one CTA per SM in waves -- pick the length that maximises (useful / total rows) x (CTAs / (waves x SMs)).
static int chanfft_pick_seg(const Partition& part) {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const long long per = part.max_out, nb = part.view.nblocks;
    int best = 64;
    double best_eff = 0.0;
    for (int seg = 24; seg <= 256; seg += 4) {
        const long long segs = (per + seg - 1) / seg;
        const long long ctas = segs * nb;
        const long long waves = (ctas + sms - 1) / sms;
        // time ~ waves x (seg + 8); work = total rows
        const double eff = (double)(per * nb) / ((double)waves * sms * (seg + 8));
        if (eff > best_eff * 1.0001) {
            best_eff = eff;
            best = seg;
        }
    }
    return best;
}

int launch_chanfft(ChanFftPlan* plan, const float2* hist, int H, const float2* in, const Partition& part, uint64_t beta_step,
                   uint64_t beta_ph0, long long abs0, float phasor_speed, const float* demod_in, float* demod_out, float* audio,
                   float2* iq, long long out_stride, cudaStream_t s) {
    const long long rows = part.total_out;
    const size_t need = (size_t)2 * rows * kCfM;
    if (need > plan->uv_cap) {
        if (plan->uv) cudaFree(plan->uv);
        plan->uv = nullptr;
        plan->uv_cap = 0;
        QDSP_CUDA_OK(cudaMalloc(&plan->uv, need * sizeof(float2)));
        plan->uv_cap = need;
    }
    ChanFftArgs a{};
    a.hist = hist;
    a.in = in;
    a.H = H;
    a.n_in = part.view.total;
    a.part = part.view;
    a.T = plan->T;
    a.pad = plan->T & 1;                 // blocks start on multiples of D (even): the window start parity is T's
    a.seg_rows = chanfft_pick_seg(part);
    a.abs0 = abs0;
    a.beta_step = beta_step;
    a.beta_ph0 = beta_ph0;
    a.gpair = plan->gpair_dev;
    a.U = plan->uv;
    a.V = plan->uv + (size_t)rows * kCfM;
    a.twist = (!plan->rotate && (plan->twob & 1)) ? 1 : 0;
    const size_t smem = (size_t)kCfStages * kCfDR * kCfM * 8 + (size_t)2 * kCfStages * 8 + 16;
    const size_t smem_b = (size_t)2 * kCfRB * 16 * kCfLd * sizeof(float2) + kCfM * sizeof(float2) + (size_t)kCfRB * (kCfM + 1) * sizeof(float);
    static bool attr_dev[64] = {};      // opt-in shared memory is a per-device function attribute
    int dev = 0;
    cudaGetDevice(&dev);
    bool& attr = attr_dev[dev & 63];
    if (!attr) {
        QDSP_CUDA_OK(cudaFuncSetAttribute(chanfft_poly_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        QDSP_CUDA_OK(cudaFuncSetAttribute(chanfft_poly_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        QDSP_CUDA_OK(cudaFuncSetAttribute(chanfft_fft_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        QDSP_CUDA_OK(cudaFuncSetAttribute(chanfft_fft_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        QDSP_CUDA_OK(cudaFuncSetAttribute(chanfft_fft_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        attr = true;
    }
    dim3 grid((part.max_out + a.seg_rows - 1) / a.seg_rows, part.view.nblocks);
    if (plan->rotate)
        chanfft_poly_kernel<true><<<grid, kCfPolyThreads, smem, s>>>(a);
    else
        chanfft_poly_kernel<false><<<grid, kCfPolyThreads, smem, s>>>(a);
    QDSP_LAUNCH_OK();
    ChanFftBArgs bb{};
    bb.U = a.U;
    bb.V = a.V;
    bb.total_out = rows;
    bb.abs0 = abs0;
    bb.T = plan->T;
    bb.pad = a.pad;
    bb.D = plan->D;
    bb.twob = plan->twob;
    bb.ph0 = plan->rotate ? 0ull : beta_ph0;
    bb.dturn = plan->dturn_dev;
    bb.dt0 = plan->dt0_dev;
    bb.delta = plan->delta_dev;
    bb.demod_in = demod_in;
    bb.demod_out = demod_out;
    bb.audio = audio;
    bb.out_stride = out_stride;
    bb.inv_speed = (float)(1.0 / (double)phasor_speed);
    bb.iq = iq;
    const unsigned nb = (unsigned)((rows + kCfNew - 1) / kCfNew);
    if (!iq)
        chanfft_fft_kernel<true, false><<<nb, kCfM, smem_b, s>>>(bb);
    else if (audio)
        chanfft_fft_kernel<true, true><<<nb, kCfM, smem_b, s>>>(bb);
    else
        chanfft_fft_kernel<false, true><<<nb, kCfM, smem_b, s>>>(bb);
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
