// qdsp_b200/csrc/api.cu — the C ABI (include/qdsp_b200.h): opaque handles, state, dispatch.
// No compute happens on the host; every process call enqueues sm_100a kernels on the caller's stream.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <vector>
#include "internal.cuh"
#include "kernels.cuh"

using namespace qdsp;

namespace {

// taps -> polyphase bank, reference src/dsp/resampling.h:137-166 (buildTapPhases):
// tapsPerPhase = ceil(tapCount / interp); phases[(I-1)-p][t] = taps[t*I + p], zero padded.
std::vector<float> build_phases(const float* taps, int T, int interp, int* tpp_out) {
    const int tpp = (T + interp - 1) / interp;
    std::vector<float> ph((size_t)interp * tpp, 0.0f);
    for (int p = 0; p < interp; p++)
        for (int t = 0; t < tpp; t++) {
            const int idx = t * interp + p;
            ph[(size_t)(interp - 1 - p) * tpp + t] = idx < T ? taps[idx] : 0.0f;
        }
    *tpp_out = tpp;
    return ph;
}

int upload_floats(float** dev, const std::vector<float>& v) {
    if (*dev) cudaFree(*dev);
    *dev = nullptr;
    QDSP_CUDA_OK(cudaMalloc(dev, sizeof(float) * (v.size() + 16)));
    QDSP_CUDA_OK(cudaMemset(*dev, 0, sizeof(float) * (v.size() + 16)));
    QDSP_CUDA_OK(cudaMemcpy(*dev, v.data(), sizeof(float) * v.size(), cudaMemcpyHostToDevice));
    return 0;
}

struct Scratch {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        QDSP_CUDA_OK(cudaMalloc(&p, bytes));
        cap = bytes;
        return 0;
    }
    ~Scratch() {
        if (p) cudaFree(p);
    }
};

// small device-resident float state with host get/set
struct DevState {
    float* p = nullptr;
    int n = 0;
    int init(int n_, const float* v) {
        n = n_;
        QDSP_CUDA_OK(cudaMalloc(&p, sizeof(float) * n));
        QDSP_CUDA_OK(cudaMemcpy(p, v, sizeof(float) * n, cudaMemcpyHostToDevice));
        return 0;
    }
    int get(float* v, int count, int offset = 0) const {
        QDSP_CUDA_OK(cudaDeviceSynchronize());
        QDSP_CUDA_OK(cudaMemcpy(v, p + offset, sizeof(float) * count, cudaMemcpyDeviceToHost));
        return 0;
    }
    int set(const float* v, int count, int offset = 0) {
        QDSP_CUDA_OK(cudaDeviceSynchronize());
        QDSP_CUDA_OK(cudaMemcpy(p + offset, v, sizeof(float) * count, cudaMemcpyHostToDevice));
        return 0;
    }
    ~DevState() {
        if (p) cudaFree(p);
    }
};

int import_tail_impl(History& hist, const void* tail_dev, int src_device, cudaStream_t s) {
    if (hist.H <= 0) return 0;
    int dev = 0;
    QDSP_CUDA_OK(cudaGetDevice(&dev));
    const size_t bytes = (size_t)hist.H * hist.elem;
    if (src_device < 0 || src_device == dev)
        QDSP_CUDA_OK(cudaMemcpyAsync(hist.buf[hist.cur], tail_dev, bytes, cudaMemcpyDeviceToDevice, s));
    else
        QDSP_CUDA_OK(cudaMemcpyPeerAsync(hist.buf[hist.cur], dev, tail_dev, src_device, bytes, s));
    return 0;
}

// the blocks that take a `dtype` read float or cf32 only (integer IQ goes through qdsp_iq_convert_process)
bool real_or_complex(int dtype, const char* who) {
    if (dtype == QDSP_F32 || dtype == QDSP_CF32) return true;
    set_last_error("%s: dtype %d is not QDSP_F32 or QDSP_CF32", who, dtype);
    return false;
}

// an integer IQ format and its conversion (include/qdsp_b200.h, qdsp_iq_convert_process)
bool iq_format_ok(int fmt, float scale, float offset, const char* who) {
    if (fmt != QDSP_CS16 && fmt != QDSP_CS8 && fmt != QDSP_CU8) {
        set_last_error("%s: format %d is not QDSP_CS16, QDSP_CS8 or QDSP_CU8", who, fmt);
        return false;
    }
    if (!isfinite(scale) || scale == 0.0f || !isfinite(offset)) {
        set_last_error("%s: scale must be finite and non-zero, offset finite (got %g, %g)", who, (double)scale, (double)offset);
        return false;
    }
    return true;
}

bool ranges_overlap(const void* a, size_t na, const void* b, size_t nb) {
    const char *pa = (const char*)a, *pb = (const char*)b;
    return pa < pb + nb && pb < pa + na;
}

// Overlapped consecutive calls (DESIGN.md §6.0f): a handle whose kernel folds the history advance into itself keeps the
// record of its last such call here. When the very next library launch is that handle's next call on the same stream,
// the handle's own rule on the buffers decides whether the two grids may overlap (programmatic dependent launch).
struct CallChain {
    long long serial = -1;      // g_launches right after the recorded launch; -1: nothing to follow
    cudaStream_t stream = nullptr;
    const void *in = nullptr, *out = nullptr;
    size_t in_bytes = 0, out_bytes = 0;

    void clear() { serial = -1; }
    bool follows(cudaStream_t s) const { return serial == g_launches.load() && stream == s; }
    void record(cudaStream_t s, const void* in_, size_t in_bytes_, const void* out_, size_t out_bytes_) {
        serial = g_launches.load();
        stream = s;
        in = in_;
        in_bytes = in_bytes_;
        out = out_;
        out_bytes = out_bytes_;
    }
};

}  // namespace

extern "C" long long qdsp_iq_convert_process(int fmt, float scale, float offset, const void* in_dev, void* out_dev,
                                             long long count, qdsp_stream_t s) {
    if (!iq_format_ok(fmt, scale, offset, "iq_convert_process")) return -1;
    if (count < 0 || (count > 0 && (!in_dev || !out_dev)) ||
        (reinterpret_cast<uintptr_t>(in_dev) % iq_pair_bytes(fmt)) != 0 || (reinterpret_cast<uintptr_t>(out_dev) & 7) != 0) {
        set_last_error("iq_convert_process: bad arguments (input aligned to its pair, output to 8 bytes)");
        return -1;
    }
    if (launch_iq_convert(fmt, IqConv{scale, offset}, in_dev, (float2*)out_dev, count, as_stream(s)) != 0) return -1;
    return count;
}

// =================================================================================================
// FIR
// =================================================================================================
struct qdsp_fir {
    int dtype = QDSP_CF32;
    int T = 0;
    float* taps_dev = nullptr;  // phases layout for I=1 == taps
    History hist;
    Partition part;
    FirPlan* plan = nullptr;
    int variant = 0;
    std::vector<float> taps;
    CallChain chain;            // the last call on the constant-bank kernels (history advance folded in)
};

extern "C" {

qdsp_fir* qdsp_fir_create(int dtype, const float* taps, int tapCount) {
    if (!taps || tapCount <= 0 || (dtype != QDSP_F32 && dtype != QDSP_CF32)) {
        set_last_error("fir_create: bad arguments");
        return nullptr;
    }
    qdsp_fir* h = new (std::nothrow) qdsp_fir();
    if (!h) return nullptr;
    h->dtype = dtype;
    if (qdsp_fir_set_taps(h, taps, tapCount) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_fir_destroy(qdsp_fir* h) {
    if (!h) return;
    if (h->taps_dev) cudaFree(h->taps_dev);
    if (h->plan) fir_plan_destroy(h->plan);
    h->hist.release();
    delete h;
}
int qdsp_fir_set_taps(qdsp_fir* h, const float* taps, int tapCount) {
    h->chain.clear();
    h->taps.assign(taps, taps + tapCount);
    if (upload_floats(&h->taps_dev, h->taps) != 0) return -1;
    if (tapCount != h->T) {
        h->T = tapCount;
        // reference filter.h:28 leaves the history uninitialised; we define it as zeros
        if (h->hist.init(tapCount - 1, h->dtype == QDSP_CF32 ? 8 : 4) != 0) return -1;
    }
    if (h->plan) fir_plan_destroy(h->plan);
    h->plan = (h->dtype == QDSP_CF32) ? fir_plan_create(taps, tapCount) : nullptr;
    return 0;
}
long long qdsp_fir_process(qdsp_fir* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (count < 0) return -1;
    if (count == 0) return 0;
    const bool dense = h->plan && h->variant != 1;
    if (dense) {
        const size_t bytes = (size_t)count * 8;
        const CallChain& prev = h->chain;
        const bool overlap_prev = prev.follows(s) && !ranges_overlap(in_dev, bytes, prev.out, prev.out_bytes) &&
                                  !ranges_overlap(out_dev, bytes, prev.in, prev.in_bytes) &&
                                  !ranges_overlap(out_dev, bytes, prev.out, prev.out_bytes);
        bool advanced = false;
        if (launch_fir_dense(h->plan, (const float2*)h->hist.ptr(), h->hist.H, (const float2*)in_dev, count, 1,
                             (float2*)out_dev, s, (float2*)h->hist.buf[h->hist.cur ^ 1], overlap_prev, &advanced) != 0)
            return -1;
        if (advanced) {              // the kernel's first CTA advanced the history tail: one launch per call
            h->hist.cur ^= 1;
            h->chain.record(s, in_dev, bytes, out_dev, bytes);
            return count;
        }
        h->chain.clear();
    } else {
        // FIR == polyphase bank with I = D = 1 read one sample later (filter.h:65 reads &buffer[i+1]);
        // y[i] = sum_j taps[j] * x[i - (T-1) + j]; the generic kernel's TPP-deep window with lead=1.
        // Blocks of <= 2^30 outputs keep per-block counts in int.
        if (h->part.build(count, nullptr, 0, 1 << 20, 1, 1, s) != 0) return -1;
        int rc;
        // history is T-1 deep; the generic kernel's virtual stream tolerates reads one element
        // further back (returns 0 there, multiplied by no tap: base index starts at -(T-1)).
        if (h->dtype == QDSP_CF32)
            rc = launch_generic_resamp<float2>((const float2*)h->hist.ptr(), h->hist.H, (const float2*)in_dev,
                                               h->taps_dev, h->T, 1, h->part, (float2*)out_dev, s);
        else
            rc = launch_generic_resamp<float>((const float*)h->hist.ptr(), h->hist.H, (const float*)in_dev,
                                              h->taps_dev, h->T, 1, h->part, (float*)out_dev, s);
        if (rc != 0) return -1;
    }
    if (h->hist.advance(in_dev, count, s) != 0) return -1;
    return count;
}
long long qdsp_fir_process_halo(qdsp_fir* h, const void* halo_dev, const void* in_dev, void* out_dev, long long count,
                                qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (!h->plan) {
        set_last_error("fir_process_halo: cf32 filters only");
        return -1;
    }
    // halo_dev == NULL: zero history (H = 0: every read before sample 0 returns zero)
    if (launch_fir_dense(h->plan, (const float2*)halo_dev, halo_dev ? h->hist.H : 0, (const float2*)in_dev, count, 1,
                         (float2*)out_dev, s) != 0)
        return -1;
    if (count >= h->hist.H) {
        if (h->hist.advance(in_dev, count, s) != 0) return -1;
    } else {   // short call: the new tail still contains halo samples
        if (halo_dev) QDSP_CUDA_OK(cudaMemcpyAsync(h->hist.buf[h->hist.cur], halo_dev, (size_t)h->hist.H * h->hist.elem, cudaMemcpyDefault, s));
        else QDSP_CUDA_OK(cudaMemsetAsync(h->hist.buf[h->hist.cur], 0, (size_t)h->hist.H * h->hist.elem, s));
        if (h->hist.advance(in_dev, count, s) != 0) return -1;
    }
    return count;
}
int qdsp_fir_history_len(qdsp_fir* h) { return h->hist.H; }
int qdsp_fir_get_history(qdsp_fir* h, void* hist_host) {
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    if (h->hist.H > 0)
        QDSP_CUDA_OK(cudaMemcpy(hist_host, h->hist.ptr(), (size_t)h->hist.H * h->hist.elem, cudaMemcpyDeviceToHost));
    return 0;
}
int qdsp_fir_set_history(qdsp_fir* h, const void* hist_host) {
    h->chain.clear();
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    if (h->hist.H > 0)
        QDSP_CUDA_OK(cudaMemcpy(h->hist.buf[h->hist.cur], hist_host, (size_t)h->hist.H * h->hist.elem,
                                cudaMemcpyHostToDevice));
    return 0;
}
int qdsp_fir_import_tail(qdsp_fir* h, const void* tail_dev, int src_device, qdsp_stream_t s) {
    h->chain.clear();
    return import_tail_impl(h->hist, tail_dev, src_device, as_stream(s));
}
int qdsp_fir_reset(qdsp_fir* h) {
    h->chain.clear();
    return h->hist.reset(nullptr);
}
int qdsp_fir_set_variant(qdsp_fir* h, int variant) {
    h->variant = variant;
    return 0;
}

}  // extern "C"

// =================================================================================================
// PolyphaseResampler
// =================================================================================================
struct qdsp_resamp {
    int dtype = QDSP_CF32;
    int T = 0, interp = 1, decim = 1, tpp = 0;
    float* phases_dev = nullptr;
    History hist;
    Partition part;
    DecimPlan* plan = nullptr;
    FirDecimPlan* fplan = nullptr;   // small decimation (2..8): dense polyphase kernel
    int variant = 0;
    std::vector<float> taps;         // host copy (kernels that take their taps as launch parameters)
    CallChain chain;                 // the last launch_firrow call (history advance folded in)
};

extern "C" {

qdsp_resamp* qdsp_resamp_create(int dtype, const float* taps, int tapCount, int interp, int decim) {
    if (!taps || tapCount <= 0 || interp <= 0 || decim <= 0 || (dtype != QDSP_F32 && dtype != QDSP_CF32)) {
        set_last_error("resamp_create: bad arguments");
        return nullptr;
    }
    qdsp_resamp* h = new (std::nothrow) qdsp_resamp();
    if (!h) return nullptr;
    h->dtype = dtype;
    h->interp = interp;
    h->decim = decim;
    if (qdsp_resamp_set_taps(h, taps, tapCount) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_resamp_destroy(qdsp_resamp* h) {
    if (!h) return;
    if (h->phases_dev) cudaFree(h->phases_dev);
    if (h->plan) decim_plan_destroy(h->plan);
    if (h->fplan) fir_decim_plan_destroy(h->fplan);
    h->hist.release();
    delete h;
}
int qdsp_resamp_set_taps(qdsp_resamp* h, const float* taps, int tapCount) {
    h->chain.clear();      // state changed from the host: the next call does not overlap its predecessor
    int tpp = 0;
    std::vector<float> ph = build_phases(taps, tapCount, h->interp, &tpp);
    if (upload_floats(&h->phases_dev, ph) != 0) return -1;
    h->T = tapCount;
    h->taps.assign(taps, taps + tapCount);
    if (tpp != h->tpp) {
        h->tpp = tpp;
        if (h->hist.init(tpp, h->dtype == QDSP_CF32 ? 8 : 4) != 0) return -1;  // zeroed, resampling.h:39
    }
    if (h->plan) decim_plan_destroy(h->plan);
    h->plan = nullptr;
    if (h->dtype == QDSP_CF32 && decim_plan_supported(tapCount, h->interp, h->decim))
        h->plan = decim_plan_create(taps, tapCount, h->decim);
    if (h->fplan) fir_decim_plan_destroy(h->fplan);
    h->fplan = nullptr;
    if (h->dtype == QDSP_CF32 && !h->plan && h->interp == 1 && h->decim >= 2 && h->decim <= 8)
        h->fplan = fir_decim_plan_create(taps, tapCount, h->decim);
    return 0;
}
int qdsp_resamp_taps_per_phase(qdsp_resamp* h) { return h->tpp; }
long long qdsp_resamp_out_count(qdsp_resamp* h, long long count) { return (count * h->interp) / h->decim; }

long long qdsp_resamp_process(qdsp_resamp* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                              int nblocks, int block_size, int* out_counts, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, h->interp, h->decim, s) != 0) return -1;
    if (out_counts) {
        for (int b = 0; b < h->part.view.nblocks; b++) {
            if (blocks) out_counts[b] = h->part.host[b].out_count;
            else {
                const long long st = (long long)b * h->part.view.block_size;
                const long long c = count - st < h->part.view.block_size ? count - st : h->part.view.block_size;
                out_counts[b] = (int)((c * h->interp) / h->decim);
            }
        }
    }
    if (count == 0) return 0;
    int rc;
    // the dense polyphase kernel works on a uniform output grid: every run() block but the last must be a
    // multiple of D (otherwise the reference's per-block schedule restart shifts the grid: generic kernel)
    bool regular = h->fplan != nullptr && h->variant != 1;
    if (regular) {
        if (blocks) {
            for (int b = 0; b + 1 < nblocks && regular; b++) regular = (blocks[b] % h->decim) == 0;
        } else {
            regular = h->part.view.nblocks <= 1 || (h->part.view.block_size % h->decim) == 0;
        }
    }
    if (regular && h->variant != 2 && h->part.total_out > 0 && firrow_supported(h->T, h->decim) &&
        (reinterpret_cast<uintptr_t>(in_dev) & 15) == 0) {
        // config 1b's geometry: row-per-lane kernel (TMA-fed, taps as uniform-register operands)
        const size_t ibytes = (size_t)count * 8, obytes = (size_t)h->part.total_out * 8;
        const CallChain& prev = h->chain;
        const bool overlap_prev = prev.follows(s) && !ranges_overlap(in_dev, ibytes, prev.out, prev.out_bytes) &&
                                  !ranges_overlap(out_dev, obytes, prev.in, prev.in_bytes) &&
                                  !ranges_overlap(out_dev, obytes, prev.out, prev.out_bytes);
        rc = launch_firrow(h->taps.data(), h->T, h->decim, (const float2*)h->hist.ptr(), (float2*)h->hist.buf[h->hist.cur ^ 1],
                           h->hist.H, (const float2*)in_dev, count, h->part.total_out, (float2*)out_dev, s, overlap_prev);
        if (rc != 0) return -1;
        h->chain.record(s, in_dev, ibytes, out_dev, obytes);
        h->hist.cur ^= 1;            // the kernel's first CTA advanced the history tail
        return h->part.total_out;
    } else if (regular) {
        rc = launch_fir_decim(h->fplan, (const float2*)h->hist.ptr(), h->hist.H, (const float2*)in_dev, count,
                              h->part.total_out, (float2*)out_dev, s);
    } else if (h->plan && h->variant != 1) {
        rc = launch_decim(h->plan, (const float2*)h->hist.ptr(), h->hist.H, (const float2*)in_dev, h->part, 0, nullptr,
                          0, 1, 0.0f, nullptr, nullptr, (float2*)out_dev, nullptr, 0, s);
    } else if (h->dtype == QDSP_CF32) {
        rc = launch_generic_resamp<float2>((const float2*)h->hist.ptr(), h->hist.H, (const float2*)in_dev,
                                           h->phases_dev, h->tpp, 0, h->part, (float2*)out_dev, s);
    } else {
        rc = launch_generic_resamp<float>((const float*)h->hist.ptr(), h->hist.H, (const float*)in_dev, h->phases_dev,
                                          h->tpp, 0, h->part, (float*)out_dev, s);
    }
    if (rc != 0) return -1;
    if (h->hist.advance(in_dev, count, s) != 0) return -1;
    return h->part.total_out;
}
long long qdsp_resamp_schedule_device(qdsp_resamp* h, long long count, const int* blocks, int nblocks, int block_size,
                                      int* phase_dev, long long* index_dev, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, h->interp, h->decim, s) != 0) return -1;
    if (launch_schedule(h->part, phase_dev, index_dev, s) != 0) return -1;
    return h->part.total_out;
}
int qdsp_resamp_history_len(qdsp_resamp* h) { return h->hist.H; }
int qdsp_resamp_get_history(qdsp_resamp* h, void* hist_host) {
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    QDSP_CUDA_OK(cudaMemcpy(hist_host, h->hist.ptr(), (size_t)h->hist.H * h->hist.elem, cudaMemcpyDeviceToHost));
    return 0;
}
int qdsp_resamp_set_history(qdsp_resamp* h, const void* hist_host) {
    h->chain.clear();
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    QDSP_CUDA_OK(cudaMemcpy(h->hist.buf[h->hist.cur], hist_host, (size_t)h->hist.H * h->hist.elem,
                            cudaMemcpyHostToDevice));
    return 0;
}
int qdsp_resamp_reset(qdsp_resamp* h) {
    h->chain.clear();
    return h->hist.reset(nullptr);
}
int qdsp_resamp_set_variant(qdsp_resamp* h, int variant) {
    h->variant = variant;
    return 0;
}

// =================================================================================================
// PowerDecimator (stateless) — reference resampling.h:220-249, including the power>1 quirk: the
// extra passes re-read the input, so the result is the first count>>(power-1) pair averages.
// =================================================================================================
long long qdsp_power_decim_process(unsigned int power, const void* in_dev, void* out_dev, long long count,
                                   qdsp_stream_t s) {
    if (count < 0) return -1;
    long long n_out;
    if (power == 0) n_out = count;
    else if (power == 1) n_out = count / 2;
    else n_out = power - 1 >= 62 ? 0 : (count >> (power - 1));
    if (launch_power_decim((const float2*)in_dev, (float2*)out_dev, n_out, power == 0, as_stream(s)) != 0) return -1;
    return n_out;
}

}  // extern "C"

// =================================================================================================
// FrequencyXlator
// =================================================================================================
struct qdsp_xlator {
    Nco nco;
    float2 inc_pow[3];
    void refresh() {
        const double th = atan2((double)nco.inc_im, (double)nco.inc_re);
        for (int j = 1; j <= 3; j++) inc_pow[j - 1] = make_float2((float)cos(th * j), (float)sin(th * j));
    }
};

extern "C" {

qdsp_xlator* qdsp_xlator_create(float sampleRate, float freq) {
    qdsp_xlator* h = new (std::nothrow) qdsp_xlator();
    if (!h) return nullptr;
    h->nco.set_freq(sampleRate, freq);
    h->nco.phase = 0;  // phase = (1, 0), processing.h:20
    h->refresh();
    return h;
}
void qdsp_xlator_destroy(qdsp_xlator* h) { delete h; }
int qdsp_xlator_set_frequency(qdsp_xlator* h, float sampleRate, float freq) {
    h->nco.set_freq(sampleRate, freq);
    h->refresh();
    return 0;
}
void qdsp_xlator_get_phase_delta(qdsp_xlator* h, float* re, float* im) {
    *re = h->nco.inc_re;
    *im = h->nco.inc_im;
}
void qdsp_xlator_get_phase(qdsp_xlator* h, float* re, float* im) { h->nco.get_phase(re, im); }
void qdsp_xlator_set_phase(qdsp_xlator* h, float re, float im) { h->nco.set_phase(re, im); }
long long qdsp_xlator_process(qdsp_xlator* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (launch_xlator((const float2*)in_dev, (float2*)out_dev, count, h->nco.phase, h->nco.step, h->inc_pow[0],
                      h->inc_pow[1], h->inc_pow[2], as_stream(s)) != 0)
        return -1;
    h->nco.advance(count);
    return count;
}

}  // extern "C"

// =================================================================================================
// FloatFMDemod / FMDemod
// =================================================================================================
struct qdsp_fmdemod {
    float phasor_speed = 1.0f;
    int stereo = 0;
    DevState st;  // [2] ping-pong
    int cur = 0;
};

static float fm_phasor_speed(float sampleRate, float deviation) {
    return (2 * QDSP_FL_M_PI) / (sampleRate / deviation);  // demodulator.h:43
}

extern "C" {

qdsp_fmdemod* qdsp_fmdemod_create(float sampleRate, float deviation, int stereo_out) {
    qdsp_fmdemod* h = new (std::nothrow) qdsp_fmdemod();
    if (!h) return nullptr;
    h->phasor_speed = fm_phasor_speed(sampleRate, deviation);
    h->stereo = stereo_out;
    const float z[2] = {0.0f, 0.0f};
    if (h->st.init(2, z) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_fmdemod_destroy(qdsp_fmdemod* h) { delete h; }
float qdsp_fmdemod_get_phase(qdsp_fmdemod* h) {
    float v = 0.0f;
    h->st.get(&v, 1, h->cur);
    return v;
}
int qdsp_fmdemod_set_phase(qdsp_fmdemod* h, float phase) { return h->st.set(&phase, 1, h->cur); }
long long qdsp_fmdemod_process(qdsp_fmdemod* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (launch_fmdemod((const float2*)in_dev, out_dev, count, h->phasor_speed, h->st.p + h->cur,
                       h->st.p + (h->cur ^ 1), h->stereo, as_stream(s)) != 0)
        return -1;
    h->cur ^= 1;
    return count;
}

}  // extern "C"

// =================================================================================================
// fused VFO -> FM demod, and the channelizer (N of them off one input)
// =================================================================================================
struct qdsp_channelizer {
    int nch = 1;
    float in_sr = 0, out_sr = 0, bw = 0, dev = 0;
    int T = 0, interp = 1, decim = 1, tpp = 0;
    float phasor_speed = 1.0f;
    std::vector<float> taps;
    std::vector<Nco> nco;        // per channel, host copy
    NcoDev* nco_dev = nullptr;   // per channel constants
    float* phases_dev = nullptr;
    History hist;                // raw (untranslated) input tail, shared by all channels
    Partition part;
    DecimPlan* plan = nullptr;
    ChanFftPlan* fftplan = nullptr;   // uniform 256-channel comb: FFT polyphase channelizer (k_chanfft.cu)
    DevState demod;              // [2][nch] ping-pong
    int cur = 0;
    long long abs_pos = 0;       // absolute index of the next input sample (NCO closed form)
    int variant = 0;
    // end-to-end staging (process_host)
    void* stage_in[2] = {nullptr, nullptr};
    float* stage_out[2] = {nullptr, nullptr};
    cudaEvent_t ev_done[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    size_t stage_samples = 0;
    // debug replay of the reference's recursive NCO (process_replay): its own state
    History hist_mixed;          // tail of the MIXED stream (resampling.h:129)
    DevState demod_replay;       // [2] ping-pong demodulator phase
    int cur_replay = 0;
    Scratch replay_scratch;      // mixed stream | resampled IQ | run table | checkpoints
    Partition part_replay;
    DecimPlan* plan_replay = nullptr;
    // bench hook: events around the dominant kernel (enable_timing), or per-launch timestamps written by the row-per-lane
    // kernel itself (enable_timing_ring): an event recorded between two launches would keep them from overlapping
    bool timing = false;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;
    unsigned long long* ring = nullptr;                     // [2 * ring_pairs]: first CTA start, last CTA end (ns)
    int ring_pairs = 0;
    long long ring_launches = 0;
    // the last row-per-lane call without IQ output; the kernel orders the carried state and its audio stores (k_rowlane.cu)
    CallChain chain;
    // element type of the input (set_input_format): integer input is converted to cf32 in `conv` (grown to the largest
    // call, so the hot path stays allocation-free) and the kernels read that
    int in_fmt = QDSP_CF32;
    IqConv in_conv{1.0f, 0.0f};
    Scratch conv;

    int set_input_format(int fmt, float scale, float offset, const char* who) {
        if (fmt != QDSP_CF32 && !iq_format_ok(fmt, scale, offset, who)) return -1;
        chain.clear();
        in_fmt = fmt;
        in_conv = fmt == QDSP_CF32 ? IqConv{1.0f, 0.0f} : IqConv{scale, offset};
        return 0;
    }

    int upload_nco() {
        chain.clear();
        std::vector<NcoDev> v(nch);
        for (int c = 0; c < nch; c++) v[c] = NcoDev{nco[c].phase, nco[c].step};
        if (!nco_dev) QDSP_CUDA_OK(cudaMalloc(&nco_dev, sizeof(NcoDev) * nch));
        QDSP_CUDA_OK(cudaDeviceSynchronize());
        QDSP_CUDA_OK(cudaMemcpy(nco_dev, v.data(), sizeof(NcoDev) * nch, cudaMemcpyHostToDevice));
        return 0;
    }
    int setup(int nch_, const float* offsets, float inSR, float outSR, float bandWidth, float deviation) {
        nch = nch_;
        in_sr = inSR;
        out_sr = outSR;
        bw = bandWidth;
        dev = deviation;
        T = qdsp_vfo_design(inSR, outSR, bandWidth, nullptr, 0, &interp, &decim);
        taps.resize(T);
        qdsp_vfo_design(inSR, outSR, bandWidth, taps.data(), T, &interp, &decim);
        std::vector<float> ph = build_phases(taps.data(), T, interp, &tpp);
        if (upload_floats(&phases_dev, ph) != 0) return -1;
        if (hist.init(tpp, 8) != 0) return -1;
        nco.resize(nch);
        for (int c = 0; c < nch; c++) {
            nco[c].set_freq(inSR, -offsets[c]);  // VFO::init: xlator.init(in, inSR, -offset), vfo.h:28
            nco[c].phase = 0;
        }
        if (upload_nco() != 0) return -1;
        phasor_speed = fm_phasor_speed(outSR, deviation);
        std::vector<float> z(2 * nch, 0.0f);
        if (demod.init(2 * nch, z.data()) != 0) return -1;
        if (decim_plan_supported(T, interp, decim)) plan = decim_plan_create(taps.data(), T, decim);
        {
            std::vector<uint64_t> steps(nch);
            for (int c = 0; c < nch; c++) steps[c] = nco[c].step;
            fftplan = chanfft_plan_create(taps.data(), T, interp, decim, nch, steps.data());   // nullptr unless a uniform comb
        }
        return 0;
    }
    long long process(const void* in_dev, float* audio, void* iq, long long out_stride, long long count,
                      const int* blocks, int nblocks, int block_size, int* out_counts, cudaStream_t s) {
        if (part.build(count, blocks, nblocks, block_size, interp, decim, s) != 0) return -1;
        if (out_counts) {
            for (int b = 0; b < part.view.nblocks; b++) {
                if (blocks) out_counts[b] = part.host[b].out_count;
                else {
                    const long long st = (long long)b * part.view.block_size;
                    const long long c = count - st < part.view.block_size ? count - st : part.view.block_size;
                    out_counts[b] = (int)((c * interp) / decim);
                }
            }
        }
        if (count == 0) return 0;
        const float* din = demod.p + (size_t)cur * nch;
        float* dout = demod.p + (size_t)(cur ^ 1) * nch;
        int rc;
        const bool events = timing && !ring;
        if (in_fmt != QDSP_CF32) {
            // integer input: convert, then the cf32 path unchanged
            if ((reinterpret_cast<uintptr_t>(in_dev) % iq_pair_bytes(in_fmt)) != 0) {
                set_last_error("process: integer input must be aligned to its pair");
                return -1;
            }
            if (conv.reserve((size_t)count * 8) != 0) return -1;
            if (launch_iq_convert(in_fmt, in_conv, in_dev, (float2*)conv.p, count, s) != 0) return -1;
            in_dev = conv.p;
        }
        if (events) QDSP_CUDA_OK(cudaEventRecord(ev_k0, s));
        bool hist_folded = false;
        int rpad = -1;
        if (fftplan && variant == 0 && !iq && chanfft_usable(fftplan, part, in_dev)) {
            // all 256 channels from one pass of column filters + two 256-point FFTs per output row
            rc = launch_chanfft(fftplan, (const float2*)hist.ptr(), hist.H, (const float2*)in_dev, part, nco[0].step, nco[0].phase,
                                abs_pos, phasor_speed, din, dout, audio, out_stride, s);
        } else if (plan && variant != 1 && nch == 1 && rowlane_supported(plan) && (reinterpret_cast<uintptr_t>(in_dev) & 15) == 0 &&
            part.max_out > 0 && (rpad = rowlane_uniform_pad(part, T)) >= 0) {
            // row-per-lane kernel; the history advance (resampling.h:129) is folded into its first CTA
            const NcoDev nh{nco[0].phase, nco[0].step};
            // overlap needs: no block-table upload between the launches (uniform partition), no IQ output (stored
            // without the wait), and no read of the previous call's audio (the input is staged before the wait)
            const bool overlap_prev = chain.follows(s) && !iq && part.view.table == nullptr &&
                                      !ranges_overlap(in_dev, (size_t)count * 8, chain.out, chain.out_bytes);
            unsigned long long* tslot = ring && ring_launches < ring_pairs ? ring + 2 * ring_launches : nullptr;
            rc = launch_decim_rowlane(plan, taps.data(), (const float2*)hist.ptr(), (float2*)hist.buf[hist.cur ^ 1], hist.H,
                                      (const float2*)in_dev, part, 1, nco_dev, &nh, abs_pos, phasor_speed, din, dout,
                                      (float2*)iq, audio, rpad, s, overlap_prev, tslot);
            if (ring && rc == 0) ring_launches++;
            hist_folded = rc == 0;
            if (hist_folded && !iq) chain.record(s, in_dev, (size_t)count * 8, audio, (size_t)part.total_out * 4);
        } else if (plan && variant != 1 && chan_supported(plan) && (reinterpret_cast<uintptr_t>(in_dev) & 15) == 0 &&
                   part.max_out > 0 && (rpad = rowlane_uniform_pad(part, T)) >= 0) {
            // wide rows: channel-per-lane kernel (32 channels share every staged sample), one launch per column slice
            rc = launch_chan(plan, taps.data(), (const float2*)hist.ptr(), hist.H, (const float2*)in_dev, part, 1, nco_dev,
                             abs_pos, nch, phasor_speed, din, dout, (float2*)iq, audio, out_stride, rpad, s);
        } else if (plan && variant != 1)
            rc = launch_decim(plan, (const float2*)hist.ptr(), hist.H, (const float2*)in_dev, part, 1, nco_dev,
                              abs_pos, nch, phasor_speed, din, dout, (float2*)iq, audio, out_stride, s);
        else
            rc = launch_generic_vfofm((const float2*)hist.ptr(), hist.H, (const float2*)in_dev, phases_dev, tpp, part,
                                      nco_dev, abs_pos, nch, phasor_speed, din, dout, audio, (float2*)iq, out_stride,
                                      s);
        if (!hist_folded || iq) chain.clear();
        if (rc != 0) return -1;
        if (events) QDSP_CUDA_OK(cudaEventRecord(ev_k1, s));
        if (part.total_out > 0) cur ^= 1;
        if (hist_folded) hist.cur ^= 1;
        else if (hist.advance(in_dev, count, s) != 0) return -1;
        abs_pos += count;
        return part.total_out;
    }
    ~qdsp_channelizer() {
        if (nco_dev) cudaFree(nco_dev);
        if (phases_dev) cudaFree(phases_dev);
        if (plan) decim_plan_destroy(plan);
        if (fftplan) chanfft_plan_destroy(fftplan);
        if (plan_replay) decim_plan_destroy(plan_replay);
        hist.release();
        hist_mixed.release();
        for (int i = 0; i < 2; i++) {
            if (stage_in[i]) cudaFree(stage_in[i]);
            if (stage_out[i]) cudaFree(stage_out[i]);
            if (ev_done[i]) cudaEventDestroy(ev_done[i]);
        }
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (ev_k0) cudaEventDestroy(ev_k0);
        if (ev_k1) cudaEventDestroy(ev_k1);
        if (ring) cudaFree(ring);
    }
};
struct qdsp_vfofm {
    qdsp_channelizer c;
};

extern "C" {

qdsp_vfofm* qdsp_vfofm_create(float offset, float inSampleRate, float outSampleRate, float bandWidth,
                              float deviation) {
    qdsp_vfofm* h = new (std::nothrow) qdsp_vfofm();
    if (!h) return nullptr;
    if (h->c.setup(1, &offset, inSampleRate, outSampleRate, bandWidth, deviation) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_vfofm_destroy(qdsp_vfofm* h) { delete h; }
int qdsp_vfofm_design(qdsp_vfofm* h, int* tapCount, int* interp, int* decim) {
    if (tapCount) *tapCount = h->c.T;
    if (interp) *interp = h->c.interp;
    if (decim) *decim = h->c.decim;
    return 0;
}
int qdsp_vfofm_set_offset(qdsp_vfofm* h, float offset) {
    // keep the phase continuous at the current position: phase(abs_pos) is preserved
    Nco& n = h->c.nco[0];
    const uint64_t cur_phase = n.phase + n.step * (uint64_t)h->c.abs_pos;
    n.set_freq(h->c.in_sr, -offset);
    n.phase = cur_phase - n.step * (uint64_t)h->c.abs_pos;
    return h->c.upload_nco();
}
void qdsp_vfofm_get_phase(qdsp_vfofm* h, float* re, float* im) {
    Nco n = h->c.nco[0];
    n.phase = n.phase + n.step * (uint64_t)h->c.abs_pos;
    n.get_phase(re, im);
}
int qdsp_vfofm_set_phase(qdsp_vfofm* h, float re, float im) {
    Nco& n = h->c.nco[0];
    n.set_phase(re, im);                              // phase at the current position ...
    n.phase -= n.step * (uint64_t)h->c.abs_pos;       // ... expressed as the constant of the closed form
    return h->c.upload_nco();
}
long long qdsp_vfofm_out_count(qdsp_vfofm* h, long long count, const int* blocks, int nblocks, int block_size) {
    Partition p;
    if (p.build(count, blocks, nblocks, block_size, h->c.interp, h->c.decim, nullptr) != 0) return -1;
    return p.total_out;
}
long long qdsp_vfofm_process(qdsp_vfofm* h, const void* in_dev, float* audio_out_dev, void* iq_out_dev,
                             long long count, const int* blocks, int nblocks, int block_size, int* out_counts,
                             qdsp_stream_t s) {
    return h->c.process(in_dev, audio_out_dev, iq_out_dev, 0, count, blocks, nblocks, block_size, out_counts,
                        as_stream(s));
}
// Host-buffer entry point: the stream is cut into chunks of whole run()-blocks; chunk i+1's H2D copy
// (copy stream) overlaps chunk i's kernel (compute stream) and chunk i-1's D2H.
long long qdsp_vfofm_process_host(qdsp_vfofm* h, const void* in_host, float* audio_out_host, long long count,
                                  int block_size, qdsp_stream_t s_) {
    qdsp_channelizer& c = h->c;
    cudaStream_t s = as_stream(s_);
    if (block_size <= 0) block_size = 1000000;
    const long long blocks_per_chunk = (8ll << 20) / block_size > 0 ? (8ll << 20) / block_size : 1;  // ~64 MiB of cf32
    const size_t chunk = (size_t)(blocks_per_chunk * block_size);
    if (c.stage_samples < chunk) {
        for (int i = 0; i < 2; i++) {
            if (c.stage_in[i]) cudaFree(c.stage_in[i]);
            if (c.stage_out[i]) cudaFree(c.stage_out[i]);
            c.stage_in[i] = nullptr;
            c.stage_out[i] = nullptr;
            QDSP_CUDA_OK(cudaMalloc(&c.stage_in[i], chunk * sizeof(float2)));   // the widest format
            QDSP_CUDA_OK(cudaMalloc((void**)&c.stage_out[i], (chunk * c.interp / c.decim + 64) * sizeof(float)));
            if (!c.ev_done[i]) QDSP_CUDA_OK(cudaEventCreateWithFlags(&c.ev_done[i], cudaEventDisableTiming));
        }
        if (!c.copy_stream) QDSP_CUDA_OK(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
        c.stage_samples = chunk;
    }
    cudaEvent_t ev_h2d[2];
    for (int i = 0; i < 2; i++) QDSP_CUDA_OK(cudaEventCreateWithFlags(&ev_h2d[i], cudaEventDisableTiming));
    const char* src = (const char*)in_host;
    const size_t E = (size_t)iq_pair_bytes(c.in_fmt);   // staged as given: 8, 4 or 2 bytes per sample cross the bus
    long long done = 0, produced = 0;
    int slot = 0;
    bool used[2] = {false, false};
    while (done < count) {
        const long long n = count - done < (long long)chunk ? count - done : (long long)chunk;
        // the slot's previous kernel + D2H must have drained before its input buffer is overwritten
        if (used[slot]) QDSP_CUDA_OK(cudaStreamWaitEvent(c.copy_stream, c.ev_done[slot], 0));
        QDSP_CUDA_OK(cudaMemcpyAsync(c.stage_in[slot], src + (size_t)done * E, (size_t)n * E, cudaMemcpyHostToDevice,
                                     c.copy_stream));
        QDSP_CUDA_OK(cudaEventRecord(ev_h2d[slot], c.copy_stream));
        QDSP_CUDA_OK(cudaStreamWaitEvent(s, ev_h2d[slot], 0));
        const long long m = c.process(c.stage_in[slot], c.stage_out[slot], nullptr, 0, n, nullptr, 0, block_size, nullptr, s);
        if (m < 0) return -1;
        c.chain.clear();   // copies and event waits go between the chunks' kernels: never overlapped
        if (m > 0)
            QDSP_CUDA_OK(cudaMemcpyAsync(audio_out_host + produced, c.stage_out[slot], (size_t)m * sizeof(float),
                                         cudaMemcpyDeviceToHost, s));
        QDSP_CUDA_OK(cudaEventRecord(c.ev_done[slot], s));
        used[slot] = true;
        produced += m;
        done += n;
        slot ^= 1;
    }
    QDSP_CUDA_OK(cudaStreamSynchronize(s));
    for (int i = 0; i < 2; i++) cudaEventDestroy(ev_h2d[i]);
    return produced;
}
long long qdsp_vfofm_process_replay(qdsp_vfofm* h, const void* in_dev, float* audio_out_dev, void* iq_out_dev,
                                    long long count, const int* blocks, int nblocks, int block_size,
                                    const float* ckpt_host, long long n_ckpt, qdsp_stream_t s_) {
    qdsp_channelizer& c = h->c;
    cudaStream_t s = as_stream(s_);
    if (c.nch != 1 || !ckpt_host) {
        set_last_error("vfofm_process_replay: bad arguments");
        return -1;
    }
    if (c.in_fmt != QDSP_CF32) {
        set_last_error("vfofm_process_replay: cf32 input only (set_input_format)");
        return -1;
    }
    if (c.part_replay.build(count, blocks, nblocks, block_size, c.interp, c.decim, s) != 0) return -1;
    if (count == 0) return 0;
    const Partition& part = c.part_replay;
    const int nb = part.view.nblocks;
    std::vector<long long> run0((size_t)nb + 1, 0);
    for (int b = 0; b < nb; b++) {
        long long cnt;
        if (blocks) cnt = part.host[b].count;
        else {
            const long long st = (long long)b * part.view.block_size;
            cnt = count - st < part.view.block_size ? count - st : part.view.block_size;
        }
        run0[b + 1] = run0[b] + (cnt + 511) / 512;
    }
    if (run0[nb] != n_ckpt) {
        set_last_error("vfofm_process_replay: %lld checkpoints given, the partition has %lld runs", n_ckpt, run0[nb]);
        return -1;
    }
    if (!c.hist_mixed.buf[0]) {
        if (c.hist_mixed.init(c.tpp, 8) != 0) return -1;
        const float z[2] = {0.f, 0.f};
        if (c.demod_replay.init(2, z) != 0) return -1;
    }
    const size_t n_out_cap = (size_t)part.total_out + 64;
    const size_t off_iq = ((size_t)count * 8 + 255) / 256 * 256;
    const size_t off_run = off_iq + (n_out_cap * 8 + 255) / 256 * 256;
    const size_t off_ck = off_run + (((size_t)nb + 1) * 8 + 255) / 256 * 256;
    if (c.replay_scratch.reserve(off_ck + (size_t)n_ckpt * 8 + 256) != 0) return -1;
    char* base = (char*)c.replay_scratch.p;
    float2* mixed = (float2*)base;
    float2* iq = iq_out_dev ? (float2*)iq_out_dev : (float2*)(base + off_iq);
    long long* run0_dev = (long long*)(base + off_run);
    float2* ck_dev = (float2*)(base + off_ck);
    QDSP_CUDA_OK(cudaMemcpyAsync(run0_dev, run0.data(), ((size_t)nb + 1) * 8, cudaMemcpyHostToDevice, s));
    QDSP_CUDA_OK(cudaMemcpyAsync(ck_dev, ckpt_host, (size_t)n_ckpt * 8, cudaMemcpyHostToDevice, s));
    QDSP_CUDA_OK(cudaStreamSynchronize(s));   // run0 / ckpt_host may be released by the caller after return
    if (launch_xlator_replay((const float2*)in_dev, mixed, part, run0_dev, ck_dev, make_float2(c.nco[0].inc_re, c.nco[0].inc_im),
                             n_ckpt, s) != 0)
        return -1;
    int rc;
    if (c.plan && c.variant != 1) {
        if (!c.plan_replay) c.plan_replay = decim_plan_create(c.taps.data(), c.T, c.decim);
        rc = launch_decim(c.plan_replay, (const float2*)c.hist_mixed.ptr(), c.hist_mixed.H, mixed, part, 0, nullptr, 0, 1, 0.0f,
                          nullptr, nullptr, iq, nullptr, 0, s);
    } else {
        rc = launch_generic_resamp<float2>((const float2*)c.hist_mixed.ptr(), c.hist_mixed.H, mixed, c.phases_dev, c.tpp, 0,
                                           part, iq, s);
    }
    if (rc != 0) return -1;
    if (c.hist_mixed.advance(mixed, count, s) != 0) return -1;
    if (part.total_out > 0) {
        if (launch_fmdemod(iq, audio_out_dev, part.total_out, c.phasor_speed, c.demod_replay.p + c.cur_replay,
                           c.demod_replay.p + (c.cur_replay ^ 1), 0, s) != 0)
            return -1;
        c.cur_replay ^= 1;
    }
    return part.total_out;
}
int qdsp_vfofm_reset(qdsp_vfofm* h) {
    qdsp_channelizer& c = h->c;
    c.chain.clear();
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    if (c.hist.reset(nullptr) != 0) return -1;
    std::vector<float> z(2 * c.nch, 0.0f);
    if (c.demod.set(z.data(), 2 * c.nch) != 0) return -1;
    c.abs_pos = 0;
    c.cur = 0;
    return 0;
}
int qdsp_vfofm_set_input_format(qdsp_vfofm* h, int fmt, float scale, float offset) {
    return h->c.set_input_format(fmt, scale, offset, "vfofm_set_input_format");
}
int qdsp_vfofm_set_variant(qdsp_vfofm* h, int variant) {
    h->c.chain.clear();
    h->c.variant = variant;
    return 0;
}
int qdsp_vfofm_seek(qdsp_vfofm* h, long long start) {
    h->c.chain.clear();
    h->c.abs_pos = start;
    return 0;
}
int qdsp_vfofm_import_tail(qdsp_vfofm* h, const void* tail_dev, int src_device, qdsp_stream_t s) {
    h->c.chain.clear();
    return import_tail_impl(h->c.hist, tail_dev, src_device, as_stream(s));
}
int qdsp_vfofm_history_len(qdsp_vfofm* h) { return h->c.hist.H; }
int qdsp_vfofm_enable_timing(qdsp_vfofm* h, int on) {
    if (on && !h->c.ev_k0) {
        QDSP_CUDA_OK(cudaEventCreate(&h->c.ev_k0));
        QDSP_CUDA_OK(cudaEventCreate(&h->c.ev_k1));
    }
    if (h->c.ring) cudaFree(h->c.ring);
    h->c.ring = nullptr;
    h->c.ring_pairs = 0;
    h->c.timing = on != 0;
    return 0;
}
// The kernel stamps its slot with %globaltimer: the first CTA's start and the last CTA's end. Launch k is reported as
// end(k) - end(k-1), the first one as end - start: completion to completion, which for launches that do not overlap is
// what an event pair around each launch measures, with nothing recorded on the stream between the launches.
int qdsp_vfofm_enable_timing_ring(qdsp_vfofm* h, int pairs) {
    if (pairs < 1) return -1;
    qdsp_channelizer& c = h->c;
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    if (c.ring) cudaFree(c.ring);
    c.ring = nullptr;
    QDSP_CUDA_OK(cudaMalloc(&c.ring, sizeof(unsigned long long) * 2 * (size_t)pairs));
    std::vector<unsigned long long> init(2 * (size_t)pairs, 0ull);
    for (int i = 0; i < pairs; i++) init[2 * (size_t)i] = ~0ull;
    QDSP_CUDA_OK(cudaMemcpy(c.ring, init.data(), sizeof(unsigned long long) * init.size(), cudaMemcpyHostToDevice));
    c.ring_pairs = pairs;
    c.ring_launches = 0;
    c.timing = true;
    return 0;
}
double qdsp_vfofm_kernel_ms_mean(qdsp_vfofm* h, int* launches) {
    qdsp_channelizer& c = h->c;
    const long long n = c.ring_launches < (long long)c.ring_pairs ? c.ring_launches : (long long)c.ring_pairs;
    if (launches) *launches = (int)n;
    if (n <= 0) return -1.0;
    std::vector<unsigned long long> t(2 * (size_t)n);
    if (cudaDeviceSynchronize() != cudaSuccess) return -1.0;
    if (cudaMemcpy(t.data(), c.ring, sizeof(unsigned long long) * t.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return -1.0;
    return (double)(t[2 * (size_t)n - 1] - t[0]) * 1e-6 / (double)n;
}
double qdsp_vfofm_kernel_ms(qdsp_vfofm* h) {
    if (!h->c.ev_k0 || h->c.ring) return -1.0;
    if (cudaEventSynchronize(h->c.ev_k1) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->c.ev_k0, h->c.ev_k1) != cudaSuccess) return -1.0;
    return (double)ms;
}

qdsp_channelizer* qdsp_channelizer_create(int nch, const float* offsets, float inSampleRate, float outSampleRate,
                                          float bandWidth, float deviation) {
    if (nch <= 0 || !offsets) {
        set_last_error("channelizer_create: bad arguments");
        return nullptr;
    }
    qdsp_channelizer* h = new (std::nothrow) qdsp_channelizer();
    if (!h) return nullptr;
    if (h->setup(nch, offsets, inSampleRate, outSampleRate, bandWidth, deviation) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_channelizer_destroy(qdsp_channelizer* h) { delete h; }
int qdsp_channelizer_design(qdsp_channelizer* h, int* tapCount, int* interp, int* decim) {
    if (tapCount) *tapCount = h->T;
    if (interp) *interp = h->interp;
    if (decim) *decim = h->decim;
    return 0;
}
long long qdsp_channelizer_process(qdsp_channelizer* h, const void* in_dev, float* audio_out_dev,
                                   long long out_stride, long long count, const int* blocks, int nblocks,
                                   int block_size, qdsp_stream_t s) {
    return h->process(in_dev, audio_out_dev, nullptr, out_stride, count, blocks, nblocks, block_size, nullptr,
                      as_stream(s));
}
int qdsp_channelizer_reset(qdsp_channelizer* h) {
    h->chain.clear();
    QDSP_CUDA_OK(cudaDeviceSynchronize());
    if (h->hist.reset(nullptr) != 0) return -1;
    std::vector<float> z(2 * h->nch, 0.0f);
    if (h->demod.set(z.data(), 2 * h->nch) != 0) return -1;
    h->abs_pos = 0;
    h->cur = 0;
    return 0;
}
int qdsp_channelizer_set_input_format(qdsp_channelizer* h, int fmt, float scale, float offset) {
    return h->set_input_format(fmt, scale, offset, "channelizer_set_input_format");
}
int qdsp_channelizer_set_variant(qdsp_channelizer* h, int variant) {
    h->chain.clear();
    h->variant = variant;
    return 0;
}
int qdsp_channelizer_seek(qdsp_channelizer* h, long long start) {
    h->chain.clear();
    h->abs_pos = start;
    return 0;
}

}  // extern "C"

// =================================================================================================
// power spectrum (an addition: the reference has none)
// =================================================================================================
struct qdsp_spectrum {
    SpectrumPlan* plan = nullptr;
};

extern "C" {

qdsp_spectrum* qdsp_spectrum_create(int fftSize, const float* window, int hop, int average) {
    if (fftSize < 64 || fftSize > 16384 || (fftSize & (fftSize - 1)) != 0 || hop < 1 || average < 1) {
        set_last_error("spectrum_create: fftSize must be a power of two in [64, 16384], hop >= 1, average >= 1 (got %d, %d, %d)",
                       fftSize, hop, average);
        return nullptr;
    }
    if (window)
        for (int i = 0; i < fftSize; i++)
            if (!isfinite(window[i])) {
                set_last_error("spectrum_create: window[%d] is not finite", i);
                return nullptr;
            }
    qdsp_spectrum* h = new (std::nothrow) qdsp_spectrum();
    if (!h) return nullptr;
    h->plan = spectrum_plan_create(fftSize, window, hop, average);
    if (!h->plan) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_spectrum_destroy(qdsp_spectrum* h) {
    if (!h) return;
    spectrum_plan_destroy(h->plan);
    delete h;
}
long long qdsp_spectrum_out_rows(qdsp_spectrum* h, long long count) { return spectrum_out_rows(h->plan, count); }
long long qdsp_spectrum_process(qdsp_spectrum* h, const void* in_dev, float* rows_out_dev, long long count, qdsp_stream_t s) {
    if (count < 0 || (reinterpret_cast<uintptr_t>(in_dev) & 7) != 0) {
        set_last_error("spectrum_process: negative count or input not aligned to 8 bytes");
        return -1;
    }
    if (count == 0) return 0;
    if (!in_dev || (!rows_out_dev && spectrum_out_rows(h->plan, count) > 0)) {
        set_last_error("spectrum_process: NULL input or output");
        return -1;
    }
    return launch_spectrum(h->plan, (const float2*)in_dev, rows_out_dev, count, as_stream(s));
}
int qdsp_spectrum_reset(qdsp_spectrum* h) {
    spectrum_plan_reset(h->plan);
    return 0;
}

}  // extern "C"

// =================================================================================================
// recurrent blocks
// =================================================================================================
struct qdsp_deemp {
    float alpha = 0.0f;
    DevState st;  // [4]: in (l, r), out (l, r)
};
struct qdsp_agc {
    float corrected = 0.0f;
    DevState st;  // [1]: level
    Partition part;
    Scratch scratch;
};
struct qdsp_cagc {
    float set_point = 1.0f, max_gain = 65535.0f, rate = 1e-3f;
    DevState st;  // [1]: gain
    Scratch scratch;
};
struct qdsp_ffagc {
    int dtype = QDSP_CF32;
    History hist;     // up to 1023 pending elements (right-aligned)
    int pending = 0;  // how many of them are real
};
struct qdsp_costas {
    int order = 4;
    float alpha = 0.0f, beta = 0.0f;
    // measured on B200 (2^26 QPSK samples, tools/_costas_sweep.py): (4096, 4096) 38 GS/s, (2048, 2048) 49 GS/s with the same
    // 4e-6 error against the sequential loop; 1536 warm-up samples: 53 GS/s but 2e-5; 1024: 1e-3 (not merged)
    int chunk = 2048, warmup = 2048;
    bool chunk_user = false;   // set_chunking(): keep; otherwise long calls use 4096-sample chunks
    DevState st;   // [4] state + [1] residual
    Scratch scratch;
};

extern "C" {

qdsp_deemp* qdsp_deemp_create(float sampleRate, float tau) {
    qdsp_deemp* h = new (std::nothrow) qdsp_deemp();
    if (!h) return nullptr;
    const float dt = 1.0f / sampleRate;  // filter.h:102-103
    h->alpha = dt / (tau + dt);
    const float z[4] = {0, 0, 0, 0};
    if (h->st.init(4, z) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_deemp_destroy(qdsp_deemp* h) { delete h; }
// the chunk-with-warm-up recurrences re-read input that a neighbouring chunk's thread overwrites when out aliases in
long long qdsp_deemp_process(qdsp_deemp* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count > 0 && ranges_overlap(in_dev, (size_t)count * 8, out_dev, (size_t)count * 8)) {
        set_last_error("deemp_process: in and out must not overlap (chunked scan with warm-up re-reads the input)");
        return -1;
    }
    if (launch_deemp((const float2*)in_dev, (float2*)out_dev, count, h->alpha, h->st.p, nullptr, 0, as_stream(s)) != 0)
        return -1;
    return count;
}
int qdsp_deemp_set_params(qdsp_deemp* h, float sampleRate, float tau) {
    // like the reference's setters (filter.h:117-127) only scalars change: handle and device state survive, the
    // next process() call picks the new alpha up
    const float dt = 1.0f / sampleRate;
    h->alpha = dt / (tau + dt);
    return 0;
}
int qdsp_deemp_get_state(qdsp_deemp* h, float* lastL, float* lastR) {
    float v[2];
    if (h->st.get(v, 2) != 0) return -1;
    *lastL = v[0];
    *lastR = v[1];
    return 0;
}
int qdsp_deemp_set_state(qdsp_deemp* h, float lastL, float lastR) {
    const float v[2] = {lastL, lastR};
    return h->st.set(v, 2);
}

qdsp_agc* qdsp_agc_create(float fallRate, float sampleRate) {
    qdsp_agc* h = new (std::nothrow) qdsp_agc();
    if (!h) return nullptr;
    h->corrected = fallRate / sampleRate;  // processing.h:92
    const float z = 0.0f;                  // level = 0, processing.h:140
    if (h->st.init(1, &z) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_agc_destroy(qdsp_agc* h) { delete h; }
long long qdsp_agc_process(qdsp_agc* h, const float* in_dev, float* out_dev, long long count, const int* blocks,
                           int nblocks, int block_size, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, 1, 1, s) != 0) return -1;
    const int nb = h->part.view.nblocks;
    if (nb == 0) return 0;
    // long batches of large run() blocks: one persistent launch, the second read of every chunk served by L2
    if (const int cb = agc_fused_chunk_blocks(h->part, in_dev, out_dev)) {
        if (h->scratch.reserve(agc_fused_scratch_bytes(cb)) != 0) return -1;
        if (launch_agc_fused(in_dev, out_dev, h->part, h->corrected, h->st.p, h->scratch.p, cb, s) == 0) return count;
        cudaGetLastError();     // a refused cooperative launch has run nothing: take the three-kernel path below
    }
    // scratch: [nb][32] partial maxima of the block-max pass, then [nb] reciprocal levels
    if (h->scratch.reserve(sizeof(float) * 33 * (size_t)nb + 64) != 0) return -1;
    float* bm = (float*)h->scratch.p;
    if (launch_agc(in_dev, out_dev, h->part, h->corrected, h->st.p, bm, bm + 32 * (size_t)nb, s) != 0) return -1;
    return count;
}
int qdsp_agc_set_params(qdsp_agc* h, float fallRate, float sampleRate) {   // processing.h:101-113
    h->corrected = fallRate / sampleRate;
    return 0;
}
int qdsp_agc_get_state(qdsp_agc* h, float* level) { return h->st.get(level, 1); }
int qdsp_agc_set_state(qdsp_agc* h, float level) { return h->st.set(&level, 1); }

qdsp_cagc* qdsp_cagc_create(float setPoint, float maxGain, float rate) {
    qdsp_cagc* h = new (std::nothrow) qdsp_cagc();
    if (!h) return nullptr;
    h->set_point = setPoint;
    h->max_gain = maxGain;
    h->rate = rate;
    const float one = 1.0f;  // _gain = 1, processing.h:291
    if (h->st.init(1, &one) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_cagc_destroy(qdsp_cagc* h) { delete h; }
long long qdsp_cagc_process(qdsp_cagc* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (h->scratch.reserve(scan_scratch_bytes(count)) != 0) return -1;
    if (launch_cagc((const float2*)in_dev, (float2*)out_dev, count, h->set_point, h->max_gain, h->rate, h->st.p,
                    h->scratch.p, h->scratch.cap, as_stream(s)) != 0)
        return -1;
    return count;
}
int qdsp_cagc_set_params(qdsp_cagc* h, float setPoint, float maxGain, float rate) {   // processing.h:258-269
    h->set_point = setPoint;
    h->max_gain = maxGain;
    h->rate = rate;
    return 0;
}
int qdsp_cagc_get_state(qdsp_cagc* h, float* gain) { return h->st.get(gain, 1); }
int qdsp_cagc_set_state(qdsp_cagc* h, float gain) { return h->st.set(&gain, 1); }

qdsp_ffagc* qdsp_ffagc_create(int dtype) {
    if (!real_or_complex(dtype, "ffagc_create")) return nullptr;
    qdsp_ffagc* h = new (std::nothrow) qdsp_ffagc();
    if (!h) return nullptr;
    h->dtype = dtype;
    if (h->hist.init(1023, dtype == QDSP_CF32 ? 8 : 4) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_ffagc_destroy(qdsp_ffagc* h) {
    if (!h) return;
    h->hist.release();
    delete h;
}
long long qdsp_ffagc_process(qdsp_ffagc* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (count < 0) return -1;
    if (count == 0) return 0;
    // virtual stream = pending ++ in; outputs while a full 1024-window exists (processing.h:189-193)
    const long long avail = h->pending + count;
    const long long n_valid = avail >= 1024 ? avail - 1023 : 0;
    if (n_valid > 0) {
        // the kernel addresses the pending samples as virtual indices -pending..-1 (right-aligned tail)
        const char* hp = (const char*)h->hist.ptr() + (size_t)(h->hist.H - h->pending) * h->hist.elem;
        if (launch_ffagc(hp, h->pending, in_dev, out_dev, n_valid, h->dtype == QDSP_CF32, s) != 0) return -1;
    }
    if (h->hist.advance(in_dev, count, s) != 0) return -1;
    h->pending = (int)(avail - n_valid < 1023 ? avail - n_valid : 1023);
    return n_valid;
}

qdsp_costas* qdsp_costas_create(int order, float loopBandwidth) {
    if (order != 2 && order != 4 && order != 8) {
        set_last_error("costas_create: order must be 2, 4 or 8");
        return nullptr;
    }
    qdsp_costas* h = new (std::nothrow) qdsp_costas();
    if (!h) return nullptr;
    h->order = order;
    // pll.h:20-23 (float/double mix as written there)
    const float damp = sqrtf(2.0f) / 2.0f;
    const float den = (float)(1.0 + 2.0 * damp * loopBandwidth + loopBandwidth * loopBandwidth);
    h->alpha = (4 * damp * loopBandwidth) / den;
    h->beta = (4 * loopBandwidth * loopBandwidth) / den;
    // default warm-up: the chunk walks start from (carried frequency, phase 0) and must have merged with the true
    // trajectory when their chunk begins. Measured against the sequential loop at loopBandwidth 0.004 (700 001 samples):
    // ORDER 4 needs 2048 samples (4e-6), the BPSK detector (error = re * im) 4096, the 8-PSK detector (the smaller branch
    // weighted by sqrt(2) - 1) 8192; the loop's time constant scales with 1 / loopBandwidth. `qdsp_costas_last_residual`
    // reports the largest boundary mismatch of every call: it is the validity check for other signals / bandwidths.
    {
        const double scale = order == 2 ? 2.0 : (order == 8 ? 4.0 : 1.0);
        double w = 8.192 / (loopBandwidth > 1e-6f ? (double)loopBandwidth : 1e-6) * scale;
        if (w < 256.0) w = 256.0;
        if (w > 65536.0) w = 65536.0;
        h->warmup = ((int)w + 15) / 16 * 16;
        h->chunk = h->warmup > 2048 ? h->warmup : 2048;
    }
    const float init[5] = {0.0f, 0.0f, 1.0f, 0.0f, 0.0f};
    if (h->st.init(5, init) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_costas_destroy(qdsp_costas* h) { delete h; }
long long qdsp_costas_process(qdsp_costas* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (ranges_overlap(in_dev, (size_t)count * 8, out_dev, (size_t)count * 8)) {
        set_last_error("costas_process: in and out must not overlap (chunked scan with warm-up re-reads the input)");
        return -1;
    }
    // the work is (1 + warmup / chunk) x the sequential loop's: with >= 32768 chunks of 4096 samples the machine is still full
    // (B200, 2^28 QPSK samples, GS/s: chunk 2048: 95, 3072: 95, 4096: 110, 8192: 103; warm-up 2048 throughout)
    const int chunk = (!h->chunk_user && count >= (1ll << 27) && h->chunk < 4096) ? 4096 : h->chunk;
    if (h->scratch.reserve(costas_scratch_bytes(count, chunk)) != 0) return -1;
    if (launch_costas((const float2*)in_dev, (float2*)out_dev, count, h->order, h->alpha, h->beta, h->st.p, chunk,
                      h->warmup, h->scratch.p, h->scratch.cap, h->st.p + 4, as_stream(s)) != 0)
        return -1;
    return count;
}
int qdsp_costas_get_state(qdsp_costas* h, float state[4]) { return h->st.get(state, 4); }
int qdsp_costas_set_state(qdsp_costas* h, const float state[4]) { return h->st.set(state, 4); }
int qdsp_costas_set_chunking(qdsp_costas* h, int chunk, int warmup) {
    if (chunk < 16 || warmup < 0 || (chunk % 16) != 0 || (warmup % 16) != 0) {
        set_last_error("costas_set_chunking: chunk must be a positive multiple of 16, warmup a non-negative multiple of 16");
        return -1;
    }
    h->chunk = chunk;
    h->warmup = warmup;
    h->chunk_user = true;
    return 0;
}
float qdsp_costas_last_residual(qdsp_costas* h) {
    float r = -1.0f;
    h->st.get(&r, 1, 4);
    return r;
}

// =================================================================================================
// StereoFMDemod (hierarchical): FloatFMDemod -> FIR<float> pilot filter -> AGC -> matrix
// =================================================================================================
}  // extern "C"
struct qdsp_stereofm {
    qdsp_fmdemod* fm = nullptr;
    qdsp_fir* fir = nullptr;
    qdsp_agc* agc = nullptr;
    Scratch scratch;   // mpx | pilot | agc'd pilot (3 x count floats)
};
extern "C" {

qdsp_stereofm* qdsp_stereofm_create(float sampleRate, float deviation) {
    qdsp_stereofm* h = new (std::nothrow) qdsp_stereofm();
    if (!h) return nullptr;
    h->fm = qdsp_fmdemod_create(sampleRate, deviation, 0);
    // win.init(1000, 1000, 19000, sampleRate), demodulator.h:212
    const int T = qdsp_blackman_tap_count(1000.0f, 1000.0f, sampleRate);
    std::vector<float> taps(T);
    qdsp_blackman_bandpass_taps(1000.0f, 1000.0f, 19000.0f, sampleRate, taps.data(), T, 1.0f);
    h->fir = qdsp_fir_create(QDSP_F32, taps.data(), T);
    h->agc = qdsp_agc_create(20.0f, sampleRate);   // agc.init(&filter.out, 20.0f, sampleRate), :214
    if (!h->fm || !h->fir || !h->agc) {
        qdsp_stereofm_destroy(h);
        return nullptr;
    }
    return h;
}
void qdsp_stereofm_destroy(qdsp_stereofm* h) {
    if (!h) return;
    if (h->fm) qdsp_fmdemod_destroy(h->fm);
    if (h->fir) qdsp_fir_destroy(h->fir);
    if (h->agc) qdsp_agc_destroy(h->agc);
    delete h;
}
long long qdsp_stereofm_process(qdsp_stereofm* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                                int nblocks, int block_size, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (h->scratch.reserve(sizeof(float) * 3 * (size_t)count + 256) != 0) return -1;
    float* mpx = (float*)h->scratch.p;
    float* pil = mpx + count;
    float* lvl = pil + count;
    if (qdsp_fmdemod_process(h->fm, in_dev, mpx, count, s) < 0) return -1;
    if (qdsp_fir_process(h->fir, mpx, pil, count, s) < 0) return -1;
    if (qdsp_agc_process(h->agc, pil, lvl, count, blocks, nblocks, block_size, s) < 0) return -1;
    if (launch_stereo_matrix(mpx, lvl, (float2*)out_dev, count, as_stream(s)) != 0) return -1;
    return count;
}
long long qdsp_stereo_matrix_process(const float* mpx_dev, const float* pilot_dev, void* out_dev, long long count,
                                     qdsp_stream_t s) {
    if (count < 0) return -1;
    if (launch_stereo_matrix(mpx_dev, pilot_dev, (float2*)out_dev, count, as_stream(s)) != 0) return -1;
    return count;
}

// =================================================================================================
// synthetic IQ + probes
// =================================================================================================
int qdsp_synth_uniform_cf32(void* out_dev, unsigned long long seed, long long start, long long count,
                            qdsp_stream_t s) {
    return launch_synth_uniform((float2*)out_dev, seed, start, count, as_stream(s));
}
int qdsp_synth_fm_cf32(void* out_dev, long long start, long long count, long long fs, long long fc, long long fm,
                       double dev, double amp, double noise_amp, unsigned long long noise_seed, qdsp_stream_t s) {
    return launch_synth_fm((float2*)out_dev, start, count, fs, fc, fm, dev, amp, noise_amp, noise_seed, as_stream(s));
}
int qdsp_synth_comb_cf32(void* out_dev, long long start, long long count, long long fs, int nch, long long spacing,
                         double dev, double amp, double noise_amp, unsigned long long noise_seed, qdsp_stream_t s) {
    return launch_synth_comb((float2*)out_dev, start, count, fs, nch, spacing, dev, amp, noise_amp, noise_seed, as_stream(s));
}
int qdsp_synth_qpsk_cf32(void* out_dev, long long start, long long count, unsigned long long seed, int sps, double freq_off,
                         double sigma, double am_depth, long long am_period, qdsp_stream_t s) {
    return launch_synth_qpsk((float2*)out_dev, start, count, seed, sps, freq_off, sigma, am_depth, am_period, as_stream(s));
}
double qdsp_measure_fp32_peak(int packed, int iters) { return run_fp32_peak(packed, iters); }

}  // extern "C"

// =================================================================================================
// element-wise / layout / per-block-statistic blocks ("next" rows): math.h, audio.h, convertion.h,
// processing.h Volume / DelayImag / Squelch / Threshold, demodulator.h AMDemod / SSBDemod
// =================================================================================================
struct qdsp_delayimag {
    DevState st;  // [2] ping-pong lastIm
    int cur = 0;
};
struct qdsp_amdemod {
    Partition part;
    Scratch scratch;
};
struct qdsp_squelch {
    float level = -50.0f;  // processing.h:486
    Partition part;
    Scratch scratch;
};
struct qdsp_sinesource {
    Nco nco;
    float2 inc_pow[3];
    void configure(float sampleRate, float freq) {
        nco.set_freq(sampleRate, freq);   // source.h:20 is the translator's expression (processing.h:21)
        const double th = atan2((double)nco.inc_im, (double)nco.inc_re);
        for (int j = 1; j <= 3; j++) inc_pow[j - 1] = make_float2((float)cos(th * j), (float)sin(th * j));
    }
};
struct qdsp_ssbdemod {
    Nco nco;
    float2 inc_pow[3];
    void configure(float sampleRate, float bandWidth, int mode) {
        // demodulator.h:403-412: float expressions, std::cos / std::sin float overloads
        float re = 1.0f, im = 0.0f;
        if (mode == QDSP_SSB_USB) {
            re = cosf((bandWidth / sampleRate) * QDSP_FL_M_PI);
            im = sinf((bandWidth / sampleRate) * QDSP_FL_M_PI);
        } else if (mode == QDSP_SSB_LSB) {
            re = cosf(-(bandWidth / sampleRate) * QDSP_FL_M_PI);
            im = sinf(-(bandWidth / sampleRate) * QDSP_FL_M_PI);
        }
        nco.set_inc(re, im);
        const double th = atan2((double)im, (double)re);
        for (int j = 1; j <= 3; j++) inc_pow[j - 1] = make_float2((float)cos(th * j), (float)sin(th * j));
    }
};

extern "C" {

long long qdsp_math_process(int op, int dtype, const void* a_dev, const void* b_dev, void* out_dev, long long count,
                            qdsp_stream_t s) {
    if (count < 0 || !real_or_complex(dtype, "math_process")) return -1;
    // math.h:32-37, 79-84, 126-131: complex/stereo add and subtract are float add/subtract over 2*count floats;
    // only Multiply<complex_t> is a complex product
    const long long nf = dtype == QDSP_CF32 ? 2 * count : count;
    if (launch_math(op, dtype == QDSP_CF32, (const float*)a_dev, (const float*)b_dev, (float*)out_dev, nf, as_stream(s)) != 0)
        return -1;
    return count;
}

long long qdsp_layout_process(int op, const void* in0_dev, const void* in1_dev, void* out0_dev, void* out1_dev,
                              long long count, qdsp_stream_t s_) {
    if (count < 0) return -1;
    cudaStream_t s = as_stream(s_);
    const float* i0 = (const float*)in0_dev;
    const float* i1 = (const float*)in1_dev;
    float* o0 = (float*)out0_dev;
    float* o1 = (float*)out1_dev;
    int rc = 0;
    switch (op) {
        case QDSP_LAYOUT_MONO_TO_STEREO: rc = launch_layout(0, i0, i0, o0, nullptr, count, s); break;        // audio.h:30
        case QDSP_LAYOUT_CHANNELS_TO_STEREO: rc = launch_layout(0, i0, i1, o0, nullptr, count, s); break;    // audio.h:80
        case QDSP_LAYOUT_STEREO_TO_MONO: rc = launch_layout(1, i0, nullptr, o0, nullptr, count, s); break;   // audio.h:129-131
        case QDSP_LAYOUT_STEREO_TO_CHANNELS: rc = launch_layout(2, i0, nullptr, o0, o1, count, s); break;    // audio.h:173
        case QDSP_LAYOUT_COMPLEX_TO_STEREO:                                                                  // convertion.h:32
            if (count > 0 && cudaMemcpyAsync(o0, i0, (size_t)count * 8, cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
                set_last_error("layout: device copy failed");
                rc = -1;
            }
            break;
        case QDSP_LAYOUT_COMPLEX_TO_REAL: rc = launch_layout(2, i0, nullptr, o0, nullptr, count, s); break;  // convertion.h:71
        case QDSP_LAYOUT_COMPLEX_TO_IMAG: rc = launch_layout(2, i0, nullptr, nullptr, o0, count, s); break;  // convertion.h:110
        case QDSP_LAYOUT_REAL_TO_COMPLEX: rc = launch_layout(0, i0, nullptr, o0, nullptr, count, s); break;  // convertion.h:157
        default:
            set_last_error("layout: unknown op %d", op);
            rc = -1;
    }
    return rc == 0 ? count : -1;
}

float qdsp_volume_level(float volume) { return powf(volume, 2); }   // Volume::setVolume, processing.h:373-374
long long qdsp_volume_process(int dtype, float level, int muted, const void* in_dev, void* out_dev, long long count,
                              qdsp_stream_t s) {
    if (count < 0 || !real_or_complex(dtype, "volume_process")) return -1;
    const long long nf = dtype == QDSP_CF32 ? 2 * count : count;
    if (muted) {   // processing.h:392-399
        if (count > 0 && cudaMemsetAsync(out_dev, 0, (size_t)nf * 4, as_stream(s)) != cudaSuccess) {
            set_last_error("volume: memset failed");
            return -1;
        }
        return count;
    }
    if (launch_scale((const float*)in_dev, (float*)out_dev, nf, level, as_stream(s)) != 0) return -1;
    return count;
}

long long qdsp_threshold_process(const float* in_dev, unsigned char* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (launch_threshold(in_dev, out_dev, count, as_stream(s)) != 0) return -1;
    return count;
}

qdsp_delayimag* qdsp_delayimag_create(void) {
    qdsp_delayimag* h = new (std::nothrow) qdsp_delayimag();
    if (!h) return nullptr;
    const float z[2] = {0.0f, 0.0f};   // lastIm = 0, processing.h:343
    if (h->st.init(2, z) != 0) {
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_delayimag_destroy(qdsp_delayimag* h) { delete h; }
long long qdsp_delayimag_process(qdsp_delayimag* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (count == 0) return 0;
    if (launch_delay_imag((const float2*)in_dev, (float2*)out_dev, count, h->st.p + h->cur, h->st.p + (h->cur ^ 1),
                          as_stream(s)) != 0)
        return -1;
    h->cur ^= 1;
    return count;
}
int qdsp_delayimag_get_state(qdsp_delayimag* h, float* lastIm) { return h->st.get(lastIm, 1, h->cur); }
int qdsp_delayimag_set_state(qdsp_delayimag* h, float lastIm) { return h->st.set(&lastIm, 1, h->cur); }

qdsp_amdemod* qdsp_amdemod_create(void) { return new (std::nothrow) qdsp_amdemod(); }
void qdsp_amdemod_destroy(qdsp_amdemod* h) { delete h; }
long long qdsp_amdemod_process(qdsp_amdemod* h, const void* in_dev, float* out_dev, long long count, const int* blocks,
                               int nblocks, int block_size, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, 1, 1, s) != 0) return -1;
    const int nb = h->part.view.nblocks;
    if (nb == 0) return 0;
    if (h->scratch.reserve(mag_scratch_bytes(nb)) != 0) return -1;
    if (launch_amdemod((const float2*)in_dev, out_dev, h->part, (double*)h->scratch.p, s) != 0) return -1;
    return count;
}

qdsp_squelch* qdsp_squelch_create(float level) {
    qdsp_squelch* h = new (std::nothrow) qdsp_squelch();
    if (h) h->level = level;
    return h;
}
void qdsp_squelch_destroy(qdsp_squelch* h) { delete h; }
void qdsp_squelch_set_level(qdsp_squelch* h, float level) { h->level = level; }
float qdsp_squelch_get_level(qdsp_squelch* h) { return h->level; }
long long qdsp_squelch_process(qdsp_squelch* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                               int nblocks, int block_size, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, 1, 1, s) != 0) return -1;
    const int nb = h->part.view.nblocks;
    if (nb == 0) return 0;
    if (h->scratch.reserve(mag_scratch_bytes(nb)) != 0) return -1;
    if (launch_squelch((const float2*)in_dev, (float2*)out_dev, h->part, (double*)h->scratch.p, h->level, s) != 0) return -1;
    return count;
}

qdsp_ssbdemod* qdsp_ssbdemod_create(float sampleRate, float bandWidth, int mode) {
    qdsp_ssbdemod* h = new (std::nothrow) qdsp_ssbdemod();
    if (!h) return nullptr;
    h->configure(sampleRate, bandWidth, mode);
    h->nco.phase = 0;   // phase = (1, 0), demodulator.h:401
    return h;
}
void qdsp_ssbdemod_destroy(qdsp_ssbdemod* h) { delete h; }
int qdsp_ssbdemod_configure(qdsp_ssbdemod* h, float sampleRate, float bandWidth, int mode) {
    h->configure(sampleRate, bandWidth, mode);
    return 0;
}
void qdsp_ssbdemod_get_phase_delta(qdsp_ssbdemod* h, float* re, float* im) {
    *re = h->nco.inc_re;
    *im = h->nco.inc_im;
}
void qdsp_ssbdemod_get_phase(qdsp_ssbdemod* h, float* re, float* im) { h->nco.get_phase(re, im); }
void qdsp_ssbdemod_set_phase(qdsp_ssbdemod* h, float re, float im) { h->nco.set_phase(re, im); }
long long qdsp_ssbdemod_process(qdsp_ssbdemod* h, const void* in_dev, float* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (launch_ssb((const float2*)in_dev, out_dev, count, h->nco.phase, h->nco.step, h->inc_pow[0], h->inc_pow[1],
                   h->inc_pow[2], as_stream(s)) != 0)
        return -1;
    h->nco.advance(count);
    return count;
}

qdsp_sinesource* qdsp_sinesource_create(float sampleRate, float freq) {
    qdsp_sinesource* h = new (std::nothrow) qdsp_sinesource();
    if (!h) return nullptr;
    h->configure(sampleRate, freq);
    h->nco.phase = 0;   // phase = (1, 0), source.h:19
    return h;
}
void qdsp_sinesource_destroy(qdsp_sinesource* h) { delete h; }
int qdsp_sinesource_configure(qdsp_sinesource* h, float sampleRate, float freq) {
    h->configure(sampleRate, freq);
    return 0;
}
void qdsp_sinesource_get_phase(qdsp_sinesource* h, float* re, float* im) { h->nco.get_phase(re, im); }
void qdsp_sinesource_set_phase(qdsp_sinesource* h, float re, float im) { h->nco.set_phase(re, im); }
long long qdsp_sinesource_process(qdsp_sinesource* h, void* out_dev, long long count, qdsp_stream_t s) {
    if (count < 0) return -1;
    if (launch_sine((float2*)out_dev, count, h->nco.phase, h->nco.step, h->inc_pow[0], h->inc_pow[1], h->inc_pow[2],
                    as_stream(s)) != 0)
        return -1;
    h->nco.advance(count);
    return count;
}

}  // extern "C"

// =================================================================================================
// MMClockRecovery<float | complex_t> ("next" row), src/dsp/clock_recovery.h:68-243
// =================================================================================================
struct qdsp_mm {
    int dtype = QDSP_CF32;
    float omega = 1.0f, gainOmega = 0.001f, muGain = 1.0f, rel = 0.005f;
    float omegaMin = 1.0f, omegaMax = 1.0f;
    DevState st;             // 44 floats, layout of oracle/port.c port_mm
    float* taps_dev = nullptr;
    Partition part;
    Scratch scratch;         // the total output count (long long) at byte 0, [nblocks] per-block counts at byte 16
    ~qdsp_mm() {
        if (taps_dev) cudaFree(taps_dev);
    }
};

extern "C" {

qdsp_mm* qdsp_mm_create(int dtype, float omega, float gainOmega, float muGain, float omegaRelLimit,
                        const float* interp_taps) {
    if (!real_or_complex(dtype, "mm_create")) return nullptr;
    if (!interp_taps) {
        set_last_error("qdsp_mm_create: the 129 x 8 interpolator table is required");
        return nullptr;
    }
    qdsp_mm* h = new (std::nothrow) qdsp_mm();
    if (!h) return nullptr;
    h->dtype = dtype;
    h->omega = omega;
    h->gainOmega = gainOmega;
    h->muGain = muGain;
    h->rel = omegaRelLimit;
    h->omegaMin = omega - (omega * omegaRelLimit);   // clock_recovery.h:83-84
    h->omegaMax = omega + (omega * omegaRelLimit);
    float st[44] = {0};
    st[0] = 0.5f;    // _mu, clock_recovery.h:234
    st[1] = omega;   // _dynOmega = _omega, :85
    if (h->st.init(44, st) != 0 || cudaMalloc(&h->taps_dev, sizeof(float) * 129 * 8) != cudaSuccess ||
        cudaMemcpy(h->taps_dev, interp_taps, sizeof(float) * 129 * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("qdsp_mm_create: device allocation failed");
        delete h;
        return nullptr;
    }
    return h;
}
void qdsp_mm_destroy(qdsp_mm* h) { delete h; }
int qdsp_mm_set_omega(qdsp_mm* h, float omega, float omegaRelLimit) {
    // MMClockRecovery::setOmega, clock_recovery.h:90-97: the limits are recomputed from the OLD omega and relLimit
    // members before omega is replaced (a reference quirk, kept); dynOmega restarts at the new omega
    h->omegaMin = h->omega - (h->omega * h->rel);
    h->omegaMax = h->omega + (h->omega * h->rel);
    h->omega = omega;
    (void)omegaRelLimit;
    return h->st.set(&omega, 1, 1);
}
int qdsp_mm_set_gains(qdsp_mm* h, float gainOmega, float muGain) {   // :99-104
    h->gainOmega = gainOmega;
    h->muGain = muGain;
    return 0;
}
int qdsp_mm_set_omega_rel_limit(qdsp_mm* h, float omegaRelLimit) {   // :106-112
    h->rel = omegaRelLimit;
    h->omegaMin = h->omega - (h->omega * h->rel);
    h->omegaMax = h->omega + (h->omega * h->rel);
    return 0;
}
int qdsp_mm_get_state(qdsp_mm* h, float state[44]) { return h->st.get(state, 44); }
int qdsp_mm_set_state(qdsp_mm* h, const float state[44]) { return h->st.set(state, 44); }
long long qdsp_mm_max_out(qdsp_mm* h, long long count) {
    // per run() block the reference caps the output count at 2 * omega * count (:135); with omega >= 1 the loop ends
    // on the input first: count / omegaMin + 1 symbols per block at most
    const double per = h->omegaMin > 0.5f ? 1.0 / (double)h->omegaMin : 2.0;
    return (long long)((double)count * per) + 16;
}
long long qdsp_mm_process(qdsp_mm* h, const void* in_dev, void* out_dev, long long count, const int* blocks, int nblocks,
                          int block_size, int* out_counts, qdsp_stream_t s_) {
    cudaStream_t s = as_stream(s_);
    if (h->part.build(count, blocks, nblocks, block_size, 1, 1, s) != 0) return -1;
    const int nb = h->part.view.nblocks;
    if (nb == 0) return 0;
    if (h->scratch.reserve(sizeof(int) * (size_t)nb + 32) != 0) return -1;
    long long* total_dev = (long long*)h->scratch.p;
    int* oc_dev = (int*)((char*)h->scratch.p + 16);
    if (launch_mm(h->dtype == QDSP_CF32, in_dev, h->part, h->taps_dev, h->omega, h->gainOmega, h->muGain, h->omegaMin,
                  h->omegaMax, h->st.p, out_dev, oc_dev, total_dev, s) != 0)
        return -1;
    // the output count is data dependent: this call waits for the kernel
    long long total = 0;
    QDSP_CUDA_OK(cudaMemcpyAsync(&total, total_dev, sizeof(total), cudaMemcpyDeviceToHost, s));
    if (out_counts) QDSP_CUDA_OK(cudaMemcpyAsync(out_counts, oc_dev, sizeof(int) * (size_t)nb, cudaMemcpyDeviceToHost, s));
    QDSP_CUDA_OK(cudaStreamSynchronize(s));
    return total;
}

}  // extern "C"

