// qdsp_b200/csrc/internal.cuh — host/device plumbing shared by the kernel files of libqdsp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <atomic>
#include <vector>
#include "common.cuh"
#include "../../include/qdsp_b200.h"

namespace qdsp {

extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
#define QDSP_LAUNCH_OK()                                                                     \
    do {                                                                                     \
        qdsp::count_launch();                                                                \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess) {                                                             \
            qdsp::set_last_error("%s:%d launch -> %s", __FILE__, __LINE__,                   \
                                 cudaGetErrorString(_e));                                    \
            return -1;                                                                       \
        }                                                                                    \
    } while (0)

inline cudaStream_t as_stream(qdsp_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Launches kern(*arg) (one kernel-parameter struct). overlap: programmatic dependent launch -- the grid may start while
// the previous grid of the stream drains, the kernel orders what it shares with it by pdl_wait() (decim_common.cuh).
// QDSP_PDL=0 never overlaps: the serialized reference of the overlapped-call tests.
inline cudaError_t launch_ex(const void* kern, dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool overlap, void* arg) {
    static const bool pdl = getenv("QDSP_PDL") ? atoi(getenv("QDSP_PDL")) != 0 : true;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (overlap && pdl) ? 1 : 0;
    void* args[1] = {arg};
    return cudaLaunchKernelExC(&cfg, kern, args);
}

// ---- block partition of a batch of run() calls ------------------------------------------------
// The reference restarts the resampler schedule (and the AGC decay) at every run() call, so the
// result is a function of (contiguous stream, partition). A partition is either uniform
// (block_size, last block short) or an explicit table living in device memory.
struct BlkInfo {
    long long in_start;   // S_b: first input sample of the block (relative to this call's input)
    long long out_start;  // O_b: first output of the block (relative to this call's output)
    int count;            // input samples in the block
    int out_count;        // outputs of the block: (count * I) / D
};
struct PartitionDev {
    const BlkInfo* table;  // explicit table, or nullptr for the uniform closed form
    long long total;       // total input samples
    long long total_out;   // total outputs of the batch
    int nblocks;
    int block_size;        // uniform: size of every block but the last
    int interp, decim;
    __device__ __forceinline__ BlkInfo get(int b) const {
        if (table) return table[b];
        BlkInfo r;
        r.in_start = (long long)b * block_size;
        const long long rem = total - r.in_start;
        r.count = rem < block_size ? (int)rem : block_size;
        const long long per = ((long long)block_size * interp) / decim;
        r.out_start = (long long)b * per;
        r.out_count = (int)(((long long)r.count * interp) / decim);
        return r;
    }
};

// Host mirror; owns the device table for explicit partitions (re-uploaded only when it changes).
struct Partition {
    std::vector<BlkInfo> host;
    std::vector<int> sizes;     // explicit sizes last uploaded
    BlkInfo* dev = nullptr;
    size_t dev_cap = 0;
    long long total_out = 0;
    int max_out = 0;            // largest per-block output count
    int max_count = 0;
    PartitionDev view{};
    // returns 0 / -1
    int build(long long count, const int* blocks, int nblocks, int block_size, int interp, int decim,
              cudaStream_t s);
    ~Partition();
};

// ---- double-buffered history tail ---------------------------------------------------------------
// hist holds the last H elements of the stream seen so far (zeros initially), i.e. the reference's
// `memmove(buffer, &buffer[count], H)` (filter.h:71 / resampling.h:129).
struct History {
    void* buf[2] = {nullptr, nullptr};
    int cur = 0;
    int H = 0;
    int elem = 8;
    int init(int H_, int elem_bytes);
    void release();
    const void* ptr() const { return buf[cur]; }
    int advance(const void* in_dev, long long count, cudaStream_t s);  // after processing `count` new elements
    int reset(cudaStream_t s);
};

// Element traits for the two stream element types.
template <typename T> struct Elem;
template <> struct Elem<float> {
    static __device__ __forceinline__ float zero() { return 0.0f; }
    static __device__ __forceinline__ float mac(float x, float t, float acc) { return fmaf(x, t, acc); }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
};
template <> struct Elem<float2> {
    static __device__ __forceinline__ float2 zero() { return make_float2(0.0f, 0.0f); }
    static __device__ __forceinline__ float2 mac(float2 x, float t, float2 acc) {
        return make_float2(fmaf(x.x, t, acc.x), fmaf(x.y, t, acc.y));
    }
    static __device__ __forceinline__ float2 add(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
};

// Virtual stream = history ++ this call's input; index i in [-H, count).
template <typename T> struct VStream {
    const T* hist;
    const T* in;
    int H;
    __device__ __forceinline__ T at(long long i) const {
        if (i >= 0) return in[i];
        if (i >= -(long long)H) return hist[H + i];
        return Elem<T>::zero();
    }
};

// ---- integer IQ input (QDSP_CS16 / QDSP_CS8 / QDSP_CU8, include/qdsp_b200.h): bytes per (re, im) pair --------------
inline int iq_pair_bytes(int fmt) {
    return fmt == QDSP_CF32 ? 8 : fmt == QDSP_CS16 ? 4 : (fmt == QDSP_CS8 || fmt == QDSP_CU8) ? 2 : 0;
}
struct IqConv {
    float scale, offset;
};

// ---- NCO bookkeeping (host) ----------------------------------------------------------------------
// phase(n) = phase0 * exp(j*n*theta), theta = arg(phaseDelta) of the reference's float32 phasor
// increment, kept as 64-bit fixed-point turns so any sample index is reachable in O(1).
struct Nco {
    float inc_re = 1.0f, inc_im = 0.0f;  // the reference's phaseDelta (processing.h:21)
    uint64_t step = 0;                    // theta in turns * 2^64
    uint64_t phase = 0;                   // current phase in turns * 2^64
    void set_freq(float sampleRate, float freq);
    void set_inc(float re, float im);     // any other float32 phasor increment (SSBDemod, demodulator.h:403-412)
    void set_phase(float re, float im);
    void get_phase(float* re, float* im) const;
    void advance(long long n) { phase += step * (uint64_t)n; }
};

}  // namespace qdsp
