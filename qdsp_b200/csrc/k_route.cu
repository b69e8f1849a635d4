// qdsp_b200/csrc/k_route.cu — per-channel delivery for the dsp:: mirror's many-output blocks (include/dsp/channelizer.h):
// the channelizer writes [nrows][src_stride] from one base pointer, and each row belongs in its own stream buffer. One
// launch copies every row to the pointer a device table holds for it (grid.y = row), so the cost per run() is one launch
// whatever the channel count. Rows are short (a run() block's outputs), so one CTA row covers a whole row in a grid-stride loop.
#include "internal.cuh"
#include "kernels.cuh"

namespace qdsp {

template <typename T>
__global__ void __launch_bounds__(256) scatter_rows_kernel(const T* __restrict__ src, long long src_stride,
                                                           T* const* __restrict__ dst, long long count) {
    const int r = blockIdx.y;
    T* d = dst[r];
    const T* s = src + (size_t)r * (size_t)src_stride;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
        d[i] = s[i];
}

int launch_scatter_rows(const void* src, long long src_stride, void* const* dst_table, int nrows, long long count, int elem_bytes,
                        cudaStream_t s) {
    if (nrows == 0 || count == 0) return 0;
    if (nrows > 65535) {
        set_last_error("scatter_rows: at most 65535 rows");
        return -1;
    }
    const long long per = (count + 255) / 256;
    const dim3 grid((unsigned)(per < 8 ? per : 8), (unsigned)nrows);
    if (elem_bytes == 8)
        scatter_rows_kernel<float2><<<grid, 256, 0, s>>>((const float2*)src, src_stride, (float2* const*)dst_table, count);
    else
        scatter_rows_kernel<float><<<grid, 256, 0, s>>>((const float*)src, src_stride, (float* const*)dst_table, count);
    QDSP_LAUNCH_OK();
    return 0;
}

}  // namespace qdsp
