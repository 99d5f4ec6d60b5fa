// Stand-alone ops of the C ABI that do not need an extractor handle.
#include "sidekit_b200.h"
#include "common.cuh"
#include "layers.cuh"

namespace skb {

// MeanStdPooling on the reference's (B, D, T) layout: one warp per (b, d) row, two-pass statistics.
__global__ void meanstd_bdt_kernel(const float* __restrict__ x, int D, int T, float* __restrict__ out, long long rows) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* p = x + row * T;
    float s = 0.f;
    for (int t = lane; t < T; t += 32) s += p[t];
    const float mean = warp_sum(s) / (float)T;
    float v = 0.f;
    for (int t = lane; t < T; t += 32) {
        const float d = p[t] - mean;
        v = fmaf(d, d, v);
    }
    v = warp_sum(v);
    if (lane == 0) {
        const long long b = row / D, d = row % D;
        out[b * 2 * D + d] = mean;
        out[b * 2 * D + D + d] = sqrtf(v / (float)(T - 1));
    }
}
}  // namespace skb

using namespace skb;

extern "C" int skb_meanstd_pool(const float* x_dev, int n_utt, int D, int T, float* out_dev, void* stream) {
    if (!x_dev || !out_dev || n_utt <= 0 || D <= 0 || T <= 0) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    const long long rows = (long long)n_utt * D;
    const int warps = 8;
    SKB_CUDA_CHECK(launch_kernel(false, meanstd_bdt_kernel, (unsigned)((rows + warps - 1) / warps), warps * 32, 0, (cudaStream_t)stream, x_dev,
                                 D, T, out_dev, rows));
    return SKB_OK;
}
