// Micro-benchmark: float64 tensor-core throughput of mma.sync.aligned.m8n8k4.f64 (SASS DMMA.8x8x4) from registers, no
// memory traffic.  (1) one CTA on one SM, 1 .. 32 warps: DMMA per clock per SM (clock64 inside the kernel); (2) every SM
// busy, 4 .. 32 warps per SM: TFLOP/s from CUDA events.  Each warp runs 8 independent accumulator chains so that the
// DMMA latency is covered.  The card name, power limit and clocks are printed first (nvidia-smi, read-only query).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/dmma_bench tools/dmma_bench.cu
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

#define CK(x)                                                                             \
    do {                                                                                  \
        cudaError_t e = (x);                                                              \
        if (e != cudaSuccess) {                                                           \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e));     \
            exit(1);                                                                      \
        }                                                                                 \
    } while (0)

constexpr int kChains = 8;

__global__ void dmma_loop(int iters, double seed, double* out, long long* cycles) {
    double a = seed + threadIdx.x, b = seed - threadIdx.x;
    double d[kChains][2];
#pragma unroll
    for (int c = 0; c < kChains; ++c) d[c][0] = d[c][1] = 0.0;
    __syncthreads();
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int c = 0; c < kChains; ++c)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(d[c][0]), "+d"(d[c][1])
                         : "d"(a), "d"(b));
    }
    __syncthreads();
    const long long t1 = clock64();
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < kChains; ++c) s += d[c][0] + d[c][1];
    if (s == 12345.678) out[threadIdx.x] = s;           // keeps the chains alive; never true for these inputs
    if (threadIdx.x == 0 && cycles) cycles[blockIdx.x] = t1 - t0;
}

int main() {
    FILE* p = popen("nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader", "r");
    char line[256] = "unknown";
    if (p) {
        if (!fgets(line, sizeof line, p)) snprintf(line, sizeof line, "unknown\n");
        pclose(p);
    }
    printf("card: %s", line);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("SMs: %d; DMMA.8x8x4 = 2 * 8 * 8 * 4 = 512 FLOP per warp instruction; %d independent chains per warp\n",
           prop.multiProcessorCount, kChains);
    double* out;
    long long* cyc;
    CK(cudaMalloc(&out, 1024 * sizeof(double)));
    CK(cudaMalloc(&cyc, 4096 * sizeof(long long)));
    const int iters = 1 << 14;

    printf("(1) one CTA on one SM\n");
    for (int warps : {1, 2, 4, 8, 16, 32}) {
        dmma_loop<<<1, warps * 32>>>(64, 1.0, out, cyc);
        CK(cudaDeviceSynchronize());
        dmma_loop<<<1, warps * 32>>>(iters, 1.0, out, cyc);
        CK(cudaDeviceSynchronize());
        long long c;
        CK(cudaMemcpy(&c, cyc, sizeof c, cudaMemcpyDeviceToHost));
        const double dmma = (double)warps * iters * kChains;
        printf("  %2d warps: %.4f DMMA / clock / SM = %.1f FLOP / clock / SM\n", warps, dmma / c, dmma * 512.0 / c);
    }

    printf("(2) every SM busy (CUDA events, best of 5)\n");
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int warps : {4, 8, 16, 32}) {
        const int ctas = prop.multiProcessorCount * 4, threads = warps * 8;     // 4 CTAs per SM of warps / 4 warps each
        dmma_loop<<<ctas, threads>>>(256, 1.0, out, nullptr);
        CK(cudaDeviceSynchronize());
        float best = 1e30f;
        for (int r = 0; r < 5; ++r) {
            CK(cudaEventRecord(e0));
            dmma_loop<<<ctas, threads>>>(iters, 1.0, out, nullptr);
            CK(cudaEventRecord(e1));
            CK(cudaEventSynchronize(e1));
            float ms;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            if (ms < best) best = ms;
        }
        const double flop = (double)ctas * (threads / 32) * iters * kChains * 512.0;
        printf("  %2d warps / SM: %.3f ms, %.2f TFLOP/s (float64, DMMA)\n", warps, best, flop / (best * 1e-3) / 1e12);
    }
    CK(cudaFree(out));
    CK(cudaFree(cyc));
    return 0;
}
