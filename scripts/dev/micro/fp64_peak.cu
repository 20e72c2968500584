// FP64 peak of one GPU, the denominator of the fp64 rollout's share of peak (scripts/dev/fp64_time.py):
// DFMA on the CUDA cores and DMMA (mma.sync m8n8k4 .f64, SASS DMMA.8x8x4) on the tensor cores, each as
// independent dependency chains in every warp of a full grid, timed with CUDA events.  Prints one JSON line.
#include <cstdio>
#include <cuda_runtime.h>

constexpr int ITERS = 4096;

__global__ void dfma_peak(double* out, double s) {
    double a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = threadIdx.x * 1e-3 + i;
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = fma(a[i], s, 1e-9);
    double r = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r += a[i];
    if (r == 12345.0) out[0] = r;        // keeps the chains alive
}

__global__ void dmma_peak(double* out, double s) {
    double c[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = threadIdx.x * 1e-3 + i;
    const double a = s, b = 1e-9 * threadIdx.x;
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
        for (int i = 0; i < 8; i += 2)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                         : "+d"(c[i]), "+d"(c[i + 1]) : "d"(a), "d"(b));
    double r = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r += c[i];
    if (r == 12345.0) out[0] = r;
}

int main() {
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    double* out;
    cudaMalloc(&out, 8);
    const int blocks = p.multiProcessorCount * 8, threads = 256;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best[2] = {1e30, 1e30};
    for (int rep = 0; rep < 6; ++rep)
        for (int k = 0; k < 2; ++k) {
            cudaEventRecord(e0);
            if (k == 0) dfma_peak<<<blocks, threads>>>(out, 0.999999);
            else dmma_peak<<<blocks, threads>>>(out, 0.999999);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float ms;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0 && ms < best[k]) best[k] = ms;   // rep 0 is the warm-up
        }
    if (cudaGetLastError() != cudaSuccess) { fprintf(stderr, "fp64_peak: CUDA error\n"); return 1; }
    const double threads_total = (double)blocks * threads;
    const double dfma_flop = threads_total * ITERS * 8 * 2;                 // 8 chains x 1 FMA
    const double dmma_flop = threads_total / 32 * ITERS * 4 * 8 * 8 * 4 * 2; // 4 MMAs of 8x8x4 per warp
    printf("{\"dfma_tflops\": %.3f, \"dmma_tflops\": %.3f, \"dfma_ms\": %.3f, \"dmma_ms\": %.3f, \"sms\": %d}\n",
           dfma_flop / best[0] / 1e9, dmma_flop / best[1] / 1e9, best[0], best[1], p.multiProcessorCount);
    return 0;
}
