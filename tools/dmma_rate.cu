// microbenchmark: FP64 issue rate on sm_100a, plain DFMA vs the FP64 tensor core (mma.sync m8n8k4 f64 = one DMMA.8x8x4)
//     nvcc -O3 -gencode arch=compute_100a,code=sm_100a tools/dmma_rate.cu -o dmma_rate && ./dmma_rate
// Prints FLOP/s and FLOP per SM clock (at the clock the card reports) for 4..16 warps per SM (32 accumulators a
// thread: 1024-thread blocks would need more registers than an SM has).
#include <cstdio>
#include <cuda_runtime.h>
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
template <int MODE> __global__ void k(double* out, double s0, double s1, int iters) {
    double acc[32];
    double x[4] = {s0 + threadIdx.x, s1, s0 * 2, s1 * 3};
    for (int i = 0; i < 32; ++i) acc[i] = i + threadIdx.x;
    for (int it = 0; it < iters; ++it) {
        if (MODE == 0) {
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = fma(acc[i], x[i & 3], x[(i + 1) & 3]);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) dmma(acc[2 * i], acc[2 * i + 1], x[i & 3], x[(i + 1) & 3]);
        }
    }
    double r = 0; for (int i = 0; i < 32; ++i) r += acc[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}
int main() {
    int clk_khz = 0, sms = 0;
    cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    double* out; cudaMalloc(&out, (size_t)sms * 32 * 32 * 8);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    printf("%d SMs, reported SM clock %.3f GHz\n", sms, clk_khz / 1e6);
    for (int warps = 4; warps <= 16; warps *= 2) for (int mode = 0; mode < 2; ++mode) {
        const int iters = 20000; float ms = 0;
        for (int rep = 0; rep < 3; ++rep) {
            cudaEventRecord(e0);
            if (mode == 0) k<0><<<sms, warps * 32>>>(out, 1.0001, 0.9999, iters); else k<1><<<sms, warps * 32>>>(out, 1.0001, 0.9999, iters);
            cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
        }
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { printf("CUDA error %s\n", cudaGetErrorString(e)); return 1; }
        // DFMA: 32 per thread per iteration, 2 FLOP each; DMMA.8x8x4: 16 per warp per iteration, 2 * 8 * 8 * 4 = 512 FLOP each
        const double flop = mode == 0 ? 2.0 * 32 * 32 * warps * (double)sms * iters : 512.0 * 16 * warps * (double)sms * iters;
        printf("warps/SM %2d %s: %8.3f ms  %6.2f TFLOP/s  %6.1f FLOP/clk/SM at the reported clock\n", warps,
               mode ? "DMMA" : "DFMA", ms, flop / ms / 1e9, flop / (ms * 1e-3) / (clk_khz * 1e3) / sms);
    }
    return 0;
}
