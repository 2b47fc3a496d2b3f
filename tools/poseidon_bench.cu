// Times the Poseidon-12 permutation device function in isolation (17 chained permutations per
// thread, like one 135-element leaf).  -DTHREADS / -DMINBLOCKS set the launch bounds:
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I plonky2_demo_b200/csrc -o pb tools/poseidon_bench.cu
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>
#include "poseidon.cuh"

#ifndef THREADS
#define THREADS 128
#endif
#ifndef MINBLOCKS
#define MINBLOCKS 1
#endif

__global__ void __launch_bounds__(THREADS, MINBLOCKS) k(uint64_t* io, size_t n, int reps) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t s[12];
#pragma unroll
    for (int k2 = 0; k2 < 12; k2++) s[k2] = io[(size_t)k2 * n + i];
    for (int r = 0; r < reps; r++) {
        pcs::poseidon12(s);
        s[0] += r;  // keep iterations distinct
    }
#pragma unroll
    for (int k2 = 0; k2 < 4; k2++) io[(size_t)k2 * n + i] = s[k2];
}

int main(int argc, char** argv) {
    size_t n = argc > 2 ? (size_t)atol(argv[2]) : (size_t)1 << 21;   // 32 = one warp: the latency of a permutation chain
    int reps = argc > 3 ? atoi(argv[3]) : 17;
    uint64_t* d;
    cudaMalloc(&d, n * 12 * 8);
    cudaMemset(d, 1, n * 12 * 8);
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, THREADS, 0);
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, k);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    k<<<(unsigned)((n + THREADS - 1) / THREADS), THREADS>>>(d, n, reps);
    cudaDeviceSynchronize();
    float best = 1e9;
    for (int it = 0; it < 3; it++) {
        cudaEventRecord(e0);
        k<<<(unsigned)((n + THREADS - 1) / THREADS), THREADS>>>(d, n, reps);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    double perms = (double)n * reps;
    double clk = best * 1e-3 * 1.965e9 * p.multiProcessorCount / perms;
    printf("{\"variant\": \"%s\", \"threads\": %d, \"regs\": %d, \"blocks_per_sm\": %d, \"ms\": %.3f, \"perms_per_s\": %.4e, "
           "\"clk_per_perm_per_sm_lane_at_1965MHz\": %.1f, \"status\": \"%s\"}\n",
           argc > 1 ? argv[1] : "default", THREADS, fa.numRegs, nb, best, perms / (best * 1e-3), clk,
           cudaGetErrorString(cudaGetLastError()));
    return 0;
}
