// Experiment (not product): a radix-16 NTT register round with its butterflies on the FP64 pipe, against the integer round the
// shipped kernel runs (run_stages in ntt.cu).  Question: can the idle FP64 pipe carry the add / sub / shift-twiddle work?
//
//   integer round (baseline): 4 constant-geometry stages, per butterfly  t = canon(mul(v, w)); (u + t, u - t)
//   FP64 round: x[a] *= g^a (one general multiplication per element), values -> pairs of exact doubles (lo + hi 2^32),
//               16-point DFT whose twiddles are powers of 2 (2^12 is a primitive 16th root: 2^96 = -1 mod p):
//               add / sub = 2 DADD each, x 2^e = exact scaling + floor-split (which renormalises), then back to u64.
// The FP64 round is checked bit-exactly against the same mathematics done with integer multiplications by 2^e.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I plonky2_demo_b200/csrc -o tools/ntt_fp64_bench tools/ntt_fp64_bench.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "gl64.cuh"

struct D2 { double l, h; };   // value = l + h * 2^32 (mod p); integers, |.| < 2^51

constexpr double TWO52 = 4503599627370496.0;
constexpr double MAGIC = 6755399441055744.0;   // 1.5 * 2^52: floor trick that also works for negative values
constexpr double T32 = 4294967296.0;

__device__ __forceinline__ double u32d(uint32_t x) { return __hiloint2double(0x43300000, (int)x) - TWO52; }
__device__ __forceinline__ D2 to_d2(uint64_t x) { return {u32d((uint32_t)x), u32d((uint32_t)(x >> 32))}; }
__device__ __forceinline__ D2 dadd(D2 a, D2 b) { return {a.l + b.l, a.h + b.h}; }
__device__ __forceinline__ D2 dsub(D2 a, D2 b) { return {a.l - b.l, a.h - b.h}; }

// x * 2^E, 0 < E < 96
template <int E>
__device__ __forceinline__ D2 mul2exp(D2 a) {
    constexpr int q = E / 32, r = E % 32;
    double Lp, Hp;
    if (r == 0) {
        Lp = a.l;
        Hp = a.h;
    } else {
        constexpr double S = (double)(1ull << r), I = S / 4294967296.0;
        const double bl = __fma_rd(a.l, I, MAGIC) - MAGIC;     // floor(l 2^r / 2^32)
        const double al = fma(bl, -T32, a.l * S);              // l 2^r mod 2^32
        const double bh = __fma_rd(a.h, I, MAGIC) - MAGIC;
        const double ah = fma(bh, -T32, a.h * S);
        // l 2^r + h 2^r 2^32 = al + (bl + ah) 2^32 + bh 2^64,  2^64 = 2^32 - 1
        Lp = al - bh;
        Hp = bl + ah + bh;
    }
    if (q == 0) return {Lp, Hp};
    if (q == 1) return {-Hp, Lp + Hp};            // x 2^32: (L, H) -> (-H, L + H)
    return {-(Lp + Hp), Lp};                      // x 2^64 = x (2^32 - 1)
}

// pair of doubles -> loose u64
__device__ __forceinline__ uint64_t from_d2(D2 a) {
    const double l1 = __fma_rd(a.l, 1.0 / T32, MAGIC) - MAGIC;
    const double l0 = fma(l1, -T32, a.l);
    const double hp = a.h + l1;
    const double h1 = __fma_rd(hp, 1.0 / T32, MAGIC) - MAGIC;
    const double h0 = fma(h1, -T32, hp);
    const uint32_t x0 = (uint32_t)__double2loint(l0 + TWO52), x1 = (uint32_t)__double2loint(h0 + TWO52);
    const uint32_t top = (uint32_t)__double2loint(h1 + (TWO52 + 4096.0));       // h1 + 4096 >= 0
    // x + (h1 + 4096) 2^64 - 4096 2^64
    return gl::sub_lc(gl::reduce96(gl::pack(x0, x1), top), 4096ull * 0xFFFFFFFFull);
}

// exponent (of 2) of the block constant: y^(2h) = 2^e in block B of stage S (compile time)
template <int S, int B> struct Blk { static constexpr int e = Blk<S - 1, B / 2>::e / 2 + ((B & 1) ? 96 : 0); };
template <int B> struct Blk<0, B> { static constexpr int e = 0; };

template <int S, int B>
__device__ __forceinline__ void blocks_fp64(D2 (&x)[16]) {
    if constexpr (B < (1 << S)) {
        constexpr int half = 8 >> S;
        constexpr int e = Blk<S, B>::e / 2;         // twiddle 2^e: the block's y^h = +- 2^e
#pragma unroll
        for (int i = 0; i < half; i++) {
            const int a = B * 2 * half + i, b = a + half;
            D2 t;
            if constexpr (e != 0) t = mul2exp<e>(x[b]); else t = x[b];
            const D2 u = x[a];
            x[a] = dadd(u, t);
            x[b] = dsub(u, t);
        }
        blocks_fp64<S, B + 1>(x);
    }
}
template <int S>
__device__ __forceinline__ void stages_fp64(D2 (&x)[16]) {
    blocks_fp64<S, 0>(x);
    if constexpr (S < 3) stages_fp64<S + 1>(x);
}
__device__ __forceinline__ void dft16_fp64(D2 (&x)[16]) { stages_fp64<0>(x); }

template <int S, int B>
__device__ __forceinline__ void blocks_int(uint64_t (&x)[16]) {   // the same mathematics, integer multiplications by 2^e
    if constexpr (B < (1 << S)) {
        constexpr int half = 8 >> S;
        constexpr int e = Blk<S, B>::e / 2;
#pragma unroll
        for (int i = 0; i < half; i++) {
            const int a = B * 2 * half + i, b = a + half;
            uint64_t t = x[b];
            if constexpr (e != 0) {
                if constexpr (e < 64) t = gl::mul(t, 1ull << e);
                else t = gl::mul(gl::mul(t, 1ull << 63), 1ull << (e - 63));
            }
            t = gl::canon(t);
            const uint64_t u = x[a];
            x[a] = gl::add_lc(u, t);
            x[b] = gl::sub_lc(u, t);
        }
        blocks_int<S, B + 1>(x);
    }
}
template <int S>
__device__ __forceinline__ void stages_int(uint64_t (&x)[16]) {
    blocks_int<S, 0>(x);
    if constexpr (S < 3) stages_int<S + 1>(x);
}
__device__ __forceinline__ void dft16_int(uint64_t (&x)[16]) { stages_int<0>(x); }

// mode 0: integer round as shipped (general twiddle per butterfly, constant geometry); 1: FP64 round; 2: integer reference of the FP64 round
template <int MODE>
__global__ void __launch_bounds__(256, 2) k_round(uint64_t* io, const uint64_t* tw_g, size_t n_threads, int reps) {
    __shared__ uint64_t tw[64];
    if (threadIdx.x < 64) tw[threadIdx.x] = tw_g[threadIdx.x];
    __syncthreads();
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_threads) return;
    uint64_t x[16];
#pragma unroll
    for (int a = 0; a < 16; a++) x[a] = io[(size_t)a * n_threads + t];
    for (int r = 0; r < reps; r++) {
        if (MODE == 0) {
#pragma unroll 1
            for (int s = 0; s < 4; s++) {
                uint64_t y[16];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint64_t tt = gl::canon(gl::mul(x[j + 8], tw[s * 8 + j]));
                    y[2 * j] = gl::add_lc(x[j], tt);
                    y[2 * j + 1] = gl::sub_lc(x[j], tt);
                }
#pragma unroll
                for (int j = 0; j < 16; j++) x[j] = y[j];
            }
        } else {
#pragma unroll
            for (int a = 1; a < 16; a++) x[a] = gl::mul(x[a], tw[32 + a]);      // pre-scale by g^a
            if (MODE == 1) {
                D2 d[16];
#pragma unroll
                for (int a = 0; a < 16; a++) d[a] = to_d2(x[a]);
                dft16_fp64(d);
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = from_d2(d[a]);
            } else {
                dft16_int(x);
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 16; a++) io[(size_t)a * n_threads + t] = gl::canon(x[a]);
}

int main() {
    const size_t n_threads = (size_t)148 * 2 * 256 * 8;
    const size_t bytes = n_threads * 16 * 8;
    uint64_t *a, *b, *c, *tw;
    cudaMalloc(&a, bytes); cudaMalloc(&b, bytes); cudaMalloc(&c, bytes); cudaMalloc(&tw, 64 * 8);
    uint64_t* h = (uint64_t*)malloc(bytes);
    uint64_t s = 0x9E3779B97F4A7C15ull;
    for (size_t i = 0; i < n_threads * 16; i++) { s ^= s << 13; s ^= s >> 7; s ^= s << 17; h[i] = s; }   // any u64, incl. non-canonical
    h[0] = ~0ull; h[1] = 0xFFFFFFFF00000001ull; h[2] = 0; h[3] = 0xFFFFFFFFull; h[4] = 0xFFFFFFFF00000000ull;
    uint64_t htw[64];
    for (int i = 0; i < 64; i++) { s ^= s << 13; s ^= s >> 7; s ^= s << 17; htw[i] = s % 0xFFFFFFFF00000001ull; }
    cudaMemcpy(tw, htw, sizeof(htw), cudaMemcpyHostToDevice);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    const unsigned grid = (unsigned)(n_threads / 256);
    // correctness: 3 chained rounds, FP64 against the integer reference of the same mathematics
    cudaMemcpy(b, h, bytes, cudaMemcpyHostToDevice); cudaMemcpy(c, h, bytes, cudaMemcpyHostToDevice);
    k_round<1><<<grid, 256>>>(b, tw, n_threads, 3);
    k_round<2><<<grid, 256>>>(c, tw, n_threads, 3);
    uint64_t* hb = (uint64_t*)malloc(bytes); uint64_t* hc = (uint64_t*)malloc(bytes);
    cudaMemcpy(hb, b, bytes, cudaMemcpyDeviceToHost); cudaMemcpy(hc, c, bytes, cudaMemcpyDeviceToHost);
    size_t bad = 0;
    for (size_t i = 0; i < n_threads * 16; i++) bad += hb[i] != hc[i];
    float ms[3];
    const int reps = 50;
    uint64_t* bufs[3] = {a, b, c};
    for (int m = 0; m < 3; m++) {
        cudaMemcpy(bufs[m], h, bytes, cudaMemcpyHostToDevice);
        for (int it = 0; it < 2; it++) {
            cudaEventRecord(e0);
            if (m == 0) k_round<0><<<grid, 256>>>(bufs[m], tw, n_threads, reps);
            if (m == 1) k_round<1><<<grid, 256>>>(bufs[m], tw, n_threads, reps);
            if (m == 2) k_round<2><<<grid, 256>>>(bufs[m], tw, n_threads, reps);
            cudaEventRecord(e1); cudaEventSynchronize(e1);
        }
        cudaEventElapsedTime(&ms[m], e0, e1);
    }
    cudaFuncAttributes f0, f1;
    cudaFuncGetAttributes(&f0, k_round<0>); cudaFuncGetAttributes(&f1, k_round<1>);
    const double elem_rounds = (double)n_threads * 16 * reps;
    printf("{\"fp64_round_equals_integer_reference\": %s, \"mismatches\": %zu, \"integer_round_ms\": %.3f, \"fp64_round_ms\": %.3f, "
           "\"integer_shift_round_ms\": %.3f, \"ps_per_element_per_4_stages\": {\"integer\": %.1f, \"fp64\": %.1f, \"integer_shift\": %.1f}, "
           "\"regs\": {\"integer\": %d, \"fp64\": %d}, \"fp64_vs_integer\": %.3f, \"status\": \"%s\"}\n",
           bad == 0 ? "true" : "false", bad, ms[0], ms[1], ms[2], ms[0] * 1e9 / elem_rounds, ms[1] * 1e9 / elem_rounds, ms[2] * 1e9 / elem_rounds,
           f0.numRegs, f1.numRegs, ms[1] / ms[0], cudaGetErrorString(cudaGetLastError()));
    return bad != 0;
}
