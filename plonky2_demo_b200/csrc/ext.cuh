// Quadratic extension of Goldilocks, F[X]/(X^2 - 7), for host and device.
//
// GPU counterpart of the reference's QuadraticExtension<GoldilocksField>
// (field/src/extension/quadratic.rs:184-192 mul, field/src/goldilocks_extensions.rs:14-28: W = 7).
// An element is the pair (a, b) = a + b*X, stored like the reference's [F; 2] (to_basefield_array).
// Device values are loose u64 like everywhere in the engine; canon() where they leave it.
#pragma once
#include <stdint.h>

#include "common.cuh"
#include "gl64.cuh"

namespace gl {

struct ext2 {
    uint64_t a, b;
};

// ---- 160-bit lazy accumulator: sum of 64x64 products, reduced once ---------------------------------
// The reference reduces such sums the same way in its extension-field kernels (goldilocks_extensions.rs:120-180
// accumulate u128 products with a carry count and reduce once); the result is the same field element.
struct acc160 {
    uint64_t lo, hi;
    uint32_t top;
};

__device__ __forceinline__ void acc_zero(acc160& A) {
    A.lo = 0;
    A.hi = 0;
    A.top = 0;
}

// A += x * y  (any u64 x, y)
__device__ __forceinline__ void acc_mac(acc160& A, uint64_t x, uint64_t y) {
    unsigned __int128 q = (unsigned __int128)x * y;
    uint64_t ql = (uint64_t)q, qh = (uint64_t)(q >> 64);
    asm("{\n\t"
        "add.cc.u64  %0, %0, %3;\n\t"
        "addc.cc.u64 %1, %1, %4;\n\t"
        "addc.u32    %2, %2, 0;\n\t"
        "}"
        : "+l"(A.lo), "+l"(A.hi), "+r"(A.top)
        : "l"(ql), "l"(qh));
}

// lo + hi*2^64 + top*2^128 -> loose u64, using 2^128 = 2^96 * 2^32 = -2^32 (mod p); top*2^32 <= p - 1 is canonical
__device__ __forceinline__ uint64_t acc_reduce(const acc160& A) {
    return sub_lc(reduce128(A.lo, A.hi), (uint64_t)A.top << 32);
}

// ---- carry-free lazy accumulation: sum_k c_k * w_k for canonical multipliers w_k held as 22-bit limbs -----------
// w = w0 + w1 2^22 + w2 2^44 (w0, w1 < 2^22, w2 < 2^20) and c = c0 + c1 2^32: the six partial products c_i w_j are
// below 2^54, so each of the six weights gets its own 64-bit accumulator and up to 1024 terms are added with one plain
// IMAD.WIDE.U32 each -- no carry chains (a 64x64 product with 160-bit accumulation costs ~20 instructions, half of them
// carry-chained; profiles/r01_fri_kernels.md).  The accumulators are recombined once per sum.
struct limbs22 {
    uint32_t w0, w1, w2;
};

__host__ __device__ __forceinline__ limbs22 split22(uint64_t w) {
    limbs22 l;
    l.w0 = (uint32_t)(w & 0x3FFFFF);
    l.w1 = (uint32_t)((w >> 22) & 0x3FFFFF);
    l.w2 = (uint32_t)(w >> 44);
    return l;
}

struct lazy6 {
    uint64_t a00, a01, a02, a10, a11, a12;   // weights 2^0, 2^22, 2^44, 2^32, 2^54, 2^76
};
constexpr int LAZY_MAX_TERMS = 1024;

__device__ __forceinline__ void lazy_zero(lazy6& A) { A.a00 = A.a01 = A.a02 = A.a10 = A.a11 = A.a12 = 0; }

// acc += a * b as ONE IMAD.WIDE.U32 (inline PTX: nvcc otherwise re-associates the sums into fresh products plus 64-bit adds)
__device__ __forceinline__ void mad_wide(uint64_t& acc, uint32_t a, uint32_t b) {
    asm("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(a), "r"(b));
}

__device__ __forceinline__ void lazy_mac(lazy6& A, uint64_t c, uint32_t w0, uint32_t w1, uint32_t w2) {
    const uint32_t c0 = (uint32_t)c, c1 = (uint32_t)(c >> 32);
    mad_wide(A.a00, c0, w0);
    mad_wide(A.a01, c0, w1);
    mad_wide(A.a02, c0, w2);
    mad_wide(A.a10, c1, w0);
    mad_wide(A.a11, c1, w1);
    mad_wide(A.a12, c1, w2);
}

// S += v << s  (0 < s < 64)
__device__ __forceinline__ void acc_add_shl(acc160& S, uint64_t v, int s) {
    uint64_t l = v << s, h = v >> (64 - s);
    asm("{\n\t"
        "add.cc.u64  %0, %0, %3;\n\t"
        "addc.cc.u64 %1, %1, %4;\n\t"
        "addc.u32    %2, %2, 0;\n\t"
        "}"
        : "+l"(S.lo), "+l"(S.hi), "+r"(S.top)
        : "l"(l), "l"(h));
}

__device__ __forceinline__ uint64_t lazy_reduce(const lazy6& A) {
    acc160 S;
    S.lo = A.a00;
    S.hi = 0;
    S.top = 0;
    acc_add_shl(S, A.a01, 22);
    acc_add_shl(S, A.a10, 32);
    acc_add_shl(S, A.a02, 44);
    acc_add_shl(S, A.a11, 54);
    {   // a12 << 76 = (a12 << 12) at weight 2^64
        uint64_t h = A.a12 << 12;
        uint32_t t = (uint32_t)(A.a12 >> 52);
        asm("{\n\t"
            "add.cc.u64  %0, %0, %2;\n\t"
            "addc.u32    %1, %1, %3;\n\t"
            "}"
            : "+l"(S.hi), "+r"(S.top)
            : "l"(h), "r"(t));
    }
    return acc_reduce(S);
}

// loose x loose -> loose.  c0 = a0 b0 + 7 a1 b1, c1 = a0 b1 + a1 b0, each as ONE lazy reduction
__device__ __forceinline__ ext2 ext_mul(ext2 x, ext2 y) {
    acc160 c0, c1;
    acc_zero(c0);
    acc_zero(c1);
    uint64_t t = canon(mul(x.b, y.b));
    acc_mac(c0, x.a, y.a);
    acc_mac(c0, t, 7);
    acc_mac(c1, x.a, y.b);
    acc_mac(c1, x.b, y.a);
    ext2 r;
    r.a = acc_reduce(c0);
    r.b = acc_reduce(c1);
    return r;
}

// loose + loose -> loose (canonicalises one operand)
__device__ __forceinline__ ext2 ext_add(ext2 x, ext2 y) {
    ext2 r;
    r.a = add_lc(x.a, canon(y.a));
    r.b = add_lc(x.b, canon(y.b));
    return r;
}

__device__ __forceinline__ ext2 ext_canon(ext2 x) {
    ext2 r;
    r.a = canon(x.a);
    r.b = canon(x.b);
    return r;
}

__device__ __forceinline__ ext2 ext_pow(ext2 base, uint64_t e) {
    ext2 acc = {1, 0};
    while (e) {
        if (e & 1) acc = ext_mul(acc, base);
        base = ext_mul(base, base);
        e >>= 1;
    }
    return ext_canon(acc);
}

}  // namespace gl

// ---- host-side extension arithmetic (setup only: powers of a few points and challenges; base field in common.cuh) -------
namespace glh {
struct ext2 {
    uint64_t a, b;
};
static inline uint64_t addmod(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a + b) % P); }
static inline ext2 ext_mul(ext2 x, ext2 y) {
    ext2 r;
    r.a = addmod(mulmod(x.a, y.a), mulmod(7, mulmod(x.b, y.b)));
    r.b = addmod(mulmod(x.a, y.b), mulmod(x.b, y.a));
    return r;
}
static inline ext2 ext_pow(ext2 x, uint64_t e) {
    ext2 acc = {1, 0};
    x.a %= P;
    x.b %= P;
    for (; e; e >>= 1) {
        if (e & 1) acc = ext_mul(acc, x);
        x = ext_mul(x, x);
    }
    return acc;
}
}  // namespace glh
