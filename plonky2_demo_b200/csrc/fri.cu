// FRI opening proof on the device (SURVEY 8f N2 / N3): the consumers of a committed batch's coefficients.
//
//   pcs_batch_eval_ext   OpeningSet::new's eval_commitment                 plonky2/src/plonk/proof.rs:316-322
//   pcs_fri_final_poly   prove_openings' batch reduction + quotients       plonky2/src/fri/oracle.rs:171-200
//   pcs_ext_coset_lde    lde_final_poly.coset_fft(shift)                   plonky2/src/fri/oracle.rs:202-207
//   pcs_fri_commit_layer one tree of fri_committed_trees                   plonky2/src/fri/prover.rs:81-87
//   pcs_fri_fold         coefficient fold between two trees                plonky2/src/fri/prover.rs:93-101
//
// Extension polynomials live COMPONENT-MAJOR on the device ([2][len]: all `a` parts, then all `b` parts) so that every
// kernel reads them coalesced and the coset LDE is the base-field NTT of two rows; the [len][2] layout of the
// reference's Vec<F::Extension> exists only at the host boundary.
//
// The two kernels that touch a whole committed batch (k_eval_ext, k_reduce_polys_base) read every coefficient once
// and should be HBM bound: the multipliers (powers of z / alpha) are held as 22-bit limbs so that a coefficient costs
// twelve plain IMAD.WIDE.U32 into twelve 64-bit accumulators -- no carry chains, no modular reduction (ext.cuh lazy6).
#include <vector>

#include "common.cuh"
#include "ext.cuh"
#include "tma.cuh"

using namespace pcs;

struct pcs_ext_poly {
    uint64_t* c = nullptr;   // [2][cap]: component e of coefficient i at c[e * cap + i]
    size_t len = 0, cap = 0;
    void* ctx = nullptr;     // the engine context (device + stream) the coefficients live on
};

namespace {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
// out[i] = base^i, i < n (canonical)
__global__ void k_ext_pow_table(gl::ext2 base, size_t n, gl::ext2* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = gl::ext_pow(base, i);
}

// [len][2] interleaved -> [2][cap] component-major (canonicalising), and back
__global__ void k_deinterleave(const uint64_t* in, size_t len, uint64_t* out, size_t cap) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) {
        out[i] = gl::canon(in[2 * i]);
        out[cap + i] = gl::canon(in[2 * i + 1]);
    }
}
__global__ void k_interleave(const uint64_t* in, size_t in_stride, size_t len, uint64_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) {
        out[2 * i] = gl::canon(in[i]);
        out[2 * i + 1] = gl::canon(in[in_stride + i]);
    }
}
// natural-order interleaved values from a leaf-order (bit-reversed) component-major LDE
__global__ void k_interleave_bitrev(const uint64_t* in, size_t n, unsigned lg_n, uint64_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        size_t r = lg_n ? (size_t)(__brevll((unsigned long long)i) >> (64 - lg_n)) : 0;
        out[2 * r] = gl::canon(in[i]);
        out[2 * r + 1] = gl::canon(in[n + i]);
    }
}

// ------------------------------------------------------------------------------------------------
// eval_commitment: P_j(z) for every polynomial of a batch, z in the extension
// ------------------------------------------------------------------------------------------------
constexpr int EV_THREADS = 256, EV_PER_THREAD = 64, EV_BATCH = 16, EV_CHUNK = EV_THREADS * EV_PER_THREAD;

// Shared tail of the two evaluation kernels: thread t holds S_t = sum_k c[t + 256 k] z^(256 k); the chunk's value is
// z^(chunk start) * sum_t z^t S_t.
__device__ __forceinline__ void eval_block_finish(gl::ext2 s, unsigned t, gl::ext2* s_red, const gl::ext2* __restrict__ pw_t,
                                                  const gl::ext2* __restrict__ pw_c, gl::ext2* __restrict__ partial) {
    s = gl::ext_canon(gl::ext_mul(s, pw_t[t]));
#pragma unroll
    for (int off = 16; off; off >>= 1) {   // warp sum (canonical adds)
        uint64_t oa = __shfl_down_sync(0xffffffffu, s.a, off), ob = __shfl_down_sync(0xffffffffu, s.b, off);
        s.a = gl::add(s.a, oa);
        s.b = gl::add(s.b, ob);
    }
    if ((t & 31) == 0) s_red[t >> 5] = s;
    __syncthreads();
    if (t == 0) {
        for (int wp = 1; wp < EV_THREADS / 32; wp++) {
            s.a = gl::add(s.a, s_red[wp].a);
            s.b = gl::add(s.b, s_red[wp].b);
        }
        partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = gl::ext_canon(gl::ext_mul(s, pw_c[blockIdx.x]));
    }
}

// grid (chunks, w).  Thread t of chunk c sums  coeff[c*16384 + t + 256 k] * (z^256)^k  over k < 64 carry-free (ext.cuh
// lazy6, loads double-buffered in batches of 16), multiplies by z^t; the block adds its 256 partial sums and scales by z^(16384 c).
__global__ void __launch_bounds__(EV_THREADS) k_eval_ext(const uint64_t* __restrict__ coeffs,
                                                         const uint64_t* const* __restrict__ poly_ptrs, size_t d,
                                                         const gl::ext2* __restrict__ pw_t /*[256] z^t*/,
                                                         const gl::ext2* __restrict__ pw_k /*[64] z^(256 k)*/,
                                                         const gl::ext2* __restrict__ pw_c /*[chunks] z^(16384 c)*/,
                                                         gl::ext2* __restrict__ partial /*[w][chunks]*/) {
    __shared__ uint32_t s_k[EV_PER_THREAD][8];   // 22-bit limbs of (z^256)^k: a part in [0..2], b part in [4..6]
    __shared__ gl::ext2 s_red[EV_THREADS / 32];
    const unsigned t = threadIdx.x;
    if (t < EV_PER_THREAD) {
        gl::ext2 w = pw_k[t];
        gl::limbs22 la = gl::split22(w.a), lb = gl::split22(w.b);
        s_k[t][0] = la.w0; s_k[t][1] = la.w1; s_k[t][2] = la.w2; s_k[t][3] = 0;
        s_k[t][4] = lb.w0; s_k[t][5] = lb.w1; s_k[t][6] = lb.w2; s_k[t][7] = 0;
    }
    __syncthreads();
    const uint64_t* poly = poly_ptrs ? poly_ptrs[blockIdx.y] : coeffs + (size_t)blockIdx.y * d;   // table: scattered polynomials
    const size_t base = (size_t)blockIdx.x * EV_CHUNK + t;
    gl::lazy6 A, B;   // 64 terms each: far below LAZY_MAX_TERMS
    gl::lazy_zero(A);
    gl::lazy_zero(B);
    // software pipeline: the loads of batch b + 1 are in flight while batch b is multiplied
    uint64_t cur[EV_BATCH], nxt[EV_BATCH];
#pragma unroll
    for (int k = 0; k < EV_BATCH; k++) {
        size_t i = base + (size_t)k * EV_THREADS;
        cur[k] = i < d ? poly[i] : 0;
    }
#pragma unroll 1
    for (int k0 = 0; k0 < EV_PER_THREAD; k0 += EV_BATCH) {
#pragma unroll
        for (int k = 0; k < EV_BATCH; k++) {
            size_t i = base + (size_t)(k0 + EV_BATCH + k) * EV_THREADS;
            nxt[k] = (k0 + EV_BATCH < EV_PER_THREAD && i < d) ? poly[i] : 0;
        }
#pragma unroll
        for (int k = 0; k < EV_BATCH; k++) {
            const uint4 wa = *reinterpret_cast<const uint4*>(&s_k[k0 + k][0]);
            const uint4 wb = *reinterpret_cast<const uint4*>(&s_k[k0 + k][4]);
            gl::lazy_mac(A, cur[k], wa.x, wa.y, wa.z);
            gl::lazy_mac(B, cur[k], wb.x, wb.y, wb.z);
        }
#pragma unroll
        for (int k = 0; k < EV_BATCH; k++) cur[k] = nxt[k];
    }
    gl::ext2 s = {gl::lazy_reduce(A), gl::lazy_reduce(B)};
    eval_block_finish(s, t, s_red, pw_t, pw_c, partial);
}

// The same sum with the coefficients staged through shared memory by the TMA unit: a block owns 128 KB of ONE polynomial
// (16384 coefficients); one elected thread streams it as bulk copies of 16 KB (8 k-steps) into a two-slot ring, each slot
// completing on its own mbarrier, so 16-32 KB per block are in flight whatever the register budget.  Needs d % 256 == 0.
constexpr int EV_GROUP = 8;                                   // k-steps (of 256 coefficients) per bulk copy
__global__ void __launch_bounds__(EV_THREADS) k_eval_ext_tma(const uint64_t* __restrict__ coeffs,
                                                             const uint64_t* const* __restrict__ poly_ptrs, size_t d,
                                                             const gl::ext2* __restrict__ pw_t, const gl::ext2* __restrict__ pw_k,
                                                             const gl::ext2* __restrict__ pw_c, gl::ext2* __restrict__ partial) {
    __shared__ __align__(128) uint64_t s_buf[2][EV_GROUP * EV_THREADS];   // 2 x 16 KB
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ uint32_t s_k[EV_PER_THREAD][8];
    __shared__ gl::ext2 s_red[EV_THREADS / 32];
    const unsigned t = threadIdx.x;
    if (t < EV_PER_THREAD) {
        gl::ext2 w = pw_k[t];
        gl::limbs22 la = gl::split22(w.a), lb = gl::split22(w.b);
        s_k[t][0] = la.w0; s_k[t][1] = la.w1; s_k[t][2] = la.w2; s_k[t][3] = 0;
        s_k[t][4] = lb.w0; s_k[t][5] = lb.w1; s_k[t][6] = lb.w2; s_k[t][7] = 0;
    }
    if (t == 0) {
        tma::mbar_init(&s_bar[0], 1);
        tma::mbar_init(&s_bar[1], 1);
        tma::fence_barrier_init();
    }
    __syncthreads();
    const uint64_t* poly = poly_ptrs ? poly_ptrs[blockIdx.y] : coeffs + (size_t)blockIdx.y * d;   // table: scattered polynomials
    const size_t base = (size_t)blockIdx.x * EV_CHUNK;
    const size_t left = d - base;                                            // > 0, multiple of 256
    const int n_steps = (int)(left < (size_t)EV_CHUNK ? left / EV_THREADS : EV_PER_THREAD);
    const int n_groups = (n_steps + EV_GROUP - 1) / EV_GROUP;
    auto issue = [&](int g) {
        const int steps = n_steps - g * EV_GROUP < EV_GROUP ? n_steps - g * EV_GROUP : EV_GROUP;
        const uint32_t bytes = (uint32_t)steps * EV_THREADS * 8;
        tma::mbar_arrive_expect_tx(&s_bar[g & 1], bytes);
        tma::bulk_load(s_buf[g & 1], poly + base + (size_t)g * EV_GROUP * EV_THREADS, bytes, &s_bar[g & 1]);
    };
    if (t == 0) {
        issue(0);
        if (n_groups > 1) issue(1);
    }
    gl::lazy6 A, B;
    gl::lazy_zero(A);
    gl::lazy_zero(B);
    for (int g = 0; g < n_groups; g++) {
        const int steps = n_steps - g * EV_GROUP < EV_GROUP ? n_steps - g * EV_GROUP : EV_GROUP;
        tma::mbar_wait(&s_bar[g & 1], (g >> 1) & 1);
        const uint64_t* buf = s_buf[g & 1];
        if (steps == EV_GROUP) {
#pragma unroll
            for (int k = 0; k < EV_GROUP; k++) {
                const uint64_t c = buf[k * EV_THREADS + t];
                const uint4 wa = *reinterpret_cast<const uint4*>(&s_k[g * EV_GROUP + k][0]);
                const uint4 wb = *reinterpret_cast<const uint4*>(&s_k[g * EV_GROUP + k][4]);
                gl::lazy_mac(A, c, wa.x, wa.y, wa.z);
                gl::lazy_mac(B, c, wb.x, wb.y, wb.z);
            }
        } else {
            for (int k = 0; k < steps; k++) {
                const uint64_t c = buf[k * EV_THREADS + t];
                const uint4 wa = *reinterpret_cast<const uint4*>(&s_k[g * EV_GROUP + k][0]);
                const uint4 wb = *reinterpret_cast<const uint4*>(&s_k[g * EV_GROUP + k][4]);
                gl::lazy_mac(A, c, wa.x, wa.y, wa.z);
                gl::lazy_mac(B, c, wb.x, wb.y, wb.z);
            }
        }
        __syncthreads();                                   // slot g & 1 has been read by everyone
        if (t == 0 && g + 2 < n_groups) issue(g + 2);
    }
    gl::ext2 s = {gl::lazy_reduce(A), gl::lazy_reduce(B)};
    eval_block_finish(s, t, s_red, pw_t, pw_c, partial);
}

// one block per polynomial: out[j] = sum over chunks
__global__ void __launch_bounds__(256) k_eval_sum(const gl::ext2* __restrict__ partial, size_t chunks, uint64_t* out) {
    __shared__ gl::ext2 s_red[8];
    const unsigned t = threadIdx.x;
    const gl::ext2* p = partial + (size_t)blockIdx.x * chunks;
    gl::ext2 s = {0, 0};
    for (size_t i = t; i < chunks; i += 256) {
        s.a = gl::add(s.a, p[i].a);
        s.b = gl::add(s.b, p[i].b);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        uint64_t oa = __shfl_down_sync(0xffffffffu, s.a, off), ob = __shfl_down_sync(0xffffffffu, s.b, off);
        s.a = gl::add(s.a, oa);
        s.b = gl::add(s.b, ob);
    }
    if ((t & 31) == 0) s_red[t >> 5] = s;
    __syncthreads();
    if (t == 0) {
        for (int wp = 1; wp < 8; wp++) {
            s.a = gl::add(s.a, s_red[wp].a);
            s.b = gl::add(s.b, s_red[wp].b);
        }
        out[2 * blockIdx.x] = s.a;
        out[2 * blockIdx.x + 1] = s.b;
    }
}

// ------------------------------------------------------------------------------------------------
// reduce_polys_base: F[i] = sum_j alpha^j f_j[i]   (util/reducing.rs:84-96)
// ------------------------------------------------------------------------------------------------
// One thread per coefficient index (coalesced over i for every polynomial), polynomials walked through a device pointer
// table, alpha powers broadcast from shared memory as 22-bit limbs, products accumulated carry-free (ext.cuh lazy6).
constexpr int RP_THREADS = 256, RP_TILE = 128, RP_GROUP = 8;   // polynomials per shared-memory tile of (pointer, alpha^j limbs)
constexpr int RP_FLUSH = 512;                   // polynomials per carry-free accumulation run (<= LAZY_MAX_TERMS)

__global__ void __launch_bounds__(RP_THREADS) k_reduce_polys_base(const uint64_t* const* __restrict__ polys, size_t n_polys,
                                                                  const gl::ext2* __restrict__ apow, size_t d,
                                                                  uint64_t* __restrict__ out /*[2][out_stride]*/,
                                                                  size_t out_stride) {
    __shared__ const uint64_t* s_ptr[RP_TILE];
    __shared__ uint32_t s_pw[RP_TILE][8];   // 22-bit limbs of alpha^j: a part in [0..2], b part in [4..6]
    const size_t i = (size_t)blockIdx.x * RP_THREADS + threadIdx.x;
    const bool live = i < d;
    uint64_t ra = 0, rb = 0;                // canonical running totals over the flushed runs
    gl::lazy6 A, B;
    gl::lazy_zero(A);
    gl::lazy_zero(B);
    size_t in_run = 0;
    for (size_t j0 = 0; j0 < n_polys; j0 += RP_TILE) {
        const int m = (int)(n_polys - j0 < RP_TILE ? n_polys - j0 : RP_TILE);
        __syncthreads();
        if ((int)threadIdx.x < m) {
            s_ptr[threadIdx.x] = polys[j0 + threadIdx.x];
            gl::ext2 w = apow[j0 + threadIdx.x];
            gl::limbs22 la = gl::split22(w.a), lb = gl::split22(w.b);
            uint32_t* q = s_pw[threadIdx.x];
            q[0] = la.w0; q[1] = la.w1; q[2] = la.w2; q[3] = 0;
            q[4] = lb.w0; q[5] = lb.w1; q[6] = lb.w2; q[7] = 0;
        }
        __syncthreads();
        if (live) {
            for (int j = 0; j < m; j += RP_GROUP) {   // eight loads in flight per thread
                uint64_t c[RP_GROUP];
#pragma unroll
                for (int u = 0; u < RP_GROUP; u++) c[u] = j + u < m ? s_ptr[j + u][i] : 0;
#pragma unroll
                for (int u = 0; u < RP_GROUP; u++) {
                    // rows past m hold stale limbs of an earlier tile, but their coefficient is 0
                    const uint4 wa = *reinterpret_cast<const uint4*>(&s_pw[j + u][0]);
                    const uint4 wb = *reinterpret_cast<const uint4*>(&s_pw[j + u][4]);
                    gl::lazy_mac(A, c[u], wa.x, wa.y, wa.z);
                    gl::lazy_mac(B, c[u], wb.x, wb.y, wb.z);
                }
            }
        }
        in_run += m;
        if (in_run + RP_TILE > RP_FLUSH) {   // uniform across the block
            ra = gl::add(ra, gl::canon(gl::lazy_reduce(A)));
            rb = gl::add(rb, gl::canon(gl::lazy_reduce(B)));
            gl::lazy_zero(A);
            gl::lazy_zero(B);
            in_run = 0;
        }
    }
    if (live) {
        out[i] = gl::add(ra, gl::canon(gl::lazy_reduce(A)));
        out[out_stride + i] = gl::add(rb, gl::canon(gl::lazy_reduce(B)));
    }
}

// The same reduction with the coefficients staged through shared memory by the TMA unit: a block owns 256 columns; one
// elected thread walks the polynomial pointer table and streams each polynomial's 2 KB slice as a bulk copy into a ring
// of two half-rings of 8 slices, each half completing on its own mbarrier; the block multiplies half h while the copies
// of the other half (and, after the release barrier, of the half after that) are in flight.  Needs d % 256 == 0.
constexpr int RT_COLS = 256, RT_HALF = 8, RT_SUPER = 256;    // RT_SUPER polynomials per carry-free run (limbs in smem)
__global__ void __launch_bounds__(RT_COLS) k_reduce_polys_base_tma(const uint64_t* const* __restrict__ polys, size_t n_polys,
                                                                   const gl::ext2* __restrict__ apow, size_t d,
                                                                   uint64_t* __restrict__ out, size_t out_stride) {
    __shared__ __align__(128) uint64_t s_buf[2][RT_HALF][RT_COLS];   // 2 x 16 KB
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ uint32_t s_pw[RT_SUPER][8];                            // 8 KB of alpha^j limbs
    const unsigned t = threadIdx.x;
    const size_t col0 = (size_t)blockIdx.x * RT_COLS;
    if (t == 0) {
        tma::mbar_init(&s_bar[0], 1);
        tma::mbar_init(&s_bar[1], 1);
        tma::fence_barrier_init();
    }
    uint64_t ra = 0, rb = 0;
    uint32_t uses = 0;                                                // completed uses of the half ring pair, for the phase parity
    for (size_t j0 = 0; j0 < n_polys; j0 += RT_SUPER) {
        const int m = (int)(n_polys - j0 < (size_t)RT_SUPER ? n_polys - j0 : RT_SUPER);
        __syncthreads();                                              // previous run's limbs / barriers are no longer in use
        for (int j = t; j < m; j += RT_COLS) {
            gl::ext2 w = apow[j0 + j];
            gl::limbs22 la = gl::split22(w.a), lb = gl::split22(w.b);
            uint32_t* q = s_pw[j];
            q[0] = la.w0; q[1] = la.w1; q[2] = la.w2; q[3] = 0;
            q[4] = lb.w0; q[5] = lb.w1; q[6] = lb.w2; q[7] = 0;
        }
        __syncthreads();
        const int n_groups = (m + RT_HALF - 1) / RT_HALF;
        auto issue = [&](int g) {
            const int cnt = m - g * RT_HALF < RT_HALF ? m - g * RT_HALF : RT_HALF;
            tma::mbar_arrive_expect_tx(&s_bar[g & 1], (uint32_t)cnt * RT_COLS * 8);
            for (int u = 0; u < cnt; u++)
                tma::bulk_load(s_buf[g & 1][u], polys[j0 + (size_t)g * RT_HALF + u] + col0, RT_COLS * 8, &s_bar[g & 1]);
        };
        if (t == 0) {
            issue(0);
            if (n_groups > 1) issue(1);
        }
        gl::lazy6 A, B;
        gl::lazy_zero(A);
        gl::lazy_zero(B);
        for (int g = 0; g < n_groups; g++) {
            const int cnt = m - g * RT_HALF < RT_HALF ? m - g * RT_HALF : RT_HALF;
            tma::mbar_wait(&s_bar[g & 1], ((uses + g) >> 1) & 1);
            if (cnt == RT_HALF) {
#pragma unroll
                for (int u = 0; u < RT_HALF; u++) {
                    const uint64_t c = s_buf[g & 1][u][t];
                    const uint4 wa = *reinterpret_cast<const uint4*>(&s_pw[g * RT_HALF + u][0]);
                    const uint4 wb = *reinterpret_cast<const uint4*>(&s_pw[g * RT_HALF + u][4]);
                    gl::lazy_mac(A, c, wa.x, wa.y, wa.z);
                    gl::lazy_mac(B, c, wb.x, wb.y, wb.z);
                }
            } else {
                for (int u = 0; u < cnt; u++) {
                    const uint64_t c = s_buf[g & 1][u][t];
                    const uint4 wa = *reinterpret_cast<const uint4*>(&s_pw[g * RT_HALF + u][0]);
                    const uint4 wb = *reinterpret_cast<const uint4*>(&s_pw[g * RT_HALF + u][4]);
                    gl::lazy_mac(A, c, wa.x, wa.y, wa.z);
                    gl::lazy_mac(B, c, wb.x, wb.y, wb.z);
                }
            }
            __syncthreads();                                          // half g & 1 has been read by everyone
            if (t == 0 && g + 2 < n_groups) issue(g + 2);
        }
        // keep the two barriers' phases in step for the next run: both halves must have been used equally often
        if (n_groups & 1) {
            if (t == 0) tma::mbar_arrive_expect_tx(&s_bar[1], 0);     // an empty use of half 1
            uses += n_groups + 1;
        } else {
            uses += n_groups;
        }
        ra = gl::add(ra, gl::canon(gl::lazy_reduce(A)));
        rb = gl::add(rb, gl::canon(gl::lazy_reduce(B)));
    }
    out[col0 + t] = ra;
    out[out_stride + col0 + t] = rb;
}

// ------------------------------------------------------------------------------------------------
// divide_by_linear: E[i] = sum_{k > i} c_k z^(k-i-1)   (division.rs:75-88, quotient padded with one zero)
// ------------------------------------------------------------------------------------------------
// Suffix scan in segments of SEG coefficients: H_s = segment Horner value, carry_s = the same scan over H with point
// z^SEG (recursion on the host), then every segment replays its Horner recurrence starting from its carry.
constexpr int SEG = 16;

__global__ void k_seg_horner(const uint64_t* __restrict__ c, size_t c_stride, size_t n, gl::ext2 z, uint64_t* h,
                             size_t h_stride, size_t n_seg) {
    size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    size_t lo = s * SEG, hi = lo + SEG < n ? lo + SEG : n;
    gl::ext2 acc = {0, 0};
    for (size_t i = hi; i-- > lo;) {
        gl::ext2 ci = {c[i], c[c_stride + i]};
        acc = gl::ext_add(gl::ext_mul(acc, z), ci);
    }
    h[s] = gl::canon(acc.a);
    h[h_stride + s] = gl::canon(acc.b);
}

// (no __restrict__: the scan runs in place, e == c, and the carries may live in the buffer being scanned one level up)
__global__ void k_seg_scan(const uint64_t* c, size_t c_stride, size_t n, gl::ext2 z, const uint64_t* carry,
                           size_t carry_stride, uint64_t* e, size_t e_stride, size_t n_seg) {
    size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    size_t lo = s * SEG, hi = lo + SEG < n ? lo + SEG : n;
    gl::ext2 acc = {0, 0};
    if (carry) {
        acc.a = carry[s];
        acc.b = carry[carry_stride + s];
    }
    for (size_t i = hi; i-- > lo;) {
        gl::ext2 ci = {c[i], c[c_stride + i]};   // read before the store: e may alias c
        e[i] = gl::canon(acc.a);
        e[e_stride + i] = gl::canon(acc.b);
        acc = gl::ext_add(gl::ext_mul(acc, z), ci);
    }
}

// acc[i] = acc[i] * s + q[i]   (shift_poly + AddAssign, oracle.rs:198-199)
__global__ void k_ext_scale_add(uint64_t* acc, size_t acc_stride, gl::ext2 s, const uint64_t* __restrict__ q,
                                size_t q_stride, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    gl::ext2 a = {acc[i], acc[acc_stride + i]}, qi = {q[i], q[q_stride + i]};
    a = gl::ext_add(gl::ext_mul(a, s), qi);
    acc[i] = gl::canon(a.a);
    acc[acc_stride + i] = gl::canon(a.b);
}

// ------------------------------------------------------------------------------------------------
// FRI commit phase
// ------------------------------------------------------------------------------------------------
// out[i] = sum_j beta^j c[i*arity + j]   (reduce_with_powers, plonk_common.rs:116-128)
__global__ void k_fri_fold(const uint64_t* __restrict__ c, size_t c_stride, unsigned arity_bits, gl::ext2 beta,
                           uint64_t* out, size_t out_stride, size_t n_out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_out) return;
    const size_t arity = (size_t)1 << arity_bits, base = i << arity_bits;
    gl::ext2 acc = {0, 0};
    for (size_t j = arity; j-- > 0;) {
        gl::ext2 cj = {c[base + j], c[c_stride + base + j]};
        acc = gl::ext_add(gl::ext_mul(acc, beta), cj);
    }
    out[i] = gl::canon(acc.a);
    out[out_stride + i] = gl::canon(acc.b);
}

// leaf k of a commit-phase tree = flatten(values'[k*arity .. (k+1)*arity)), values' in bit-reversed order = the LDE's
// leaf order: column 2m + e of leaf k is component e of position k*arity + m.  cols [2*arity][n_leaves] poly-major.
__global__ void k_fri_leaf_columns(const uint64_t* __restrict__ lde /*[2][n]*/, size_t n, unsigned arity_bits,
                                   uint64_t* cols, size_t n_leaves) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // = e * n + position
    if (idx >= 2 * n) return;
    size_t e = idx / n, pos = idx - e * n;
    size_t k = pos >> arity_bits, m = pos & (((size_t)1 << arity_bits) - 1);
    cols[(2 * m + e) * n_leaves + k] = lde[idx];
}

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// E = suffix scan of c (both [2][stride] component-major, n elements) at point z; e may alias c
int ext_suffix_scan(const uint64_t* c, size_t c_stride, size_t n, glh::ext2 z, uint64_t* e, size_t e_stride,
                    cudaStream_t st) {
    gl::ext2 zd = {z.a, z.b};
    if (n <= (size_t)SEG) {
        k_seg_scan<<<1, 32, 0, st>>>(c, c_stride, n, zd, nullptr, 0, e, e_stride, 1);
        PCS_CUDA(cudaGetLastError());
        return PCS_OK;
    }
    size_t n_seg = (n + SEG - 1) / SEG;
    DevBuf h;
    PCS_CUDA(h.alloc(2 * n_seg * 8, st));
    k_seg_horner<<<blocks_for(n_seg, 128), 128, 0, st>>>(c, c_stride, n, zd, h.u64(), n_seg, n_seg);
    PCS_CUDA(cudaGetLastError());
    int rc = ext_suffix_scan(h.u64(), n_seg, n_seg, glh::ext_pow(z, SEG), h.u64(), n_seg, st);   // carries, in place
    if (rc) return rc;
    k_seg_scan<<<blocks_for(n_seg, 128), 128, 0, st>>>(c, c_stride, n, zd, h.u64(), n_seg, e, e_stride, n_seg);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

int pow_table(glh::ext2 base, size_t n, gl::ext2* out, cudaStream_t st) {
    gl::ext2 b = {base.a % glh::P, base.b % glh::P};
    k_ext_pow_table<<<blocks_for(n, 128), 128, 0, st>>>(b, n, out);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------
// coeffs: contiguous [w][d] device matrix, or (coeffs == nullptr) polys: HOST array of w device pointers
static int eval_ext_common(const uint64_t* coeffs, const uint64_t* const* polys, size_t w, unsigned lg_d,
                           const uint64_t point[2], uint64_t* out) {
    cudaStream_t st = (cudaStream_t)pcs_stream();
    const size_t d = (size_t)1 << lg_d, chunks = (d + EV_CHUNK - 1) / EV_CHUNK;
    glh::ext2 z = {point[0] % glh::P, point[1] % glh::P};
    DevBuf tabs, partial, res, table;
    bool aligned = true;
    if (!coeffs) {
        for (size_t j = 0; j < w; j++) {
            if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
            aligned = aligned && ((uintptr_t)polys[j] % 16 == 0);
        }
        PCS_CUDA(table.alloc(w * sizeof(uint64_t*), st));
        PCS_CUDA(cudaMemcpyAsync(table.p, polys, w * sizeof(uint64_t*), cudaMemcpyHostToDevice, st));
    }
    const uint64_t* const* ptrs = coeffs ? nullptr : (const uint64_t* const*)table.p;
    PCS_CUDA(tabs.alloc((EV_THREADS + EV_PER_THREAD + chunks) * sizeof(gl::ext2), st));
    PCS_CUDA(partial.alloc(w * chunks * sizeof(gl::ext2), st));
    PCS_CUDA(res.alloc(w * 16, st));
    gl::ext2* pw_t = (gl::ext2*)tabs.p;
    gl::ext2* pw_k = pw_t + EV_THREADS;
    gl::ext2* pw_c = pw_k + EV_PER_THREAD;
    int rc;
    if ((rc = pow_table(z, EV_THREADS, pw_t, st))) return rc;
    if ((rc = pow_table(glh::ext_pow(z, EV_THREADS), EV_PER_THREAD, pw_k, st))) return rc;
    if ((rc = pow_table(glh::ext_pow(z, EV_CHUNK), chunks, pw_c, st))) return rc;
    if (d % EV_THREADS == 0 && aligned)   // TMA-staged (rows of a [w][d] matrix with d >= 256 are 16-byte aligned)
        k_eval_ext_tma<<<dim3((unsigned)chunks, (unsigned)w), EV_THREADS, 0, st>>>(coeffs, ptrs, d, pw_t, pw_k, pw_c,
                                                                                   (gl::ext2*)partial.p);
    else
        k_eval_ext<<<dim3((unsigned)chunks, (unsigned)w), EV_THREADS, 0, st>>>(coeffs, ptrs, d, pw_t, pw_k, pw_c,
                                                                               (gl::ext2*)partial.p);
    PCS_CUDA(cudaGetLastError());
    k_eval_sum<<<(unsigned)w, 256, 0, st>>>((const gl::ext2*)partial.p, chunks, res.u64());
    PCS_CUDA(cudaGetLastError());
    PCS_CUDA(cudaMemcpyAsync(out, res.p, w * 16, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_eval_ext(const pcs_batch* b, const uint64_t point[2], uint64_t* out) {
    if (int rc = need_init()) return rc;
    if (!b || !point || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (!b->coeffs) return fail(PCS_ERR_ARG, "coefficients were not kept (PCS_KEEP_COEFFS)");
    BatchScope scope(b);
    return eval_ext_common(b->coeffs, nullptr, b->w, b->lg_d, point, out);
}

int pcs_eval_ext_dev(const uint64_t* const* polys_dev, size_t w, unsigned lg_d, const uint64_t point[2], uint64_t* out) {
    if (int rc = need_init()) return rc;
    if (w == 0) return PCS_OK;
    if (!polys_dev || !point || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (int rc = check_two_adicity(lg_d)) return rc;
    return eval_ext_common(nullptr, polys_dev, w, lg_d, point, out);
}

// ------------------------------------------------------------------------------------------------
static int ext_poly_alloc(size_t len, pcs_ext_poly** out, cudaStream_t st) {
    pcs_ext_poly* p = new pcs_ext_poly();
    p->len = len;
    p->cap = len ? len : 1;
    p->ctx = cur_ctx();
    cudaError_t e = cudaMallocAsync((void**)&p->c, 2 * p->cap * 8, st);
    if (e != cudaSuccess) {
        delete p;
        set_error(std::string("cudaMallocAsync: ") + cudaGetErrorString(e));
        return PCS_ERR_CUDA;
    }
    *out = p;
    return PCS_OK;
}

int pcs_ext_poly_new(const uint64_t* coeffs, size_t len, pcs_ext_poly** out) {
    if (int rc = need_init()) return rc;
    if (!out || (len && !coeffs)) return fail(PCS_ERR_ARG, "NULL pointer");
    *out = nullptr;
    cudaStream_t st = (cudaStream_t)pcs_stream();
    pcs_ext_poly* p = nullptr;
    int rc = ext_poly_alloc(len, &p, st);
    if (rc) return rc;
    if (len) {
        DevBuf tmp;
        cudaError_t e = tmp.alloc(len * 16, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(tmp.p, coeffs, len * 16, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) {
            k_deinterleave<<<blocks_for(len, 256), 256, 0, st>>>(tmp.u64(), len, p->c, p->cap);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // the caller may reuse `coeffs`
        if (e != cudaSuccess) {
            pcs_ext_poly_free(p);
            set_error(std::string("pcs_ext_poly_new: ") + cudaGetErrorString(e));
            return PCS_ERR_CUDA;
        }
    }
    *out = p;
    return PCS_OK;
}

int pcs_ext_poly_len(const pcs_ext_poly* p, size_t* len) {
    if (!p || !len) return fail(PCS_ERR_ARG, "NULL pointer");
    *len = p->len;
    return PCS_OK;
}

int pcs_ext_poly_read(const pcs_ext_poly* p, uint64_t* coeffs) {
    if (!p) return fail(PCS_ERR_ARG, "NULL pointer");
    if (p->len == 0) return PCS_OK;
    if (!coeffs) return fail(PCS_ERR_ARG, "NULL pointer");
    CtxScope scope(p->ctx);
    cudaStream_t st = (cudaStream_t)pcs_stream();
    DevBuf tmp;
    PCS_CUDA(tmp.alloc(p->len * 16, st));
    k_interleave<<<blocks_for(p->len, 256), 256, 0, st>>>(p->c, p->cap, p->len, tmp.u64());
    PCS_CUDA(cudaGetLastError());
    PCS_CUDA(cudaMemcpyAsync(coeffs, tmp.p, p->len * 16, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

void pcs_ext_poly_free(pcs_ext_poly* p) {
    if (!p) return;
    CtxScope scope(p->ctx);
    if (p->c) cudaFreeAsync(p->c, (cudaStream_t)pcs_stream());
    delete p;
}

// ------------------------------------------------------------------------------------------------
// ptrs: `total` device pointers to d = 2^lg_d coefficients each, batch after batch
static int final_poly_common(const std::vector<const uint64_t*>& ptrs, unsigned lg_d, size_t n_batches, const uint64_t* points,
                             const size_t* batch_len, const uint64_t alpha[2], pcs_ext_poly** out) {
    cudaStream_t st = (cudaStream_t)pcs_stream();
    const size_t d = (size_t)1 << lg_d, total = ptrs.size();
    size_t longest = 0;
    bool aligned = true;
    for (size_t i = 0; i < n_batches; i++) longest = batch_len[i] > longest ? batch_len[i] : longest;
    for (auto q : ptrs) aligned = aligned && ((uintptr_t)q % 16 == 0);
    const glh::ext2 a = {alpha[0] % glh::P, alpha[1] % glh::P};
    pcs_ext_poly* fin = nullptr;
    int rc = ext_poly_alloc(d, &fin, st);
    if (rc) return rc;
    struct Guard { pcs_ext_poly* p; bool armed = true; ~Guard() { if (armed) pcs_ext_poly_free(p); } } guard{fin};
    DevBuf table, apow, comp;
    PCS_CUDA(table.alloc(total * sizeof(uint64_t*), st));
    PCS_CUDA(apow.alloc(longest * sizeof(gl::ext2), st));
    PCS_CUDA(comp.alloc(2 * d * 8, st));
    PCS_CUDA(cudaMemcpyAsync(table.p, ptrs.data(), total * sizeof(uint64_t*), cudaMemcpyHostToDevice, st));
    if ((rc = pow_table(a, longest, (gl::ext2*)apow.p, st))) return rc;
    PCS_CUDA(cudaMemsetAsync(fin->c, 0, 2 * fin->cap * 8, st));   // PolynomialCoeffs::empty()
    size_t first = 0;
    for (size_t i = 0; i < n_batches; i++) {
        const size_t m = batch_len[i];
        if (d % RT_COLS == 0 && aligned)   // TMA-staged
            k_reduce_polys_base_tma<<<(unsigned)(d / RT_COLS), RT_COLS, 0, st>>>(
                (const uint64_t* const*)table.p + first, m, (const gl::ext2*)apow.p, d, comp.u64(), d);
        else
            k_reduce_polys_base<<<blocks_for(d, RP_THREADS), RP_THREADS, 0, st>>>(
                (const uint64_t* const*)table.p + first, m, (const gl::ext2*)apow.p, d, comp.u64(), d);
        PCS_CUDA(cudaGetLastError());
        const glh::ext2 z = {points[2 * i] % glh::P, points[2 * i + 1] % glh::P};
        if ((rc = ext_suffix_scan(comp.u64(), d, d, z, comp.u64(), d, st))) return rc;     // quotient, last coefficient 0
        const glh::ext2 s = glh::ext_pow(a, m);                                             // alpha^count
        k_ext_scale_add<<<blocks_for(d, 256), 256, 0, st>>>(fin->c, fin->cap, gl::ext2{s.a, s.b}, comp.u64(), d, d);
        PCS_CUDA(cudaGetLastError());
        first += m;
    }
    PCS_CUDA(cudaStreamSynchronize(st));   // `ptrs` (host) was copied asynchronously
    guard.armed = false;
    *out = fin;
    return PCS_OK;
}

int pcs_fri_final_poly(const pcs_batch* const* oracles, size_t n_oracles, size_t n_batches, const uint64_t* points,
                       const size_t* batch_len, const uint32_t* oracle_index, const uint32_t* poly_index,
                       const uint64_t alpha[2], pcs_ext_poly** out) {
    if (int rc = need_init()) return rc;
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!oracles || !n_oracles || !n_batches || !points || !batch_len || !oracle_index || !poly_index || !alpha)
        return fail(PCS_ERR_ARG, "NULL pointer or empty instance");
    for (size_t o = 0; o < n_oracles; o++) {
        if (!oracles[o]) return fail(PCS_ERR_ARG, "NULL oracle");
        if (!oracles[o]->coeffs) return fail(PCS_ERR_ARG, "coefficients were not kept (PCS_KEEP_COEFFS)");
        if (oracles[o]->lg_d != oracles[0]->lg_d) return fail(PCS_ERR_ARG, "oracles of different degrees");
    }
    for (size_t o = 1; o < n_oracles; o++)
        if (oracles[o]->ctx != oracles[0]->ctx) return fail(PCS_ERR_ARG, "oracles live on different devices");
    BatchScope scope(oracles[0]);
    const unsigned lg_d = oracles[0]->lg_d;
    const size_t d = (size_t)1 << lg_d;
    size_t total = 0;
    for (size_t i = 0; i < n_batches; i++) {
        if (batch_len[i] == 0) return fail(PCS_ERR_ARG, "empty FRI batch");
        total += batch_len[i];
    }
    std::vector<const uint64_t*> ptrs(total);
    for (size_t k = 0; k < total; k++) {
        if (oracle_index[k] >= n_oracles) return fail(PCS_ERR_ARG, "oracle index out of bounds");
        const pcs_batch* o = oracles[oracle_index[k]];
        if (poly_index[k] >= o->w) return fail(PCS_ERR_ARG, "polynomial index out of bounds");
        ptrs[k] = o->coeffs + (size_t)poly_index[k] * d;
    }
    return final_poly_common(ptrs, lg_d, n_batches, points, batch_len, alpha, out);
}

int pcs_fri_final_poly_dev(const uint64_t* const* polys_dev, unsigned lg_d, size_t n_batches, const uint64_t* points,
                           const size_t* batch_len, const uint64_t alpha[2], pcs_ext_poly** out) {
    if (int rc = need_init()) return rc;
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!polys_dev || !n_batches || !points || !batch_len || !alpha) return fail(PCS_ERR_ARG, "NULL pointer or empty instance");
    if (int rc = check_two_adicity(lg_d)) return rc;
    size_t total = 0;
    for (size_t i = 0; i < n_batches; i++) {
        if (batch_len[i] == 0) return fail(PCS_ERR_ARG, "empty FRI batch");
        total += batch_len[i];
    }
    std::vector<const uint64_t*> ptrs(polys_dev, polys_dev + total);
    for (auto q : ptrs)
        if (!q) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
    return final_poly_common(ptrs, lg_d, n_batches, points, batch_len, alpha, out);
}

// ------------------------------------------------------------------------------------------------
// LDE of both components into lde [2][n] (leaf order)
static int ext_lde(const pcs_ext_poly* p, unsigned rate_bits, uint64_t shift, uint64_t* lde, unsigned* lg_n_out,
                   cudaStream_t st) {
    int lg_d = ilog2_strict(p->len);
    if (lg_d < 0) return fail(PCS_ERR_NOT_POW2, "Not a power of two: " + std::to_string(p->len));
    if (int rc = check_two_adicity((unsigned)lg_d + rate_bits)) return rc;
    if (int rc = check_shift(shift)) return rc;
    NttPlan* plan = ntt_plan_get((unsigned)lg_d, rate_bits, false, shift % glh::P, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    const size_t n = p->len << rate_bits;
    PCS_CUDA(ntt_lde(plan, p->c, p->cap, lde, n, 2, st));
    *lg_n_out = (unsigned)lg_d + rate_bits;
    return PCS_OK;
}

int pcs_ext_coset_lde(const pcs_ext_poly* p, unsigned rate_bits, uint64_t shift, uint64_t* values) {
    if (int rc = need_init()) return rc;
    if (!p || !values) return fail(PCS_ERR_ARG, "NULL pointer");
    CtxScope scope(p->ctx);
    cudaStream_t st = (cudaStream_t)pcs_stream();
    if (p->len == 0) return fail(PCS_ERR_ARG, "empty polynomial");
    const size_t n = p->len << rate_bits;
    DevBuf lde, o;
    PCS_CUDA(lde.alloc(2 * n * 8, st));
    PCS_CUDA(o.alloc(2 * n * 8, st));
    unsigned lg_n = 0;
    int rc = ext_lde(p, rate_bits, shift, lde.u64(), &lg_n, st);
    if (rc) return rc;
    k_interleave_bitrev<<<blocks_for(n, 256), 256, 0, st>>>(lde.u64(), n, lg_n, o.u64());
    PCS_CUDA(cudaGetLastError());
    PCS_CUDA(cudaMemcpyAsync(values, o.p, 2 * n * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_fri_commit_layer(const pcs_ext_poly* p, unsigned rate_bits, uint64_t shift, unsigned arity_bits,
                         unsigned cap_height, uint64_t* cap_out, pcs_batch** tree) {
    if (int rc = need_init()) return rc;
    if (!tree) return fail(PCS_ERR_ARG, "tree is NULL");
    *tree = nullptr;
    if (!p || p->len == 0) return fail(PCS_ERR_ARG, "NULL or empty polynomial");
    CtxScope scope(p->ctx);           // the tree is built (and its batch bound) where the polynomial lives
    cudaStream_t st = (cudaStream_t)pcs_stream();
    int lg_d = ilog2_strict(p->len);
    if (lg_d < 0) return fail(PCS_ERR_NOT_POW2, "Not a power of two: " + std::to_string(p->len));
    const unsigned lg_n = (unsigned)lg_d + rate_bits;
    if (arity_bits > lg_n) return fail(PCS_ERR_ARG, "arity larger than the LDE");
    const unsigned lg_leaves = lg_n - arity_bits;
    const size_t n = (size_t)1 << lg_n, n_leaves = (size_t)1 << lg_leaves, width = (size_t)2 << arity_bits;
    const size_t n_cap = (size_t)1 << cap_height;
    BatchOwner b;   // a tree over rows written here, without phase events
    if (int rc = batch_begin(width, 0, lg_leaves, 0, 0, 0, cap_height, BATCH_ROWS | BATCH_UNTIMED, b)) return rc;
    DevBuf lde;
    PCS_CUDA(lde.alloc(2 * n * 8, st));
    unsigned lg_n2 = 0;
    int rc = ext_lde(p, rate_bits, shift, lde.u64(), &lg_n2, st);
    if (rc) return rc;
    k_fri_leaf_columns<<<blocks_for(2 * n, 256), 256, 0, st>>>(lde.u64(), n, arity_bits, b->lde, n_leaves);
    PCS_CUDA(cudaGetLastError());
    rc = build_tree_dev(b->lde, n_leaves, width, lg_leaves, cap_height, b->digests, b->cap, st, nullptr);
    if (rc) return rc;
    if (cap_out) {
        PCS_CUDA(cudaMemcpyAsync(cap_out, b->cap, n_cap * 32, cudaMemcpyDeviceToHost, st));
        PCS_CUDA(cudaStreamSynchronize(st));
    }
    *tree = b.release();
    return PCS_OK;
}

int pcs_fri_fold(pcs_ext_poly* p, unsigned arity_bits, const uint64_t beta[2]) {
    if (int rc = need_init()) return rc;
    if (!p || !beta) return fail(PCS_ERR_ARG, "NULL pointer");
    if (arity_bits == 0) return PCS_OK;
    if (arity_bits > 31 || (p->len & (((size_t)1 << arity_bits) - 1)) || p->len == 0)
        return fail(PCS_ERR_ARG, "polynomial length is not a multiple of the arity (par_chunks_exact would drop coefficients)");
    CtxScope scope(p->ctx);
    cudaStream_t st = (cudaStream_t)pcs_stream();
    const size_t n_out = p->len >> arity_bits;
    DevBuf o;
    PCS_CUDA(o.alloc(2 * n_out * 8, st));
    gl::ext2 b = {beta[0] % glh::P, beta[1] % glh::P};
    k_fri_fold<<<blocks_for(n_out, 128), 128, 0, st>>>(p->c, p->cap, arity_bits, b, o.u64(), n_out, n_out);
    PCS_CUDA(cudaGetLastError());
    PCS_CUDA(cudaMemcpyAsync(p->c, o.p, n_out * 8, cudaMemcpyDeviceToDevice, st));
    PCS_CUDA(cudaMemcpyAsync(p->c + p->cap, o.u64() + n_out, n_out * 8, cudaMemcpyDeviceToDevice, st));
    p->len = n_out;
    return PCS_OK;
}

}  // extern "C"
