// Rows of an on-demand batch (PCS_LDE_ON_DEMAND) at a few leaves, evaluated from its kept coefficients instead of a
// regenerated LDE: rows[k][j] = P_j(x_k) = sum_i c_j[i] x_k^i with x_k = 7 * w_N^{brev_{log N}(leaf_k)}, the point of leaf k
// (the leaf order is the bit-reversed natural order of the coset 7 <w_N>, oracle.rs:84).  This serves the FRI query phase
// (fri/prover.rs:183-216: num_query_rounds rows per initial tree), where regenerating the LDE would cost a whole LDE.
//
// The sum is the base-field form of eval_commitment's (fri.cu k_eval_ext): a block owns 16384 coefficients of one
// polynomial, thread t sums c[t + 256 k] (x^256)^k over k < 64 with the multipliers held as 22-bit limbs in shared memory, so
// a coefficient costs six IMAD.WIDE.U32 per point into carry-free accumulators (ext.cuh lazy6).  A block serves RE_POINTS
// points per coefficient it loads: 48 multiply-adds per 8-byte load make the kernel compute bound, so the loads are plain
// coalesced ones, not TMA-staged like k_eval_ext_tma's (which does 12 multiply-adds per load and is bound by HBM).
#include "common.cuh"
#include "ext.cuh"

namespace pcs {
namespace {

constexpr int RE_THREADS = 256, RE_PER_THREAD = 64, RE_CHUNK = RE_THREADS * RE_PER_THREAD;
constexpr int RE_POINTS = 8;    // points per tile: 8 accumulators of 12 registers; -Xptxas -v: 128 registers (two blocks per SM), no spills
constexpr int RE_BATCH = 2;     // coefficients loaded ahead of their multiply-adds (4 spills at RE_POINTS = 8)
// per point: x^t (t < 256), x^(256 k) (k < 64), then x^(16384 c) for every chunk c
constexpr size_t TAB_T = 0, TAB_K = RE_THREADS, TAB_C = RE_THREADS + RE_PER_THREAD;

// tabs[k][..] for every point k (leaf idx[k], or leaf 0 for the padding of the last tile)
__global__ void k_point_tables(const uint64_t* __restrict__ idx, size_t n, size_t n_pad, unsigned lg_n, uint64_t root,
                               size_t chunks, uint64_t* __restrict__ tabs) {
    const size_t per = TAB_C + chunks;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad * per) return;
    const size_t k = i / per, e = i % per;
    const size_t leaf = k < n ? idx[k] : 0;
    const uint64_t br = brev_bits(leaf, lg_n);
    const uint64_t x = gl::canon(gl::mul(7, gl::pow(root, br)));   // F::coset_shift() = 7 (types.rs:437)
    const uint64_t ex = e < TAB_K ? e : e < TAB_C ? (uint64_t)(e - TAB_K) * RE_THREADS : (uint64_t)(e - TAB_C) * RE_CHUNK;
    tabs[i] = gl::pow(x, ex);
}

// grid (chunks, polynomials, tiles): block (c, j, tile) writes partial[k][j][c] = x_k^(16384 c) sum_t x_k^t S_t for the
// RE_POINTS points k of the tile, S_t = sum_k' c_j[16384 c + t + 256 k'] (x_k^256)^k'.
__global__ void __launch_bounds__(RE_THREADS, 2) k_rows_eval(const uint64_t* __restrict__ coeffs, size_t d,
                                                             const uint64_t* __restrict__ tabs, size_t chunks, size_t w,
                                                             size_t j_first, uint64_t* __restrict__ partial) {
    __shared__ uint4 s_k[RE_POINTS][RE_PER_THREAD];   // 22-bit limbs of (x_p^256)^k
    __shared__ uint64_t s_red[RE_POINTS][RE_THREADS / 32];
    const unsigned t = threadIdx.x;
    const size_t per = TAB_C + chunks, p0 = (size_t)blockIdx.z * RE_POINTS, j = j_first + blockIdx.y;
    for (unsigned i = t; i < RE_POINTS * RE_PER_THREAD; i += RE_THREADS) {
        const unsigned p = i / RE_PER_THREAD, k = i % RE_PER_THREAD;
        const gl::limbs22 l = gl::split22(tabs[(p0 + p) * per + TAB_K + k]);
        s_k[p][k] = make_uint4(l.w0, l.w1, l.w2, 0);
    }
    __syncthreads();
    const uint64_t* poly = coeffs + j * d;
    const size_t base = (size_t)blockIdx.x * RE_CHUNK + t;
    gl::lazy6 A[RE_POINTS];   // 64 terms each: far below LAZY_MAX_TERMS
#pragma unroll
    for (int p = 0; p < RE_POINTS; p++) gl::lazy_zero(A[p]);
#pragma unroll 1
    for (int k0 = 0; k0 < RE_PER_THREAD; k0 += RE_BATCH) {
        uint64_t c[RE_BATCH];
#pragma unroll
        for (int k = 0; k < RE_BATCH; k++) {
            const size_t i = base + (size_t)(k0 + k) * RE_THREADS;
            c[k] = i < d ? poly[i] : 0;
        }
#pragma unroll
        for (int k = 0; k < RE_BATCH; k++)
#pragma unroll
            for (int p = 0; p < RE_POINTS; p++) {
                const uint4 l = s_k[p][k0 + k];
                gl::lazy_mac(A[p], c[k], l.x, l.y, l.z);
            }
    }
#pragma unroll
    for (int p = 0; p < RE_POINTS; p++) {
        uint64_t s = gl::canon(gl::mul(gl::canon(gl::lazy_reduce(A[p])), tabs[(p0 + p) * per + TAB_T + t]));
#pragma unroll
        for (int off = 16; off; off >>= 1) s = gl::add(s, __shfl_down_sync(0xffffffffu, s, off));
        if ((t & 31) == 0) s_red[p][t >> 5] = s;
    }
    __syncthreads();
    if (t < RE_POINTS) {
        uint64_t s = s_red[t][0];
        for (int wp = 1; wp < RE_THREADS / 32; wp++) s = gl::add(s, s_red[t][wp]);
        partial[((p0 + t) * w + j) * chunks + blockIdx.x] = gl::canon(gl::mul(s, tabs[(p0 + t) * per + TAB_C + blockIdx.x]));
    }
}

// one warp per (point k, column j): rows[k][j] = sum of the chunks' partials; salt columns j >= w are gathered from the
// batch's salt rows (leaf order, canonical)
__global__ void k_rows_sum(const uint64_t* __restrict__ partial, size_t chunks, size_t w, size_t salt_w,
                           const uint64_t* __restrict__ salts, size_t n_leaves, const uint64_t* __restrict__ idx, size_t n,
                           uint64_t* __restrict__ rows) {
    const size_t wt = w + salt_w, wid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const unsigned lane = threadIdx.x & 31;
    if (wid >= n * wt) return;
    const size_t k = wid / wt, j = wid % wt;
    if (j >= w) {
        if (lane == 0) rows[k * wt + j] = salts[(j - w) * n_leaves + idx[k]];
        return;
    }
    const uint64_t* p = partial + (k * w + j) * chunks;
    uint64_t s = 0;
    for (size_t i = lane; i < chunks; i += 32) s = gl::add(s, p[i]);
#pragma unroll
    for (int off = 16; off; off >>= 1) s = gl::add(s, __shfl_down_sync(0xffffffffu, s, off));
    if (lane == 0) rows[k * wt + j] = s;
}

}  // namespace

int rows_eval(const pcs_batch* b, const uint64_t* idx_dev, size_t n, uint64_t* out_dev, cudaStream_t st) {
    if (n == 0) return PCS_OK;
    const size_t d = (size_t)1 << b->lg_d, chunks = (d + RE_CHUNK - 1) / RE_CHUNK;
    const size_t tiles = (n + RE_POINTS - 1) / RE_POINTS, n_pad = tiles * RE_POINTS, per = TAB_C + chunks;
    const unsigned lg_n = b->lg_d + b->rate_bits;
    const uint64_t root = glh::primitive_root_of_unity(lg_n);
    DevBuf tabs, partial;
    PCS_CUDA(tabs.alloc(n_pad * per * 8, st));
    PCS_CUDA(partial.alloc(n_pad * b->w * chunks * 8, st));
    k_point_tables<<<(unsigned)((n_pad * per + 255) / 256), 256, 0, st>>>(idx_dev, n, n_pad, lg_n, root, chunks, tabs.u64());
    PCS_CUDA(cudaGetLastError());
    for (size_t t0 = 0; t0 < tiles; t0 += 65535)
        for (size_t j0 = 0; j0 < b->w; j0 += 65535) {
            const size_t nt = tiles - t0 < 65535 ? tiles - t0 : 65535, nj = b->w - j0 < 65535 ? b->w - j0 : 65535;
            k_rows_eval<<<dim3((unsigned)chunks, (unsigned)nj, (unsigned)nt), RE_THREADS, 0, st>>>(
                b->coeffs, d, tabs.u64() + t0 * RE_POINTS * per, chunks, b->w, j0, partial.u64() + t0 * RE_POINTS * b->w * chunks);
            PCS_CUDA(cudaGetLastError());
        }
    const size_t warps = n * (b->w + b->salt_w);
    k_rows_sum<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(partial.u64(), chunks, b->w, b->salt_w, b->salts, b->n, idx_dev, n,
                                                         out_dev);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

}  // namespace pcs
