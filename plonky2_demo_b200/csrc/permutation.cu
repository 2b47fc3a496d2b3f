// The permutation argument's Z and partial-product polynomials on the device:
//
//   pcs_permutation_partial_products   all_wires_permutation_partial_products    plonky2/src/plonk/prover.rs
//                                      = wires_permutation_partial_products_and_zs per challenge (plonk/prover.rs),
//                                        quotient_chunk_products / partial_products_and_z_gx (util/partial_products.rs)
//
// Three steps, all challenges of a launch from ONE read of the wire and sigma columns:
//   1. k_perm_rows   row i, challenge c: the chunk products N_k = prod num_j and D_k = prod den_j over the wires of chunk k,
//                    their prefixes NP_k, DP_k, and ONE inversion of DP_{K-1} per row (shared by the challenges of the launch
//                    through Montgomery's trick).  Walking back, 1/DP_k = 1/DP_{k+1} * D_{k+1}, so the row-local prefixes
//                    Q_0 .. Q_k = NP_k / DP_k go to the partial-product outputs and the row total T_i = NP_{K-1} / DP_{K-1}
//                    to a [C][n] scratch.  Exact field arithmetic: inverting the chunk denominators' product instead of
//                    every den_j (batch_multiplicative_inverse) gives the same values, and the product is zero exactly when
//                    one den_j is, which raises the device flag behind "Tried to invert zero".
//   2. the scan      Z(x_0) = 1, Z(x_{i+1}) = Z(x_i) T_i: an exclusive multiplicative reduce-then-scan over tiles of 4096 rows
//                    (tile products, one block scanning the tile products, each tile rescanned with its prefix).
//   3. k_mul_z       pp_k(x_i) = Z(x_i) * (Q_0 .. Q_k)(x_i), canonical.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "gl64.cuh"

using namespace pcs;

namespace {

constexpr int ROW_THREADS_MAX = 256;
constexpr size_t ROW_SMEM_TARGET = 64u << 10;   // per block: several blocks per SM
constexpr int MAX_NC = 4;                        // challenges per pass over the inputs
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 16, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;
constexpr int PART_THREADS = 1024;

// out[i] = base^i, i < n (canonical)
__global__ void k_pow_table(uint64_t base, size_t n, uint64_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = gl::pow(base, i);
}

// Step 1 for NC challenges.  wires / sigmas: device tables of R column pointers; bk [NC][R] = beta_c k_j, beta / gamma [NC]
// (all canonical); pp: device table of NC * P column pointers (challenge-major); T [NC][n].  Shared memory per thread and
// challenge: NP_k and D_{k+1} for k < P, at sm[((k * NC + c) * 2 + e) * blockDim + tid] (conflict-free).
template <int NC>
__global__ void __launch_bounds__(ROW_THREADS_MAX) k_perm_rows(
    const uint64_t* const* __restrict__ wires, const uint64_t* const* __restrict__ sigmas, unsigned R, unsigned D, unsigned P,
    size_t n, const uint64_t* __restrict__ x_lo, const uint64_t* __restrict__ x_hi, const uint64_t* __restrict__ bk,
    const uint64_t* __restrict__ beta, const uint64_t* __restrict__ gamma, uint64_t* const* __restrict__ pp,
    uint64_t* __restrict__ T, unsigned* zero_flag) {
    extern __shared__ uint64_t sm[];
    const unsigned tid = threadIdx.x, bd = blockDim.x;
    const size_t i = (size_t)blockIdx.x * bd + tid;
    if (i >= n) return;
    const uint64_t x = subgroup_point(x_lo, x_hi, i);
    uint64_t np[NC], dp[NC], b[NC], g[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) {
        np[c] = 1;
        dp[c] = 1;
        b[c] = beta[c];
        g[c] = gamma[c];
    }
    unsigned j = 0;
    for (unsigned k = 0; k <= P; k++) {
        const unsigned j1 = min(j + D, R);
        uint64_t nk[NC], dk[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) nk[c] = dk[c] = 1;
#pragma unroll 2
        for (; j < j1; j++) {
            const uint64_t w = gl::canon(__ldg(wires[j] + i)), s = gl::canon(__ldg(sigmas[j] + i));
#pragma unroll
            for (int c = 0; c < NC; c++) {
                const uint64_t wg = gl::add_lc(w, g[c]);
                const uint64_t num = gl::add_lc(wg, gl::canon(gl::mul(bk[c * R + j], x)));   // w + beta k_j x + gamma
                const uint64_t den = gl::add_lc(wg, gl::canon(gl::mul(b[c], s)));            // w + beta sigma_j + gamma
                nk[c] = gl::mul(nk[c], num);
                dk[c] = gl::mul(dk[c], den);
            }
        }
#pragma unroll
        for (int c = 0; c < NC; c++) {
            np[c] = gl::mul(np[c], nk[c]);
            dp[c] = gl::mul(dp[c], dk[c]);
            if (k < P) sm[((k * NC + c) * 2) * bd + tid] = np[c];
            if (k > 0) sm[(((k - 1) * NC + c) * 2 + 1) * bd + tid] = dk[c];
        }
    }
    // one inversion for the NC row denominators (Montgomery's trick)
    uint64_t pre[NC], acc = 1;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        pre[c] = acc;
        acc = gl::mul(acc, dp[c]);
    }
    acc = gl::canon(acc);
    if (acc == 0) *zero_flag = 1;
    uint64_t inv = inverse(acc), inv_c[NC];
#pragma unroll
    for (int c = NC - 1; c >= 0; c--) {
        inv_c[c] = gl::mul(inv, pre[c]);   // 1 / DP_{K-1} of challenge c
        inv = gl::mul(inv, dp[c]);
    }
#pragma unroll
    for (int c = 0; c < NC; c++) {
        T[c * n + i] = gl::mul(np[c], inv_c[c]);
        uint64_t v = inv_c[c];
        for (int k = (int)P - 1; k >= 0; k--) {
            v = gl::mul(v, sm[(((unsigned)k * NC + c) * 2 + 1) * bd + tid]);   // 1 / DP_k
            pp[c * P + k][i] = gl::mul(sm[(((unsigned)k * NC + c) * 2) * bd + tid], v);
        }
    }
}

// Multiplicative scans over a block (blockDim.x = 32 * warps, warps <= 32): returns the exclusive prefix of v, *total the
// product of all v.  ws: 32 words of shared memory.
__device__ __forceinline__ uint64_t block_exclusive_scan(uint64_t v, uint64_t* ws, uint64_t* total) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint64_t inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint64_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= (unsigned)off) inc = gl::mul(inc, o);
    }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint64_t t = lane < nw ? ws[lane] : 1;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint64_t o = __shfl_up_sync(0xffffffffu, t, off);
            if (lane >= (unsigned)off) t = gl::mul(t, o);
        }
        ws[lane] = t;   // inclusive over warps
    }
    __syncthreads();
    uint64_t exc = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) exc = 1;
    if (warp > 0) exc = gl::mul(exc, ws[warp - 1]);
    *total = ws[nw - 1];
    __syncthreads();   // ws is reused by the caller's next scan
    return exc;
}

// product of each tile of SCAN_TILE rows of T[c] -> part[c][tile]
__global__ void __launch_bounds__(SCAN_THREADS) k_tile_product(const uint64_t* __restrict__ T, size_t n, size_t tiles,
                                                               uint64_t* __restrict__ part) {
    __shared__ uint64_t ws[32];
    const unsigned c = blockIdx.y;
    const size_t base = (size_t)blockIdx.x * SCAN_TILE;
    uint64_t acc = 1;
    for (unsigned r = threadIdx.x; r < SCAN_TILE; r += SCAN_THREADS)
        if (base + r < n) acc = gl::mul(acc, T[c * n + base + r]);
    uint64_t total;
    block_exclusive_scan(acc, ws, &total);
    if (threadIdx.x == 0) part[c * tiles + blockIdx.x] = total;
}

// exclusive scan of part[c][0 .. tiles) in place, one block per challenge
__global__ void __launch_bounds__(PART_THREADS) k_scan_parts(uint64_t* part, size_t tiles) {
    __shared__ uint64_t ws[32];
    uint64_t* p = part + (size_t)blockIdx.x * tiles;
    uint64_t carry = 1;
    for (size_t base = 0; base < tiles; base += PART_THREADS) {
        const size_t r = base + threadIdx.x;
        uint64_t total;
        const uint64_t exc = block_exclusive_scan(r < tiles ? p[r] : 1, ws, &total);
        if (r < tiles) p[r] = gl::mul(carry, exc);
        carry = gl::mul(carry, total);
    }
}

// Z of every row: tile `blockIdx.x` of T[c] rescanned from its prefix part[c][tile]; z[c] = device column pointers.
// Thread t owns rows [16 t, 16 t + 16) of the tile, staged in shared memory with one pad word per 16 (no bank conflicts).
__global__ void __launch_bounds__(SCAN_THREADS) k_tile_scan(const uint64_t* __restrict__ T, size_t n, size_t tiles,
                                                            const uint64_t* __restrict__ part, uint64_t* const* __restrict__ z) {
    __shared__ uint64_t tile[SCAN_TILE + SCAN_TILE / SCAN_ITEMS];
    __shared__ uint64_t ws[32];
    const unsigned c = blockIdx.y, t = threadIdx.x;
    const size_t base = (size_t)blockIdx.x * SCAN_TILE;
    auto slot = [](unsigned r) { return r + r / SCAN_ITEMS; };
    for (unsigned r = t; r < SCAN_TILE; r += SCAN_THREADS) tile[slot(r)] = base + r < n ? T[c * n + base + r] : 1;
    __syncthreads();
    uint64_t own = 1;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) own = gl::mul(own, tile[slot(t * SCAN_ITEMS + k)]);
    uint64_t total;
    uint64_t run = gl::mul(block_exclusive_scan(own, ws, &total), part[c * tiles + blockIdx.x]);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        const unsigned s = slot(t * SCAN_ITEMS + k);
        const uint64_t v = tile[s];
        tile[s] = gl::canon(run);
        run = gl::mul(run, v);
    }
    __syncthreads();
    uint64_t* out = z[c];
    for (unsigned r = t; r < SCAN_TILE; r += SCAN_THREADS)
        if (base + r < n) out[base + r] = tile[slot(r)];
}

// Step 3: cols = the C (1 + P) output columns in prove() order: pp of challenge c, product k <- Z_c * pp (canonical)
__global__ void k_mul_z(uint64_t* const* __restrict__ cols, unsigned C, unsigned P, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (unsigned c = 0; c < C; c++) {
        const uint64_t zc = cols[c][i];
        for (unsigned k = 0; k < P; k++) {
            uint64_t* col = cols[C + c * P + k];
            col[i] = gl::canon(gl::mul(col[i], zc));
        }
    }
}

}  // namespace

cudaError_t pcs::launch_pow_table(uint64_t base, size_t n, uint64_t* out, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_pow_table<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(base, n, out);
    return cudaGetLastError();
}

int pcs::point_tables(uint64_t root, size_t n, DevBuf& buf, cudaStream_t st) {
    const size_t n_lo = (size_t)1 << X_LO_BITS, n_hi = (n + n_lo - 1) / n_lo;
    PCS_CUDA(buf.alloc((n_lo + n_hi) * 8, st));
    PCS_CUDA(launch_pow_table(root, std::min(n, n_lo), buf.u64(), st));
    PCS_CUDA(launch_pow_table(glh::powmod(root, n_lo), n_hi, buf.u64() + n_lo, st));
    return PCS_OK;
}

int pcs::stage_host_columns(const uint64_t* const* cols, size_t R, size_t n, uint64_t* dst, cudaStream_t st) {
    if (is_pageable_host(cols[0])) return stage_pageable(cols, R, n, dst, st);
    for (size_t j = 0; j < R; j++) PCS_CUDA(cudaMemcpyAsync(dst + j * n, cols[j], n * 8, cudaMemcpyHostToDevice, st));
    return PCS_OK;
}

extern "C" {

int pcs_permutation_partial_products(const uint64_t* const* wires, const uint64_t* const* sigmas, size_t num_routed_wires,
                                     unsigned lg_n, const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas,
                                     size_t num_challenges, unsigned quotient_degree_factor, unsigned flags,
                                     uint64_t* const* out) {
    if (int rc = need_init()) return rc;
    const size_t R = num_routed_wires, C = num_challenges, D = quotient_degree_factor;
    if (D < 2) return fail(PCS_ERR_ARG, "quotient_degree_factor must be at least 2");
    if (R == 0) return fail(PCS_ERR_ARG, "num_routed_wires is 0");
    if (C == 0) return fail(PCS_ERR_ARG, "num_challenges is 0");
    if (R > 0xFFFFFFFFu) return fail(PCS_ERR_ARG, "num_routed_wires too large");
    if (!wires || !sigmas || !k_is || !betas || !gammas || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (int rc = check_two_adicity(lg_n)) return rc;
    const size_t n = (size_t)1 << lg_n, K = (R + D - 1) / D, P = K - 1, W = C * (1 + P);
    for (size_t j = 0; j < R; j++)
        if (!wires[j] || !sigmas[j]) return fail(PCS_ERR_ARG, "NULL column pointer");
    for (size_t j = 0; j < W; j++)
        if (!out[j]) return fail(PCS_ERR_ARG, "NULL output pointer");
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    cudaStream_t st = (cudaStream_t)pcs_stream();

    // launch shape of step 1: per thread 2 P NC words of shared memory
    int dev = 0, smem_max = 0;
    PCS_CUDA(cudaGetDevice(&dev));
    PCS_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const size_t nc_max = std::min<size_t>(C, MAX_NC);
    auto smem_of = [&](int threads, size_t nc) { return 2 * P * nc * 8 * (size_t)threads; };
    int threads = ROW_THREADS_MAX;
    while (threads > 32 && smem_of(threads, nc_max) > ROW_SMEM_TARGET) threads /= 2;
    if (smem_of(threads, nc_max) > (size_t)smem_max)
        return fail(PCS_ERR_ARG, "too many partial products: " + std::to_string(P) + " per challenge");

    // small tables: x_lo / x_hi, beta_c k_j, beta, gamma (canonical)
    std::vector<uint64_t> consts(C * R + 2 * C);
    for (size_t c = 0; c < C; c++) {
        const uint64_t b = betas[c] % glh::P;
        for (size_t j = 0; j < R; j++) consts[c * R + j] = glh::mulmod(b, k_is[j] % glh::P);
        consts[C * R + c] = b;
        consts[C * R + C + c] = gammas[c] % glh::P;
    }
    DevBuf xt, cb, tscr, part, flag, in_buf, out_buf, t_wires, t_sigmas, t_out;
    if (int rc = point_tables(glh::primitive_root_of_unity(lg_n), n, xt, st)) return rc;
    if (int rc = upload_table(consts.data(), consts.size(), cb, st)) return rc;
    PCS_CUDA(flag.alloc(sizeof(unsigned), st));
    PCS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(unsigned), st));

    // inputs and outputs: device column tables (host inputs are staged into [R][n] blocks, outputs into [W][n])
    std::vector<const uint64_t*> wp(wires, wires + R), sp(sigmas, sigmas + R);
    std::vector<uint64_t*> op(out, out + W);
    if (!dev_ptrs) {
        PCS_CUDA(in_buf.alloc(2 * R * n * 8, st));
        PCS_CUDA(out_buf.alloc(W * n * 8, st));
        if (int rc = stage_host_columns(wires, R, n, in_buf.u64(), st)) return rc;
        if (int rc = stage_host_columns(sigmas, R, n, in_buf.u64() + R * n, st)) return rc;
        for (size_t j = 0; j < R; j++) {
            wp[j] = in_buf.u64() + j * n;
            sp[j] = in_buf.u64() + (R + j) * n;
        }
        for (size_t j = 0; j < W; j++) op[j] = out_buf.u64() + j * n;
    }
    if (int rc = upload_table(wp.data(), R, t_wires, st)) return rc;
    if (int rc = upload_table(sp.data(), R, t_sigmas, st)) return rc;
    if (int rc = upload_table(op.data(), W, t_out, st)) return rc;
    uint64_t* const* cols = (uint64_t* const*)t_out.p;

    // step 1, NC <= 4 challenges per pass over the inputs
    PCS_CUDA(tscr.alloc(C * n * 8, st));
    const uint64_t* bk = cb.u64();
    for (size_t c0 = 0; c0 < C; c0 += MAX_NC) {
        const size_t nc = std::min<size_t>(C - c0, MAX_NC);
        const uint64_t *bkc = bk + c0 * R, *beta = bk + C * R + c0, *gamma = bk + C * R + C + c0;
        uint64_t* const* ppc = cols + C + c0 * P;
        uint64_t* T = tscr.u64() + c0 * n;
        const size_t smem = smem_of(threads, nc);
        PCS_CUDA(dispatch_width(nc, [&](auto NC) {
            if (smem > (48u << 10)) {
                cudaError_t e = cudaFuncSetAttribute(k_perm_rows<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
            }
            k_perm_rows<NC><<<(unsigned)((n + threads - 1) / threads), threads, smem, st>>>(
                (const uint64_t* const*)t_wires.p, (const uint64_t* const*)t_sigmas.p, (unsigned)R, (unsigned)D, (unsigned)P, n,
                xt.u64(), xt.u64() + (1u << X_LO_BITS), bkc, beta, gamma, ppc, T, (unsigned*)flag.p);
            return cudaGetLastError();
        }));
    }

    // step 2: Z = exclusive product scan of T; step 3: partial products times Z
    const size_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    PCS_CUDA(part.alloc(C * tiles * 8, st));
    k_tile_product<<<dim3((unsigned)tiles, (unsigned)C), SCAN_THREADS, 0, st>>>(tscr.u64(), n, tiles, part.u64());
    PCS_CUDA(cudaGetLastError());
    k_scan_parts<<<(unsigned)C, PART_THREADS, 0, st>>>(part.u64(), tiles);
    PCS_CUDA(cudaGetLastError());
    k_tile_scan<<<dim3((unsigned)tiles, (unsigned)C), SCAN_THREADS, 0, st>>>(tscr.u64(), n, tiles, part.u64(), cols);
    PCS_CUDA(cudaGetLastError());
    if (P) {
        k_mul_z<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cols, (unsigned)C, (unsigned)P, n);
        PCS_CUDA(cudaGetLastError());
    }

    unsigned zero = 0;
    PCS_CUDA(cudaMemcpyAsync(&zero, flag.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    if (zero) return fail(PCS_ERR_ARG, "Tried to invert zero");
    if (!dev_ptrs)
        for (size_t j = 0; j < W; j++)
            if (int rc = d2h_pageable(out[j], out_buf.u64() + j * n, n * 8, st)) return rc;
    return PCS_OK;
}

}  // extern "C"
