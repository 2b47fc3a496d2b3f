// prove()'s quotient polynomials on the device, from the three committed batches' LDE rows read in place:
//
//   pcs_quotient_polys   compute_quotient_polys                  plonky2/src/plonk/prover.rs:576-744
//                          eval_vanishing_poly_base_batch         plonk/vanishing_poly.rs (without the gate constraints)
//                          ZeroPolyOnCoset::eval_l_0 / eval_inverse   plonk/plonk_common.rs
//                          check_partial_products                 util/partial_products.rs
//                          reduce_with_powers_multi               plonk/plonk_common.rs
//                        + prove()'s trim_to_len(quotient_degree) and chunks(degree)   plonk/prover.rs
//
// With n = 2^lg_d, r = rate_bits, q = log2_ceil(D), M = n 2^q, the quotient domain is the points x_i = 7 w_M^i, i < M, read
// by the reference at LDE index m = i 2^(r-q).  In leaf order that is leaf brev_{lg M}(i): exactly leaves [0, M) of every
// batch, its first 2^q coset blocks (DESIGN §3).  Leaf l = b n + t (block b, position t) is the natural point
// i = brev_n(t) 2^q + brev_q(b), so Z_H(x_i) = 7^n w_{2^q}^{brev_q(b)} - 1 is one constant per block, and Z(g x_i) (point
// i + 2^q) sits in the same block at position brev_n(brev_n(t) + 1 mod n).
//
//   1. k_quotient_points  leaf l, all alphas of a launch from ONE read of the wire, sigma, Z and partial-product columns:
//                         the C terms L_0(x)(Z_c(x) - 1), then per challenge the K terms prev * prod num - next * prod den,
//                         reduced with powers of each alpha (Horner over each challenge's K terms, the blocks put together with
//                         alpha^offset), plus alpha^(C (P + 2)) times the caller's tail, times Z_H(x)^-1.  The inversions of
//                         n (x - 1) behind L_0 are shared by a thread's PT_ITEMS points (Montgomery's trick).  Output [C][M]
//                         in leaf order = the bit-reversed natural vectors of the size-M domain.
//   2. launch_bitrev_permute + coset_intt_dev (api.cu): coset_ifft(7) of the natural-order vectors.
//   3. k_trim_check       coefficients [D n, M) must be zero (trim_to_len), else a device flag.
//   4. the D chunks of n coefficients of every alpha copied out, alpha-major.
#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"
#include "gl64.cuh"

using namespace pcs;

namespace {

constexpr int PT_THREADS = 128;
constexpr int PT_ITEMS = 4;        // points per thread, strided by PT_THREADS (coalesced): one inversion for all of them
constexpr int MAX_NC = 4;          // challenges (and alphas) per pass over the inputs

struct PointArgs {
    const uint64_t* sigmas;   // sigma column j at sigmas[j * stride + l]
    const uint64_t* wires;    // wire column j
    const uint64_t* zs;       // Z_c at column c, pp_{c,k} at column C + c P + k
    size_t stride;            // N = n << rate_bits (the batches' column length)
    unsigned R, D, K, C, lg_n, lg_m;
    uint64_t n_f;             // n as a field element
    const uint64_t* x_lo;     // point_tables of w_M: x_i = 7 w_M^i
    const uint64_t* x_hi;
    const uint64_t* zh;       // [2^q] Z_H(x) of coset block b
    const uint64_t* zh_inv;   // [2^q] Z_H(x)^-1
    const uint64_t* bk;       // [C][R] beta_c k_j
    const uint64_t* beta;     // [C]
    const uint64_t* gamma;    // [C]
    const uint64_t* alpha;    // [C]
    const uint64_t* apow;     // [C][2 C + 1]: alpha_a^c, alpha_a^(C + c K) (c < C), alpha_a^(C (K + 1))
    const uint64_t* const* tail;   // NULL or C device columns of M values, natural order
    uint64_t* out;            // [C][M] leaf order
};

// Challenges [c0, c0 + nc) and alphas [a0, a0 + na), nc, na <= N.  The pass with c0 == 0 writes out[a] (and adds the tail),
// the others add to it: every pass's share is already multiplied by Z_H^-1.
template <int N>
__global__ void __launch_bounds__(PT_THREADS) k_quotient_points(const PointArgs A, unsigned c0, unsigned nc, unsigned a0,
                                                                unsigned na) {
    const size_t M = (size_t)1 << A.lg_m, n = (size_t)1 << A.lg_n, st = A.stride;
    const size_t base = (size_t)blockIdx.x * (PT_THREADS * PT_ITEMS) + threadIdx.x;
    const unsigned C = A.C, R = A.R, D = A.D, K = A.K, P = K - 1;

    // 1 / (n (x - 1)) of every point of the thread, one inversion
    uint64_t xs[PT_ITEMS], dinv[PT_ITEMS], pre[PT_ITEMS], acc = 1;
#pragma unroll
    for (int k = 0; k < PT_ITEMS; k++) {
        const size_t l = base + (size_t)k * PT_THREADS;
        uint64_t d = 1;
        xs[k] = 0;
        if (l < M) {
            const size_t i = brev_bits(l, A.lg_m);
            xs[k] = gl::mul(subgroup_point(A.x_lo, A.x_hi, i), 7);
            d = gl::mul(A.n_f, gl::canon(gl::sub_lc(xs[k], 1)));
        }
        pre[k] = acc;
        acc = gl::mul(acc, d);
        dinv[k] = d;
    }
    uint64_t inv = inverse(gl::canon(acc));   // x - 1 != 0 on the coset 7 <w_M>: 7 is not in a subgroup of order <= 2^32
#pragma unroll
    for (int k = PT_ITEMS - 1; k >= 0; k--) {
        const uint64_t d = dinv[k];
        dinv[k] = gl::mul(inv, pre[k]);
        inv = gl::mul(inv, d);
    }

    uint64_t al[N], bt[N], gm[N];
#pragma unroll
    for (int a = 0; a < N; a++) al[a] = a < (int)na ? A.alpha[a0 + a] : 0;
#pragma unroll
    for (int c = 0; c < N; c++) {
        bt[c] = c < (int)nc ? A.beta[c0 + c] : 0;
        gm[c] = c < (int)nc ? A.gamma[c0 + c] : 0;
    }

#pragma unroll 1
    for (int k = 0; k < PT_ITEMS; k++) {
        const size_t l = base + (size_t)k * PT_THREADS;
        if (l >= M) break;
        const size_t b = l >> A.lg_n, t = l & (n - 1);
        const size_t l_next = (b << A.lg_n) | brev_bits((brev_bits(t, A.lg_n) + 1) & (n - 1), A.lg_n);
        const uint64_t x = xs[0];
        const uint64_t l0 = gl::mul(A.zh[b], dinv[0]);   // L_0(x) = Z_H(x) / (n (x - 1))
#pragma unroll
        for (int s = 0; s + 1 < PT_ITEMS; s++) {   // point k + 1 to the front: registers, not a local array
            xs[s] = xs[s + 1];
            dinv[s] = dinv[s + 1];
        }

        uint64_t res[N];
#pragma unroll
        for (int a = 0; a < N; a++) res[a] = 0;
        uint64_t zc[N], nxt[N], S[N][N];
#pragma unroll
        for (int c = 0; c < N; c++) {
            if (c < (int)nc) {
                zc[c] = gl::canon(__ldg(A.zs + (size_t)(c0 + c) * st + l));
                nxt[c] = gl::canon(__ldg(A.zs + (size_t)(c0 + c) * st + l_next));   // Z_c(g x)
                const uint64_t term = gl::canon(gl::mul(l0, gl::sub_lc(zc[c], 1)));
#pragma unroll
                for (int a = 0; a < N; a++)   // alpha_a^(c0 + c) L_0(x) (Z_c(x) - 1)
                    if (a < (int)na) res[a] = gl::add_lc(res[a], gl::canon(gl::mul(term, A.apow[(a0 + a) * (2 * C + 1) + c0 + c])));
            }
#pragma unroll
            for (int a = 0; a < N; a++) S[c][a] = 0;
        }
        // check_partial_products, chunks from the last to the first (Horner in reverse, as reduce_with_powers_multi)
        for (int kk = (int)K - 1; kk >= 0; kk--) {
            const unsigned j0 = (unsigned)kk * D, j1 = min(j0 + D, R);
            uint64_t nk[N], dk[N];
#pragma unroll
            for (int c = 0; c < N; c++) nk[c] = dk[c] = 1;
#pragma unroll 2
            for (unsigned j = j0; j < j1; j++) {
                const uint64_t w = gl::canon(__ldg(A.wires + (size_t)j * st + l));
                const uint64_t s = gl::canon(__ldg(A.sigmas + (size_t)j * st + l));
#pragma unroll
                for (int c = 0; c < N; c++) {
                    if (c < (int)nc) {
                        const uint64_t wg = gl::add_lc(w, gm[c]);
                        const uint64_t num = gl::add_lc(wg, gl::canon(gl::mul(__ldg(A.bk + (size_t)(c0 + c) * R + j), x)));
                        const uint64_t den = gl::add_lc(wg, gl::canon(gl::mul(bt[c], s)));
                        nk[c] = gl::mul(nk[c], num);
                        dk[c] = gl::mul(dk[c], den);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < N; c++) {
                if (c < (int)nc) {
                    // accumulators [Z_c(x), pp_c,0 .. pp_c,P-1, Z_c(g x)]: prev of chunk kk, next = prev of chunk kk + 1
                    const uint64_t prev =
                        kk == 0 ? zc[c] : gl::canon(__ldg(A.zs + (size_t)(C + (c0 + c) * P + kk - 1) * st + l));
                    const uint64_t term =
                        gl::canon(gl::sub_lc(gl::mul(prev, nk[c]), gl::canon(gl::mul(nxt[c], dk[c]))));
#pragma unroll
                    for (int a = 0; a < N; a++) S[c][a] = gl::add_lc(gl::mul(S[c][a], al[a]), term);
                    nxt[c] = prev;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < N; c++)
            if (c < (int)nc)
#pragma unroll
                for (int a = 0; a < N; a++)
                    if (a < (int)na)
                        res[a] = gl::add_lc(
                            res[a], gl::canon(gl::mul(S[c][a], A.apow[(a0 + a) * (2 * C + 1) + C + c0 + c])));
        const uint64_t zhi = A.zh_inv[b];
        const size_t i = brev_bits(l, A.lg_m);
#pragma unroll
        for (int a = 0; a < N; a++) {
            if (a < (int)na) {
                uint64_t r = res[a];
                if (c0 == 0 && A.tail)   // alpha^(C (P + 2)) * the caller's reduced remainder of the vanishing terms
                    r = gl::add_lc(r, gl::canon(gl::mul(A.apow[(a0 + a) * (2 * C + 1) + 2 * C], A.tail[a0 + a][i])));
                uint64_t* o = A.out + (size_t)(a0 + a) * M + l;
                r = gl::canon(gl::mul(r, zhi));
                *o = c0 == 0 ? r : gl::add(r, *o);
            }
        }
    }
}

// trim_to_len(D n): coefficients [from, M) of every column of vals [C][M] must be zero
__global__ void k_trim_check(const uint64_t* __restrict__ vals, size_t M, size_t from, unsigned* flag) {
    const size_t i = from + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M && vals[(size_t)blockIdx.y * M + i] != 0) *flag = 1;
}

// resident, whole, committed LDE rows (what the quotient-domain kernels read in place), or the reason why not
const char* unusable(const pcs_batch* b) {
    if (b->on_demand) return "a PCS_LDE_ON_DEMAND batch keeps no LDE rows";
    if (b->rows_only || b->coset_first != 0 || b->full_rate_bits != b->rate_bits) return "a shard batch holds part of the LDE";
    if (!b->lde || !b->committed) return "the batch is not committed";
    return nullptr;
}

unsigned log2_ceil(size_t v) {
    unsigned q = 0;
    while (((size_t)1 << q) < v) q++;
    return q;
}

}  // namespace

int pcs::check_quotient_domain(std::initializer_list<const pcs_batch*> batches, size_t D, size_t C, unsigned& lg_n, unsigned& q) {
    const pcs_batch* b0 = *batches.begin();
    for (const pcs_batch* b : batches)
        if (b->ctx != b0->ctx) return fail(PCS_ERR_ARG, "the batches belong to different contexts");
    if (D < 2) return fail(PCS_ERR_ARG, "quotient_degree_factor must be at least 2");
    if (C == 0) return fail(PCS_ERR_ARG, "num_challenges is 0");
    for (const pcs_batch* b : batches)
        if (const char* why = unusable(b)) return fail(PCS_ERR_ARG, why);
    for (const pcs_batch* b : batches)
        if (b->lg_d != b0->lg_d || b->rate_bits != b0->rate_bits) return fail(PCS_ERR_ARG, "the batches differ in degree or rate");
    lg_n = b0->lg_d;
    q = log2_ceil(D);
    if (q > b0->rate_bits)   // compute_quotient_polys' assertion
        return fail(PCS_ERR_ARG, "Having constraints of degree higher than the rate is not supported yet. "
                                 "quotient_degree_factor " + std::to_string(D) + " needs rate_bits >= " + std::to_string(q));
    return PCS_OK;
}

extern "C" {

int pcs_quotient_polys(const pcs_batch* constants_sigmas, const pcs_batch* wires, const pcs_batch* zs_partial_products,
                       size_t num_constants, size_t num_routed_wires, const uint64_t* k_is, const uint64_t* betas,
                       const uint64_t* gammas, const uint64_t* alphas, size_t num_challenges, unsigned quotient_degree_factor,
                       const uint64_t* const* gate_terms, unsigned flags, uint64_t* const* out) {
    const pcs_batch *cs = constants_sigmas, *wb = wires, *zb = zs_partial_products;
    if (!cs || !wb || !zb || !k_is || !betas || !gammas || !alphas || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    BatchScope scope(cs);
    if (int rc = need_init()) return rc;
    const size_t R = num_routed_wires, C = num_challenges, D = quotient_degree_factor;
    unsigned lg_n, q;
    if (int rc = check_quotient_domain({cs, wb, zb}, D, C, lg_n, q)) return rc;
    if (R == 0) return fail(PCS_ERR_ARG, "num_routed_wires is 0");
    if (R > 0xFFFFFFFFu || C > 0xFFFFu) return fail(PCS_ERR_ARG, "num_routed_wires or num_challenges too large");
    const size_t K = (R + D - 1) / D, P = K - 1;
    if (num_constants + R > cs->w || num_constants > cs->w)
        return fail(PCS_ERR_ARG, "constants_sigmas has " + std::to_string(cs->w) + " polynomials, the sigmas end at " +
                                     std::to_string(num_constants + R));
    if (R > wb->w) return fail(PCS_ERR_ARG, "wires has " + std::to_string(wb->w) + " polynomials, fewer than num_routed_wires");
    if (C * (1 + P) > zb->w)
        return fail(PCS_ERR_ARG, "zs_partial_products has " + std::to_string(zb->w) + " polynomials, the partial products end at " +
                                     std::to_string(C * (1 + P)));
    for (size_t j = 0; j < C * D; j++)
        if (!out[j]) return fail(PCS_ERR_ARG, "NULL output pointer");
    if (gate_terms)
        for (size_t a = 0; a < C; a++)
            if (!gate_terms[a]) return fail(PCS_ERR_ARG, "NULL gate_terms column");
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    cudaStream_t st = (cudaStream_t)pcs_stream();
    const unsigned lg_m = lg_n + q;
    const size_t n = (size_t)1 << lg_n, M = (size_t)1 << lg_m, blocks = (size_t)1 << q;

    // small tables (canonical): bk [C][R], beta, gamma, alpha [C], apow [C][2C + 1], zh, zh_inv [2^q]
    const uint64_t w_m = glh::primitive_root_of_unity(lg_m);
    std::vector<uint64_t> consts(C * R + 3 * C + C * (2 * C + 1) + 2 * blocks);
    uint64_t* h = consts.data();
    uint64_t *h_bk = h, *h_beta = h_bk + C * R, *h_gamma = h_beta + C, *h_alpha = h_gamma + C, *h_apow = h_alpha + C,
             *h_zh = h_apow + C * (2 * C + 1), *h_zhi = h_zh + blocks;
    for (size_t c = 0; c < C; c++) {
        h_beta[c] = betas[c] % glh::P;
        h_gamma[c] = gammas[c] % glh::P;
        h_alpha[c] = alphas[c] % glh::P;
        for (size_t j = 0; j < R; j++) h_bk[c * R + j] = glh::mulmod(h_beta[c], k_is[j] % glh::P);
    }
    for (size_t a = 0; a < C; a++) {
        uint64_t* ap = h_apow + a * (2 * C + 1);
        for (size_t c = 0; c < C; c++) {
            ap[c] = glh::powmod(h_alpha[a], c);
            ap[C + c] = glh::powmod(h_alpha[a], C + c * K);
        }
        ap[2 * C] = glh::powmod(h_alpha[a], C * (K + 1));
    }
    const uint64_t g_n = glh::powmod(7, n), w_q = glh::powmod(w_m, n);   // 7^n, w_{2^q}
    for (size_t b = 0; b < blocks; b++) {   // ZeroPolyOnCoset: block b holds the points i = brev_q(b) mod 2^q
        size_t br = 0;
        for (unsigned s = 0; s < q; s++) br |= ((b >> s) & 1) << (q - 1 - s);
        const uint64_t v = glh::mulmod(g_n, glh::powmod(w_q, br));
        h_zh[b] = v ? v - 1 : glh::P - 1;
        h_zhi[b] = glh::inverse(h_zh[b]);
    }
    DevBuf cb, xt, flag, tails, t_tails, pts, nat;   // released in stream order on every return
    if (int rc = upload_table(consts.data(), consts.size(), cb, st)) return rc;
    if (int rc = point_tables(w_m, M, xt, st)) return rc;
    PCS_CUDA(flag.alloc(sizeof(unsigned), st));
    PCS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(unsigned), st));

    // the caller's tails: a device table of C columns (host columns staged into [C][M] first)
    const uint64_t* const* tail_dev = nullptr;
    if (gate_terms) {
        std::vector<const uint64_t*> tp(gate_terms, gate_terms + C);
        if (!dev_ptrs) {
            PCS_CUDA(tails.alloc(C * M * 8, st));
            if (int rc = stage_host_columns(gate_terms, C, M, tails.u64(), st)) return rc;
            for (size_t a = 0; a < C; a++) tp[a] = tails.u64() + a * M;
        }
        if (int rc = upload_table(tp.data(), C, t_tails, st)) return rc;
        tail_dev = (const uint64_t* const*)t_tails.p;
    }

    // 1. the point kernel, N <= 4 challenges and alphas per pass
    PCS_CUDA(pts.alloc(C * M * 8, st));
    PointArgs A;
    A.sigmas = cs->lde + num_constants * cs->n;
    A.wires = wb->lde;
    A.zs = zb->lde;
    A.stride = cs->n;
    A.R = (unsigned)R, A.D = (unsigned)D, A.K = (unsigned)K, A.C = (unsigned)C, A.lg_n = lg_n, A.lg_m = lg_m;
    A.n_f = n % glh::P;
    A.x_lo = xt.u64(), A.x_hi = xt.u64() + (1u << X_LO_BITS);
    const uint64_t* dc = cb.u64();
    A.bk = dc, A.beta = dc + (h_beta - h), A.gamma = dc + (h_gamma - h), A.alpha = dc + (h_alpha - h);
    A.apow = dc + (h_apow - h), A.zh = dc + (h_zh - h), A.zh_inv = dc + (h_zhi - h);
    A.tail = tail_dev;
    A.out = pts.u64();
    for (size_t c0 = 0; c0 < C; c0 += MAX_NC)
        for (size_t a0 = 0; a0 < C; a0 += MAX_NC) {
            const unsigned nc = (unsigned)std::min<size_t>(C - c0, MAX_NC), na = (unsigned)std::min<size_t>(C - a0, MAX_NC);
            PCS_CUDA(dispatch_width(C, [&](auto N) {
                const size_t per_block = PT_THREADS * PT_ITEMS;
                k_quotient_points<N><<<(unsigned)((M + per_block - 1) / per_block), PT_THREADS, 0, st>>>(A, (unsigned)c0, nc,
                                                                                                       (unsigned)a0, na);
                return cudaGetLastError();
            }));
        }
    tails.release();

    // 2. leaf order -> natural order, coset_ifft(7)
    PCS_CUDA(nat.alloc(C * M * 8, st));
    PCS_CUDA(launch_bitrev_permute(pts.u64(), M, nat.u64(), M, C, lg_m, st));
    pts.release();
    if (int rc = coset_intt_dev(nat.u64(), C, lg_m, 7, st)) return rc;

    // 3. trim_to_len(D n); 4. chunks(n), alpha-major
    if (D * n < M) {
        const size_t tail_len = M - D * n;
        k_trim_check<<<dim3((unsigned)((tail_len + 255) / 256), (unsigned)C), 256, 0, st>>>(nat.u64(), M, D * n, (unsigned*)flag.p);
        PCS_CUDA(cudaGetLastError());
    }
    if (dev_ptrs)
        for (size_t j = 0; j < C * D; j++)
            PCS_CUDA(cudaMemcpyAsync(out[j], nat.u64() + (j / D) * M + (j % D) * n, n * 8, cudaMemcpyDeviceToDevice, st));
    unsigned bad = 0;
    PCS_CUDA(cudaMemcpyAsync(&bad, flag.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    if (bad) return fail(PCS_ERR_ARG, "Quotient has failed, the vanishing polynomial is not divisible by Z_H");
    if (!dev_ptrs)
        for (size_t j = 0; j < C * D; j++)
            if (int rc = d2h_pageable(out[j], nat.u64() + (j / D) * M + (j % D) * n, n * 8, st)) return rc;
    return PCS_OK;
}

}  // extern "C"
