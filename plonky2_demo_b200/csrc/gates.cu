// The gate constraints of prove()'s quotient step on the device, from the constants and wires batches' LDE rows read in place:
//
//   pcs_gate_constraint_terms   evaluate_gate_constraints_base_batch   plonk/vanishing_poly.rs
//                                 compute_filter                      gates/gate.rs
//                                 NoopGate, ConstantGate, PublicInputGate, ArithmeticGate, PoseidonGate   gates/*.rs
//                               + reduce_with_powers per alpha       plonk/plonk_common.rs
//
// The quotient domain x_i = 7 w_M^i, i < M = n 2^q, is leaves [0, M) of each batch's leaf-order LDE (quotient.cu, DESIGN §3),
// so one thread per leaf reads every column coalesced.  By linearity, slot k's sum over the gates reduced with alpha^k equals
// sum_g filter_g sum_k c_{g,k} alpha^k: each gate's constraints are reduced as they are produced (alpha^k from a table read
// uniformly across the warp), then multiplied by the gate's filter once.  The loop over the gate table is uniform too.
//
//   1. k_gate_points     leaf l -> out[a][l] for the alphas [a0, a0 + na) of a pass (N <= 4 at a time), [C][M] in leaf order.
//   2. launch_bitrev_permute: leaf order -> natural order of the size-M domain, into the caller's columns.
//
// PoseidonGate runs the naive permutation with the witness substituted where the reference constrains it: constant layer, S-box
// on every lane (full rounds) or on lane 0 (partial rounds), MDS.  The MDS layers are the leaf hash's FP64 network
// (mds_layer_fp64), which adds the next round's constants where they are round_addends (full rounds); behind the other layers
// the constants RC[r + 1] are added lane by lane.  The reference writes the partial rounds in the fast form; both forms give the
// same constraints for any witness, which tests/test_gate_oracle.py checks against the CPU oracle's fast form.
#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"
#include "gl64.cuh"
#include "poseidon.cuh"

using namespace pcs;

namespace {

constexpr int GT_THREADS = 128;
constexpr int MAX_NA = 4;                     // alphas per pass over the inputs
constexpr unsigned POSEIDON_WIRES = 135, POSEIDON_CONSTRAINTS = 123;
constexpr uint64_t UNUSED_SELECTOR = 0xFFFFFFFFull;   // gates/selectors.rs

// loose - loose, loose + loose -> loose
__device__ __forceinline__ uint64_t sub_ll(uint64_t a, uint64_t b) { return gl::sub_lc(a, gl::canon(b)); }
__device__ __forceinline__ uint64_t add_ll(uint64_t a, uint64_t b) { return gl::add_lc(a, gl::canon(b)); }

struct GateArgs {
    const uint64_t* consts;   // constant k at consts[k * stride + l]
    const uint64_t* wires;    // wire k
    size_t stride;            // N = n << rate_bits
    const uint32_t* gates;    // [G][5]: kind, param, selector_index, group start, group end
    unsigned G, num_selectors, NK;
    bool many;                // num_selectors > 1
    const uint64_t* pih;      // [4] canonical
    const uint64_t* apow;     // [C][NK] alpha_a^k, canonical
    unsigned lg_m;
    uint64_t* out;            // [C][M] leaf order
};

// the alpha-reduced constraints of one gate: acc[a] += c alpha_a^k
template <int N>
struct Reducer {
    uint64_t acc[N];
    const uint64_t* ap;   // apow + a0 NK
    unsigned NK, na;
    __device__ __forceinline__ void emit(unsigned k, uint64_t c) {
#pragma unroll
        for (int a = 0; a < N; a++)
            if (a < (int)na) acc[a] = gl::add_lc(acc[a], gl::canon(gl::mul(c, __ldg(ap + (size_t)a * NK + k))));
    }
};

// the state after MDS layer r and the constants of round r + 1 (none after round 29)
__device__ __forceinline__ void mds_and_next_constants(uint64_t (&s)[12], int r) {
    using namespace pconst;
    if (r < 3 || r >= 26) {   // round_addends[r] = RC[r + 1] (0 for r = 29): the network adds them
        mds_layer_fp64(s, &ROUND_ADD_D[24 * r]);
    } else {
        mds_layer_fp64(s, &ROUND_ADD_D[24 * 29]);
#pragma unroll
        for (int i = 0; i < 12; i++) s[i] = gl::add_lc_wide(s[i], RC[12 * (r + 1) + i]);
    }
}

// PoseidonGate::eval_unfiltered (gates/poseidon.rs): w = this leaf's wire column base
template <int N>
__device__ __forceinline__ void poseidon_gate(const uint64_t* __restrict__ w, size_t st, Reducer<N>& red) {
    using namespace pconst;
    auto W = [&](unsigned j) { return __ldg(w + (size_t)j * st); };
    unsigned k = 0;
    const uint64_t swap = W(24);
    red.emit(k++, gl::mul(swap, gl::sub_lc(swap, 1)));
    uint64_t s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint64_t lhs = W(i), rhs = W(i + 4), delta = W(25 + i);
        red.emit(k++, sub_ll(gl::mul(swap, sub_ll(rhs, lhs)), delta));
        s[i] = add_ll(lhs, delta);
        s[i + 4] = sub_ll(rhs, delta);
    }
#pragma unroll
    for (int i = 8; i < 12; i++) s[i] = W(i);
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = gl::add_lc_wide(s[i], RC[i]);
    // rounds 0..3 (full, wires from round 1 on), 4..25 (partial), 26..29 (full)
#pragma unroll 1
    for (int r = 0; r < 30; r++) {
        const bool full = r < 4 || r >= 26;
        if (full) {
            if (r != 0) {
                const unsigned w0 = r < 4 ? 29 + 12 * (r - 1) : 87 + 12 * (r - 26);
#pragma unroll
                for (int i = 0; i < 12; i++) {
                    const uint64_t sb = W(w0 + i);
                    red.emit(k++, sub_ll(s[i], sb));
                    s[i] = sb;
                }
            }
#pragma unroll
            for (int i = 0; i < 12; i++) s[i] = sbox7(s[i]);
        } else {
            const uint64_t sb = W(65 + (r - 4));
            red.emit(k++, sub_ll(s[0], sb));
            s[0] = sbox7(sb);
        }
        mds_and_next_constants(s, r);
    }
#pragma unroll
    for (int i = 0; i < 12; i++) red.emit(k++, sub_ll(s[i], W(12 + i)));
}

template <int N>
__global__ void __launch_bounds__(GT_THREADS) k_gate_points(const GateArgs A, unsigned a0, unsigned na) {
    const size_t M = (size_t)1 << A.lg_m, st = A.stride;
    const size_t l = (size_t)blockIdx.x * GT_THREADS + threadIdx.x;
    if (l >= M) return;
    const uint64_t* c = A.consts + l;
    const uint64_t* w = A.wires + l;
    auto Cn = [&](unsigned j) { return __ldg(c + (size_t)j * st); };
    auto W = [&](unsigned j) { return __ldg(w + (size_t)j * st); };
    const unsigned ns = A.num_selectors;
    uint64_t res[N];
#pragma unroll
    for (int a = 0; a < N; a++) res[a] = 0;
    Reducer<N> red;
    red.ap = A.apow + (size_t)a0 * A.NK;
    red.NK = A.NK;
    red.na = na;
#pragma unroll 1
    for (unsigned g = 0; g < A.G; g++) {
        const uint32_t* e = A.gates + 5 * g;
        const uint32_t kind = e[0], param = e[1];
        if (kind == PCS_GATE_NOOP) continue;
#pragma unroll
        for (int a = 0; a < N; a++) red.acc[a] = 0;
        switch (kind) {
            case PCS_GATE_CONSTANT:
#pragma unroll 1
                for (unsigned j = 0; j < param; j++) red.emit(j, sub_ll(Cn(ns + j), W(j)));
                break;
            case PCS_GATE_PUBLIC_INPUT:
#pragma unroll
                for (unsigned j = 0; j < 4; j++) red.emit(j, gl::sub_lc(W(j), A.pih[j]));
                break;
            case PCS_GATE_ARITHMETIC: {
                const uint64_t c0 = Cn(ns), c1 = Cn(ns + 1);
#pragma unroll 1
                for (unsigned j = 0; j < param; j++) {
                    const uint64_t prod = gl::mul(gl::mul(W(4 * j), W(4 * j + 1)), c0);
                    red.emit(j, sub_ll(W(4 * j + 3), add_ll(prod, gl::mul(W(4 * j + 2), c1))));
                }
                break;
            }
            default:   // PCS_GATE_POSEIDON
                poseidon_gate<N>(w, st, red);
                break;
        }
        // compute_filter(g, group, s, many)
        const uint64_t s = gl::canon(Cn(e[2]));
        uint64_t f = A.many ? gl::sub_lc(UNUSED_SELECTOR, s) : 1;
#pragma unroll 1
        for (uint32_t i = e[3]; i < e[4]; i++)
            if (i != g) f = gl::mul(f, gl::sub_lc(i, s));
#pragma unroll
        for (int a = 0; a < N; a++) res[a] = gl::add_lc(res[a], gl::canon(gl::mul(f, red.acc[a])));
    }
#pragma unroll
    for (int a = 0; a < N; a++)
        if (a < (int)na) A.out[(size_t)(a0 + a) * M + l] = gl::canon(res[a]);
}

}  // namespace

extern "C" {

int pcs_gate_constraint_terms(const pcs_batch* constants_sigmas, const pcs_batch* wires, const uint32_t* gates, size_t num_gates,
                              const size_t* selector_groups, size_t num_selectors, size_t num_lookup_selectors,
                              size_t num_constants, const uint64_t* public_inputs_hash, const uint64_t* alphas,
                              size_t num_challenges, unsigned quotient_degree_factor, unsigned flags, uint64_t* const* out) {
    const pcs_batch *cs = constants_sigmas, *wb = wires;
    if (!cs || !wb || (num_gates && !gates) || (num_selectors && !selector_groups) || !public_inputs_hash || !alphas || !out)
        return fail(PCS_ERR_ARG, "NULL pointer");
    BatchScope scope(cs);
    if (int rc = need_init()) return rc;
    const size_t C = num_challenges, D = quotient_degree_factor, G = num_gates, S = num_selectors;
    unsigned lg_n, q;
    if (int rc = check_quotient_domain({cs, wb}, D, C, lg_n, q)) return rc;
    if (C > 0xFFFFu || G > 0xFFFFu) return fail(PCS_ERR_ARG, "num_challenges or num_gates too large");
    if (num_lookup_selectors) return fail(PCS_ERR_ARG, "lookups are not supported: num_lookup_selectors must be 0");
    if (num_constants > cs->w)
        return fail(PCS_ERR_ARG, "constants_sigmas has " + std::to_string(cs->w) + " polynomials, fewer than num_constants");
    if (S > num_constants) return fail(PCS_ERR_ARG, "num_selectors exceeds num_constants");
    for (size_t j = 0; j < C; j++)
        if (!out[j]) return fail(PCS_ERR_ARG, "NULL output pointer");
    for (size_t t = 0; t < S; t++) {
        const size_t a = selector_groups[2 * t], b = selector_groups[2 * t + 1];
        if (a >= b || b > G)
            return fail(PCS_ERR_ARG, "selector group " + std::to_string(t) + " is not a non-empty range of the " +
                                         std::to_string(G) + " gates");
    }
    // gate table [G][5] (kind, param, selector, group start, end) and the number of constraint slots
    std::vector<uint32_t> table(5 * G + 1);
    size_t NK = 1;
    for (size_t g = 0; g < G; g++) {
        const uint32_t kind = gates[3 * g], param = gates[3 * g + 1];
        const size_t sel = gates[3 * g + 2];
        const std::string at = "gate " + std::to_string(g) + ": ";
        if (kind > PCS_GATE_POSEIDON) return fail(PCS_ERR_ARG, at + "unknown gate kind " + std::to_string(kind));
        if (sel >= S) return fail(PCS_ERR_ARG, at + "selector_index " + std::to_string(sel) + " >= num_selectors");
        if (g < selector_groups[2 * sel] || g >= selector_groups[2 * sel + 1])
            return fail(PCS_ERR_ARG, at + "outside its selector group");
        size_t need_w = 0, need_c = S, nk = 0;
        switch (kind) {
            case PCS_GATE_CONSTANT: need_w = param, need_c = S + param, nk = param; break;
            case PCS_GATE_PUBLIC_INPUT: need_w = 4, nk = 4; break;
            case PCS_GATE_ARITHMETIC: need_w = 4 * (size_t)param, need_c = S + 2, nk = param; break;
            case PCS_GATE_POSEIDON: need_w = POSEIDON_WIRES, nk = POSEIDON_CONSTRAINTS; break;
            default: break;
        }
        if (need_w > wb->w)
            return fail(PCS_ERR_ARG, at + "needs " + std::to_string(need_w) + " wires, the wires batch has " +
                                         std::to_string(wb->w));
        if (need_c > num_constants)
            return fail(PCS_ERR_ARG, at + "needs num_selectors + " + std::to_string(need_c - S) + " constants, num_constants is " +
                                         std::to_string(num_constants));
        NK = std::max(NK, nk);
        uint32_t* e = &table[5 * g];
        e[0] = kind, e[1] = param, e[2] = (uint32_t)sel;
        e[3] = (uint32_t)selector_groups[2 * sel], e[4] = (uint32_t)selector_groups[2 * sel + 1];
    }
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    cudaStream_t st = (cudaStream_t)pcs_stream();
    const unsigned lg_m = lg_n + q;
    const size_t M = (size_t)1 << lg_m;

    // small tables (canonical): public_inputs_hash [4], alpha_a^k [C][NK]
    std::vector<uint64_t> consts(4 + C * NK);
    for (int j = 0; j < 4; j++) consts[j] = public_inputs_hash[j] % glh::P;
    for (size_t a = 0; a < C; a++) {
        const uint64_t al = alphas[a] % glh::P;
        uint64_t p = 1;
        for (size_t k = 0; k < NK; k++, p = glh::mulmod(p, al)) consts[4 + a * NK + k] = p;
    }
    DevBuf cb, tb, pts, nat;   // released in stream order on every return
    if (int rc = upload_table(consts.data(), consts.size(), cb, st)) return rc;
    if (int rc = upload_table(table.data(), table.size(), tb, st)) return rc;

    // 1. the point kernel, N <= 4 alphas per pass
    PCS_CUDA(pts.alloc(C * M * 8, st));
    GateArgs A;
    A.consts = cs->lde;
    A.wires = wb->lde;
    A.stride = cs->n;
    A.gates = (const uint32_t*)tb.p;
    A.G = (unsigned)G, A.num_selectors = (unsigned)S, A.NK = (unsigned)NK;
    A.many = S > 1;
    A.pih = cb.u64();
    A.apow = cb.u64() + 4;
    A.lg_m = lg_m;
    A.out = pts.u64();
    for (size_t a0 = 0; a0 < C; a0 += MAX_NA) {
        const unsigned na = (unsigned)std::min<size_t>(C - a0, MAX_NA);
        PCS_CUDA(dispatch_width(C, [&](auto N) {
            k_gate_points<N><<<(unsigned)((M + GT_THREADS - 1) / GT_THREADS), GT_THREADS, 0, st>>>(A, (unsigned)a0, na);
            return cudaGetLastError();
        }));
    }

    // 2. leaf order -> natural order, straight into device outputs or through one staging block to the host
    if (dev_ptrs) {
        for (size_t a = 0; a < C; a++) PCS_CUDA(launch_bitrev_permute(pts.u64() + a * M, M, out[a], M, 1, lg_m, st));
        return PCS_OK;
    }
    PCS_CUDA(nat.alloc(C * M * 8, st));
    PCS_CUDA(launch_bitrev_permute(pts.u64(), M, nat.u64(), M, C, lg_m, st));
    pts.release();
    for (size_t a = 0; a < C; a++)
        if (int rc = d2h_pageable(out[a], nat.u64() + a * M, M * 8, st)) return rc;
    return PCS_OK;
}

}  // extern "C"
