// Poseidon-12 permutation over Goldilocks, one permutation per thread, state in registers.
//
// GPU counterpart of Poseidon::poseidon (plonky2/src/hash/poseidon.rs:599-609):
//   4 full rounds -> 22 partial rounds -> 4 full rounds, S-box x^7, MDS = circ(17,15,41,16,2,28,
//   13,13,39,18,34,20) + diag(8,0,..) (poseidon_goldilocks.rs:24-25).
// Output is bit-identical (after canonicalisation) to the reference for every input; the
// reference's own `consistency` test (poseidon.rs:777-790) licenses any algebraically equal
// evaluation order, and tests/ pin this kernel to the reference KATs (poseidon_goldilocks.rs:461-482).
//
// Design for the B200 integer and FP64 pipes.  Measured rates (profiles/r01_intpipe.md): IADD3 128/clk/SM,
// IMAD/LOP3/SHF 64, IMAD.WIDE 32 -- so the wide multiplier is the scarce unit and is reserved for the S-boxes
// (4 IMAD.WIDE per modmul):
//  * MDS layer = add/shift network, zero multiplies, run on the FP64 pipe (mds_layer_fp64).  Each lane is split in
//    32-bit halves; the 12-point circulant product of a half is computed exactly in doubles through the factorisation
//    x^12 - 1 = prod over zeta in {1,-1,i,-i} of (x^3 - zeta) with x^4 = zeta (three 4-point DFTs, three 3x3 twisted
//    products whose constants are (2+i), (-4-i), (16-i), [16,32,16], [-1,-8,2] -- the MDS matrix was designed to have
//    these -- and three inverse DFTs).  Same mathematics as the reference's x86 path (poseidon_goldilocks.rs:217-248,
//    307-441), derived and verified independently in tests/golden/make_golden.py:mds_network_check.
//    The next round's constant is folded into the network's last additions, so constant_layer costs nothing; one
//    96-bit fold per lane (gl::fold_halves_biased) brings the result back to 64 bits.
//  * partial rounds use the same network's middle stage alone, with the state kept in its transform
//    domain (crt_mid_half) and the scalar FAST_PARTIAL_ROUND_CONSTANTS[r] added to lane 0 after
//    its S-box; the sparse "fast" matrices of poseidon.rs:584-596 would need 23 full 64x64
//    multiplies per round on the scarce pipe.
#pragma once
#include "gl64.cuh"
#include "poseidon_constants.cuh"

namespace pcs {

constexpr int SPONGE_WIDTH = 12;
constexpr int SPONGE_RATE = 8;

__device__ __forceinline__ uint64_t sbox7(uint64_t x) {
    uint64_t x2 = gl::sqr(x);
    uint64_t x4 = gl::sqr(x2);
    uint64_t x3 = gl::mul(x, x2);
    return gl::mul(x3, x4);
}

// ------------------------------------------------------------------------------------------------
// The MDS network on the FP64 pipe.
//
// B200 has a full-rate FP64 pipe (measured 61 DFMA/clk/SM, co-issuing with the integer pipes at
// 121 instr/clk/SM, profiles/r01_fp64pipe.md) that integer code leaves idle, while the integer
// version of the network saturates the ALU pipe (profiles/r01_poseidon_unified.md).  Every value in
// the network is an integer of magnitude < 2^45 and every operation is an add, a subtract or a
// multiplication by 2, 4, 8 or 16 -- all EXACT in IEEE double (53-bit significand), in any
// evaluation order and rounding mode.  One DADD/DFMA replaces the IADD3 + IADD3.X pair of a 64-bit
// integer add, and fused shift-adds are free.
//   in : a 32-bit half x enters as the double with bit pattern 0x43300000_xxxxxxxx = 2^52 + x
//        (no conversion instruction); differences of two such values are exact, and
//        (2^52 + x) - 2^52 recovers x where a sum needs it.
//   out: the last addition adds the pre-biased round constant 2^52 + c (ROUND_ADD_D), so the result
//        2^52 + y has y's low 32 bits in its low word and y >> 32 in its high word - 0x43300000.
// ------------------------------------------------------------------------------------------------
constexpr double TWO52 = 4503599627370496.0;

__device__ __forceinline__ void mds_half_fp64(const uint32_t (&s)[12], const double* __restrict__ addb /*stride 2*/,
                                              uint32_t (&ylo)[12], uint32_t (&yhi)[12]) {
    double A[3], B[3], P[3], Q[3];
    double s0d;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        double v0 = __hiloint2double(0x43300000, (int)s[j]), v3 = __hiloint2double(0x43300000, (int)s[j + 3]);
        double v6 = __hiloint2double(0x43300000, (int)s[j + 6]), v9 = __hiloint2double(0x43300000, (int)s[j + 9]);
        double d6 = v6 - TWO52, d9 = v9 - TWO52;  // s6, s9 as exact doubles
        P[j] = v0 - v6;                           // s0 - s6
        Q[j] = v3 - v9;                           // s3 - s9
        double u = fma(d6, 2.0, P[j]);            // s0 + s6
        double v = fma(d9, 2.0, Q[j]);            // s3 + s9
        A[j] = u + v;
        B[j] = u - v;
        if (j == 0) s0d = P[0] + d6;              // s0 itself, for the diagonal term
    }
    double t = A[0] + A[1] + A[2];
    double Ya[3] = {t + A[2], t + A[0], t + A[1]};  // times 16, applied below
    double Yb[3] = {fma(B[1], -2.0, fma(B[2], 8.0, -B[0])),
                    fma(B[2], -2.0, fma(B[0], -8.0, -B[1])),
                    fma(B[1], -8.0, fma(B[0], 2.0, -B[2]))};
    double re[3], im[3];
    re[0] = fma(Q[2], 4.0, fma(Q[1], -16.0, fma(P[0], 2.0, -Q[0]) + P[1]) + P[2]);
    im[0] = fma(P[2], -4.0, fma(P[1], 16.0, fma(Q[0], 2.0, P[0]) + Q[1]) + Q[2]);
    re[1] = fma(Q[2], -16.0, fma(P[1], 2.0, fma(P[0], -4.0, Q[0]) - Q[1]) + P[2]);
    im[1] = fma(P[2], 16.0, fma(Q[1], 2.0, fma(Q[0], -4.0, -P[0]) + P[1]) + Q[2]);
    re[2] = fma(P[2], 2.0, fma(P[1], -4.0, fma(P[0], 16.0, Q[0]) + Q[1]) - Q[2]);
    im[2] = fma(Q[2], 2.0, fma(Q[1], -4.0, fma(Q[0], 16.0, -P[0]) - P[1]) + P[2]);
#pragma unroll
    for (int j = 0; j < 3; j++) {
        double e1 = fma(Ya[j], 16.0, Yb[j]), e2 = fma(Ya[j], 16.0, -Yb[j]);
        double y0 = e1 + re[j];
        if (j == 0) y0 = fma(s0d, 8.0, y0);       // MDS_MATRIX_DIAG[0] = 8
        double r0 = y0 + addb[2 * j];
        double r3 = (e2 + im[j]) + addb[2 * (j + 3)];
        double r6 = (e1 - re[j]) + addb[2 * (j + 6)];
        double r9 = (e2 - im[j]) + addb[2 * (j + 9)];
        ylo[j] = (uint32_t)__double2loint(r0);     yhi[j] = (uint32_t)__double2hiint(r0);
        ylo[j + 3] = (uint32_t)__double2loint(r3); yhi[j + 3] = (uint32_t)__double2hiint(r3);
        ylo[j + 6] = (uint32_t)__double2loint(r6); yhi[j + 6] = (uint32_t)__double2hiint(r6);
        ylo[j + 9] = (uint32_t)__double2loint(r9); yhi[j + 9] = (uint32_t)__double2hiint(r9);
    }
}

// s <- MDS * s + add[r]  on the FP64 pipe; rcd = &ROUND_ADD_D[24 * r] (add[r]: see full_round)
__device__ __forceinline__ void mds_layer_fp64(uint64_t (&s)[12], const uint64_t* __restrict__ rcd) {
    const double* addb = reinterpret_cast<const double*>(rcd);
    uint32_t lo[12], hi[12];
#pragma unroll
    for (int i = 0; i < 12; i++) {
        lo[i] = (uint32_t)s[i];
        hi[i] = (uint32_t)(s[i] >> 32);
    }
    uint32_t l0[12], l1[12], h0[12], h1[12];
    mds_half_fp64(lo, addb, l0, l1);
    mds_half_fp64(hi, addb + 1, h0, h1);
#pragma unroll
    for (int r = 0; r < 12; r++) s[r] = gl::fold_halves_biased(l0[r], l1[r], h0[r], h1[r]);
}

// ------------------------------------------------------------------------------------------------
// Partial rounds in the FP64 network's TRANSFORM domain.
//
// The network factors circ through the CRT of x^12 - 1 in three stages.  Per 32-bit half, the forward stage F maps
// the 12 lanes to three groups of (A, B, P, Q):
//     A_j = s_j + s_j+3 + s_j+6 + s_j+9,  B_j = s_j - s_j+3 + s_j+6 - s_j+9,  P_j = s_j - s_j+6,  Q_j = s_j+3 - s_j+9,
// the middle stage G is the three twisted 3-point products (Ya, Yb, re/im) and the inverse stage H gives the lanes back,
// with  F(circ s) = S G(F s),  S = diag(4, 4, 2, 2) on the (A, B, P, Q) blocks.  In the 22 partial rounds only lane 0
// passes an S-box, so the state stays in this domain as U = F(circ part of the state), the diagonal term 8 x_prev
// (MDS_MATRIX_DIAG[0] = 8) is kept aside, and a round is S G alone -- F and H drop out of the loop:
//     ext = (A_0 + B_0 + 2 P_0) / 4           lane 0 of the circulant part (read off G's outputs before S: no division)
//     s_0 = ext + 8 x_prev                    x_prev: previous round's S-box output + constant, 0 on entry
//     x   = sbox(s_0) + PARTIAL_RC[r]
//     U  <- S G(U + (x - ext) tau)            tau: + to A_0, B_0 and P_0
// The 22nd round runs G and then the network's inverse stage H instead of S, which yields the lanes (+ 8 x e_0) directly.
// The injected value is formed as (x - s_0) + 8 x_prev from the FOLDED s_0 (halves < 2^32), so it stays below 2^36 in
// magnitude however large ext's double representation is.
// The values are signed integers held exactly in doubles.  Per round A grows by the L1 row norm 256 of S G, B by 44,
// P/Q by 50, so all 12 (lo, hi) pairs are renormalised every two rounds (renorm_d, valid for either sign), and lane 0
// is folded with a positive multiple of p added (fold_signed_d).  tests/test_partial_crt.py proves every intermediate
// an integer below 2^53 over the full signed input ranges and replays the whole permutation on integers.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double u32_as_double(uint32_t x) { return __hiloint2double(0x43300000, (int)x) - TWO52; }
__device__ __forceinline__ double u32_biased(uint32_t x) { return __hiloint2double(0x43300000, (int)x); }   // 2^52 + x

// y = circ-correlation(s) + 8*s0*e0 on exact doubles (no constants), the whole network in the lane domain, as the pipe
// benchmarks in tools/ run it.  ZERO0: lane 0 is taken as 0.
template <bool ZERO0>
__device__ __forceinline__ void mds_net_d(const double (&s)[12], double (&y)[12]) {
    double A[3], B[3], P[3], Q[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const bool z = ZERO0 && j == 0;
        double u = z ? s[6] : s[j] + s[j + 6], v = s[j + 3] + s[j + 9];
        A[j] = u + v;
        B[j] = u - v;
        P[j] = z ? -s[6] : s[j] - s[j + 6];
        Q[j] = s[j + 3] - s[j + 9];
    }
    double t = A[0] + A[1] + A[2];
    double Ya[3] = {t + A[2], t + A[0], t + A[1]};  // times 16, applied below
    double Yb[3] = {fma(B[1], -2.0, fma(B[2], 8.0, -B[0])),
                    fma(B[2], -2.0, fma(B[0], -8.0, -B[1])),
                    fma(B[1], -8.0, fma(B[0], 2.0, -B[2]))};
    double re[3], im[3];
    re[0] = fma(Q[2], 4.0, fma(Q[1], -16.0, fma(P[0], 2.0, -Q[0]) + P[1]) + P[2]);
    im[0] = fma(P[2], -4.0, fma(P[1], 16.0, fma(Q[0], 2.0, P[0]) + Q[1]) + Q[2]);
    re[1] = fma(Q[2], -16.0, fma(P[1], 2.0, fma(P[0], -4.0, Q[0]) - Q[1]) + P[2]);
    im[1] = fma(P[2], 16.0, fma(Q[1], 2.0, fma(Q[0], -4.0, -P[0]) + P[1]) + Q[2]);
    re[2] = fma(P[2], 2.0, fma(P[1], -4.0, fma(P[0], 16.0, Q[0]) + Q[1]) - Q[2]);
    im[2] = fma(Q[2], 2.0, fma(Q[1], -4.0, fma(Q[0], 16.0, -P[0]) - P[1]) + P[2]);
#pragma unroll
    for (int j = 0; j < 3; j++) {
        double e1 = fma(Ya[j], 16.0, Yb[j]), e2 = fma(Ya[j], 16.0, -Yb[j]);
        y[j] = e1 + re[j];
        y[j + 3] = e2 + im[j];
        y[j + 6] = e1 - re[j];
        y[j + 9] = e2 - im[j];
    }
    if (!ZERO0) y[0] = fma(s[0], 8.0, y[0]);  // MDS_MATRIX_DIAG[0] = 8
}

// u = F(s) for one 32-bit half of the 12 lanes; u = (A_0..2, B_0..2, P_0..2, Q_0..2)
__device__ __forceinline__ void crt_forward_d(const uint32_t (&s)[12], double (&u)[12]) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
        double v0 = u32_biased(s[j]), v3 = u32_biased(s[j + 3]), v6 = u32_biased(s[j + 6]), v9 = u32_biased(s[j + 9]);
        double P = v0 - v6, Q = v3 - v9;
        double a = fma(v6 - TWO52, 2.0, P);   // s_j + s_j+6
        double b = fma(v9 - TWO52, 2.0, Q);   // s_j+3 + s_j+9
        u[j] = a + b;
        u[j + 3] = a - b;
        u[j + 6] = P;
        u[j + 9] = Q;
    }
}

// G on one half: w = G(u + g tau) = (4 Ya, Yb, re, im), the A block already carrying its factor 4 of S (it folds into
// the FMAs); the other blocks get theirs in crt_scale_half, or go through H unscaled in the last round (crt_lanes_half).
__device__ __forceinline__ void crt_mid_half(const double (&u)[12], double g, double (&w)[12]) {
    const double A0 = u[0] + g, A1 = u[1], A2 = u[2];
    const double B0 = u[3] + g, B1 = u[4], B2 = u[5];
    const double P0 = u[6] + g, P1 = u[7], P2 = u[8];
    const double Q0 = u[9], Q1 = u[10], Q2 = u[11];
    const double T = ((A1 + A2) + A0) * 64.0;              // 4 * 16 * (A_0 + A_1 + A_2)
    w[0] = fma(A2, 64.0, T);
    w[1] = fma(A0, 64.0, T);
    w[2] = fma(A1, 64.0, T);
    w[3] = fma(B1, -2.0, fma(B2, 8.0, -B0));
    w[4] = fma(B2, -2.0, fma(B0, -8.0, -B1));
    w[5] = fma(B1, -8.0, fma(B0, 2.0, -B2));
    w[6] = fma(Q2, 4.0, fma(Q1, -16.0, fma(P0, 2.0, -Q0) + P1) + P2);
    w[7] = fma(Q2, -16.0, fma(P1, 2.0, fma(P0, -4.0, Q0) - Q1) + P2);
    w[8] = fma(P2, 2.0, fma(P1, -4.0, fma(P0, 16.0, Q0) + Q1) - Q2);
    w[9] = fma(P2, -4.0, fma(P1, 16.0, fma(Q0, 2.0, P0) + Q1) + Q2);
    w[10] = fma(P2, 16.0, fma(Q1, 2.0, fma(Q0, -4.0, -P0) + P1) + Q2);
    w[11] = fma(Q2, 2.0, fma(Q1, -4.0, fma(Q0, 16.0, -P0) - P1) + P2);
}

// u <- S G = the rest of S applied to w.  Returns ext = (A_0 + B_0 + 2 P_0) / 4 of the new u, formed before the scaling.
__device__ __forceinline__ double crt_scale_half(const double (&w)[12], double (&u)[12]) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
        u[j] = w[j];
        u[j + 3] = w[j + 3] * 4.0;
        u[j + 6] = w[j + 6] * 2.0;
        u[j + 9] = w[j + 9] * 2.0;
    }
    return fma(w[0], 0.25, w[3] + w[6]);
}

// The last round's lanes: y = H w (the network's own inverse stage: circ part of the state) + bias + rcd, with rcd the
// biased constants 2^52 + half of the next full round (stride 2).
__device__ __forceinline__ void crt_lanes_half(const double (&w)[12], double bias, const double* __restrict__ rcd,
                                               double (&y)[12]) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
        double e1 = fma(w[j], 0.25, w[j + 3] + bias), e2 = fma(w[j], 0.25, bias - w[j + 3]);   // Ya +- Yb
        y[j] = (e1 + w[j + 6]) + rcd[2 * j];
        y[j + 6] = (e1 - w[j + 6]) + rcd[2 * (j + 6)];
        y[j + 3] = (e2 + w[j + 9]) + rcd[2 * (j + 3)];
        y[j + 9] = (e2 - w[j + 9]) + rcd[2 * (j + 9)];
    }
}

// (lo, hi), |lo|, |hi| < 2^51  ->  equivalent pair with both halves in [-2^20, 2^32 + 2^20]:
//   l1 = floor(lo / 2^32), h1 = floor(hi / 2^32) (round-down FMA onto 1.5 * 2^52, where doubles are spaced 1 apart for
//   either sign of the quotient),  lo' = lo - l1 2^32 - h1,  hi' = hi - h1 (2^32 - 1) + l1,  lo' + hi' 2^32 = lo + hi 2^32 - h1 p.
__device__ __forceinline__ void renorm_d(double& lo, double& hi) {
    const double C = 6755399441055744.0, INV32 = 1.0 / 4294967296.0;
    double l1 = __fma_rd(lo, INV32, C) - C;
    double h1 = __fma_rd(hi, INV32, C) - C;
    double lo2 = fma(l1, -4294967296.0, lo) - h1;
    double hi2 = fma(h1, -4294967295.0, hi) + l1;
    lo = lo2;
    hi = hi2;
}

// (BIAS_LO, BIAS_HI) = 2^19 p as lo + hi 2^32: added to a signed pair with |lo|, |hi| < 2^51 - 2^20 it makes both halves
// non-negative and below 2^52, the range fold_halves_biased reads from the bit pattern of 2^52 + half.
constexpr double BIAS_LO = 2251799813685248.0 + 524288.0;    // 2^51 + 2^19
constexpr double BIAS_HI = 2251799813685248.0 - 1048576.0;   // 2^51 - 2^20

// signed lane value lo + hi 2^32 as a loose u64
__device__ __forceinline__ uint64_t fold_signed_d(double lo, double hi) {
    double bl = lo + (TWO52 + BIAS_LO), bh = hi + (TWO52 + BIAS_HI);
    return gl::fold_halves_biased((uint32_t)__double2loint(bl), (uint32_t)__double2hiint(bl),
                                  (uint32_t)__double2loint(bh), (uint32_t)__double2hiint(bh));
}

// Lane 0 of one partial round: s_0 = ext + 8 x_prev through its S-box; (gl, gh) = x - ext as halves, to be injected;
// (el, eh): ext of the current U, (xl, xh): x_prev, becomes x; rc = PARTIAL_RC[r].
__device__ __forceinline__ void lane0_crt(double el, double eh, double& xl, double& xh, uint64_t rc, double& gl, double& gh) {
    const uint64_t s0 = fold_signed_d(fma(xl, 8.0, el), fma(xh, 8.0, eh));
    const uint64_t x = gl::add_lc_wide(sbox7(s0), rc);
    // x - ext = (x - s_0) + 8 x_prev
    gl = fma(xl, 8.0, u32_biased((uint32_t)x) - u32_biased((uint32_t)s0));
    gh = fma(xh, 8.0, u32_biased((uint32_t)(x >> 32)) - u32_biased((uint32_t)(s0 >> 32)));
    xl = u32_as_double((uint32_t)x);
    xh = u32_as_double((uint32_t)(x >> 32));
}

// The permutation.  Input lanes: any u64 (loose); output lanes: canonical (CANON_OUT) or loose -- a sponge feeds the state
// straight into the next permutation and canonicalises only the digest it finally emits.
//
// A full round is  "12 s-boxes ; s = M s + add[r]"  where add[r] is the constant needed by the NEXT s-box layer moved behind
// the linear layer (tests/golden/make_golden.py:round_addends), held as biased doubles in ROUND_ADD_D and absorbed by the
// network's last additions.  The code must stay resident in the SM's instruction cache (with separate loop bodies for
// every round group the kernel was instruction-fetch bound, profiles/r01_leafhash_v2.md), so the two groups of full rounds
// share one loop body.
__device__ __forceinline__ void full_round(uint64_t (&s)[12], int r) {
    using namespace pconst;
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = sbox7(s[i]);
    mds_layer_fp64(s, &ROUND_ADD_D[24 * r]);
}

template <bool CANON_OUT = true>
__device__ __forceinline__ void poseidon12(uint64_t (&s)[12]) {
    using namespace pconst;
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = gl::add_lc_wide(s[i], RC[i]);
    // rounds 0..3 (full), 4..25 (partial, FP64 transform domain), 26..29 (full): the two full-round groups share
    // ONE loop body (phase 0 and phase 1) so that the code stays small enough for the instruction cache
#pragma unroll 1
    for (int phase = 0; phase < 2; phase++) {
#pragma unroll 1
        for (int r = 0; r < 4; r++) full_round(s, 26 * phase + r);
        if (phase == 0) {
            // rounds 4..25 in the transform domain (see crt_mid_half); entry: U = F(s), ext = s_0, x_prev = 0
            double ul[12], uh[12];
            {
                uint32_t lo[12], hi[12];
#pragma unroll
                for (int i = 0; i < 12; i++) {
                    lo[i] = (uint32_t)s[i];
                    hi[i] = (uint32_t)(s[i] >> 32);
                }
                crt_forward_d(lo, ul);
                crt_forward_d(hi, uh);
            }
            double el = u32_as_double((uint32_t)s[0]), eh = u32_as_double((uint32_t)(s[0] >> 32));
            double xl = 0.0, xh = 0.0;
            // the 22nd round runs G then H (the lanes, + RC[26] as 2^52 + halves of add[25]) instead of S G
            const double* rcd = reinterpret_cast<const double*>(&ROUND_ADD_D[24 * 25]);
#pragma unroll 1
            for (int k = 0; k < 11; k++) {
                double gl, gh, wl[12], wh[12];
                lane0_crt(el, eh, xl, xh, PARTIAL_RC[2 * k], gl, gh);
                crt_mid_half(ul, gl, wl);
                crt_mid_half(uh, gh, wh);
                el = crt_scale_half(wl, ul);
                eh = crt_scale_half(wh, uh);
                lane0_crt(el, eh, xl, xh, PARTIAL_RC[2 * k + 1], gl, gh);
                crt_mid_half(ul, gl, wl);
                crt_mid_half(uh, gh, wh);
                if (k < 10) {
                    el = crt_scale_half(wl, ul);
                    eh = crt_scale_half(wh, uh);
#pragma unroll
                    for (int i = 0; i < 12; i++) renorm_d(ul[i], uh[i]);
                } else {
                    crt_lanes_half(wl, BIAS_LO, rcd, ul);
                    crt_lanes_half(wh, BIAS_HI, rcd + 1, uh);
                    ul[0] = fma(xl, 8.0, ul[0]);               // + 8 x_last (MDS_MATRIX_DIAG[0])
                    uh[0] = fma(xh, 8.0, uh[0]);
                }
            }
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const double bl = ul[i], bh = uh[i];
                s[i] = gl::fold_halves_biased((uint32_t)__double2loint(bl), (uint32_t)__double2hiint(bl),
                                              (uint32_t)__double2loint(bh), (uint32_t)__double2hiint(bh));
            }
        }
    }
    if (CANON_OUT) {
#pragma unroll
        for (int i = 0; i < 12; i++) s[i] = gl::canon(s[i]);
    }
}

}  // namespace pcs
