/*
 * ORACLE (test infrastructure, NOT the product): CPU restatement of the gate-constraint tail of compute_quotient_polys
 * (plonk/prover.rs:576-744), following the reference item by item:
 *   plonk/vanishing_poly.rs: evaluate_gate_constraints_base_batch   num_gate_constraints slots, gate g's constraint k times its
 *                                                    filter added into slot k, gates in common_data.gates order
 *   gates/gate.rs: compute_filter                    prod over the group of (i - s), i != g, times (UNUSED_SELECTOR - s) when
 *                                                    there is more than one selector
 *   gates/noop.rs, constant.rs, public_input.rs, arithmetic_base.rs, poseidon.rs   eval_unfiltered
 *   plonk/plonk_common.rs: reduce_with_powers        Horner over the slots in reverse, per alpha
 * PoseidonGate is written in the reference's fast form (partial_first_constant_layer, mds_partial_layer_init,
 * FAST_PARTIAL_ROUND_CONSTANTS, mds_partial_layer_fast) with the tables of oracle/poseidon_constants.h, and the full rounds' MDS
 * as the plain circulant sums (mds_row_shf): the device evaluates another form.  Field arithmetic is oracle/gl64.h (any u64
 * accepted).  Points run in parallel (OpenMP).
 *
 *   gcc -O3 -march=x86-64-v3 -fopenmp -fPIC -shared -I oracle -o libgate_oracle.so gate_oracle.c
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "gl64.h"
#include "poseidon_constants.h"

#define EXPORT __attribute__((visibility("default")))

enum { GATE_NOOP = 0, GATE_CONSTANT = 1, GATE_PUBLIC_INPUT = 2, GATE_ARITHMETIC = 3, GATE_POSEIDON = 4 };
#define PW 12
#define POSEIDON_WIRES 135
#define POSEIDON_CONSTRAINTS 123
static const uint64_t UNUSED_SELECTOR = 0xFFFFFFFFull;

static unsigned log2_ceil(size_t v) {
    unsigned q = 0;
    while (((size_t)1 << q) < v) q++;
    return q;
}

static gl_t sbox(gl_t x) {
    const gl_t x2 = gl_sqr(x), x4 = gl_sqr(x2), x3 = gl_mul(x, x2);
    return gl_mul(x3, x4);
}

static void constant_layer(gl_t* s, int round) {
    for (int i = 0; i < PW; i++) s[i] = gl_add(s[i], ALL_ROUND_CONSTANTS[i + PW * round]);
}

/* mds_layer_field: out_r = sum_i s[(i + r) % 12] circ[i] + s[r] diag[r] */
static void mds_layer(gl_t* s) {
    gl_t out[PW];
    for (int r = 0; r < PW; r++) {
        gl_t acc = gl_mul(s[r], MDS_MATRIX_DIAG[r]);
        for (int i = 0; i < PW; i++) acc = gl_add(acc, gl_mul(s[(i + r) % PW], MDS_MATRIX_CIRC[i]));
        out[r] = acc;
    }
    memcpy(s, out, sizeof(out));
}

/* mds_partial_layer_init */
static void mds_partial_layer_init(gl_t* s) {
    gl_t res[PW] = {s[0]};
    for (int r = 1; r < PW; r++)
        for (int c = 1; c < PW; c++) res[c] = gl_add(res[c], gl_mul(s[r], FAST_PARTIAL_ROUND_INITIAL_MATRIX[(r - 1) * 11 + (c - 1)]));
    memcpy(s, res, sizeof(res));
}

/* mds_partial_layer_fast(state, r) */
static void mds_partial_layer_fast(gl_t* s, int r) {
    gl_t d = gl_mul(s[0], MDS_MATRIX_CIRC[0] + MDS_MATRIX_DIAG[0]);
    for (int i = 1; i < PW; i++) d = gl_add(d, gl_mul(s[i], FAST_PARTIAL_ROUND_W_HATS[r * 11 + i - 1]));
    for (int i = 1; i < PW; i++) s[i] = gl_add(s[i], gl_mul(s[0], FAST_PARTIAL_ROUND_VS[r * 11 + i - 1]));
    s[0] = d;
}

/* PoseidonGate::eval_unfiltered on one row of 135 wires -> its 123 constraints, in order */
EXPORT void ref_poseidon_gate_constraints(const uint64_t* w, uint64_t* out) {
    size_t k = 0;
    const gl_t swap = w[24];
    out[k++] = gl_mul(swap, gl_sub(swap, 1));
    for (int i = 0; i < 4; i++) out[k++] = gl_sub(gl_mul(swap, gl_sub(w[i + 4], w[i])), w[25 + i]);
    gl_t s[PW];
    for (int i = 0; i < 4; i++) {
        s[i] = gl_add(w[i], w[25 + i]);
        s[i + 4] = gl_sub(w[i + 4], w[25 + i]);
    }
    for (int i = 8; i < PW; i++) s[i] = w[i];
    int round = 0;
    for (int r = 0; r < 4; r++, round++) {
        constant_layer(s, round);
        if (r != 0)
            for (int i = 0; i < PW; i++) {
                const gl_t sb = w[29 + 12 * (r - 1) + i];
                out[k++] = gl_sub(s[i], sb);
                s[i] = sb;
            }
        for (int i = 0; i < PW; i++) s[i] = sbox(s[i]);
        mds_layer(s);
    }
    for (int i = 0; i < PW; i++) s[i] = gl_add(s[i], FAST_PARTIAL_FIRST_ROUND_CONSTANT[i]);   /* partial_first_constant_layer */
    mds_partial_layer_init(s);
    for (int r = 0; r < 22; r++) {
        const gl_t sb = w[65 + r];
        out[k++] = gl_sub(s[0], sb);
        s[0] = sbox(sb);
        if (r < 21) s[0] = gl_add(s[0], FAST_PARTIAL_ROUND_CONSTANTS[r]);
        mds_partial_layer_fast(s, r);
    }
    round += 22;
    for (int r = 0; r < 4; r++, round++) {
        constant_layer(s, round);
        for (int i = 0; i < PW; i++) {
            const gl_t sb = w[87 + 12 * r + i];
            out[k++] = gl_sub(s[i], sb);
            s[i] = sb;
        }
        for (int i = 0; i < PW; i++) s[i] = sbox(s[i]);
        mds_layer(s);
    }
    for (int i = 0; i < PW; i++) out[k++] = gl_sub(s[i], w[12 + i]);
    for (size_t j = 0; j < k; j++) out[j] = gl_canon(out[j]);
}

/* Gate terms of compute_quotient_polys: out[a][i] = reduce_with_powers(constraints(x_i), alphas[a]) at every point i < n 2^q of
 * the quotient domain (LDE index i * 2^(rate_bits - q)).  cs [cs_w][N], wires [w_w][N]: the batches' LDEs in NATURAL order.
 * gates [G][3] = kind, param, selector_index; groups [S][2]; pih [4]; out [C][n 2^q].  Returns 0, or -1 on an argument the
 * engine refuses (unknown kind, selector or group out of range, a column beyond its batch, q > rate_bits). */
EXPORT int ref_gate_terms(const uint64_t* cs, size_t cs_w, const uint64_t* wires, size_t w_w, unsigned lg_n, unsigned rate_bits,
                          const uint32_t* gates, size_t G, const size_t* groups, size_t S, size_t num_constants,
                          const uint64_t* pih, const uint64_t* alphas, size_t C, unsigned D, uint64_t* out) {
    const unsigned q = log2_ceil(D);
    if (q > rate_bits || num_constants > cs_w || S > num_constants) return -1;
    const size_t n = (size_t)1 << lg_n, N = n << rate_bits, M = n << q, step = (size_t)1 << (rate_bits - q);
    size_t NK = 0;
    for (size_t g = 0; g < G; g++) {
        const uint32_t kind = gates[3 * g], param = gates[3 * g + 1], sel = gates[3 * g + 2];
        if (sel >= S || g < groups[2 * sel] || g >= groups[2 * sel + 1]) return -1;
        size_t nk = 0, need_w = 0, need_c = S;
        switch (kind) {
            case GATE_NOOP: break;
            case GATE_CONSTANT: nk = need_w = param, need_c = S + param; break;
            case GATE_PUBLIC_INPUT: nk = need_w = 4; break;
            case GATE_ARITHMETIC: nk = param, need_w = 4 * (size_t)param, need_c = S + 2; break;
            case GATE_POSEIDON: nk = POSEIDON_CONSTRAINTS, need_w = POSEIDON_WIRES; break;
            default: return -1;
        }
        if (need_w > w_w || need_c > num_constants) return -1;
        if (nk > NK) NK = nk;
    }
#pragma omp parallel
    {
        gl_t* slots = (gl_t*)malloc((NK + POSEIDON_CONSTRAINTS + 1) * sizeof(gl_t));
        gl_t* pc = slots + NK;
        gl_t lw[POSEIDON_WIRES];
#pragma omp for schedule(static)
        for (size_t i = 0; i < M; i++) {
            const size_t m = i * step;
            for (size_t k = 0; k < NK; k++) slots[k] = 0;
            for (size_t g = 0; g < G; g++) {
                const uint32_t kind = gates[3 * g], param = gates[3 * g + 1], sel = gates[3 * g + 2];
                const gl_t s = cs[sel * N + m];
                gl_t filter = 1;
                for (size_t t = groups[2 * sel]; t < groups[2 * sel + 1]; t++)
                    if (t != g) filter = gl_mul(filter, gl_sub(t, s));
                if (S > 1) filter = gl_mul(filter, gl_sub(UNUSED_SELECTOR, s));
#define CONST(k) cs[(S + (k)) * N + m]
#define WIRE(k) wires[(k) * N + m]
                switch (kind) {
                    case GATE_CONSTANT:
                        for (size_t k = 0; k < param; k++) slots[k] = gl_add(slots[k], gl_mul(filter, gl_sub(CONST(k), WIRE(k))));
                        break;
                    case GATE_PUBLIC_INPUT:
                        for (size_t k = 0; k < 4; k++) slots[k] = gl_add(slots[k], gl_mul(filter, gl_sub(WIRE(k), pih[k])));
                        break;
                    case GATE_ARITHMETIC:
                        for (size_t k = 0; k < param; k++) {
                            const gl_t computed = gl_add(gl_mul(gl_mul(WIRE(4 * k), WIRE(4 * k + 1)), CONST(0)),
                                                         gl_mul(WIRE(4 * k + 2), CONST(1)));
                            slots[k] = gl_add(slots[k], gl_mul(filter, gl_sub(WIRE(4 * k + 3), computed)));
                        }
                        break;
                    case GATE_POSEIDON:
                        for (size_t k = 0; k < POSEIDON_WIRES; k++) lw[k] = WIRE(k);
                        ref_poseidon_gate_constraints(lw, pc);
                        for (size_t k = 0; k < POSEIDON_CONSTRAINTS; k++) slots[k] = gl_add(slots[k], gl_mul(filter, pc[k]));
                        break;
                    default: break;
                }
#undef CONST
#undef WIRE
            }
            for (size_t a = 0; a < C; a++) {
                gl_t acc = 0;
                for (size_t k = NK; k-- > 0;) acc = gl_add(gl_mul(acc, alphas[a]), slots[k]);
                out[a * M + i] = gl_canon(acc);
            }
        }
        free(slots);
    }
    return 0;
}

EXPORT void ref_gate_set_num_threads(int n) {
#ifdef _OPENMP
    extern void omp_set_num_threads(int);
    omp_set_num_threads(n);
#else
    (void)n;
#endif
}
