/*
 * ORACLE (test infrastructure, NOT the product): CPU restatement of compute_quotient_polys (plonk/prover.rs:576-744)
 * without the gate constraints, following the reference item by item:
 *   plonk/prover.rs: compute_quotient_polys          points x_i = 7 w^i of the size n 2^q domain, LDE index i * step,
 *                                                    next index (i + next_step) mod lde_size
 *   plonk/vanishing_poly.rs: eval_vanishing_poly_base_batch   L_0(x)(Z(x) - 1) per challenge, numerator / denominator
 *                                                    values, check_partial_products per challenge
 *   util/partial_products.rs: check_partial_products acc * prod num chunk - new_acc * prod den chunk, acc from Z(x) through
 *                                                    the partial products to Z(gx)
 *   plonk/plonk_common.rs: ZeroPolyOnCoset           eval_l_0 = Z_H(x) * (n (x - 1)).inverse(), eval_inverse(i)
 *   plonk/plonk_common.rs: reduce_with_powers_multi  Horner over the terms in reverse
 *   field/src/polynomial/mod.rs: coset_ifft          ifft, then coefficient k times shift^-k
 * The caller's tail (the alpha-reduced gate constraints) follows the permutation terms: res += alpha^T tail.  Field
 * arithmetic is oracle/gl64.h (any u64 accepted).  Points run in parallel (OpenMP).
 *
 *   gcc -O3 -march=x86-64-v3 -fopenmp -fPIC -shared -I oracle -o libquotient_oracle.so quotient_oracle.c
 */
#include <stdint.h>
#include <stdlib.h>

#include "gl64.h"

#define EXPORT __attribute__((visibility("default")))

static unsigned log2_ceil(size_t v) {
    unsigned q = 0;
    while (((size_t)1 << q) < v) q++;
    return q;
}

/* Quotient VALUES of compute_quotient_polys before the coset_ifft.  cs [cs_w][N], wires [w_w][N], zs [z_w][N]: the
 * batches' LDEs in NATURAL order (N = n << rate_bits).  tails: NULL or [C][n 2^q] (natural order).  out [C][n 2^q].
 * Returns 0, or -1 when a column range exceeds its batch or q > rate_bits. */
EXPORT int ref_quotient_values(const uint64_t* cs, size_t cs_w, const uint64_t* wires, size_t w_w, const uint64_t* zs,
                               size_t z_w, unsigned lg_n, unsigned rate_bits, size_t num_constants, size_t R,
                               const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, const uint64_t* alphas,
                               size_t C, unsigned D, const uint64_t* tails, uint64_t* out) {
    const unsigned q = log2_ceil(D);
    if (q > rate_bits) return -1;
    const size_t n = (size_t)1 << lg_n, N = n << rate_bits, M = n << q, K = (R + D - 1) / D, P = K - 1, T = C * (P + 2);
    if (num_constants + R > cs_w || R > w_w || C * (1 + P) > z_w) return -1;
    const size_t step = (size_t)1 << (rate_bits - q), next_step = (size_t)1 << q;
    const gl_t w_m = gl_primitive_root_of_unity(lg_n + q), w_q = gl_primitive_root_of_unity(q);
    const gl_t g_n = gl_pow(GL_COSET_SHIFT, n);
#pragma omp parallel
    {
        gl_t* terms = (gl_t*)malloc((T + 2 * R) * sizeof(gl_t));
        gl_t *num = terms + T, *den = num + R;
#pragma omp for schedule(static)
        for (size_t i = 0; i < M; i++) {
            const gl_t x = gl_mul(GL_COSET_SHIFT, gl_pow(w_m, i));   /* shifted_x */
            const size_t m = i * step, m_next = ((i + next_step) % M) * step;
            /* ZeroPolyOnCoset: evals[i mod 2^q] = g^n w_{2^q}^i - 1 */
            const gl_t zh = gl_sub(gl_mul(g_n, gl_pow(w_q, i % next_step)), 1);
            const gl_t l_0 = gl_mul(zh, gl_pow(gl_mul(n % GL_P, gl_sub(x, 1)), GL_P - 2));   /* eval_l_0 */
            size_t t = 0;
            for (size_t c = 0; c < C; c++) terms[t++] = gl_mul(l_0, gl_sub(zs[c * N + m], 1));
            for (size_t c = 0; c < C; c++) {
                for (size_t j = 0; j < R; j++) {
                    const gl_t wire_value = wires[j * N + m];
                    const gl_t s_id = gl_mul(k_is[j], x);
                    num[j] = gl_add(gl_add(wire_value, gl_mul(betas[c], s_id)), gammas[c]);
                    den[j] = gl_add(gl_add(wire_value, gl_mul(betas[c], cs[(num_constants + j) * N + m])), gammas[c]);
                }
                /* check_partial_products(num, den, partials_c, z_x, z_gx, D) */
                gl_t acc = zs[c * N + m];
                for (size_t k = 0; k < K; k++) {
                    gl_t np = 1, dp = 1;
                    for (size_t j = k * D; j < (k + 1) * D && j < R; j++) {
                        np = gl_mul(np, num[j]);
                        dp = gl_mul(dp, den[j]);
                    }
                    const gl_t new_acc = k < P ? zs[(C + c * P + k) * N + m] : zs[c * N + m_next];
                    terms[t++] = gl_sub(gl_mul(acc, np), gl_mul(new_acc, dp));
                    acc = new_acc;
                }
            }
            const gl_t zh_inv = gl_pow(zh, GL_P - 2);   /* eval_inverse */
            for (size_t a = 0; a < C; a++) {
                gl_t cumul = 0;   /* reduce_with_powers_multi: terms in reverse */
                for (size_t u = T; u-- > 0;) cumul = gl_add(gl_mul(cumul, alphas[a]), terms[u]);
                if (tails) cumul = gl_add(cumul, gl_mul(gl_pow(alphas[a], T), tails[a * M + i]));
                out[a * M + i] = gl_canon(gl_mul(cumul, zh_inv));
            }
        }
        free(terms);
    }
    return 0;
}

/* PolynomialValues::coset_ifft(shift) on w vectors [w][2^lg_m] in place: radix-2 inverse FFT (natural order in and out),
 * times 1/M, coefficient k times shift^-k. */
EXPORT void ref_coset_ifft(uint64_t* v, size_t w, unsigned lg_m, uint64_t shift) {
    const size_t M = (size_t)1 << lg_m;
    const gl_t w_inv = gl_pow(gl_primitive_root_of_unity(lg_m), M - 1), m_inv = gl_inverse_2exp(lg_m);
    const gl_t s_inv = gl_pow(shift, GL_P - 2);
#pragma omp parallel for schedule(static)
    for (size_t c = 0; c < w; c++) {
        gl_t* a = v + c * M;
        for (size_t i = 1, j = 0; i < M; i++) {   /* bit reversal */
            size_t bit = M >> 1;
            for (; j & bit; bit >>= 1) j ^= bit;
            j ^= bit;
            if (i < j) {
                const gl_t t = a[i];
                a[i] = a[j];
                a[j] = t;
            }
        }
        for (size_t len = 2; len <= M; len <<= 1) {
            const gl_t wl = gl_pow(w_inv, M / len);
            for (size_t s = 0; s < M; s += len) {
                gl_t tw = 1;
                for (size_t k = 0; k < len / 2; k++) {
                    const gl_t u = a[s + k], x = gl_mul(a[s + k + len / 2], tw);
                    a[s + k] = gl_add(u, x);
                    a[s + k + len / 2] = gl_sub(u, x);
                    tw = gl_mul(tw, wl);
                }
            }
        }
        gl_t f = m_inv;
        for (size_t k = 0; k < M; k++) {
            a[k] = gl_canon(gl_mul(a[k], f));
            f = gl_mul(f, s_inv);
        }
    }
}

EXPORT void ref_quot_set_num_threads(int n) {
#ifdef _OPENMP
    extern void omp_set_num_threads(int);
    omp_set_num_threads(n);
#else
    (void)n;
#endif
}
