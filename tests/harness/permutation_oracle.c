/*
 * ORACLE (test infrastructure, NOT the product): CPU restatement of the permutation argument of prove(),
 * following the reference item by item:
 *   plonk/prover.rs: all_wires_permutation_partial_products      one call per challenge
 *   plonk/prover.rs: wires_permutation_partial_products_and_zs   per row: numerators, denominators,
 *                                                                batch_multiplicative_inverse, quotient values
 *   util/partial_products.rs: quotient_chunk_products            product of each chunk of quotient_degree_factor values
 *   util/partial_products.rs: partial_products_and_z_gx          running product from Z(x); the last one is Z(gx) and is
 *                                                                swapped with Z(x)
 *   field/src/batch_util / Field::batch_multiplicative_inverse   prefix products, one inversion, walk back; panics with
 *                                                                "Tried to invert zero" on a zero element
 * Field arithmetic is oracle/gl64.h (the reference's GoldilocksField, any u64 accepted).  The rows are independent up to
 * quotient_chunk_products and run in parallel (OpenMP); partial_products_and_z_gx carries Z(x) from row to row and runs
 * in row order, as the reference's loop does.
 *
 *   gcc -O3 -march=x86-64-v3 -fopenmp -fPIC -shared -I oracle -o libpermutation_oracle.so permutation_oracle.c
 */
#include <stdint.h>
#include <stdlib.h>

#include "gl64.h"

#define EXPORT __attribute__((visibility("default")))

/* Field::batch_multiplicative_inverse on x[0 .. len): 1 when an element is zero (the reference panics), else 0 */
static int batch_multiplicative_inverse(const gl_t* x, size_t len, gl_t* prefix, gl_t* out) {
    gl_t acc = 1;
    for (size_t j = 0; j < len; j++) {
        if (gl_canon(x[j]) == 0) return 1;
        prefix[j] = acc;
        acc = gl_mul(acc, x[j]);
    }
    gl_t inv = gl_pow(acc, GL_P - 2);
    for (size_t j = len; j-- > 0;) {
        out[j] = gl_mul(inv, prefix[j]);
        inv = gl_mul(inv, x[j]);
    }
    return 0;
}

/* quotient_chunk_products: products of the chunks [kD, min((k+1)D, len)) */
static size_t quotient_chunk_products(const gl_t* q, size_t len, unsigned D, gl_t* out) {
    size_t k = 0;
    for (size_t j0 = 0; j0 < len; j0 += D, k++) {
        gl_t acc = 1;
        for (size_t j = j0; j < j0 + D && j < len; j++) acc = gl_mul(acc, q[j]);
        out[k] = acc;
    }
    return k;
}

/* all_wires_permutation_partial_products.  wires, sigmas: [R][n] (wire j at row i = wires[j n + i]); k_is [R]; betas,
 * gammas [C]; out [C][P + 1][n]: per challenge the reference's return value [pp_0 .. pp_{P-1}, Z], canonical.
 * Returns 0, or -1 when a denominator is zero ("Tried to invert zero"). */
EXPORT int ref_permutation_partial_products(const uint64_t* wires, const uint64_t* sigmas, size_t R, unsigned lg_n,
                                            const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, size_t C,
                                            unsigned D, uint64_t* out) {
    const size_t n = (size_t)1 << lg_n, K = (R + D - 1) / D, P = K - 1;
    const gl_t omega = gl_primitive_root_of_unity(lg_n);
    gl_t* chunks = (gl_t*)malloc(n * K * sizeof(gl_t));   /* quotient_chunk_products of every row, one challenge */
    if (!chunks) return -2;
    int err = 0;
    for (size_t c = 0; c < C && !err; c++) {
        const gl_t beta = betas[c], gamma = gammas[c];
#pragma omp parallel reduction(| : err)
        {
            gl_t* num = (gl_t*)malloc(4 * R * sizeof(gl_t));
            gl_t *den = num + R, *inv = den + R, *scratch = inv + R;
#pragma omp for schedule(static)
            for (size_t i = 0; i < n; i++) {
                /* x = subgroup[i]: the powers of omega restarted every 4096 rows to keep the loop parallel */
                const gl_t x = gl_mul(gl_pow(omega, i & ~(size_t)4095), gl_pow(omega, i & 4095));
                for (size_t j = 0; j < R; j++) {
                    const gl_t wire_value = wires[j * n + i];
                    const gl_t s_id = gl_mul(k_is[j], x);
                    num[j] = gl_add(gl_add(wire_value, gl_mul(beta, s_id)), gamma);
                    den[j] = gl_add(gl_add(wire_value, gl_mul(beta, sigmas[j * n + i])), gamma);
                }
                if (batch_multiplicative_inverse(den, R, scratch, inv)) {
                    err |= 1;
                    continue;
                }
                for (size_t j = 0; j < R; j++) num[j] = gl_mul(num[j], inv[j]);   /* quotient_values */
                quotient_chunk_products(num, R, D, chunks + i * K);
            }
            free(num);
        }
        if (err) break;
        /* partial_products_and_z_gx(z_x, quotient_partials) and the swap, row after row */
        uint64_t* res = out + c * (P + 1) * n;
        gl_t z_x = 1;
        for (size_t i = 0; i < n; i++) {
            gl_t acc = z_x;
            for (size_t k = 0; k < K; k++) {
                acc = gl_mul(acc, chunks[i * K + k]);
                if (k < P) res[k * n + i] = gl_canon(acc);
            }
            res[P * n + i] = gl_canon(z_x);   /* swap: Z(x) is returned, Z(gx) carried to the next row */
            z_x = acc;
        }
    }
    free(chunks);
    return err ? -1 : 0;
}

EXPORT void ref_perm_set_num_threads(int n) {
#ifdef _OPENMP
    extern void omp_set_num_threads(int);
    omp_set_num_threads(n);
#else
    (void)n;
#endif
}
