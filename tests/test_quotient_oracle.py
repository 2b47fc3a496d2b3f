"""The quotient step's CPU oracle (tests/harness/quotient_oracle.c), no GPU needed:

- it equals a literal big-integer restatement of compute_quotient_polys without the gate constraints (eval_l_0,
  check_partial_products, reduce_with_powers_multi, the Z_H division, coset_ifft) on edge shapes: n = 1 .. 16, P = 0 and a short
  last chunk, D = 2, 3, 5, 8 with q < rate_bits and q = rate_bits, one to five challenges, non-canonical inputs, scalars and tails;
- on a witness that satisfies copy constraints, committed through the oracle with a zero tail, the trim succeeds at D = 5 and
  the plonk verifier's identity vanishing(z) = Z_H(z) sum_k z^(k n) chunk_k(z) holds at random points, with the vanishing terms
  recomputed from the polynomials at z and g z; one changed wire value makes the trim fail at D = 5 and the identity fail at
  D = 8 (this pins what L_0, x_i, Z(g x) and the term order mean independently of any restatement)."""
import os
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))

import permutation_oracle as po  # noqa: E402
import quotient_oracle as qo  # noqa: E402
from helpers import noncanonical  # noqa: E402
from test_permutation_oracle import copy_constrained_witness  # noqa: E402

P = 0xFFFFFFFF00000001
GEN = 1753635133440165772   # POWER_OF_TWO_GENERATOR


def omega(lg):
    return pow(GEN, 1 << (32 - lg), P)


def inv(a):
    return pow(a % P, P - 2, P)


# ---- literal big-int restatement of the reference ------------------------------------------------------------------------
def check_partial_products(numerators, denominators, partials, z_x, z_gx, max_degree):
    acc, res = z_x, []
    for k, new_acc in enumerate(list(partials) + [z_gx]):
        num = den = 1
        for v in numerators[k * max_degree:(k + 1) * max_degree]:
            num = num * v % P
        for v in denominators[k * max_degree:(k + 1) * max_degree]:
            den = den * v % P
        res.append((acc * num - new_acc * den) % P)
        acc = new_acc
    return res


def reduce_with_powers_multi(terms, alphas):
    cumul = [0] * len(alphas)
    for t in reversed(terms):
        cumul = [(c * a + t) % P for c, a in zip(cumul, alphas)]
    return cumul


def big_reference(cs, wires, zs, rate_bits, num_constants, R, k_is, betas, gammas, alphas, D, tails):
    """compute_quotient_polys on natural-order LDEs, the tail appended as alpha^T tail; -> [C][M] coefficients"""
    N = cs.shape[1]
    n = N >> rate_bits
    q = (D - 1).bit_length()
    M, step, next_step = n << q, 1 << (rate_bits - q), 1 << q
    C = len(betas)
    K = -(-R // D)
    Pn = K - 1
    T = C * (Pn + 2)
    betas, gammas, alphas = [int(v) % P for v in betas], [int(v) % P for v in gammas], [int(v) % P for v in alphas]
    w_m = omega((n << q).bit_length() - 1)
    zh_on_coset = [(pow(7, n, P) * pow(omega(q), k, P) - 1) % P for k in range(next_step)]   # ZeroPolyOnCoset
    values = [[0] * M for _ in range(C)]
    for i in range(M):
        x = 7 * pow(w_m, i, P) % P
        m, m_next = i * step, ((i + next_step) % M) * step
        l_0 = zh_on_coset[i % next_step] * inv(n * (x - 1)) % P
        z1, pp_terms = [], []
        for c in range(C):
            z_x, z_gx = int(zs[c][m]), int(zs[c][m_next])
            z1.append(l_0 * (z_x - 1) % P)
            num = [(int(wires[j][m]) + betas[c] * (int(k_is[j]) * x % P) + gammas[c]) % P for j in range(R)]
            den = [(int(wires[j][m]) + betas[c] * int(cs[num_constants + j][m]) + gammas[c]) % P for j in range(R)]
            partials = [int(zs[C + c * Pn + k][m]) for k in range(Pn)]
            pp_terms += check_partial_products(num, den, partials, z_x, z_gx, D)
        res = reduce_with_powers_multi(z1 + pp_terms, alphas)
        for a in range(C):
            r = res[a]
            if tails is not None:
                r = (r + pow(alphas[a], T, P) * int(tails[a][i])) % P
            values[a][i] = r * inv(zh_on_coset[i % next_step]) % P
    # coset_ifft(7): c_k = 7^-k / M sum_i v_i w^-ik
    w_inv, m_inv, s_inv = inv(w_m), inv(M), inv(7)
    out = np.empty((C, M), dtype=np.uint64)
    for a in range(C):
        for k in range(M):
            wk = pow(w_inv, k, P)
            acc, pw = 0, 1
            for v in values[a]:
                acc = (acc + v * pw) % P
                pw = pw * wk % P
            out[a, k] = acc * m_inv % P * pow(s_inv, k, P) % P
    return out


SHAPES = [   # (R, lg_n, C, D, rate_bits, num_constants, with_tail)
    (3, 0, 1, 2, 1, 0, False),     # n = 1
    (5, 2, 1, 8, 3, 1, True),      # P = 0 (R < D), q = rate_bits
    (8, 1, 2, 8, 3, 0, False),     # P = 0, R == D
    (7, 3, 3, 3, 3, 2, True),      # short last chunk, q = 2 < rate_bits
    (9, 4, 2, 2, 2, 0, True),      # D = 2, q < rate_bits
    (20, 3, 5, 5, 4, 3, True),     # five challenges, D = 5 (q = 3)
    (12, 2, 4, 5, 3, 0, False),    # q = rate_bits with D < 2^q
]


@pytest.mark.parametrize("R,lg_n,C,D,rate_bits,nc,with_tail", SHAPES)
def test_oracle_equals_big_int_restatement(R, lg_n, C, D, rate_bits, nc, with_tail):
    rng = np.random.default_rng(7 * R + 100 * lg_n + C + 1000 * D)
    n, q = 1 << lg_n, (D - 1).bit_length()
    N, M, K = n << rate_bits, n << q, -(-R // D)
    cs = noncanonical(rng, (nc + R + 1, N))
    wires = noncanonical(rng, (R + 2, N))
    zs = noncanonical(rng, (C * K + 1, N))
    k_is, betas, gammas, alphas = (noncanonical(rng, s) for s in (R, C, C, C))
    tails = noncanonical(rng, (C, M)) if with_tail else None
    got = qo.compute_quotient_polys(cs, wires, zs, rate_bits, nc, R, k_is, betas, gammas, alphas, D, tails)
    want = big_reference(cs, wires, zs, rate_bits, nc, R, k_is, betas, gammas, alphas, D, tails)
    assert got.shape == (C, M)
    assert np.array_equal(got, want)


def test_oracle_coset_ifft_matches_the_existing_oracle():
    rng = np.random.default_rng(3)
    coeffs = rng.integers(0, P, (3, 64), dtype=np.uint64)
    values = oracle.coset_lde(coeffs, 0)   # evaluations on 7 <w_64>, natural order
    v = np.ascontiguousarray(values)
    qo.lib().ref_coset_ifft(v.ctypes.data_as(qo.u64p), 3, 6, 7)
    assert np.array_equal(v, coeffs)


# ---- the plonk verifier's identity on a satisfiable copy-constraint instance ---------------------------------------------
def _commit_natural(values, rate_bits):
    """values [w][n] -> (coefficients [w][n], natural-order LDE [w][n << rate_bits])"""
    coeffs = oracle.fft(values, inverse=True)
    return coeffs, oracle.coset_lde(coeffs, rate_bits)


def _instance(rng, R, lg_n, C, nc, rate_bits, change_wire):
    n = 1 << lg_n
    wires, sigmas, k_is, x, last_cycle = copy_constrained_witness(rng, R, lg_n, n_cycles=min(8, R * n // 6))
    if change_wire:
        i, j = last_cycle[0]
        wires = wires.copy()
        wires[j][i] = (int(wires[j][i]) + 1) % P
    betas = rng.integers(1, P, C, dtype=np.uint64)
    gammas = rng.integers(1, P, C, dtype=np.uint64)
    consts = rng.integers(0, P, (nc, n), dtype=np.uint64)
    cs_c, cs_lde = _commit_natural(np.vstack([consts, sigmas]), rate_bits)
    w_c, w_lde = _commit_natural(wires, rate_bits)
    return dict(k_is=k_is, betas=betas, gammas=gammas, cs=(cs_c, cs_lde), w=(w_c, w_lde))


def _zs(inst, R, D, rate_bits):
    nc_ = inst["cs"][0].shape[0] - R
    n = inst["w"][0].shape[1]
    wires = oracle.fft(inst["w"][0], inverse=False)[:R]
    sigmas = oracle.fft(inst["cs"][0][nc_:], inverse=False)
    zs = po.prove_order(po.all_wires_permutation_partial_products(wires, sigmas, inst["k_is"], inst["betas"], inst["gammas"], D))
    assert zs.shape[1] == n
    return _commit_natural(zs, rate_bits)


def _eval(coeffs, z):
    return [oracle.poly_eval(c, z) for c in coeffs]


def vanishing_at(inst, zs_c, R, nc, D, alphas, z):
    """eval_vanishing_poly at an arbitrary point z from the polynomials at z and g z (no gate constraints)"""
    n = zs_c.shape[1]
    C = len(inst["betas"])
    K = -(-R // D)
    Pn = K - 1
    w = _eval(inst["w"][0][:R], z)
    s = _eval(inst["cs"][0][nc:nc + R], z)
    zv = _eval(zs_c, z)
    z_g = _eval(zs_c[:C], z * omega(n.bit_length() - 1) % P)
    l_0 = (pow(z, n, P) - 1) * inv(n * (z - 1)) % P
    z1, pp = [], []
    for c in range(C):
        b, g = int(inst["betas"][c]), int(inst["gammas"][c])
        num = [(w[j] + b * int(inst["k_is"][j]) * z + g) % P for j in range(R)]
        den = [(w[j] + b * s[j] + g) % P for j in range(R)]
        z1.append(l_0 * (zv[c] - 1) % P)
        pp += check_partial_products(num, den, zv[C + c * Pn:C + (c + 1) * Pn], zv[c], z_g[c], D)
    return reduce_with_powers_multi(z1 + pp, [int(a) % P for a in alphas])


def _quotient(inst, zs_lde, R, nc, D, rate_bits, alphas):
    return qo.compute_quotient_polys(inst["cs"][1], inst["w"][1], zs_lde, rate_bits, nc, R, inst["k_is"], inst["betas"],
                                     inst["gammas"], alphas, D)


@pytest.mark.parametrize("R,lg_n,D", [(7, 3, 5), (7, 3, 8), (12, 4, 5)])
def test_verifier_identity_holds_on_a_satisfied_instance(R, lg_n, D):
    rng = np.random.default_rng(R * 31 + lg_n + D)
    C, nc, rate_bits = 2, 2, 3
    n = 1 << lg_n
    inst = _instance(rng, R, lg_n, C, nc, rate_bits, change_wire=False)
    zs_c, zs_lde = _zs(inst, R, D, rate_bits)
    alphas = rng.integers(1, P, C, dtype=np.uint64)
    chunks = qo.quotient_poly_chunks(_quotient(inst, zs_lde, R, nc, D, rate_bits, alphas), n, D)   # the trim succeeds
    assert chunks.shape == (C * D, n)
    for z in (int(v) for v in rng.integers(2, P, 3, dtype=np.uint64)):
        van = vanishing_at(inst, zs_c, R, nc, D, alphas, z)
        for a in range(C):
            t = sum(pow(z, k * n, P) * oracle.poly_eval(chunks[a * D + k], z) for k in range(D)) % P
            assert van[a] == (pow(z, n, P) - 1) * t % P, (a, z)


def test_changed_wire_fails_the_trim_and_the_identity():
    R, lg_n, C, nc, rate_bits = 7, 3, 2, 2, 3
    n = 1 << lg_n
    rng = np.random.default_rng(99)
    inst = _instance(rng, R, lg_n, C, nc, rate_bits, change_wire=True)
    alphas = rng.integers(1, P, C, dtype=np.uint64)
    zs_c, zs_lde = _zs(inst, R, 5, rate_bits)
    with pytest.raises(ValueError, match="Quotient has failed, the vanishing polynomial is not divisible by Z_H"):
        qo.quotient_poly_chunks(_quotient(inst, zs_lde, R, nc, 5, rate_bits, alphas), n, 5)
    # D = 8 = 2^q: nothing to trim, but the chunks no longer satisfy the verifier's identity
    zs_c, zs_lde = _zs(inst, R, 8, rate_bits)
    chunks = qo.quotient_poly_chunks(_quotient(inst, zs_lde, R, nc, 8, rate_bits, alphas), n, 8)
    z = int(rng.integers(2, P, dtype=np.uint64))
    van = vanishing_at(inst, zs_c, R, nc, 8, alphas, z)
    t = sum(pow(z, k * n, P) * oracle.poly_eval(chunks[k], z) for k in range(8)) % P
    assert van[0] != (pow(z, n, P) - 1) * t % P
