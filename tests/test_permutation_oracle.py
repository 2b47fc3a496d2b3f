"""The permutation argument's CPU oracle (tests/harness/permutation_oracle.c), no GPU needed:

- it equals a literal big-integer restatement of wires_permutation_partial_products_and_zs, batch_multiplicative_inverse,
  quotient_chunk_products and partial_products_and_z_gx on small shapes with every edge (n = 1, P = 0, a short last chunk,
  D = 2, one and three challenges, non-canonical inputs);
- on a witness that satisfies copy constraints, Z starts at 1, the check_partial_products identities hold at every row and
  the running product wraps around to 1, and a single changed wire value breaks the wrap-around (this pins what k_j, x_i
  and sigma mean independently of any restatement);
- get_unique_coset_shifts returns 7^j and refuses more shifts than there are cosets."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))

import permutation_oracle as po  # noqa: E402
from helpers import noncanonical  # noqa: E402

P = 0xFFFFFFFF00000001
GEN = 1753635133440165772   # POWER_OF_TWO_GENERATOR


def omega(lg_n):
    return pow(GEN, 1 << (32 - lg_n), P)


# ---- literal big-int restatement of the reference ------------------------------------------------------------------------
def batch_multiplicative_inverse(xs):
    if any(x % P == 0 for x in xs):
        raise ZeroDivisionError("Tried to invert zero")
    return [pow(x, P - 2, P) for x in xs]


def prod(xs):
    acc = 1
    for v in xs:
        acc = acc * v % P
    return acc


def quotient_chunk_products(quotient_values, max_degree):
    return [prod(quotient_values[i:i + max_degree]) for i in range(0, len(quotient_values), max_degree)]


def partial_products_and_z_gx(z_x, quotient_chunk_products_):
    res, acc = [], z_x
    for q in quotient_chunk_products_:
        acc = acc * q % P
        res.append(acc)
    return res


def wires_permutation_partial_products_and_zs(wires, sigmas, k_is, beta, gamma, degree_factor):
    R, n = len(wires), len(wires[0])
    w = omega(n.bit_length() - 1)
    num_prods = -(-R // degree_factor) - 1
    z_x, rows = 1, []
    for i in range(n):
        x = pow(w, i, P)
        numerators = [(int(wires[j][i]) + beta * (int(k_is[j]) * x) + gamma) % P for j in range(R)]
        denominators = [(int(wires[j][i]) + beta * int(sigmas[j][i]) + gamma) % P for j in range(R)]
        invs = batch_multiplicative_inverse(denominators)
        quotient_values = [numerators[j] * invs[j] % P for j in range(R)]
        partials = quotient_chunk_products(quotient_values, degree_factor)
        pp = partial_products_and_z_gx(z_x, partials)
        z_x, pp[num_prods] = pp[num_prods], z_x   # swap: Z(x) is returned, Z(gx) carried on
        rows.append(pp)
    return np.array(rows, dtype=np.uint64).T   # [P + 1][n]


def big_reference(wires, sigmas, k_is, betas, gammas, degree_factor):
    return np.stack([wires_permutation_partial_products_and_zs(wires, sigmas, k_is, int(b) % P, int(g) % P, degree_factor)
                     for b, g in zip(betas, gammas)])


SHAPES = [   # (R, lg_n, C, D)
    (3, 0, 1, 2),     # n = 1
    (5, 3, 1, 8),     # P = 0 (R <= D)
    (8, 2, 2, 8),     # P = 0, R == D
    (7, 3, 3, 3),     # short last chunk, three challenges
    (9, 4, 1, 2),     # D = 2, odd R
    (20, 3, 2, 8),    # 3 chunks, the last of 4
    (80, 3, 2, 8),    # the m = 2 demo shape
]


@pytest.mark.parametrize("R,lg_n,C,D", SHAPES)
def test_oracle_equals_big_int_restatement(R, lg_n, C, D):
    rng = np.random.default_rng(1000 * R + 10 * lg_n + C)
    n = 1 << lg_n
    wires, sigmas = noncanonical(rng, (R, n)), noncanonical(rng, (R, n))
    k_is, betas, gammas = noncanonical(rng, R), noncanonical(rng, C), noncanonical(rng, C)
    got = po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D)
    want = big_reference(wires, sigmas, k_is, betas, gammas, D)
    assert got.shape == (C, -(-R // D), n)
    assert np.array_equal(got, want)
    assert (got < np.uint64(P)).all()
    assert (got[:, -1, 0] == 1).all()   # Z(x_0) = 1


def test_oracle_zero_denominator():
    rng = np.random.default_rng(5)
    R, n = 6, 4
    wires, sigmas = rng.integers(0, P, (R, n), dtype=np.uint64), rng.integers(0, P, (R, n), dtype=np.uint64)
    beta = 11
    gamma = (P - (int(wires[4][2]) + beta * int(sigmas[4][2])) % P) % P   # den_4(x_2) = 0
    with pytest.raises(ZeroDivisionError, match="Tried to invert zero"):
        po.all_wires_permutation_partial_products(wires, sigmas, np.arange(1, R + 1), [beta], [gamma], 2)
    with pytest.raises(ZeroDivisionError):
        big_reference(wires, sigmas, np.arange(1, R + 1), [beta], [gamma], 2)


# ---- the copy-constraint property --------------------------------------------------------------------------------------
def copy_constrained_witness(rng, R, lg_n, n_cycles):
    """A witness with random copy-constraint cycles over (row, wire) cells: every cell of a cycle holds the same value, and
    sigma(i, j) = k_{j'} x_{i'} for the next cell (i', j') of its cycle (the identity k_j x_i for a singleton)."""
    n = 1 << lg_n
    k_is = [pow(7, j, P) for j in range(R)]
    x = [pow(omega(lg_n), i, P) for i in range(n)]
    wires = rng.integers(0, P, (R, n), dtype=np.uint64)
    sigmas = np.array([[k_is[j] * x[i] % P for i in range(n)] for j in range(R)], dtype=np.uint64)
    cells = [(i, j) for j in range(R) for i in range(n)]
    rng.shuffle(cells)
    pos = 0
    for _ in range(n_cycles):
        size = int(rng.integers(2, 6))
        cyc = [tuple(c) for c in cells[pos:pos + size]]
        pos += size
        v = int(rng.integers(0, P, dtype=np.uint64))
        for t, (i, j) in enumerate(cyc):
            wires[j][i] = v
            ni, nj = cyc[(t + 1) % len(cyc)]
            sigmas[j][i] = k_is[nj] * x[ni] % P
    return wires, sigmas, np.array(k_is, dtype=np.uint64), x, cyc


def _num_den(wires, sigmas, k_is, x, beta, gamma, i):
    R = wires.shape[0]
    num = [(int(wires[j][i]) + beta * int(k_is[j]) * x[i] + gamma) % P for j in range(R)]
    den = [(int(wires[j][i]) + beta * int(sigmas[j][i]) + gamma) % P for j in range(R)]
    return num, den


@pytest.mark.parametrize("R,lg_n,D", [(80, 3, 8), (7, 4, 3), (4, 5, 2)])
def test_copy_constraints_satisfied(R, lg_n, D):
    rng = np.random.default_rng(R + lg_n)
    n = 1 << lg_n
    wires, sigmas, k_is, x, last_cycle = copy_constrained_witness(rng, R, lg_n, n_cycles=min(8, R * n // 6))
    betas, gammas = [int(v) for v in rng.integers(1, P, 2, dtype=np.uint64)], [int(v) for v in rng.integers(1, P, 2, dtype=np.uint64)]
    out = po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D)
    K = -(-R // D)
    for c, (beta, gamma) in enumerate(zip(betas, gammas)):
        z = [int(v) for v in out[c, K - 1]]
        assert z[0] == 1
        wrap = z[-1]
        for i in range(n):
            num, den = _num_den(wires, sigmas, k_is, x, beta, gamma, i)
            # check_partial_products (util/partial_products.rs): prev * prod(num chunk) == next * prod(den chunk), from
            # Z(x) through the partial products to Z(gx)
            chain = [z[i]] + [int(out[c, k, i]) for k in range(K - 1)] + [z[(i + 1) % n]]
            for k in range(K):
                nk = prod(num[k * D:(k + 1) * D])
                dk = prod(den[k * D:(k + 1) * D])
                if i == n - 1 and k == K - 1:
                    wrap = chain[k] * nk * pow(dk, P - 2, P) % P
                else:
                    assert chain[k] * nk % P == chain[k + 1] * dk % P, (c, i, k)
        assert wrap == 1   # the running product returns to 1 after row n - 1

    # one changed wire value breaks the wrap-around
    i, j = last_cycle[0]
    wires2 = wires.copy()
    wires2[j][i] = (int(wires2[j][i]) + 1) % P
    out2 = po.all_wires_permutation_partial_products(wires2, sigmas, k_is, betas, gammas, D)
    for c, (beta, gamma) in enumerate(zip(betas, gammas)):
        num, den = _num_den(wires2, sigmas, k_is, x, beta, gamma, n - 1)
        tail = int(out2[c, K - 1, n - 1]) * prod(num) * pow(prod(den), P - 2, P) % P
        assert tail != 1


# ---- get_unique_coset_shifts ---------------------------------------------------------------------------------------------
def test_get_unique_coset_shifts():
    from plonky2_demo_b200.permutation import get_unique_coset_shifts

    assert get_unique_coset_shifts(1 << 20, 80).tolist() == [pow(7, j, P) for j in range(80)]
    assert get_unique_coset_shifts(8, 0).size == 0
    order = (P - 1) // 5   # a subgroup with (p - 1) / |H| = 5 cosets (Lagrange)
    assert get_unique_coset_shifts(order, 5).tolist() == [pow(7, j, P) for j in range(5)]
    with pytest.raises(ValueError, match="The subgroup does not have enough distinct cosets"):
        get_unique_coset_shifts(order, 6)
    with pytest.raises(ValueError, match="The subgroup does not have enough distinct cosets"):
        get_unique_coset_shifts(1 << 32, (P - 1) // (1 << 32) + 1)


def test_num_partial_products():
    from plonky2_demo_b200.permutation import num_partial_products

    assert num_partial_products(80, 8) == 9     # standard_recursion_config: 2 (1 + 9) = 20 polynomials in commitment #2
    assert num_partial_products(8, 8) == 0
    assert num_partial_products(9, 2) == 4
