"""The permutation argument's Z and partial-product polynomials, computed on the GPU (pcs_permutation_partial_products).

Mirror of the step of prove() between commitment #1 (wires) and commitment #2 (Zs and partial products):

    get_unique_coset_shifts                      field/src/cosets.rs
    wires_permutation_partial_products_and_zs    plonk/prover.rs  (one challenge)
    all_wires_permutation_partial_products       plonk/prover.rs  (every challenge)
    zs_partial_products_values                   the values prove() commits as #2, in zs_range / partial_products_range order

Inputs are host arrays: `wire_values` [num_wires][n] (witness.get_wire(i, j) = wire_values[j][i]; only the first
num_routed_wires are read), `sigma_values` [num_routed_wires][n] (the j-th sigma polynomial's values, i.e.
prover_data.sigmas[i][j] = sigma_values[j][i]), `k_is` = common_data.k_is.  Any u64 is accepted; outputs are canonical.
A zero denominator raises PcsError "Tried to invert zero", where the reference panics.
"""
import numpy as np

from . import _ffi
from .polynomial import GOLDILOCKS_ORDER, log2_strict

MULTIPLICATIVE_GROUP_GENERATOR = 7   # field/src/goldilocks_field.rs


def get_unique_coset_shifts(subgroup_size, num_shifts):
    """field/src/cosets.rs: g^0 .. g^(num_shifts - 1) for the multiplicative group's generator g = 7; the cosets g^i H are
    distinct while num_shifts <= (p - 1) / |H| (Lagrange)."""
    num_cosets = (GOLDILOCKS_ORDER - 1) // int(subgroup_size)
    if int(num_shifts) > num_cosets:
        raise ValueError("The subgroup does not have enough distinct cosets")
    return np.array([pow(MULTIPLICATIVE_GROUP_GENERATOR, i, GOLDILOCKS_ORDER) for i in range(int(num_shifts))], dtype=np.uint64)


def num_partial_products(num_routed_wires, quotient_degree_factor):
    """common_data.num_partial_products: ceil(R / D) chunks of quotient values, all but the last kept."""
    return -(-int(num_routed_wires) // int(quotient_degree_factor)) - 1


def _run(wire_values, sigma_values, k_is, betas, gammas, quotient_degree_factor, num_routed_wires, out_rows):
    """One engine call; out_rows(C, P, n) -> (result array, its C (1 + P) rows in prove() order)."""
    sigmas = _ffi.as_u64(sigma_values)
    R = sigmas.shape[0] if num_routed_wires is None else int(num_routed_wires)
    wires = _ffi.as_u64(wire_values)
    if wires.ndim != 2 or sigmas.ndim != 2 or wires.shape[0] < R or sigmas.shape[0] < R or wires.shape[1] != sigmas.shape[1]:
        raise ValueError("wire_values / sigma_values: [>= num_routed_wires][n] each")
    n = wires.shape[1]
    lg_n = log2_strict(n)
    k = _ffi.as_u64(k_is)
    b, g = _ffi.as_u64(np.atleast_1d(betas)), _ffi.as_u64(np.atleast_1d(gammas))
    if k.shape[0] < R or b.shape != g.shape:
        raise ValueError("k_is needs num_routed_wires entries, betas and gammas one per challenge")
    C = b.shape[0]
    P = num_partial_products(R, quotient_degree_factor) if R and quotient_degree_factor >= 2 else 0
    res, rows = out_rows(C, P, n)
    _ffi.check(_ffi.lib().pcs_permutation_partial_products(
        _ffi.ptr_array([wires[j] for j in range(R)]), _ffi.ptr_array([sigmas[j] for j in range(R)]), R, lg_n, _ffi.ptr(k),
        _ffi.ptr(b), _ffi.ptr(g), C, int(quotient_degree_factor), 0, _ffi.ptr_array(rows)))
    return res


def _per_challenge(C, P, n):
    out = np.empty((C, P + 1, n), dtype=np.uint64)
    return out, [out[c, P] for c in range(C)] + [out[c, k] for c in range(C) for k in range(P)]


def all_wires_permutation_partial_products(wire_values, sigma_values, k_is, betas, gammas, quotient_degree_factor,
                                           num_routed_wires=None):
    """plonk/prover.rs: [C][P + 1][n], challenge c = wires_permutation_partial_products_and_zs(betas[c], gammas[c])."""
    return _run(wire_values, sigma_values, k_is, betas, gammas, quotient_degree_factor, num_routed_wires, _per_challenge)


def wires_permutation_partial_products_and_zs(wire_values, sigma_values, k_is, beta, gamma, quotient_degree_factor,
                                              num_routed_wires=None):
    """plonk/prover.rs: [P + 1][n] = [pp_0 .. pp_{P-1}, Z] for one (beta, gamma)."""
    return _run(wire_values, sigma_values, k_is, [beta], [gamma], quotient_degree_factor, num_routed_wires, _per_challenge)[0]


def zs_partial_products_values(wire_values, sigma_values, k_is, betas, gammas, quotient_degree_factor, num_routed_wires=None):
    """[C (1 + P)][n] in prove()'s order for commitment #2 (Z of every challenge, then the partial products
    challenge-major): the matrix PolynomialBatch.from_values takes."""
    def rows(C, P, n):
        out = np.empty((C * (1 + P), n), dtype=np.uint64)
        return out, [out[j] for j in range(out.shape[0])]

    return _run(wire_values, sigma_values, k_is, betas, gammas, quotient_degree_factor, num_routed_wires, rows)
