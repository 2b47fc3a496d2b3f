"""prove()'s quotient polynomials, computed on the GPU from the committed batches (pcs_quotient_polys).

Mirror of the step of prove() between commitment #2 (Zs and partial products) and commitment #3 (the quotient chunks):

    compute_quotient_polys    plonk/prover.rs:576-744, without the gate constraints (the caller supplies them reduced)
    quotient_poly_chunks      prove()'s trim_to_len(quotient_degree) and chunks(degree): the input of commitment #3

The three batches are the PolynomialBatch objects of prove(): `constants_sigmas` (sigma j = polynomial num_constants + j),
`wires` (commitment #1) and `zs_partial_products` (commitment #2 in zs_partial_products_values' order).  Their LDE rows are read
in place on the device.  `gate_terms` is None or [C][n 2^q]: per alpha a, the remainder of the vanishing terms after the
permutation terms, reduced with powers of alphas[a] from alpha^0 (sum_j constraint_j(x_i) alphas[a]^j, lookup terms first when
the circuit has them), at every point of the quotient domain in natural order.  Any u64 is accepted; outputs are canonical.  A
vanishing polynomial that Z_H does not divide raises PcsError "Quotient has failed, the vanishing polynomial is not divisible
by Z_H", where the reference panics.
"""
import numpy as np

from . import _ffi
from .polynomial import log2_ceil


def quotient_poly_chunks(constants_sigmas, wires, zs_partial_products, num_constants, num_routed_wires, k_is, betas, gammas,
                         alphas, quotient_degree_factor, gate_terms=None):
    """[C D][n]: chunk k of quotient polynomial a at row a D + k, as prove() passes them to from_coeffs for commitment #3."""
    b, g, a = (_ffi.as_u64(np.atleast_1d(v)) for v in (betas, gammas, alphas))
    k = _ffi.as_u64(k_is)
    C, D, R = b.shape[0], int(quotient_degree_factor), int(num_routed_wires)
    if g.shape != b.shape or a.shape != b.shape or k.shape[0] < R:
        raise ValueError("betas, gammas and alphas need one entry per challenge, k_is num_routed_wires entries")
    n = 1 << constants_sigmas.degree_log
    tails = None
    if gate_terms is not None:
        gt = _ffi.as_u64(gate_terms)
        if gt.shape != (C, n << log2_ceil(D)):
            raise ValueError("gate_terms: [num_challenges][n 2^log2_ceil(quotient_degree_factor)]")
        tails = _ffi.ptr_array([gt[j] for j in range(C)])
    out = np.empty((C * max(D, 0), n), dtype=np.uint64)
    _ffi.check(_ffi.lib().pcs_quotient_polys(
        constants_sigmas._h, wires._h, zs_partial_products._h, int(num_constants), R, _ffi.ptr(k), _ffi.ptr(b), _ffi.ptr(g),
        _ffi.ptr(a), C, D, tails, 0, _ffi.ptr_array([out[j] for j in range(out.shape[0])])))
    return out


def compute_quotient_polys(constants_sigmas, wires, zs_partial_products, num_constants, num_routed_wires, k_is, betas, gammas,
                           alphas, quotient_degree_factor, gate_terms=None):
    """plonk/prover.rs:576-744: [C][n 2^q] coefficients of the quotient polynomials, q = log2_ceil(quotient_degree_factor), as
    the reference returns them before prove() trims them (coefficients from D n on are zero, which the engine checks)."""
    chunks = quotient_poly_chunks(constants_sigmas, wires, zs_partial_products, num_constants, num_routed_wires, k_is, betas,
                                  gammas, alphas, quotient_degree_factor, gate_terms)
    D, n = int(quotient_degree_factor), 1 << constants_sigmas.degree_log
    C = chunks.shape[0] // D
    out = np.zeros((C, n << log2_ceil(D)), dtype=np.uint64)
    out[:, :D * n] = chunks.reshape(C, D * n)
    return out
