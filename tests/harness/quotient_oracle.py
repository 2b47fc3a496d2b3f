"""ORACLE -- test infrastructure, NOT the product: ctypes front-end of quotient_oracle.c, the CPU restatement of
compute_quotient_polys (plonk/prover.rs:576-744) without the gate constraints, and of prove()'s trim_to_len / chunks.  The library is
built by c_oracle.  Its inputs are the batches' LDEs in natural order, as oracle.coset_lde returns them."""
import ctypes as C

import c_oracle
import numpy as np
from c_oracle import u64, u64p

_lib = None

QUOTIENT_FAILED = "Quotient has failed, the vanishing polynomial is not divisible by Z_H"


def build():
    """Compile (if needed) and return the path of the shared library."""
    return c_oracle.build("quotient_oracle")


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ref_quotient_values.argtypes = [u64p, C.c_size_t, u64p, C.c_size_t, u64p, C.c_size_t, C.c_uint, C.c_uint, C.c_size_t,
                                          C.c_size_t, u64p, u64p, u64p, u64p, C.c_size_t, C.c_uint, u64p, u64p]
        L.ref_quotient_values.restype = C.c_int
        L.ref_coset_ifft.argtypes = [u64p, C.c_size_t, C.c_uint, C.c_uint64]
        L.ref_coset_ifft.restype = None
        L.ref_quot_set_num_threads.argtypes = [C.c_int]
        L.ref_quot_set_num_threads.restype = None
        _lib = L
    return _lib


def use_all_cores():
    return c_oracle.use_all_cores(lib().ref_quot_set_num_threads)


def log2_ceil(v):
    return (int(v) - 1).bit_length()


def compute_quotient_polys(cs_lde, wires_lde, zs_lde, rate_bits, num_constants, num_routed_wires, k_is, betas, gammas, alphas,
                           quotient_degree_factor, gate_terms=None):
    """Natural-order LDEs [w][n << rate_bits] of constants_sigmas, wires and zs_partial_products -> [C][n 2^q] coefficients of
    the quotient polynomials (coset_ifft(7) of the quotient values), before the trim."""
    cs, w, z = u64(cs_lde), u64(wires_lde), u64(zs_lde)
    k, b, g, a = (u64(np.atleast_1d(v)) for v in (k_is, betas, gammas, alphas))
    N = cs.shape[1]
    assert w.shape[1] == N and z.shape[1] == N and b.shape == g.shape == a.shape
    n = N >> rate_bits
    lg_n = n.bit_length() - 1
    q = log2_ceil(quotient_degree_factor)
    M = n << q
    tails = None if gate_terms is None else u64(gate_terms)
    assert tails is None or tails.shape == (b.size, M)
    out = np.empty((b.size, M), dtype=np.uint64)
    p = lambda x: x.ctypes.data_as(u64p) if x is not None else None  # noqa: E731
    rc = lib().ref_quotient_values(p(cs), cs.shape[0], p(w), w.shape[0], p(z), z.shape[0], lg_n, rate_bits, num_constants,
                                   num_routed_wires, p(k), p(b), p(g), p(a), b.size, quotient_degree_factor, p(tails), p(out))
    assert rc == 0, rc
    lib().ref_coset_ifft(p(out), b.size, lg_n + q, 7)
    return out


def quotient_poly_chunks(quotient_polys, n, quotient_degree_factor):
    """prove(): trim_to_len(D n) of every quotient polynomial (ValueError with the reference's message when a coefficient
    beyond it is not zero), then chunks(n): [C D][n], alpha-major."""
    qp = u64(quotient_polys)
    D = quotient_degree_factor
    if qp[:, D * n:].any():
        raise ValueError(QUOTIENT_FAILED)
    return qp[:, :D * n].reshape(-1, n).copy()
