"""ORACLE -- test infrastructure, NOT the product: ctypes front-end of permutation_oracle.c, the CPU restatement of
all_wires_permutation_partial_products (plonk/prover.rs).  The library is built by c_oracle."""
import ctypes as C

import c_oracle
import numpy as np
from c_oracle import u64, u64p

_lib = None


def build():
    """Compile (if needed) and return the path of the shared library."""
    return c_oracle.build("permutation_oracle")


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ref_permutation_partial_products.argtypes = [u64p, u64p, C.c_size_t, C.c_uint, u64p, u64p, u64p, C.c_size_t,
                                                       C.c_uint, u64p]
        L.ref_permutation_partial_products.restype = C.c_int
        L.ref_perm_set_num_threads.argtypes = [C.c_int]
        L.ref_perm_set_num_threads.restype = None
        _lib = L
    return _lib


def use_all_cores():
    return c_oracle.use_all_cores(lib().ref_perm_set_num_threads)


def all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, quotient_degree_factor):
    """wires, sigmas [R][n]; k_is [R]; betas, gammas [C] -> [C][P + 1][n]: per challenge [pp_0 .. pp_{P-1}, Z], the order
    wires_permutation_partial_products_and_zs returns.  Raises ZeroDivisionError("Tried to invert zero") where the
    reference panics."""
    w, s, k, b, g = (u64(a) for a in (wires, sigmas, k_is, betas, gammas))
    R, n = w.shape
    assert s.shape == (R, n) and k.shape == (R,) and b.shape == g.shape
    lg_n = n.bit_length() - 1
    assert n == 1 << lg_n and quotient_degree_factor >= 2
    P = -(-R // quotient_degree_factor) - 1
    out = np.empty((b.size, P + 1, n), dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(u64p)  # noqa: E731
    rc = lib().ref_permutation_partial_products(p(w), p(s), R, lg_n, p(k), p(b), p(g), b.size, quotient_degree_factor, p(out))
    if rc == -1:
        raise ZeroDivisionError("Tried to invert zero")
    assert rc == 0, rc
    return out


def prove_order(per_challenge):
    """[C][P + 1][n] -> [C (1 + P)][n] in the order of prove()'s commitment #2: the Zs, then the partial products
    challenge-major."""
    return np.concatenate([per_challenge[:, -1, :], per_challenge[:, :-1, :].reshape(-1, per_challenge.shape[2])])
