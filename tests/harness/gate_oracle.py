"""ORACLE -- test infrastructure, NOT the product: ctypes front-end of gate_oracle.c, the CPU restatement of
evaluate_gate_constraints_base_batch (plonk/vanishing_poly.rs) for NoopGate, ConstantGate, PublicInputGate, ArithmeticGate and
PoseidonGate, reduced with powers of each alpha: the gate-constraint tail of compute_quotient_polys.  The library is built by
c_oracle.  Its inputs are the batches' LDEs in natural order, as oracle.coset_lde returns them."""
import ctypes as C

import c_oracle
import numpy as np
from c_oracle import u64, u64p

_lib = None

NOOP, CONSTANT, PUBLIC_INPUT, ARITHMETIC, POSEIDON = range(5)


def build():
    """Compile (if needed) and return the path of the shared library."""
    return c_oracle.build("gate_oracle", ("gl64.h", "poseidon_constants.h"))


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ref_gate_terms.argtypes = [u64p, C.c_size_t, u64p, C.c_size_t, C.c_uint, C.c_uint, C.POINTER(C.c_uint32), C.c_size_t,
                                     C.POINTER(C.c_size_t), C.c_size_t, C.c_size_t, u64p, u64p, C.c_size_t, C.c_uint, u64p]
        L.ref_gate_terms.restype = C.c_int
        L.ref_poseidon_gate_constraints.argtypes = [u64p, u64p]
        L.ref_poseidon_gate_constraints.restype = None
        L.ref_gate_set_num_threads.argtypes = [C.c_int]
        L.ref_gate_set_num_threads.restype = None
        _lib = L
    return _lib


def use_all_cores():
    return c_oracle.use_all_cores(lib().ref_gate_set_num_threads)


def set_num_threads(n):
    lib().ref_gate_set_num_threads(int(n))


def poseidon_gate_constraints(wires_row):
    """PoseidonGate::eval_unfiltered on one row of 135 wire values (fast form) -> its 123 constraints"""
    w = u64(wires_row)
    assert w.shape == (135,)
    out = np.empty(123, dtype=np.uint64)
    lib().ref_poseidon_gate_constraints(w.ctypes.data_as(u64p), out.ctypes.data_as(u64p))
    return out


def gate_terms(cs_lde, wires_lde, rate_bits, gates, groups, num_constants, public_inputs_hash, alphas, quotient_degree_factor):
    """Natural-order LDEs [w][n << rate_bits] of constants_sigmas and wires; gates [(kind, param, selector_index)], groups
    [(start, end)] -> [C][n 2^q] gate terms in natural order of the quotient domain"""
    cs, w = u64(cs_lde), u64(wires_lde)
    N = cs.shape[1]
    assert w.shape[1] == N
    n = N >> rate_bits
    q = (int(quotient_degree_factor) - 1).bit_length()
    M = n << q
    g = np.ascontiguousarray(np.array(gates, dtype=np.uint32).reshape(-1, 3))
    gr = np.ascontiguousarray(np.array(groups, dtype=np.uintp).reshape(-1, 2))
    pih, a = u64(np.asarray(public_inputs_hash).reshape(4)), u64(np.atleast_1d(alphas))
    out = np.empty((a.size, M), dtype=np.uint64)
    rc = lib().ref_gate_terms(cs.ctypes.data_as(u64p), cs.shape[0], w.ctypes.data_as(u64p), w.shape[0], n.bit_length() - 1,
                              rate_bits, g.ctypes.data_as(C.POINTER(C.c_uint32)), g.shape[0],
                              gr.ctypes.data_as(C.POINTER(C.c_size_t)), gr.shape[0], num_constants, pih.ctypes.data_as(u64p),
                              a.ctypes.data_as(u64p), a.size, int(quotient_degree_factor), out.ctypes.data_as(u64p))
    assert rc == 0, rc
    return out
