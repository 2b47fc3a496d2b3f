"""The gate constraints of prove()'s quotient step, evaluated on the GPU (pcs_gate_constraint_terms).

Mirror of evaluate_gate_constraints_base_batch (plonk/vanishing_poly.rs) for the gates of the matmul demo, reduced with powers of
each alpha: gate_constraint_terms(...)[a][i] = sum_j constraint_j(x_i) alphas[a]^j at every point x_i = 7 w^i of the quotient
domain (size n 2^log2_ceil(quotient_degree_factor)), in natural order.  That is the `gate_terms` tail of quotient_poly_chunks, so

    terms = gate_constraint_terms(constants_sigmas, wires, gates, selectors_info, num_constants, pi_hash, alphas, D)
    chunks = quotient_poly_chunks(constants_sigmas, wires, zs_partial_products, ..., alphas, D, gate_terms=terms)

is the whole quotient step of a circuit built from these gates (no lookups):

    NoopGate, ConstantGate(num_consts), PublicInputGate, ArithmeticGate(num_ops), PoseidonGate     plonky2/src/gates/*.rs
    SelectorsInfo(selector_indices, groups)                                                          gates/selectors.rs

The batches are the PolynomialBatch objects of prove(): `constants_sigmas` (constant k = polynomial k, the selectors first) and
`wires` (commitment #1); their LDE rows are read in place on the device.  Any u64 is accepted; outputs are canonical.
"""
from dataclasses import dataclass

import numpy as np

from . import _ffi
from .polynomial import log2_ceil


@dataclass(frozen=True)
class NoopGate:
    pass


@dataclass(frozen=True)
class ConstantGate:
    num_consts: int


@dataclass(frozen=True)
class PublicInputGate:
    pass


@dataclass(frozen=True)
class ArithmeticGate:
    num_ops: int


@dataclass(frozen=True)
class PoseidonGate:
    pass


@dataclass(frozen=True)
class SelectorsInfo:
    """selector_indices[g]: the selector polynomial of gate g; groups[s]: the (start, end) gate range selector s covers."""
    selector_indices: tuple
    groups: tuple

    def num_selectors(self):
        return len(self.groups)


def _gate_entry(gate):
    if isinstance(gate, NoopGate):
        return _ffi.PCS_GATE_NOOP, 0
    if isinstance(gate, ConstantGate):
        return _ffi.PCS_GATE_CONSTANT, int(gate.num_consts)
    if isinstance(gate, PublicInputGate):
        return _ffi.PCS_GATE_PUBLIC_INPUT, 0
    if isinstance(gate, ArithmeticGate):
        return _ffi.PCS_GATE_ARITHMETIC, int(gate.num_ops)
    if isinstance(gate, PoseidonGate):
        return _ffi.PCS_GATE_POSEIDON, 0
    raise ValueError(f"no device evaluation for gate {gate!r}")


def gate_table(gates, selectors_info):
    """(gates [G][3] uint32: kind, param, selector_index; groups [S][2] size_t) as pcs_gate_constraint_terms takes them"""
    if len(selectors_info.selector_indices) != len(gates):
        raise ValueError("selectors_info.selector_indices needs one entry per gate")
    table = np.array([(*_gate_entry(g), int(s)) for g, s in zip(gates, selectors_info.selector_indices)],
                     dtype=np.uint32).reshape(-1, 3)
    groups = np.array([(int(r[0]), int(r[1])) for r in selectors_info.groups], dtype=np.uintp).reshape(-1, 2)
    return table, groups


def gate_constraint_terms(constants_sigmas, wires, gates, selectors_info, num_constants, public_inputs_hash, alphas,
                          quotient_degree_factor):
    """[C][n 2^q] uint64: per alpha, the gate constraints reduced with its powers at every point of the quotient domain."""
    table, groups = gate_table(gates, selectors_info)
    pih = _ffi.as_u64(np.asarray(public_inputs_hash).reshape(-1))
    a = _ffi.as_u64(np.atleast_1d(alphas))
    if pih.shape != (4,):
        raise ValueError("public_inputs_hash: 4 elements")
    D = int(quotient_degree_factor)
    n = 1 << constants_sigmas.degree_log
    out = np.empty((a.shape[0], n << log2_ceil(D)), dtype=np.uint64)
    _ffi.check(_ffi.lib().pcs_gate_constraint_terms(
        constants_sigmas._h, wires._h, table.ctypes.data_as(_ffi.C.POINTER(_ffi.C.c_uint32)), table.shape[0],
        groups.ctypes.data_as(_ffi.C.POINTER(_ffi.sz)), groups.shape[0], 0, int(num_constants), _ffi.ptr(pih), _ffi.ptr(a),
        a.shape[0], D, 0, _ffi.ptr_array([out[j] for j in range(out.shape[0])])))
    return out
