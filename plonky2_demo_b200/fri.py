"""FRI oracle: mirror of plonky2/src/fri/{mod,oracle,reduction_strategies}.rs.

PolynomialBatch.from_values / from_coeffs run the whole commit (IFFT, coset LDE, leaf hashing,
Merkle levels) on the GPU through pcs_commit_from_values / pcs_commit_from_coeffs and return a
DEVICE-RESIDENT batch: the 9 GB of LDE rows never visit the host unless asked for.  The
reference's public fields stay available (`polynomials`, `merkle_tree.cap / .digests / .leaves`,
`degree_log`, `rate_bits`, `blinding`) and are fetched lazily.
"""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _ffi
from .hashing import MerkleCap, MerkleProof
from .polynomial import PolynomialCoeffs, PolynomialValues, log2_strict, reverse_bits

SALT_SIZE = 4  # oracle.rs:26


class FriReductionStrategy:
    """reduction_strategies.rs:11-26 (Fixed and ConstantArityBits; MinSize is an offline search
    that is out of the commit path's scope)."""

    def __init__(self, kind, *args):
        self.kind, self.args = kind, args

    @classmethod
    def Fixed(cls, arity_bits):
        return cls("Fixed", list(arity_bits))

    @classmethod
    def ConstantArityBits(cls, arity_bits, final_poly_bits):
        return cls("ConstantArityBits", arity_bits, final_poly_bits)

    def reduction_arity_bits(self, degree_bits, rate_bits, cap_height, num_queries):
        """reduction_strategies.rs:30-57"""
        if self.kind == "Fixed":
            return list(self.args[0])
        arity_bits, final_poly_bits = self.args
        result = []
        while degree_bits > final_poly_bits and degree_bits + rate_bits - arity_bits >= cap_height:
            result.append(arity_bits)
            assert degree_bits >= arity_bits
            degree_bits -= arity_bits
        return result

    def __eq__(self, other):
        return self.kind == other.kind and self.args == other.args

    def __repr__(self):
        return f"FriReductionStrategy.{self.kind}{self.args}"


@dataclass
class FriConfig:
    """fri/mod.rs:19-32"""

    rate_bits: int
    cap_height: int
    proof_of_work_bits: int
    reduction_strategy: FriReductionStrategy
    num_query_rounds: int

    def rate(self):
        return 1.0 / (1 << self.rate_bits)

    def fri_params(self, degree_bits, hiding):
        """fri/mod.rs:39-52"""
        return FriParams(
            config=self,
            hiding=hiding,
            degree_bits=degree_bits,
            reduction_arity_bits=self.reduction_strategy.reduction_arity_bits(
                degree_bits, self.rate_bits, self.cap_height, self.num_query_rounds
            ),
        )

    def num_cap_elements(self):
        return 1 << self.cap_height


@dataclass
class FriParams:
    """fri/mod.rs:62-103"""

    config: FriConfig
    hiding: bool
    degree_bits: int
    reduction_arity_bits: List[int]

    def total_arities(self):
        return sum(self.reduction_arity_bits)

    def max_arity_bits(self):
        return max(self.reduction_arity_bits) if self.reduction_arity_bits else None

    def lde_bits(self):
        return self.degree_bits + self.config.rate_bits

    def lde_size(self):
        return 1 << self.lde_bits()

    def final_poly_bits(self):
        return self.degree_bits - self.total_arities()

    def final_poly_len(self):
        return 1 << self.final_poly_bits()


def fri_proof_of_work(sponge_state, input_buffer, config):
    """fri/prover.rs:115-160 on the GPU.  `sponge_state`: the challenger's 12-lane state, `input_buffer`: its pending
    inputs (len < 12, overwritten into the state first, :136-138).  Returns the PoW witness (smallest valid one)."""
    st = _ffi.as_u64(sponge_state, copy=True).reshape(12)
    buf = _ffi.as_u64(input_buffer).reshape(-1)
    if buf.shape[0] >= 12:
        raise ValueError("input_buffer.len() < WIDTH is an invariant of Challenger")
    st[: buf.shape[0]] = buf
    min_leading_zeros = config.proof_of_work_bits + (64 - 64)   # (64 - F::order().bits()) = 0 for Goldilocks, :119
    w = C.c_uint64()
    _ffi.check(_ffi.lib().pcs_pow_grind(_ffi.ptr(st), buf.shape[0], min_leading_zeros, C.byref(w)))
    return int(w.value)


class _DeviceLeaves:
    """`merkle_tree.leaves` of a device-resident batch: rows are gathered on demand."""

    def __init__(self, batch):
        self._b = batch

    def __len__(self):
        return self._b.n_leaves

    def __getitem__(self, i):
        if isinstance(i, slice):
            start, stop, step = i.indices(len(self))
            if step == 1:
                return self._b.leaves_range(start, stop - start)
            return self._b.get_rows(range(start, stop, step))
        if i < 0:
            i += len(self)
        return self._b.get_rows([i])[0]


class _DeviceMerkleTree:
    """MerkleTree view (merkle_tree.rs:39-55) over a device-resident batch."""

    def __init__(self, batch):
        self._b = batch
        self.cap = MerkleCap(batch._cap)
        self.leaves = _DeviceLeaves(batch)
        self._digests = None

    @property
    def digests(self):
        if self._digests is None:
            out = np.empty((self._b.n_digests, 4), dtype=np.uint64)
            _ffi.check(_ffi.lib().pcs_batch_digests(self._b._h, _ffi.ptr(out)))
            self._digests = out
        return self._digests

    def get(self, i):
        """merkle_tree.rs:168"""
        return self.leaves[i]

    def prove(self, leaf_index):
        """merkle_tree.rs:173-207, gathered on the device"""
        k = log2_strict(self._b.n_leaves) - self._b.cap_height
        sib = np.empty((k, 4), dtype=np.uint64)
        _ffi.check(_ffi.lib().pcs_batch_prove(self._b._h, int(leaf_index), _ffi.ptr(sib)))
        return MerkleProof(sib)


class PolynomialBatch:
    """oracle.rs:30-37.  Construct with from_values / from_coeffs."""

    def __init__(self):
        self._h = None

    # ---- constructors -------------------------------------------------------------------------
    @classmethod
    def from_values(cls, values, rate_bits, blinding, cap_height, timing=None, fft_root_table=None, salts=None,
                    lde_on_demand=False):
        """oracle.rs:43-65.  `values`: list of PolynomialValues / arrays, or a [w][d] matrix.
        `timing` (a dict or None) receives the reference's TimingTree scope names with device times
        in ms; `fft_root_table` is accepted and ignored (the engine owns its twiddles).
        lde_on_demand: keep no LDE rows on the device (PCS_LDE_ON_DEMAND); the same commitment, and every accessor
        recomputes the rows it returns from the kept coefficients."""
        return cls._commit(values, True, rate_bits, blinding, cap_height, timing, salts, lde_on_demand=lde_on_demand)

    @classmethod
    def from_coeffs(cls, polynomials, rate_bits, blinding, cap_height, timing=None, fft_root_table=None, salts=None,
                    keep_coeffs=False, lde_on_demand=False):
        """oracle.rs:68-98.  keep_coeffs: also keep `polynomials` on the device (PCS_KEEP_COEFFS), which the opening
        proof (fri_prover.prove_openings, eval_commitment) reads; the host copy the caller passed stays referenced
        either way.  lde_on_demand: as in from_values (implies keep_coeffs)."""
        return cls._commit(polynomials, False, rate_bits, blinding, cap_height, timing, salts, keep_coeffs, lde_on_demand)

    @classmethod
    def _rows(cls, polys):
        if isinstance(polys, np.ndarray) and polys.ndim == 2:
            m = _ffi.as_u64(polys)
            return [m[j] for j in range(m.shape[0])]
        rows = []
        for p in polys:
            a = p.values if isinstance(p, PolynomialValues) else p.coeffs if isinstance(p, PolynomialCoeffs) else p
            rows.append(_ffi.as_u64(a).reshape(-1))
        return rows

    @classmethod
    def _commit(cls, polys, is_values, rate_bits, blinding, cap_height, timing, salts, keep_coeffs=False, lde_on_demand=False):
        rows = cls._rows(polys)
        if len(rows) == 0:
            raise IndexError("index out of bounds: the len is 0 but the index is 0")  # oracle.rs:76 polynomials[0]
        d = rows[0].shape[0]
        lg_d = log2_strict(d)
        for r in rows:
            if r.shape[0] != d:
                raise ValueError("assertion failed: all polynomials must have the same length")  # oracle.rs:114
        n = d << rate_bits
        salt_rows = []
        if blinding:
            if salts is None:
                # oracle.rs:119-123 draws SALT_SIZE columns from OsRng; os.urandom is the same source
                rnd = np.frombuffer(__import__("os").urandom(8 * SALT_SIZE * n), dtype=np.uint64)
                salts = (rnd % np.uint64(0xFFFFFFFF00000001)).reshape(SALT_SIZE, n)
            salt_rows = [_ffi.as_u64(s).reshape(-1) for s in salts]
            assert len(salt_rows) == SALT_SIZE and all(s.shape[0] == n for s in salt_rows)
        self = cls()
        self.degree_log, self.rate_bits, self.blinding, self.cap_height = lg_d, rate_bits, bool(blinding), cap_height
        self.n_polys, self.salt_w, self.n_leaves = len(rows), len(salt_rows), n
        self.n_digests = 2 * (n - (1 << cap_height)) if cap_height <= lg_d + rate_bits else 0
        cap = np.empty((1 << min(cap_height, 40), 4), dtype=np.uint64) if cap_height <= lg_d + rate_bits else None
        h = C.c_void_p()
        pp = _ffi.ptr_array(rows)
        sp = _ffi.ptr_array(salt_rows) if salt_rows else None
        L = _ffi.lib()
        on_demand = _ffi.PCS_LDE_ON_DEMAND if lde_on_demand else 0
        if is_values:
            # the coefficients stay on the device with the batch (PCS_KEEP_COEFFS) and are fetched when
            # `polynomials` is first read, like the leaves
            rc = L.pcs_commit_from_values(pp, len(rows), lg_d, rate_bits, cap_height, sp, len(salt_rows),
                                          _ffi.PCS_KEEP_COEFFS | on_demand, None, _ffi.ptr(cap), C.byref(h))
            self._coeffs_host = None
        else:
            rc = L.pcs_commit_from_coeffs(pp, len(rows), lg_d, rate_bits, cap_height, sp, len(salt_rows),
                                          (_ffi.PCS_KEEP_COEFFS if keep_coeffs else 0) | on_demand, _ffi.ptr(cap), C.byref(h))
            self._coeffs_host = rows
        if rc == _ffi_cap_height_code():
            raise ValueError(L.pcs_last_error().decode())  # merkle_tree.rs:136-142 message
        _ffi.check(rc)
        self._h = h
        self._cap = cap
        self.merkle_tree = _DeviceMerkleTree(self)
        if timing is not None:
            ms = (C.c_float * 5)()
            _ffi.check(L.pcs_batch_timings(h, ms))
            if is_values:
                timing["IFFT"] = ms[0]
            timing["FFT + blinding"] = ms[1]
            timing["transpose LDEs"] = ms[2]
            timing["build Merkle tree"] = ms[3] + ms[4]
        return self

    # ---- reference fields / accessors ------------------------------------------------------------
    @property
    def polynomials(self):
        """oracle.rs:33: Vec<PolynomialCoeffs<F>> (coefficient form)."""
        if self._coeffs_host is None:
            out = np.empty((self.n_polys, 1 << self.degree_log), dtype=np.uint64)
            _ffi.check(_ffi.lib().pcs_batch_all_coeffs(self._h, _ffi.ptr(out)))
            self._coeffs_host = out
        return [PolynomialCoeffs(c) for c in self._coeffs_host]

    def prove_many(self, leaf_indices):
        """MerkleTree::prove for several leaves in one device round trip -> list of MerkleProof."""
        idx = np.ascontiguousarray(np.fromiter(leaf_indices, dtype=np.uint64))
        k = log2_strict(self.n_leaves) - self.cap_height
        sib = np.empty((idx.shape[0], k, 4), dtype=np.uint64)
        _ffi.check(_ffi.lib().pcs_batch_prove_many(self._h, _ffi.ptr(idx), idx.shape[0], _ffi.ptr(sib)))
        return [MerkleProof(s) for s in sib]

    def get_rows(self, indices):
        idx = np.ascontiguousarray(np.fromiter(indices, dtype=np.uint64))
        out = np.empty((idx.shape[0], self.n_polys + self.salt_w), dtype=np.uint64)
        _ffi.check(_ffi.lib().pcs_batch_get_rows(self._h, _ffi.ptr(idx), idx.shape[0], _ffi.ptr(out)))
        return out

    def leaves_range(self, first, count):
        out = np.empty((count, self.n_polys + self.salt_w), dtype=np.uint64)
        _ffi.check(_ffi.lib().pcs_batch_leaves(self._h, first, count, _ffi.ptr(out)))
        return out

    def get_lde_values(self, index, step):
        """oracle.rs:128-133"""
        index = reverse_bits(index * step, self.degree_log + self.rate_bits)
        row = self.merkle_tree.leaves[index]
        return row[: row.shape[0] - (SALT_SIZE if self.blinding else 0)]

    def get_lde_values_packed(self, index_start, step, width):
        """oracle.rs:137-159: `width` consecutive points, returned column-major [leaf_len][width]."""
        idx = [reverse_bits((index_start + i) * step, self.degree_log + self.rate_bits) for i in range(width)]
        rows = self.get_rows(idx)
        if self.blinding:
            rows = rows[:, : rows.shape[1] - SALT_SIZE]
        return np.ascontiguousarray(rows.T)

    def lde_values_natural(self, index_start, step, count):
        """get_lde_values(index_start + k, step) for k < count in one device call: [count][n_polys] (salts dropped) -- the rows
        compute_quotient_polys walks (plonk/prover.rs:576-744), prefetched in bulk instead of 32 points at a time."""
        out = np.empty((count, self.n_polys), dtype=np.uint64)
        _ffi.check(_ffi.lib().pcs_batch_lde_natural(self._h, index_start, step, count, _ffi.ptr(out)))
        return out

    def timings(self):
        ms = (C.c_float * 5)()
        _ffi.check(_ffi.lib().pcs_batch_timings(self._h, ms))
        return list(ms)

    def free(self):
        if self._h is not None:
            _ffi.lib().pcs_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _ffi_cap_height_code():
    return -3
