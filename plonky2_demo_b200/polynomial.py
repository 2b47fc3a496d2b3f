"""PolynomialValues / PolynomialCoeffs and the (i)FFT entry points.

Mirror of field/src/polynomial/mod.rs and field/src/fft.rs for F = GoldilocksField; the
transforms run on the GPU (pcs_ntt / pcs_coset_lde).
"""
import numpy as np

from . import _ffi

GOLDILOCKS_ORDER = 0xFFFFFFFF00000001
TWO_ADICITY = 32          # field/src/goldilocks_field.rs:76
COSET_SHIFT = 7           # F::coset_shift(), field/src/types.rs:437-439


def log2_strict(n):
    """util/src/lib.rs:35 -- panics (here: ValueError) if n is not a power of two."""
    n = int(n)
    if n <= 0 or n & (n - 1):
        raise ValueError(f"Not a power of two: {n}")
    return n.bit_length() - 1


def log2_ceil(n):
    """util/src/lib.rs log2_ceil: the least q with 2^q >= n."""
    return (int(n) - 1).bit_length()


def reverse_bits(n, num_bits):
    """plonky2/src/util/mod.rs:30-38"""
    return int(format(n, f"0{num_bits}b")[::-1], 2) if num_bits else 0


def reverse_index_bits(arr):
    """util/src/lib.rs:62: out[brev(i)] = arr[i] (host-side index shuffle of a small array)."""
    arr = np.asarray(arr)
    lg = log2_strict(arr.shape[0])
    idx = np.arange(arr.shape[0], dtype=np.uint64)
    rev = np.zeros_like(idx)
    for b in range(lg):
        rev |= ((idx >> np.uint64(b)) & np.uint64(1)) << np.uint64(lg - 1 - b)
    out = np.empty_like(arr)
    out[rev.astype(np.int64)] = arr
    return out


class PolynomialCoeffs:
    """field/src/polynomial/mod.rs:118 -- coefficient form, `coeffs` is a uint64 vector."""

    def __init__(self, coeffs):
        self.coeffs = _ffi.as_u64(coeffs)
        assert self.coeffs.ndim == 1

    def __len__(self):
        return self.coeffs.shape[0]

    def lde(self, rate_bits):
        """:201-203 zero-pad to len << rate_bits."""
        return self.padded(len(self) << rate_bits)

    def padded(self, new_len):
        """:216-220"""
        if new_len < len(self):
            raise ValueError(f"Trying to pad a polynomial of length {len(self)} to a length of {new_len}.")
        out = np.zeros(new_len, dtype=np.uint64)
        out[: len(self)] = self.coeffs
        return PolynomialCoeffs(out)

    def fft_with_options(self, zero_factor=None, root_table=None):
        return fft_with_options(self, zero_factor, root_table)

    def fft(self):
        return fft_with_options(self, None, None)

    def coset_fft_with_options(self, shift, zero_factor=None, root_table=None):
        """:282-295 evaluations on shift*H in natural order.  `zero_factor` only promises that the
        top (1 - 2^-zero_factor) coefficients are zero (fft.rs:165-168); it lets the engine skip
        them, the result is identical either way."""
        n = len(self)
        lg_n = log2_strict(n)
        r = int(zero_factor or 0)
        if r:
            d = n >> r
            if np.any(self.coeffs[d:] % np.uint64(GOLDILOCKS_ORDER)):
                raise ValueError("zero_factor promises zero high coefficients")
        else:
            d = n
        c = np.ascontiguousarray(self.coeffs[:d])
        out = np.empty(n, dtype=np.uint64)
        ptrs = _ffi.ptr_array([c])
        _ffi.check(_ffi.lib().pcs_coset_lde(ptrs, 1, lg_n - r, r, int(shift) % GOLDILOCKS_ORDER, _ffi.ptr(out), 0))
        return PolynomialValues(out)

    def coset_fft(self, shift):
        return self.coset_fft_with_options(shift, None, None)


class PolynomialValues:
    """field/src/polynomial/mod.rs:23 -- point-value form over the subgroup of order len."""

    def __init__(self, values):
        self.values = _ffi.as_u64(values)
        assert self.values.ndim == 1
        if log2_strict(self.values.shape[0]) > TWO_ADICITY:  # :30 debug_assert
            raise ValueError("polynomial too long for the field's two-adicity")

    def __len__(self):
        return self.values.shape[0]

    def ifft(self):
        return ifft_with_options(self, None, None)

    def coset_ifft(self, shift):
        """:63-73 coefficients from evaluations on shift*H (natural order)."""
        v = _ffi.as_u64(self.values, copy=True).reshape(1, -1)
        _ffi.check(_ffi.lib().pcs_coset_intt(_ffi.ptr(v), 1, log2_strict(v.shape[1]), int(shift) % GOLDILOCKS_ORDER))
        return PolynomialCoeffs(v[0])

    def lde(self, rate_bits):
        """:79-82 evaluations of the same polynomial on the 2^rate_bits times larger subgroup."""
        return self.ifft().lde(rate_bits).coset_fft_with_options(1, rate_bits, None)

    def lde_onto_coset(self, rate_bits):
        """:85-88"""
        return self.ifft().lde(rate_bits).coset_fft_with_options(COSET_SHIFT, rate_bits, None)


def fft_with_options(poly, zero_factor=None, root_table=None):
    """field/src/fft.rs:57-65.  `root_table` is accepted for signature compatibility; the engine
    keeps its own twiddle tables in HBM."""
    return poly.coset_fft_with_options(1, zero_factor, root_table)


def ifft_with_options(poly, zero_factor=None, root_table=None):
    """field/src/fft.rs:72-95"""
    v = _ffi.as_u64(poly.values, copy=True).reshape(1, -1)
    lg_n = log2_strict(v.shape[1])
    _ffi.check(_ffi.lib().pcs_ntt(_ffi.ptr(v), 1, lg_n, 1))
    return PolynomialCoeffs(v[0])


def ntt_batch(polys, inverse=False):
    """Batched fft/ifft on a [w][n] matrix (natural order in and out)."""
    a = _ffi.as_u64(polys, copy=True)
    w, n = a.shape
    _ffi.check(_ffi.lib().pcs_ntt(_ffi.ptr(a), w, log2_strict(n), int(bool(inverse))))
    return a
