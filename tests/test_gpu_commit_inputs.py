"""Every way a commitment's input reaches the engine (-m gpu), through the C ABI: device polynomials read in place, staged or
followed through a pointer table, host polynomials staged at once, chunk by chunk from pinned memory or through the pinned
ring from pageable memory, values transformed on the device, salts from the host or the device, full commits and shards.
Each case commits seeded polynomials; cap, digests and every leaf must equal the CPU oracle's.

Left out because another test pins them exactly: small host coefficients (test_gpu_parity.py::test_from_coeffs), host salts
of a full commit (test_gpu_parity.py::test_from_coeffs_blinding_salts), scattered device pointers with lg_d >= 1 read through
the pointer table (test_sharded.py::test_cuda_commit_from_scattered_device_pointers)."""
import ctypes as C
import functools

import numpy as np
import pytest

import oracle
from helpers import seeded_polys, splitmix64_stream

pytestmark = pytest.mark.gpu

SMALL = (24, 10, 2, 3)    # (w, lg_d, rate_bits, cap_height): 8 KB per polynomial, staged through pinned memory at once
LARGE = (48, 16, 1, 4)    # 24 MB of host input: two H2D chunks (32 + 16 polynomials), a sponge absorb between them
TINY = (9, 0, 3, 2)       # lg_d == 0: no NTT pass to follow a pointer table
SALT_W = 4

CASES = [
    # (id, shape, input, from_values, coeffs_out, salts, shard)
    ("dev_contiguous", SMALL, "device", False, False, None, False),
    ("dev_contiguous_keep", SMALL, "device_keep", False, False, None, False),
    ("dev_scattered_keep", SMALL, "scattered_keep", False, False, None, False),
    ("dev_scattered_lg_d0", TINY, "scattered", False, False, None, False),
    ("host_pinned_chunks", LARGE, "pinned", False, False, None, False),
    ("host_pageable_ring", LARGE, "host", False, False, None, False),
    ("values_dev", SMALL, "device", True, False, None, False),
    ("values_dev_coeffs_out", SMALL, "device", True, True, None, False),
    ("values_host_small", SMALL, "host", True, False, None, False),
    ("values_host_small_coeffs_out", SMALL, "host", True, True, None, False),
    ("values_host_large", LARGE, "host", True, False, None, False),
    ("values_host_large_coeffs_out", LARGE, "host", True, True, None, False),
    ("salts_dev", SMALL, "device", False, False, "device", False),
    ("shard_salts_host", SMALL, "host", False, False, "host", True),
    ("shard_salts_dev", SMALL, "device", False, False, "device", True),
]


@pytest.fixture(scope="module")
def L():
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    p.init(0)
    yield _ffi.lib()
    p.shutdown()


@functools.lru_cache(maxsize=None)
def _reference(shape, from_values, salted):
    w, lg_d, r, cap = shape
    x = seeded_polys(w, 1 << lg_d, base_seed=0xC0DE + 64 * lg_d)
    salts = splitmix64_stream(0x5A175, SALT_W << (lg_d + r)).reshape(SALT_W, -1) if salted else None
    commit = oracle.commit_from_values if from_values else oracle.commit_from_coeffs
    return x, salts, commit(x, r, cap, salts=salts)


def _dev_ptrs(tensors):
    from plonky2_demo_b200 import _ffi

    return (_ffi.u64p * len(tensors))(*[C.cast(C.c_void_p(t.data_ptr()), _ffi.u64p) for t in tensors])


def _inputs(kind, x, keep):
    """(u64** over the rows of x, flags, owners to keep alive) for one input kind."""
    import torch

    from plonky2_demo_b200 import _ffi

    w, d = x.shape
    if kind in ("device", "device_keep"):
        t = torch.from_numpy(x.view(np.int64).copy()).cuda()
        return _ffi.dev_ptr_array(t.data_ptr(), w, d), _ffi.PCS_DEVICE_PTRS | keep, [t]
    if kind in ("scattered", "scattered_keep"):
        rows = [torch.from_numpy(x[j].view(np.int64).copy()).cuda() for j in reversed(range(w))][::-1]
        return _dev_ptrs(rows), _ffi.PCS_DEVICE_PTRS | keep, rows
    if kind == "pinned":
        t = torch.from_numpy(x.view(np.int64).copy()).pin_memory()
        return (_ffi.u64p * w)(*[C.cast(C.c_void_p(t.data_ptr() + 8 * j * d), _ffi.u64p) for j in range(w)]), keep, [t]
    rows = [np.ascontiguousarray(x[j]) for j in range(w)]
    return _ffi.ptr_array(rows), keep, rows


def _check_batch(L, h, cap_out, leaves, digests, cap):
    from plonky2_demo_b200 import _ffi

    got_cap, got_dig, got_leaves = np.empty_like(cap), np.empty_like(digests), np.empty_like(leaves)
    _ffi.check(L.pcs_batch_cap(h, _ffi.ptr(got_cap)))
    _ffi.check(L.pcs_batch_digests(h, _ffi.ptr(got_dig)))
    _ffi.check(L.pcs_batch_leaves(h, 0, leaves.shape[0], _ffi.ptr(got_leaves)))
    assert np.array_equal(cap_out, cap)
    assert np.array_equal(got_cap, cap)
    assert np.array_equal(got_dig, digests)
    assert np.array_equal(got_leaves, leaves)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_commit_input_kind(L, case):
    import torch

    from plonky2_demo_b200 import _ffi

    _, shape, kind, from_values, want_coeffs, salt_src, shard = case
    w, lg_d, r, cap_h = shape
    d = 1 << lg_d
    x, salts, ref = _reference(shape, from_values, salt_src is not None)
    keep = _ffi.PCS_KEEP_COEFFS if kind.endswith("_keep") else 0
    polys, flags, owners = _inputs(kind, x, keep)
    leaves, digests, cap = ref["leaves"], ref["digests"], ref["cap"]
    lg_cosets, coset_first = r, 0
    if shard:
        # the second half of the cosets; its salt rows are the shard's own leaf range, in leaf order
        lg_cosets, coset_first = r - 1, 1 << (r - 1)
        lo, hi = coset_first * d, (coset_first << lg_d) + (d << lg_cosets)
        leaves = np.ascontiguousarray(leaves[lo:hi])
        cap_h -= 1
        digests, cap = oracle.merkle_build(leaves, cap_h)
        salts = np.ascontiguousarray(leaves[:, w:].T)
    salt_ptrs = None
    if salt_src == "host":
        salt_rows = [np.ascontiguousarray(s) for s in salts]
        salt_ptrs = _ffi.ptr_array(salt_rows)
    elif salt_src == "device":
        salt_rows = [torch.from_numpy(s.view(np.int64).copy()).cuda() for s in salts]
        salt_ptrs = _dev_ptrs(salt_rows)
    salt_w = SALT_W if salt_src else 0
    cap_out = np.empty_like(cap)
    h = C.c_void_p()
    if shard:
        _ffi.check(L.pcs_commit_shard_from_coeffs(polys, w, lg_d, r, coset_first, lg_cosets, cap_h, salt_ptrs, salt_w, flags,
                                                  _ffi.ptr(cap_out), C.byref(h)))
    elif from_values:
        coeffs_out = np.zeros_like(x) if want_coeffs else None
        out_rows = [coeffs_out[j] for j in range(w)] if want_coeffs else None
        _ffi.check(L.pcs_commit_from_values(polys, w, lg_d, r, cap_h, salt_ptrs, salt_w, flags,
                                            _ffi.ptr_array(out_rows) if want_coeffs else None, _ffi.ptr(cap_out), C.byref(h)))
        if want_coeffs:
            assert np.array_equal(coeffs_out, ref["coeffs"])
    else:
        _ffi.check(L.pcs_commit_from_coeffs(polys, w, lg_d, r, cap_h, salt_ptrs, salt_w, flags, _ffi.ptr(cap_out), C.byref(h)))
    try:
        _check_batch(L, h, cap_out, leaves, digests, cap)
        if from_values or keep:   # PolynomialBatch.polynomials stays on the device
            kept = np.empty_like(x)
            _ffi.check(L.pcs_batch_all_coeffs(h, _ffi.ptr(kept)))
            assert np.array_equal(kept, ref["coeffs"] if from_values else x)
        else:
            assert not L.pcs_batch_coeffs_dev(h)
    finally:
        L.pcs_batch_free(h)
    del owners
