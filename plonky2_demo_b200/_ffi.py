"""ctypes binding of libpcs.so (include/pcs.h).  Fails loudly when the CUDA engine is missing:
there is no CPU fallback in this package."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCS_LIB") or os.path.join(_HERE, "libpcs.so")   # PCS_LIB: A/B builds of the same engine

u64p = C.POINTER(C.c_uint64)
u64pp = C.POINTER(u64p)
sz = C.c_size_t

PCS_DEVICE_PTRS = 1
PCS_KEEP_COEFFS = 2
PCS_MULTI_CE_GATHER = 4
PCS_LDE_ON_DEMAND = 8

# every symbol include/pcs.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "pcs_init": (C.c_int, [C.c_int, C.c_void_p]),
    "pcs_device": (C.c_int, []),
    "pcs_shutdown": (None, []),
    "pcs_last_error": (C.c_char_p, []),
    "pcs_stream": (C.c_void_p, []),
    "pcs_synchronize": (C.c_int, []),
    "pcs_field_op": (C.c_int, [C.c_int, u64p, u64p, sz, u64p]),
    "pcs_poseidon_permute": (C.c_int, [u64p, sz]),
    "pcs_pow_grind": (C.c_int, [u64p, C.c_uint, C.c_uint, u64p]),
    "pcs_hash_or_noop": (C.c_int, [u64p, sz, sz, u64p]),
    "pcs_two_to_one": (C.c_int, [u64p, u64p, sz, u64p]),
    "pcs_ntt": (C.c_int, [u64p, sz, C.c_uint, C.c_int]),
    "pcs_coset_intt": (C.c_int, [u64p, sz, C.c_uint, C.c_uint64]),
    "pcs_ntt_dev": (C.c_int, [C.c_void_p, sz, C.c_uint, C.c_int]),
    "pcs_coset_intt_dev": (C.c_int, [C.c_void_p, sz, C.c_uint, C.c_uint64]),
    "pcs_coset_lde": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint64, u64p, C.c_int]),
    "pcs_coset_lde_dev": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint64, C.c_void_p]),
    "pcs_merkle_build": (C.c_int, [u64p, sz, sz, C.c_uint, u64p, u64p]),
    "pcs_commit_from_coeffs": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint, u64pp, sz, C.c_uint, u64p, C.POINTER(C.c_void_p)]),
    "pcs_commit_shard_from_coeffs": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint, u64pp, sz, C.c_uint, u64p, C.POINTER(C.c_void_p)]),
    "pcs_shard_begin": (C.c_int, [sz, sz, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_void_p)]),
    "pcs_shard_begin_rows": (C.c_int, [sz, sz, C.c_uint, C.c_uint, C.POINTER(C.c_void_p)]),
    "pcs_shard_set_rows": (C.c_int, [C.c_void_p, sz, sz, u64pp, C.c_int]),
    "pcs_shard_extend": (C.c_int, [C.c_void_p, sz, sz, u64pp]),
    "pcs_shard_finish": (C.c_int, [C.c_void_p, u64p]),
    "pcs_commit_from_values": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint, u64pp, sz, C.c_uint, u64pp, u64p, C.POINTER(C.c_void_p)]),
    "pcs_batch_shape": (C.c_int, [C.c_void_p, C.POINTER(sz), C.POINTER(sz), C.POINTER(sz), C.POINTER(C.c_uint)]),
    "pcs_batch_cap": (C.c_int, [C.c_void_p, u64p]),
    "pcs_batch_digests": (C.c_int, [C.c_void_p, u64p]),
    "pcs_batch_leaves": (C.c_int, [C.c_void_p, sz, sz, u64p]),
    "pcs_batch_get_rows": (C.c_int, [C.c_void_p, u64p, sz, u64p]),
    "pcs_batch_lde_natural": (C.c_int, [C.c_void_p, sz, sz, sz, u64p]),
    "pcs_batch_prove": (C.c_int, [C.c_void_p, sz, u64p]),
    "pcs_batch_prove_many": (C.c_int, [C.c_void_p, u64p, sz, u64p]),
    "pcs_batch_coeffs": (C.c_int, [C.c_void_p, sz, u64p]),
    "pcs_batch_all_coeffs": (C.c_int, [C.c_void_p, u64p]),
    "pcs_batch_lde_dev": (C.c_void_p, [C.c_void_p]),
    "pcs_batch_coeffs_dev": (C.c_void_p, [C.c_void_p]),
    "pcs_batch_digests_dev": (C.c_void_p, [C.c_void_p]),
    "pcs_batch_cap_dev": (C.c_void_p, [C.c_void_p]),
    "pcs_batch_timings": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pcs_batch_free": (None, [C.c_void_p]),
    "pcs_timing_totals": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_uint), C.c_int]),
    # one commitment over several GPUs from one process
    "pcs_multi_init": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "pcs_multi_devices": (C.c_int, [C.POINTER(C.c_int)]),
    "pcs_multi_commit_from_coeffs": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint, u64pp, sz, C.c_uint, u64p, C.POINTER(C.c_void_p)]),
    "pcs_multi_commit_from_values": (C.c_int, [u64pp, sz, C.c_uint, C.c_uint, C.c_uint, u64pp, sz, C.c_uint, u64pp, u64p, C.POINTER(C.c_void_p)]),
    "pcs_multi_batch_shape": (C.c_int, [C.c_void_p, C.POINTER(sz), C.POINTER(sz), C.POINTER(C.c_int), C.POINTER(C.c_uint)]),
    "pcs_multi_batch_cap": (C.c_int, [C.c_void_p, u64p]),
    "pcs_multi_batch_get_rows": (C.c_int, [C.c_void_p, u64p, sz, u64p]),
    "pcs_multi_batch_prove": (C.c_int, [C.c_void_p, sz, u64p]),
    "pcs_multi_batch_shard": (C.c_void_p, [C.c_void_p, C.c_int]),
    "pcs_multi_batch_poly_ptrs": (C.c_int, [C.c_void_p, u64pp]),
    "pcs_multi_batch_timings": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pcs_multi_batch_free": (None, [C.c_void_p]),
    # FRI opening proof (SURVEY 8f N2 / N3)
    "pcs_batch_eval_ext": (C.c_int, [C.c_void_p, u64p, u64p]),
    "pcs_eval_ext_dev": (C.c_int, [u64pp, sz, C.c_uint, u64p, u64p]),
    "pcs_fri_final_poly_dev": (C.c_int, [u64pp, C.c_uint, sz, u64p, C.POINTER(sz), u64p, C.POINTER(C.c_void_p)]),
    "pcs_ext_poly_new": (C.c_int, [u64p, sz, C.POINTER(C.c_void_p)]),
    "pcs_ext_poly_len": (C.c_int, [C.c_void_p, C.POINTER(sz)]),
    "pcs_ext_poly_read": (C.c_int, [C.c_void_p, u64p]),
    "pcs_ext_poly_free": (None, [C.c_void_p]),
    "pcs_fri_final_poly": (C.c_int, [C.POINTER(C.c_void_p), sz, sz, u64p, C.POINTER(sz), C.POINTER(C.c_uint32),
                                     C.POINTER(C.c_uint32), u64p, C.POINTER(C.c_void_p)]),
    "pcs_ext_coset_lde": (C.c_int, [C.c_void_p, C.c_uint, C.c_uint64, u64p]),
    "pcs_fri_commit_layer": (C.c_int, [C.c_void_p, C.c_uint, C.c_uint64, C.c_uint, C.c_uint, u64p, C.POINTER(C.c_void_p)]),
    "pcs_fri_fold": (C.c_int, [C.c_void_p, C.c_uint, u64p]),
}

_lib = None


class PcsError(RuntimeError):
    """Non-zero pcs_status.  The reference panics in the same situations."""

    def __init__(self, code, msg):
        super().__init__(f"pcs error {code}: {msg}")
        self.code = code
        self.msg = msg


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA engine with `python -m plonky2_demo_b200.build` "
                "(this package has no CPU fallback)"
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise PcsError(rc, (lib().pcs_last_error() or b"").decode())
    return rc


def ptr(a):
    return a.ctypes.data_as(u64p) if a is not None else None


def as_u64(a, copy=False):
    if copy:
        return np.array(a, dtype=np.uint64, order="C", copy=True)
    return np.ascontiguousarray(a, dtype=np.uint64)


def ptr_array(arrays):
    """u64** over a list of contiguous uint64 numpy arrays (kept alive by the caller)."""
    arr = (u64p * len(arrays))()
    for i, a in enumerate(arrays):
        arr[i] = a.ctypes.data_as(u64p)
    return arr


def dev_ptr_array(base, count, stride_elems):
    """u64** over `count` device pointers base + j*stride (a contiguous device matrix)."""
    arr = (u64p * count)()
    for j in range(count):
        arr[j] = C.cast(C.c_void_p(base + 8 * j * stride_elems), u64p)
    return arr
