"""Commitments that keep no LDE rows in HBM (PCS_LDE_ON_DEMAND, -m gpu).  Every check is exact equality.

Small shapes are checked against the CPU oracle through every input path: the cap, every digest, leaf ranges that cross coset
boundaries, get_rows on both sides of the crossover between evaluating rows from the coefficients and regenerating the LDE,
natural-order windows and Merkle paths.  The benchmark shape is checked against a resident commit of the same data, after a
decoy commit of other data has left wrong values in the pool memory the on-demand commit's scratch comes from.  Opening proofs
over on-demand oracles must equal the oracle's and verify.  135 x 2^24 (about 172 GB as a resident batch) commits on one GPU."""
import ctypes as C
import functools
import random

import numpy as np
import pytest

import oracle
from helpers import P, as_oracle_proof, assert_same_proof, brev, seeded_polys, splitmix64_stream
from oracle import fri_ref as fr

pytestmark = pytest.mark.gpu

SALT_W = 4
ROWS_EVAL_MAX = 128            # csrc/common.cuh: get_rows above this many rows regenerates the LDE
ERR_ARG = -5

CASES = [
    # (id, (w, lg_d, rate_bits, cap_height), input, from_values, coeffs_out, salts: where they live, as the input does)
    ("lgd0_r3_w9", (9, 0, 3, 2), "device", False, False, None),
    ("lgd0_r0_w1_unhashed", (1, 0, 0, 0), "host", False, False, None),
    ("lgd1_r4_w5_cap_logn", (5, 1, 4, 5), "device", False, False, "device"),
    ("lgd5_r2_w17_cap_eq_rate", (17, 5, 2, 2), "scattered", False, False, None),
    ("lgd5_r1_w8_cap_above_rate", (8, 5, 1, 3), "host", False, False, "host"),
    ("lgd12_r3_w135", (135, 12, 3, 4), "device", False, False, None),
    ("lgd12_r0_w24_last_group_on_rate", (24, 12, 0, 2), "device", True, False, None),
    ("lgd15_r1_w4_cap0_unhashed", (4, 15, 1, 0), "device", False, False, None),
    ("lgd15_r2_w4_salted", (4, 15, 2, 1), "host", False, False, "host"),
    ("lgd10_r2_w9_scattered_salted", (9, 10, 2, 3), "scattered", False, False, "device"),
    ("host_pinned_chunks", (48, 16, 1, 4), "pinned", False, False, None),
    ("host_pageable_ring", (48, 16, 1, 4), "host", False, False, "host"),
    ("values_host_large_coeffs_out", (48, 16, 1, 4), "host", True, True, None),
    ("values_host_small_coeffs_out", (24, 10, 2, 3), "host", True, True, "host"),
    ("values_dev_coeffs_out", (9, 10, 3, 3), "device", True, True, None),
    ("values_host_small", (17, 8, 1, 2), "host", True, False, "host"),
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
    x = seeded_polys(w, 1 << lg_d, base_seed=0x0D0D + 64 * lg_d + w)
    salts = splitmix64_stream(0x5A17 + w, SALT_W << (lg_d + r)).reshape(SALT_W, -1) if salted else None
    commit = oracle.commit_from_values if from_values else oracle.commit_from_coeffs
    return x, salts, commit(x, r, cap, salts=salts)


def _ptrs(tensors):
    from plonky2_demo_b200 import _ffi

    return (_ffi.u64p * len(tensors))(*[C.cast(C.c_void_p(t.data_ptr()), _ffi.u64p) for t in tensors])


def _inputs(kind, x):
    """(u64** over the rows of x, flags, owners to keep alive) for one input kind."""
    import torch

    from plonky2_demo_b200 import _ffi

    w, d = x.shape
    flags = _ffi.PCS_LDE_ON_DEMAND
    if kind == "device":
        t = torch.from_numpy(x.view(np.int64).copy()).cuda()
        return _ffi.dev_ptr_array(t.data_ptr(), w, d), flags | _ffi.PCS_DEVICE_PTRS, [t]
    if kind == "scattered":
        rows = [torch.from_numpy(x[j].view(np.int64).copy()).cuda() for j in reversed(range(w))][::-1]
        return _ptrs(rows), flags | _ffi.PCS_DEVICE_PTRS, rows
    if kind == "pinned":
        t = torch.from_numpy(x.view(np.int64).copy()).pin_memory()
        return (_ffi.u64p * w)(*[C.cast(C.c_void_p(t.data_ptr() + 8 * j * d), _ffi.u64p) for j in range(w)]), flags, [t]
    rows = [np.ascontiguousarray(x[j]) for j in range(w)]
    return _ffi.ptr_array(rows), flags, rows


def _salt_ptrs(src, salts):
    import torch

    from plonky2_demo_b200 import _ffi

    if src is None:
        return None, []
    if src == "host":
        rows = [np.ascontiguousarray(s) for s in salts]
        return _ffi.ptr_array(rows), rows
    rows = [torch.from_numpy(s.view(np.int64).copy()).cuda() for s in salts]
    return _ptrs(rows), rows


def _leaves(L, h, first, count, wt):
    from plonky2_demo_b200 import _ffi

    out = np.empty((count, wt), dtype=np.uint64)
    _ffi.check(L.pcs_batch_leaves(h, first, count, _ffi.ptr(out)))
    return out


def _get_rows(L, h, idx, wt):
    from plonky2_demo_b200 import _ffi

    idx = np.ascontiguousarray(idx, dtype=np.uint64)
    out = np.empty((idx.shape[0], wt), dtype=np.uint64)
    _ffi.check(L.pcs_batch_get_rows(h, _ffi.ptr(idx), idx.shape[0], _ffi.ptr(out)))
    return out


def _lde_natural(L, h, start, step, count, w):
    from plonky2_demo_b200 import _ffi

    out = np.empty((count, w), dtype=np.uint64)
    _ffi.check(L.pcs_batch_lde_natural(h, start, step, count, _ffi.ptr(out)))
    return out


def _prove_many(L, h, idx, depth):
    from plonky2_demo_b200 import _ffi

    idx = np.ascontiguousarray(idx, dtype=np.uint64)
    out = np.empty((idx.shape[0], depth, 4), dtype=np.uint64)
    _ffi.check(L.pcs_batch_prove_many(h, _ffi.ptr(idx), idx.shape[0], _ffi.ptr(out)))
    return out


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_on_demand_commit_matches_oracle(L, case):
    from plonky2_demo_b200 import _ffi

    _, shape, kind, from_values, want_coeffs, salt_src = case
    w, lg_d, r, cap_h = shape
    d, n = 1 << lg_d, 1 << (lg_d + r)
    x, salts, ref = _reference(shape, from_values, salt_src is not None)
    leaves, digests, cap = ref["leaves"], ref["digests"], ref["cap"]
    wt = leaves.shape[1]
    polys, flags, owners = _inputs(kind, x)
    salt_ptrs, salt_owners = _salt_ptrs(salt_src, salts)
    salt_w = SALT_W if salt_src else 0
    cap_out = np.empty_like(cap)
    h = C.c_void_p()
    if from_values:
        coeffs_out = np.zeros_like(x) if want_coeffs else None
        out_rows = _ffi.ptr_array([coeffs_out[j] for j in range(w)]) if want_coeffs else None
        _ffi.check(L.pcs_commit_from_values(polys, w, lg_d, r, cap_h, salt_ptrs, salt_w, flags, out_rows, _ffi.ptr(cap_out),
                                            C.byref(h)))
        if want_coeffs:
            assert np.array_equal(coeffs_out, ref["coeffs"])
    else:
        _ffi.check(L.pcs_commit_from_coeffs(polys, w, lg_d, r, cap_h, salt_ptrs, salt_w, flags, _ffi.ptr(cap_out), C.byref(h)))
    del owners, salt_owners   # the batch keeps its own copies
    try:
        assert not L.pcs_batch_lde_dev(h)
        got_cap, got_dig = np.empty_like(cap), np.empty_like(digests)
        _ffi.check(L.pcs_batch_cap(h, _ffi.ptr(got_cap)))
        _ffi.check(L.pcs_batch_digests(h, _ffi.ptr(got_dig)))
        assert np.array_equal(cap_out, cap) and np.array_equal(got_cap, cap)
        assert np.array_equal(got_dig, digests)
        kept = np.empty_like(x)
        _ffi.check(L.pcs_batch_all_coeffs(h, _ffi.ptr(kept)))
        assert np.array_equal(kept, ref["coeffs"] if from_values else x)
        # leaf ranges: all of them, and one that starts inside a coset and crosses into the next
        assert np.array_equal(_leaves(L, h, 0, n, wt), leaves)
        first = max(d - 3, 0) if n > d else 0
        count = min(n - first, d + 6)
        assert np.array_equal(_leaves(L, h, first, count, wt), leaves[first:first + count])
        # get_rows evaluated from the coefficients (<= ROWS_EVAL_MAX rows) and gathered from the regenerated LDE (more)
        rng = np.random.default_rng(w * 1000 + lg_d)
        for m in (1, 28, ROWS_EVAL_MAX, ROWS_EVAL_MAX + 1, 700):
            idx = rng.integers(0, n, size=m).astype(np.uint64)
            idx[0] = n - 1
            assert np.array_equal(_get_rows(L, h, idx, wt), leaves[idx.astype(np.int64)]), m
        # natural-order windows (salt columns dropped)
        for step in (1, 2, 8):
            if step > n:
                continue
            start = 1 if n // step > 1 else 0
            count = n // step - start
            want = leaves[[brev((start + k) * step, lg_d + r) for k in range(count)], :w]
            assert np.array_equal(_lde_natural(L, h, start, step, count, w), want), step
        depth = lg_d + r - cap_h
        if depth:
            idx = rng.integers(0, n, size=16).astype(np.uint64)
            sib = _prove_many(L, h, idx, depth)
            for k, i in enumerate(idx):
                assert np.array_equal(sib[k], oracle.merkle_prove(digests, n, cap_h, int(i)))
    finally:
        L.pcs_batch_free(h)


def test_on_demand_refusals(L):
    import torch

    from plonky2_demo_b200 import _ffi

    w, lg_d, r, cap_h = 9, 6, 2, 2
    d, n = 1 << lg_d, 1 << (lg_d + r)
    x = seeded_polys(w, d, base_seed=0xFEED)
    rows = [np.ascontiguousarray(x[j]) for j in range(w)]
    pp = _ffi.ptr_array(rows)
    h = C.c_void_p()
    flags = _ffi.PCS_LDE_ON_DEMAND
    assert L.pcs_commit_shard_from_coeffs(pp, w, lg_d, r, 0, 1, cap_h - 1, None, 0, flags, None, C.byref(h)) == ERR_ARG
    assert b"PCS_LDE_ON_DEMAND" in L.pcs_last_error()
    assert not h.value
    mh = C.c_void_p()
    assert L.pcs_multi_commit_from_coeffs(pp, w, lg_d, r, cap_h, None, 0, flags, None, C.byref(mh)) == ERR_ARG
    assert L.pcs_multi_commit_from_values(pp, w, lg_d, r, cap_h, None, 0, flags, None, None, C.byref(mh)) == ERR_ARG
    assert not mh.value
    t = torch.from_numpy(x.view(np.int64).copy()).cuda()
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(t.data_ptr(), w, d), w, lg_d, r, cap_h, None, 0,
                                        flags | _ffi.PCS_DEVICE_PTRS, None, C.byref(h)))
    try:
        assert not L.pcs_batch_lde_dev(h)
        assert L.pcs_batch_coeffs_dev(h)                 # implied PCS_KEEP_COEFFS
        out = np.empty((2, w), dtype=np.uint64)
        for bad in ([n], [0, n + 5]):
            idx = np.array(bad, dtype=np.uint64)
            assert L.pcs_batch_get_rows(h, _ffi.ptr(idx), idx.shape[0], _ffi.ptr(out)) == ERR_ARG
            assert b"leaf index out of bounds" in L.pcs_last_error()
        big = np.zeros(ROWS_EVAL_MAX + 1, dtype=np.uint64)
        big[-1] = n
        out_big = np.empty((big.shape[0], w), dtype=np.uint64)
        assert L.pcs_batch_get_rows(h, _ffi.ptr(big), big.shape[0], _ffi.ptr(out_big)) == ERR_ARG
        assert L.pcs_batch_leaves(h, n - 1, 2, _ffi.ptr(out)) == ERR_ARG
        assert L.pcs_batch_lde_natural(h, n // 2, 2, 1, _ffi.ptr(out)) == ERR_ARG
        sib = np.empty((lg_d + r - cap_h, 4), dtype=np.uint64)
        assert L.pcs_batch_prove(h, n, _ffi.ptr(sib)) == ERR_ARG
    finally:
        L.pcs_batch_free(h)


# ---------------------------------------------------------------------------------------------
# opening proofs over on-demand oracles (prove_openings reads rows through get_rows)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_d,rate_bits,cap_height,arities,widths,n_queries", [
    (7, 3, 4, [4], [6, 9, 3, 2], 28),           # few query rows: evaluated from the coefficients
    (9, 2, 2, [2, 2], [17, 5, 24, 3], 300),     # more than ROWS_EVAL_MAX: the LDE is regenerated
])
def test_prove_openings_over_on_demand_oracles(L, lg_d, rate_bits, cap_height, arities, widths, n_queries):
    import plonky2_demo_b200 as pcs
    from plonky2_demo_b200.fri_prover import (Challenger, FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo,
                                              eval_commitment, prove_openings)

    d, pow_bits = 1 << lg_d, 4
    coeffs = [seeded_polys(w, d, 0xA11CE + 31 * k) for k, w in enumerate(widths)]
    cpu = []
    for c in coeffs:
        o = oracle.commit_from_coeffs(c, rate_bits, cap_height)
        o["coeffs"], o["cap_height"] = c, cap_height
        cpu.append(o)
    rng = random.Random(lg_d)
    zeta = (rng.randrange(P), rng.randrange(P))
    zeta_next = fr.ext_mul((fr.primitive_root_of_unity(lg_d), 0), zeta)
    all_polys = [(k, j) for k, w in enumerate(widths) for j in range(w)]
    batches = [(zeta, all_polys), (zeta_next, [(len(widths) - 2, 0), (len(widths) - 2, 1)])]
    inst = FriInstanceInfo(oracles=[FriOracleInfo(w, False) for w in widths],
                           batches=[FriBatchInfo(pt, [FriPolynomialInfo(o, j) for o, j in ps]) for pt, ps in batches])
    cfg = pcs.FriConfig(rate_bits, cap_height, pow_bits, pcs.FriReductionStrategy.Fixed(arities), n_queries)
    params = cfg.fri_params(lg_d, False)
    for on_demand in (True, False):
        gpu = [pcs.PolynomialBatch.from_coeffs(c, rate_bits, False, cap_height, keep_coeffs=True, lde_on_demand=on_demand)
               for c in coeffs]
        openings = [[tuple(int(v) for v in eval_commitment(pt, gpu[o])[j]) for o, j in ps] for pt, ps in batches]
        ch, och = Challenger(), fr.Challenger()
        for c in (ch, och):
            for o in cpu:
                c.observe_cap(o["cap"])
            for vals in openings:
                c.observe_extension_elements(vals)
        verifier_ch = och.clone()
        got = prove_openings(inst, gpu, ch, params)
        want = fr.prove_openings(cpu, batches, och, rate_bits, cap_height, arities, pow_bits, n_queries)
        assert_same_proof(got, want)
        assert fr.verify_fri_proof(batches, openings, verifier_ch, [o["cap"] for o in cpu], as_oracle_proof(got), rate_bits,
                                   cap_height, arities, pow_bits, n_queries, lg_d)
        for b in gpu:
            b.free()


def test_python_accessors_and_serialization(L):
    """The Python mirror: leaves, get_lde_values(_packed), lde_values_natural, prove and serialisation are the resident
    batch's."""
    import plonky2_demo_b200 as pcs
    from plonky2_demo_b200 import serialization

    w, lg_d, r, cap_h = 11, 9, 2, 3
    vals = oracle.fft(seeded_polys(w, 1 << lg_d, base_seed=0xC0FFEE))
    salts = splitmix64_stream(0xB1D, SALT_W << (lg_d + r)).reshape(SALT_W, -1)
    res = pcs.PolynomialBatch.from_values(vals, r, True, cap_h, salts=salts)
    od = pcs.PolynomialBatch.from_values(vals, r, True, cap_h, salts=salts, lde_on_demand=True)
    try:
        assert np.array_equal(od.merkle_tree.cap.hashes, res.merkle_tree.cap.hashes)
        assert np.array_equal(od.merkle_tree.digests, res.merkle_tree.digests)
        assert np.array_equal(od.merkle_tree.leaves[5:300], res.merkle_tree.leaves[5:300])
        assert np.array_equal(od.merkle_tree.leaves[7], res.merkle_tree.leaves[7])
        assert np.array_equal(od.get_lde_values(13, 2), res.get_lde_values(13, 2))
        assert np.array_equal(od.get_lde_values_packed(32, 1, 32), res.get_lde_values_packed(32, 1, 32))
        assert np.array_equal(od.lde_values_natural(0, 4, 512), res.lde_values_natural(0, 4, 512))
        assert np.array_equal(od.merkle_tree.prove(77).siblings, res.merkle_tree.prove(77).siblings)
        assert [p.siblings.tolist() for p in od.prove_many([1, 2, 2047])] == [p.siblings.tolist() for p in res.prove_many([1, 2, 2047])]
        assert all(np.array_equal(a.coeffs, b.coeffs) for a, b in zip(od.polynomials, res.polynomials))
        assert serialization.polynomial_batch_to_bytes(od) == serialization.polynomial_batch_to_bytes(res)
    finally:
        od.free()
        res.free()


# ---------------------------------------------------------------------------------------------
# benchmark size, against a resident commit of the same data
# ---------------------------------------------------------------------------------------------
def test_headline_shape_matches_resident_commit(L):
    import torch

    from plonky2_demo_b200 import _ffi

    w, lg_d, r, cap_h = 135, 20, 3, 4
    d, n = 1 << lg_d, 1 << (lg_d + r)
    if torch.cuda.mem_get_info()[0] < (24 << 30):
        pytest.skip("the benchmark shape needs 24 GiB of free HBM")
    gen = torch.Generator(device="cuda").manual_seed(0x0D)
    x = torch.randint(0, 1 << 62, (w, d), dtype=torch.int64, device="cuda", generator=gen)
    decoy = torch.randint(0, 1 << 62, (w, d), dtype=torch.int64, device="cuda", generator=gen)
    flags = _ffi.PCS_DEVICE_PTRS
    cap_r, cap_o = np.empty((16, 4), dtype=np.uint64), np.empty((16, 4), dtype=np.uint64)
    hr, hd, ho = C.c_void_p(), C.c_void_p(), C.c_void_p()
    # resident commit first (kept alive, so its buffers cannot hand the right values to the on-demand commit), then a decoy
    # on-demand commit of other data freed in stream order, then the checked commit with no host sync in between
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(x.data_ptr(), w, d), w, lg_d, r, cap_h, None, 0, flags,
                                        _ffi.ptr(cap_r), C.byref(hr)))
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(decoy.data_ptr(), w, d), w, lg_d, r, cap_h, None, 0,
                                        flags | _ffi.PCS_LDE_ON_DEMAND, None, C.byref(hd)))
    L.pcs_batch_free(hd)
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(x.data_ptr(), w, d), w, lg_d, r, cap_h, None, 0,
                                        flags | _ffi.PCS_LDE_ON_DEMAND, None, C.byref(ho)))
    try:
        _ffi.check(L.pcs_batch_cap(ho, _ffi.ptr(cap_o)))
        assert np.array_equal(cap_o, cap_r)
        nd = 2 * (n - 16)
        dr, do = np.empty((nd, 4), dtype=np.uint64), np.empty((nd, 4), dtype=np.uint64)
        _ffi.check(L.pcs_batch_digests(hr, _ffi.ptr(dr)))
        _ffi.check(L.pcs_batch_digests(ho, _ffi.ptr(do)))
        assert np.array_equal(do, dr)
        del dr, do
        rng = np.random.default_rng(28)
        for m in (28, 1000):
            idx = rng.integers(0, n, size=m).astype(np.uint64)
            assert np.array_equal(_get_rows(L, ho, idx, w), _get_rows(L, hr, idx, w)), m
        assert np.array_equal(_lde_natural(L, ho, 12345, 2, 1 << 16, w), _lde_natural(L, hr, 12345, 2, 1 << 16, w))
        first = 3 * d - 1000
        assert np.array_equal(_leaves(L, ho, first, 5000, w), _leaves(L, hr, first, 5000, w))
    finally:
        L.pcs_batch_free(ho)
        L.pcs_batch_free(hr)


def _mem_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def test_large_commit_on_one_gpu(L):
    """135 x 2^24 at rate 3: 145 GB of LDE rows as a resident batch, which does not fit one B200.  Rows equal direct
    evaluation and Merkle paths verify against the cap.  Then configs[4]'s opening proof over it (bench.py's instance at
    degree 2^24: all at zeta, the first 20 at g * zeta, arities [4] x 5, 28 queries, 16 PoW bits) against fri_ref: the CPU
    cannot build this commitment's tree, so the transcript observes the device's cap, initial-tree rows come from direct
    evaluation and initial-tree paths from pcs_batch_prove_many (the verifier checks them against the cap); everything else
    must be equal: openings, the 2^24-coefficient final polynomial and its 2^27-point LDE, 5 commit-phase caps, the final
    polynomial, the PoW witness and every query step."""
    import torch

    import plonky2_demo_b200 as pcs
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.fri import _DeviceMerkleTree
    from plonky2_demo_b200.fri_prover import (Challenger, FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo,
                                              eval_commitment, final_poly, prove_openings)

    w, lg_d, r, cap_h = 135, 24, 3, 4
    d, n = 1 << lg_d, 1 << (lg_d + r)
    free, host_mem = torch.cuda.mem_get_info()[0], _mem_available_bytes()
    if free < (80 << 30):
        pytest.skip(f"135 x 2^24 on demand needs 80 GiB of free HBM ({free >> 30} GiB free)")
    if host_mem < (40 << 30):
        pytest.skip(f"the 135 x 2^24 CPU reference needs 40 GiB of host memory ({host_mem >> 30} GiB available)")
    gen = torch.Generator(device="cuda").manual_seed(0x24)
    x = torch.randint(0, 1 << 62, (w, d), dtype=torch.int64, device="cuda", generator=gen)
    cap = np.empty((1 << cap_h, 4), dtype=np.uint64)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(x.data_ptr(), w, d), w, lg_d, r, cap_h, None, 0,
                                        _ffi.PCS_DEVICE_PTRS | _ffi.PCS_LDE_ON_DEMAND, _ffi.ptr(cap), C.byref(h)))
    b = pcs.PolynomialBatch()
    b._h, b._coeffs_host, b._cap = h, [], cap
    b.degree_log, b.rate_bits, b.blinding, b.cap_height = lg_d, r, False, cap_h
    b.n_polys, b.salt_w, b.n_leaves, b.n_digests = w, 0, n, 2 * (n - (1 << cap_h))
    b.merkle_tree = _DeviceMerkleTree(b)
    try:
        coeffs = x.cpu().numpy().view(np.uint64)                 # 18 GB: the CPU reference's input
        del x
        torch.cuda.empty_cache()
        rng = np.random.default_rng(24)
        idx = np.concatenate([[0, n - 1], rng.integers(0, n, size=6)]).astype(np.uint64)
        rows = _get_rows(L, h, idx, w)
        g = oracle.primitive_root_of_unity(lg_d + r)
        for k, leaf in enumerate(idx):
            xk = oracle.gl_mul(7, oracle.gl_pow(g, brev(int(leaf), lg_d + r)))
            for j in [0, 1, 67, 134]:
                assert int(rows[k, j]) == oracle.poly_eval(coeffs[j], xk), (int(leaf), j)
        idx = rng.integers(0, n, size=64).astype(np.uint64)
        rows = _get_rows(L, h, idx, w)
        sib = _prove_many(L, h, idx, lg_d + r - cap_h)
        for k, leaf in enumerate(idx):
            assert oracle.merkle_verify(rows[k], int(leaf), cap, sib[k])

        # configs[4]'s opening proof
        zeta = (0x0123456789ABCDEF % P, 0x0FEDCBA987654321 % P)
        batches = [(zeta, [(0, j) for j in range(w)]),
                   (fr.ext_mul((fr.primitive_root_of_unity(lg_d), 0), zeta), [(0, j) for j in range(20)])]
        inst = FriInstanceInfo([FriOracleInfo(w, False)],
                               [FriBatchInfo(pt, [FriPolynomialInfo(o, j) for o, j in ps]) for pt, ps in batches])
        openings = [[tuple(int(v) for v in row) for row in eval_commitment(pt, b)[:len(ps)]] for pt, ps in batches]
        for (pt, ps), vals in zip(batches, openings):
            assert vals == [tuple(int(v) for v in row) for row in fr.eval_base_polys_ext(coeffs[:len(ps)], pt)], pt
        cfg = pcs.CircuitConfig.standard_recursion_config().fri_config
        params = cfg.fri_params(lg_d, False)
        assert (cfg.rate_bits, cfg.cap_height, params.reduction_arity_bits) == (r, cap_h, [4] * 5)
        ch, och = Challenger(), fr.Challenger()
        for c in (ch, och):
            c.observe_cap(cap)
            for vals in openings:
                c.observe_extension_elements(vals)
        verifier_ch = och.clone()
        got = prove_openings(inst, [b], ch, params)

        def eval_row(i):
            xi = fr.COSET_SHIFT * pow(g, brev(i, lg_d + r), P) % P
            return fr.eval_base_polys_ext(coeffs, (xi, 0))[:, 0]

        entry = {"coeffs": coeffs, "cap_height": cap_h, "rows": eval_row,
                 "path": lambda i: np.asarray(b.prove_many([i])[0].siblings).reshape(-1, 4)}
        want = fr.prove_openings([entry], batches, och, r, cap_h, params.reduction_arity_bits, cfg.proof_of_work_bits,
                                 cfg.num_query_rounds)
        assert_same_proof(got, want)
        assert ch.get_challenge() == och.get_challenge()
        assert fr.verify_fri_proof(batches, openings, verifier_ch, [cap], as_oracle_proof(got), r, cap_h,
                                   params.reduction_arity_bits, cfg.proof_of_work_bits, cfg.num_query_rounds, lg_d)
        fin = final_poly(inst, [b], want["_alpha"])
        try:
            assert np.array_equal(fin.coeffs, want["_final_poly_full"])
            assert np.array_equal(fin.lde_coset_fft(r), want["_lde_values"])
        finally:
            fin.free()
    finally:
        b.free()
