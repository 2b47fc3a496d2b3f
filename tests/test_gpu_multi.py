"""GPU tests (-m gpu) of the round-2 entry points: the device field-op grid (prime_field_testing.rs:7-17), shards that
take LDE rows / salt columns, and pcs_multi_* -- one commitment over several GPUs from ONE process -- against the CPU
oracle and against the single-GPU engine.  Tests that need more than one GPU skip themselves on a 1-GPU box; everything
else (pcs_multi_* over ONE device included) runs there."""
import ctypes as C

import numpy as np
import pytest

import oracle
from helpers import P, brev, canon, field_grid, seeded_polys

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcs():
    import plonky2_demo_b200 as p

    p.init(0)
    yield p
    p.shutdown()


def _gpu_count():
    import torch

    return torch.cuda.device_count()


# ---------------------------------------------------------------------------------------------
# K1: GoldilocksField ops on the device vs big-int arithmetic on the reference's input grid
# (field/src/prime_field_testing.rs:7-17,78-125)
# ---------------------------------------------------------------------------------------------
def _field_op(op, a, b=None):
    from plonky2_demo_b200 import _ffi

    a = np.ascontiguousarray(a, dtype=np.uint64)
    out = np.empty_like(a)
    bb = None if b is None else np.ascontiguousarray(b, dtype=np.uint64)
    _ffi.check(_ffi.lib().pcs_field_op(op, _ffi.ptr(a), _ffi.ptr(bb), a.size, _ffi.ptr(out)))
    return out


def test_device_field_grid_vs_bigint(pcs):
    g = field_grid()
    # the reference's grid is canonical; add the non-canonical representatives the engine must accept (goldilocks_field.rs:33-37)
    g = sorted(set(g + [P, P + 1, P + 9, (1 << 64) - 1, (1 << 64) - 2, (1 << 64) - (1 << 32), 0xFFFFFFFF, 0xFFFFFFFF00000000]))
    a = np.array([x for x in g for _ in g], dtype=np.uint64)
    b = np.array([y for _ in g for y in g], dtype=np.uint64)
    ai, bi = [int(x) for x in a], [int(y) for y in b]
    ops = {0: lambda x, y: (x + y) % P, 1: lambda x, y: (x - y) % P, 2: lambda x, y: x * y % P}
    for op, f in ops.items():
        want = np.array([f(x, y) for x, y in zip(ai, bi)], dtype=np.uint64)
        got = _field_op(op, a, b)
        assert np.array_equal(got, want), f"op {op}: first mismatch at {int(np.flatnonzero(got != want)[0])}"
    ga = np.array(g, dtype=np.uint64)
    gi = [int(x) for x in ga]
    assert np.array_equal(_field_op(4, ga), np.array([x * x % P for x in gi], dtype=np.uint64))
    assert np.array_equal(_field_op(5, ga), np.array([x % P for x in gi], dtype=np.uint64))
    assert np.array_equal(_field_op(6, ga), np.array([(-x) % P for x in gi], dtype=np.uint64))
    # reduce96: x + top * 2^64 for 32-bit tops
    tops = np.array([0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], dtype=np.uint64)
    a2 = np.array([x for x in gi for _ in tops], dtype=np.uint64)
    t2 = np.array([int(t) for _ in gi for t in tops], dtype=np.uint64)
    want = np.array([(int(x) + (int(t) << 64)) % P for x, t in zip(a2, t2)], dtype=np.uint64)
    assert np.array_equal(_field_op(7, a2, t2), want)
    # x * 2^k, k = 0..191 (2 has order 192: inverse_2exp, types.rs:227-262)
    ks = np.arange(192, dtype=np.uint64)
    for x in (1, 7, P - 1, (1 << 63) + 5, (1 << 64) - 1):
        got = _field_op(8, np.full(192, x, dtype=np.uint64), ks)
        assert np.array_equal(got, np.array([x * pow(2, int(k), P) % P for k in ks], dtype=np.uint64))
    # 3 names no operation (it was retired without renumbering the others): refused like any unknown op
    from plonky2_demo_b200 import _ffi

    for op in (3, 9, -1):
        with pytest.raises(_ffi.PcsError, match=r"pcs error -5: unknown field operation"):
            _field_op(op, ga, ga)


def test_device_field_random_products_vs_bigint(pcs):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 1 << 64, size=200_000, dtype=np.uint64)
    b = rng.integers(0, 1 << 64, size=200_000, dtype=np.uint64)
    want = np.array([int(x) * int(y) % P for x, y in zip(a, b)], dtype=np.uint64)
    assert np.array_equal(_field_op(2, a, b), want)
    # products whose high limbs stress the borrow / carry fix-ups: (2^32 - 1) * 2^32 multiples, p - 1 squares, tiny * huge
    edge = np.array([0xFFFFFFFF, 0xFFFFFFFF00000000, P - 1, P - 2, 1 << 32, (1 << 32) + 1, (1 << 63), 1, 0, (1 << 64) - 1], dtype=np.uint64)
    ea = np.repeat(edge, edge.size)
    eb = np.tile(edge, edge.size)
    want = np.array([int(x) * int(y) % P for x, y in zip(ea, eb)], dtype=np.uint64)
    assert np.array_equal(_field_op(2, ea, eb), want)


# ---------------------------------------------------------------------------------------------
# shards that take rows: salt columns of a coset shard, and a tree over externally computed LDE rows
# ---------------------------------------------------------------------------------------------
def _dev(arr):
    import torch

    return torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).cuda()


@pytest.mark.parametrize("w,lg_d,r,cap_h,n_shards", [(5, 6, 3, 4, 2), (9, 5, 2, 1, 4), (12, 7, 1, 0, 2)])
def test_shard_with_salt_rows(pcs, w, lg_d, r, cap_h, n_shards):
    """blinding in sharded mode: every shard = coset LDE of the polynomials + its leaf-order slice of the salt columns"""
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.sharded import ShardPlan

    L = _ffi.lib()
    d, n = 1 << lg_d, 1 << (lg_d + r)
    coeffs = seeded_polys(w, d, base_seed=0xA11CE)
    salts = seeded_polys(4, n, base_seed=0x5A17)
    salts[0, :3] = [P, P + 5, (1 << 64) - 1]                      # non-canonical salts are canonicalised
    ref = oracle.commit_from_coeffs(coeffs, r, cap_h, salts=salts)
    plan = ShardPlan(w, lg_d, r, cap_h, n_shards)
    dc = _dev(coeffs)
    salt_leaf = np.stack([salts[k][[brev(i, lg_d + r) for i in range(n)]] for k in range(4)])
    caps = []
    for k in range(n_shards):
        lo, hi = plan.leaf_range(k)
        h = C.c_void_p()
        _ffi.check(L.pcs_shard_begin(w, 4, lg_d, r, plan.coset_first(k), plan.lg_cosets, plan.local_cap_height, C.byref(h)))
        _ffi.check(L.pcs_shard_extend(h, 0, w, _ffi.dev_ptr_array(dc.data_ptr(), w, d)))
        ds = _dev(salt_leaf[:, lo:hi])
        _ffi.check(L.pcs_shard_set_rows(h, w, 4, _ffi.dev_ptr_array(ds.data_ptr(), 4, hi - lo), 0))
        cap = np.empty((plan.local_cap_len(), 4), dtype=np.uint64)
        _ffi.check(L.pcs_shard_finish(h, _ffi.ptr(cap)))
        rows = np.empty((hi - lo, w + 4), dtype=np.uint64)
        _ffi.check(L.pcs_batch_leaves(h, 0, hi - lo, _ffi.ptr(rows)))
        assert np.array_equal(rows, canon(ref["leaves"][lo:hi]))     # the oracle keeps the salts as given, the engine emits canonical values
        caps.append(cap)
        L.pcs_batch_free(h)
    from plonky2_demo_b200.hashing import PoseidonHash

    cap = plan.assemble_cap(caps, lambda a, b: PoseidonHash.two_to_one_batch(np.ascontiguousarray(a), np.ascontiguousarray(b)))
    assert np.array_equal(cap, ref["cap"])


@pytest.mark.parametrize("w,lg_d,r,cap_h,lg_parts", [(7, 6, 2, 3, 3), (135, 8, 3, 4, 4), (3, 4, 1, 0, 2)])
def test_shard_from_rows_sub_coset_ranges(pcs, w, lg_d, r, cap_h, lg_parts):
    """pcs_shard_begin_rows: trees over leaf ranges SMALLER than a coset block (more shards than 2^rate_bits), fed with the
    rows of a full LDE -- the all-to-all partition's per-GPU half; the pieces assemble to the reference tree."""
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.hashing import PoseidonHash

    L = _ffi.lib()
    d, n = 1 << lg_d, 1 << (lg_d + r)
    coeffs = seeded_polys(w, d, base_seed=0xB0B)
    ref = oracle.commit_from_coeffs(coeffs, r, cap_h)
    import torch

    dc = _dev(coeffs)
    lde = torch.empty((w, n), dtype=torch.int64, device="cuda")
    _ffi.check(L.pcs_coset_lde_dev(_ffi.dev_ptr_array(dc.data_ptr(), w, d), w, lg_d, r, 7, C.c_void_p(lde.data_ptr())))
    _ffi.check(L.pcs_synchronize())
    parts = 1 << lg_parts
    n_loc = n >> lg_parts
    lch = max(cap_h - lg_parts, 0)
    roots = []
    for k in range(parts):
        h = C.c_void_p()
        _ffi.check(L.pcs_shard_begin_rows(w, 0, lg_d + r - lg_parts, lch, C.byref(h)))
        ptrs = (_ffi.u64p * w)(*[C.cast(C.c_void_p(lde.data_ptr() + 8 * (j * n + k * n_loc)), _ffi.u64p) for j in range(w)])
        _ffi.check(L.pcs_shard_set_rows(h, 0, w, ptrs, 1))
        cap = np.empty((1 << lch, 4), dtype=np.uint64)
        _ffi.check(L.pcs_shard_finish(h, _ffi.ptr(cap)))
        rows = np.empty((n_loc, w), dtype=np.uint64)
        _ffi.check(L.pcs_batch_leaves(h, 0, n_loc, _ffi.ptr(rows)))
        assert np.array_equal(rows, ref["leaves"][k * n_loc:(k + 1) * n_loc])
        assert L.pcs_shard_extend(h, 0, 1, ptrs) != 0            # row shards do not take polynomials
        roots.append(cap)
        L.pcs_batch_free(h)
    level = np.concatenate(roots).reshape(-1, 4)
    while level.shape[0] > (1 << cap_h):
        level = PoseidonHash.two_to_one_batch(np.ascontiguousarray(level[0::2]), np.ascontiguousarray(level[1::2]))
    assert np.array_equal(level, ref["cap"])


# ---------------------------------------------------------------------------------------------
# pcs_multi_*: one process, several GPUs (or one)
# ---------------------------------------------------------------------------------------------
def _multi_commit(L, _ffi, polys, lg_d, r, cap_h, salts=None, from_values=False, flags=0, coeffs_out=None):
    w = polys.shape[0] if hasattr(polys, "shape") else len(polys)
    cap = np.empty((1 << cap_h, 4), dtype=np.uint64)
    h = C.c_void_p()
    pp = _ffi.ptr_array([polys[j] for j in range(w)])
    sp = _ffi.ptr_array([salts[k] for k in range(salts.shape[0])]) if salts is not None else None
    sw = salts.shape[0] if salts is not None else 0
    if from_values:
        co = _ffi.ptr_array([coeffs_out[j] for j in range(w)]) if coeffs_out is not None else None
        _ffi.check(L.pcs_multi_commit_from_values(pp, w, lg_d, r, cap_h, sp, sw, flags, co, _ffi.ptr(cap), C.byref(h)))
    else:
        _ffi.check(L.pcs_multi_commit_from_coeffs(pp, w, lg_d, r, cap_h, sp, sw, flags, _ffi.ptr(cap), C.byref(h)))
    return h, cap


def _check_multi_against_oracle(L, _ffi, h, cap, ref, w_total, lg_n, cap_h, rng):
    n = 1 << lg_n
    assert np.array_equal(cap, ref["cap"])
    cap2 = np.empty_like(cap)
    _ffi.check(L.pcs_multi_batch_cap(h, _ffi.ptr(cap2)))
    assert np.array_equal(cap2, cap)
    idx = np.array(sorted(set([0, n - 1] + [int(x) for x in rng.integers(0, n, size=12)])), dtype=np.uint64)
    rows = np.empty((idx.size, w_total), dtype=np.uint64)
    _ffi.check(L.pcs_multi_batch_get_rows(h, _ffi.ptr(idx), idx.size, _ffi.ptr(rows)))
    assert np.array_equal(rows, ref["leaves"][idx.astype(np.int64)])
    for k, leaf in enumerate(idx):
        sib = np.empty((lg_n - cap_h, 4), dtype=np.uint64)
        _ffi.check(L.pcs_multi_batch_prove(h, int(leaf), _ffi.ptr(sib)))
        assert np.array_equal(sib, oracle.merkle_prove(ref["digests"], n, cap_h, int(leaf)))
        assert oracle.merkle_verify(rows[k], int(leaf), cap, sib)


@pytest.mark.parametrize("n_dev", [1, 2, 4, 8])
def test_multi_commit_matches_oracle(pcs, n_dev):
    from plonky2_demo_b200 import _ffi

    if _gpu_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    L = _ffi.lib()
    L.pcs_shutdown()                                   # a fresh multi-GPU state for this device count
    _ffi.check(L.pcs_multi_init(None, n_dev))
    assert L.pcs_multi_devices(None) == n_dev
    rng = np.random.default_rng(100 + n_dev)
    try:
        # shapes: whole cap subtrees per device, one root per device + top levels (n_dev > 2^cap_height), ragged widths, chunked H2D
        for (w, lg_d, r, cap_h) in [(135, 10, 3, 4), (7, 6, 3, 0), (20, 12, 3, 2), (3, 3, 3, 4), (64, 14, 3, 4),
                                     (1, 0, 3, 0), (2, 1, 3, 3), (5, 2, 3, 4), (40, 16, 3, 4)]:   # single coefficients, fewer polynomials than devices, several H2D groups
            coeffs = seeded_polys(w, 1 << lg_d, base_seed=0xC0FFEE + w)
            coeffs[0, : min(2, coeffs.shape[1])] = [P + 3, (1 << 64) - 1][: min(2, coeffs.shape[1])]       # non-canonical input coefficients
            ref = oracle.commit_from_coeffs(coeffs, r, cap_h)
            # the other exchange: copy-engine gathers instead of peer loads fused into the first NTT pass
            h, cap = _multi_commit(L, _ffi, coeffs, lg_d, r, cap_h, flags=_ffi.PCS_MULTI_CE_GATHER)
            assert np.array_equal(cap, ref["cap"])
            L.pcs_multi_batch_free(h)
            h, cap = _multi_commit(L, _ffi, coeffs, lg_d, r, cap_h)
            _check_multi_against_oracle(L, _ffi, h, cap, ref, w, lg_d + r, cap_h, rng)
            nl, ll, ns, ch = C.c_size_t(), C.c_size_t(), C.c_int(), C.c_uint()
            _ffi.check(L.pcs_multi_batch_shape(h, C.byref(nl), C.byref(ll), C.byref(ns), C.byref(ch)))
            assert (nl.value, ll.value, ns.value, ch.value) == (1 << (lg_d + r), w, n_dev, cap_h)
            if n_dev <= (1 << cap_h):                    # the shards' digests are contiguous slices of the reference's
                nd = ref["digests"].shape[0] // n_dev
                for g in range(n_dev):
                    dg = np.empty((nd, 4), dtype=np.uint64)
                    _ffi.check(L.pcs_batch_digests(L.pcs_multi_batch_shard(h, g), _ffi.ptr(dg)))
                    assert np.array_equal(dg, ref["digests"][g * nd:(g + 1) * nd])
            L.pcs_multi_batch_free(h)
        # from_values (+ coefficients returned), blinding salts, kept coefficients + openings over peer pointers
        w, lg_d, r, cap_h = 9, 9, 3, 3
        coeffs = seeded_polys(w, 1 << lg_d, base_seed=0xFACE)
        salts = seeded_polys(4, 1 << (lg_d + r), base_seed=0x5EA)
        ref = oracle.commit_from_coeffs(coeffs, r, cap_h, salts=salts)
        out = np.zeros_like(coeffs)
        h, cap = _multi_commit(L, _ffi, oracle.fft(coeffs), lg_d, r, cap_h, salts=salts, from_values=True, coeffs_out=out)
        assert np.array_equal(out, coeffs)
        _check_multi_against_oracle(L, _ffi, h, cap, ref, w + 4, lg_d + r, cap_h, rng)
        ptrs = (_ffi.u64p * w)()
        _ffi.check(L.pcs_multi_batch_poly_ptrs(h, ptrs))
        z = np.array([0x123456789, 0x987654321], dtype=np.uint64)
        ev = np.empty((w, 2), dtype=np.uint64)
        _ffi.check(L.pcs_init(0, None))
        _ffi.check(L.pcs_eval_ext_dev(ptrs, w, lg_d, _ffi.ptr(z), _ffi.ptr(ev)))
        from oracle import fri_ref

        assert np.array_equal(ev, fri_ref.eval_base_polys_ext(coeffs, (int(z[0]), int(z[1]))))
        L.pcs_multi_batch_free(h)
        # more devices than coset blocks (rate_bits < log2 n_dev): polynomial-partitioned LDE + peer pulls of LDE rows into row
        # shards; leaf ranges are fractions of a coset block
        if n_dev > 1:
            lg_dev = n_dev.bit_length() - 1
            for (w, lg_d, r, cap_h, blind) in [(7, 6, lg_dev - 1, 1, False), (3, 5, 0, 0, True), (20, 9, lg_dev - 1, 4, False),
                                                (1, 3, 0, 2, False)]:
                if cap_h > lg_d + r:
                    continue
                coeffs = seeded_polys(w, 1 << lg_d, base_seed=0xA2A + w)
                salts = seeded_polys(4, 1 << (lg_d + r), base_seed=0x77 + w) if blind else None
                ref = oracle.commit_from_coeffs(coeffs, r, cap_h, salts=salts)
                h, cap = _multi_commit(L, _ffi, coeffs, lg_d, r, cap_h, salts=salts)
                _check_multi_against_oracle(L, _ffi, h, cap, ref, w + (4 if blind else 0), lg_d + r, cap_h, rng)
                L.pcs_multi_batch_free(h)
                out = np.zeros_like(coeffs)
                h, cap = _multi_commit(L, _ffi, oracle.fft(coeffs), lg_d, r, cap_h, salts=salts, from_values=True, coeffs_out=out)
                assert np.array_equal(cap, ref["cap"]) and np.array_equal(out, coeffs)
                L.pcs_multi_batch_free(h)
        # errors: more devices than leaves, empty batch
        if n_dev > 2:
            hh = C.c_void_p()
            c1 = seeded_polys(2, 1)
            assert L.pcs_multi_commit_from_coeffs(_ffi.ptr_array([c1[0], c1[1]]), 2, 0, 1, 0, None, 0, 0, None, C.byref(hh)) != 0
        hh = C.c_void_p()
        assert L.pcs_multi_commit_from_coeffs(None, 0, 4, 3, 0, None, 0, 0, None, C.byref(hh)) != 0
    finally:
        L.pcs_shutdown()
        pcs.init(0)


def test_multi_commit_device_pointers_and_single_gpu_equivalence(pcs):
    """device-resident inputs spread over the devices are read in place (peer loads); the cap equals the 1-GPU engine's"""
    import torch

    from plonky2_demo_b200 import _ffi

    n_dev = 2 if _gpu_count() >= 2 else 1
    L = _ffi.lib()
    L.pcs_shutdown()
    _ffi.check(L.pcs_multi_init(None, n_dev))
    try:
        w, lg_d, r, cap_h = 33, 17, 3, 4          # 35 MB: several polynomial groups in the gather pipeline
        d = 1 << lg_d
        coeffs = seeded_polys(w, d, base_seed=0xDE71CE)
        tens = [torch.from_numpy(coeffs[j].view(np.int64)).to(f"cuda:{j % n_dev}") for j in range(w)]
        for g in range(n_dev):
            torch.cuda.synchronize(g)
        ptrs = (_ffi.u64p * w)(*[C.cast(C.c_void_p(t.data_ptr()), _ffi.u64p) for t in tens])
        cap = np.empty((1 << cap_h, 4), dtype=np.uint64)
        h = C.c_void_p()
        _ffi.check(L.pcs_multi_commit_from_coeffs(ptrs, w, lg_d, r, cap_h, None, 0, _ffi.PCS_DEVICE_PTRS | _ffi.PCS_MULTI_CE_GATHER,
                                                  _ffi.ptr(cap), C.byref(h)))
        cap_peer = cap.copy()
        L.pcs_multi_batch_free(h)
        _ffi.check(L.pcs_multi_commit_from_coeffs(ptrs, w, lg_d, r, cap_h, None, 0, _ffi.PCS_DEVICE_PTRS, _ffi.ptr(cap), C.byref(h)))
        assert np.array_equal(cap, cap_peer)
        ms = (C.c_float * 5)()
        _ffi.check(L.pcs_multi_batch_timings(h, ms))
        assert ms[3] > 0
        L.pcs_multi_batch_free(h)
        _ffi.check(L.pcs_init(0, None))
        one = pcs.PolynomialBatch.from_coeffs(coeffs, r, False, cap_h)
        assert np.array_equal(cap, one.merkle_tree.cap.hashes)
        assert np.array_equal(cap, oracle.commit_from_coeffs(coeffs, r, cap_h)["cap"])
        one.free()
    finally:
        L.pcs_shutdown()
        pcs.init(0)


def test_contexts_per_device_keep_batches_alive(pcs):
    """pcs_init(other device) switches the current context; batches of the first device stay valid and are served on it"""
    from plonky2_demo_b200 import _ffi

    if _gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    L = _ffi.lib()
    coeffs = seeded_polys(6, 1 << 8, base_seed=77)
    ref = oracle.commit_from_coeffs(coeffs, 2, 1)
    b0 = pcs.PolynomialBatch.from_coeffs(coeffs, 2, False, 1)
    assert L.pcs_device() == 0
    _ffi.check(L.pcs_init(1, None))
    assert L.pcs_device() == 1
    b1 = pcs.PolynomialBatch.from_coeffs(coeffs, 2, False, 1)
    assert np.array_equal(b1.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b0.merkle_tree.leaves[:], ref["leaves"])      # served by device 0's context
    assert L.pcs_device() == 1
    b0.free()
    b1.free()
    _ffi.check(L.pcs_init(0, None))


# ---------------------------------------------------------------------------------------------
# the C ABI without Python: tests/c_abi_smoke.c built with gcc, commit + rows + paths + multi-GPU vs the oracle
# ---------------------------------------------------------------------------------------------
def build_c_smoke(tmp_path):
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    oracle.build()
    exe = str(tmp_path / "c_abi_smoke")
    subprocess.check_call(["gcc", "-O2", "-Wall", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "c_abi_smoke.c"),
                           "-o", exe, "-L", os.path.join(root, "plonky2_demo_b200"), "-lpcs", "-L", os.path.join(root, "oracle"),
                           "-loracle", f"-Wl,-rpath,{os.path.join(root, 'plonky2_demo_b200')}", f"-Wl,-rpath,{os.path.join(root, 'oracle')}"])
    return exe


@pytest.mark.parametrize("lg_d", [3, 12, 16])
def test_c_abi_smoke_binary(tmp_path, lg_d):
    import json
    import subprocess

    exe = build_c_smoke(tmp_path)
    n_dev = 1
    for k in (8, 4, 2):
        if _gpu_count() >= k:
            n_dev = k
            break
    r = subprocess.run([exe, str(n_dev), str(lg_d)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout, r.stderr)
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["c_abi_smoke"] is True and out["multi_devices"] == n_dev, out


# ---------------------------------------------------------------------------------------------
# SURVEY 8f N1: the consumers of a committed batch in compute_quotient_polys (plonk/prover.rs:576-744)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,lg_d,r,blinding", [(135, 10, 3, False), (20, 12, 3, True), (7, 5, 1, False), (3, 3, 2, True)])
def test_lde_natural_matches_get_lde_values(pcs, w, lg_d, r, blinding):
    """pcs_batch_lde_natural == get_lde_values(index, step) row by row (oracle.rs:128-133), for every step the prover uses
    (step = 2^(rate_bits - quotient_degree_bits)) and for windows of the domain"""
    d, n = 1 << lg_d, 1 << (lg_d + r)
    coeffs = seeded_polys(w, d, base_seed=0x1DE)
    salts = seeded_polys(4, n, base_seed=0x5A) if blinding else None
    ref = oracle.commit_from_coeffs(coeffs, r, 0, salts=salts)
    b = pcs.PolynomialBatch.from_coeffs(coeffs, r, blinding, 0, salts=salts)
    lg_n = lg_d + r
    for s in range(r + 1):
        step = 1 << s
        m = n // step
        want = ref["leaves"][[brev(k * step, lg_n) for k in range(m)]][:, :w]
        assert np.array_equal(b.lde_values_natural(0, step, m), want)
        # a window in the middle, and the packed accessor's 32-point batches
        lo, cnt = m // 3, min(37, m - m // 3)
        assert np.array_equal(b.lde_values_natural(lo, step, cnt), want[lo:lo + cnt])
        assert np.array_equal(b.get_lde_values(5 % m, step), want[5 % m])
    from plonky2_demo_b200 import _ffi

    out = np.empty((2, w), dtype=np.uint64)
    assert _ffi.lib().pcs_batch_lde_natural(b._h, n - 1, 1, 2, _ffi.ptr(out)) != 0      # past the end of the domain
    assert _ffi.lib().pcs_batch_lde_natural(b._h, 0, 3, 1, _ffi.ptr(out)) != 0          # step must be a power of two
    b.free()


def test_lde_natural_streams_large_tables(pcs):
    """more than one 16 MB piece: the pinned double buffering must not reorder or drop rows"""
    w, lg_d, r = 135, 14, 3
    coeffs = seeded_polys(w, 1 << lg_d, base_seed=0xB16)
    b = pcs.PolynomialBatch.from_coeffs(coeffs, r, False, 4)
    n = 1 << (lg_d + r)
    got = b.lde_values_natural(0, 1, n)                      # 141 MB
    rng = np.random.default_rng(3)
    idx = rng.integers(0, n, size=64)
    rows = b.get_rows([brev(int(k), lg_d + r) for k in idx])
    assert np.array_equal(got[idx], rows)
    # natural order: row k is P_j(7 * w^k); check a few against direct evaluation
    wN = oracle.primitive_root_of_unity(lg_d + r)
    for k in (0, 1, int(idx[0])):
        x = 7 * pow(wN, k, P) % P
        assert int(got[k][3]) == oracle.poly_eval(coeffs[3], x)
    b.free()


@pytest.mark.parametrize("w,lg_n", [(16, 15), (3, 4), (1, 0), (5, 11)])
def test_coset_intt_dev_matches_host_entry_point(pcs, w, lg_n):
    """pcs_coset_intt_dev (device pointer, asynchronous) == pcs_coset_intt == the oracle's coset_ifft; both use the
    table-driven shift^-i scaling and the tiled bit-reversal"""
    import torch

    from plonky2_demo_b200 import _ffi

    n = 1 << lg_n
    coeffs = seeded_polys(w, n, base_seed=0xC05E7)
    shift = 7
    pw = np.array([pow(shift, i, P) for i in range(n)], dtype=object)
    scaled = np.array([[int(c) * int(p) % P for c, p in zip(row, pw)] for row in coeffs], dtype=np.uint64)
    vals = oracle.fft(scaled)                                # values of P on shift * <w_n>
    t = torch.from_numpy(vals.view(np.int64).copy()).cuda()
    _ffi.check(_ffi.lib().pcs_coset_intt_dev(C.c_void_p(t.data_ptr()), w, lg_n, shift))
    _ffi.check(_ffi.lib().pcs_synchronize())
    assert np.array_equal(t.cpu().numpy().view(np.uint64), coeffs)
    host = vals.copy()
    _ffi.check(_ffi.lib().pcs_coset_intt(_ffi.ptr(host), w, lg_n, shift))
    assert np.array_equal(host, coeffs)


# ---------------------------------------------------------------------------------------------
# the latency form of Poseidon (one permutation per half-warp, poseidon_coop.cuh): every entry point that switches to it below
# 8192 permutations per launch must agree with the throughput form and with the oracle
# ---------------------------------------------------------------------------------------------
def test_cooperative_poseidon_matches_oracle_and_throughput_form(pcs):
    from plonky2_demo_b200.hashing import PoseidonHash, poseidon

    rng = np.random.default_rng(21)
    g = np.array(field_grid(), dtype=np.uint64)
    nc = np.array([P, P + 1, (1 << 64) - 1, (1 << 64) - 2, 0xFFFFFFFF, 0xFFFFFFFF00000000, 0], dtype=np.uint64)
    for n in (1, 2, 3, 7, 8, 33, 4097, 8192):            # <= 8192: latency form; odd counts leave half a warp idle
        x = np.concatenate([rng.integers(0, 1 << 64, size=(n, 12), dtype=np.uint64)[: max(n - 2, 0)],
                            g[rng.integers(0, g.size, size=(1, 12))], nc[rng.integers(0, nc.size, size=(1, 12))]])[:n]
        assert np.array_equal(poseidon(x), oracle.poseidon(x)), n
    big = rng.integers(0, 1 << 64, size=(8193, 12), dtype=np.uint64)     # throughput form
    assert np.array_equal(poseidon(big)[:100], poseidon(big[:100]))
    # two_to_one and hash_or_noop on both sides of the switch
    for n in (5, 8192, 8193):
        l = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
        r = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
        assert np.array_equal(PoseidonHash.two_to_one_batch(l, r), oracle.two_to_one(l, r))
    for ln in (1, 4, 5, 8, 9, 135):
        rows = rng.integers(0, 1 << 64, size=(100, ln), dtype=np.uint64)
        assert np.array_equal(PoseidonHash.hash_or_noop_batch(rows), oracle.hash_or_noop(rows))


@pytest.mark.parametrize("log_n,leaf_len,cap_height", [(13, 7, 0), (13, 135, 4), (14, 9, 0), (14, 32, 4), (16, 5, 2), (12, 135, 12), (7, 135, 1)])
def test_merkle_trees_across_the_latency_switch(pcs, log_n, leaf_len, cap_height):
    """trees whose leaf level / node levels sit on either side of the 8192-permutation switch between the throughput kernels
    and the latency kernels (incl. the fused top-of-tree launches): digests and cap == oracle"""
    rng = np.random.default_rng(log_n * 100 + leaf_len)
    leaves = rng.integers(0, 1 << 64, size=(1 << log_n, leaf_len), dtype=np.uint64)
    t = pcs.MerkleTree.new(leaves, cap_height)
    digests, cap = oracle.merkle_build(leaves, cap_height)
    assert np.array_equal(t.cap.hashes, cap)
    assert np.array_equal(t.digests, digests)
