"""Benchmark-size commitments (-m gpu), exact against the CPU oracle on every input path.

bench.py's flagship workload is a from_coeffs commit of 135 x 2^20 at rate 3 with cap height 4: 2^23 leaves and 9 GB of LDE
rows.  Several paths only run at that size: the pinned ring of pageable host input wraps ~22 times, the streaming sponge parks
its state at columns 8 and 48, and from_values hands more than 512 MB of coefficients back one polynomial at a time.  Each
case here must reproduce the oracle's cap and every digest (the hash of every leaf) exactly, plus a fixed sample of LDE rows.

The oracle runs once per shape for the whole module (about a minute on 8 host cores at the headline shape, 17 GB of host
memory at its peak); other cap heights are rebuilt from its leaf digests.

Every checked commit follows a decoy: other data of the same shape, committed through the other leaf-hashing form (one hash
kernel over the whole leaf, or the streaming sponge over groups of columns), freed in stream order, with no host sync before
the checked commit is enqueued, as in bench.py's timed loop.  Whatever the checked commit fails to write then holds the
decoy's values.  The decoy takes the other form because a write skipped by one path is skipped by a decoy on that path too,
and the memory can still hold the right values from an earlier case that committed the same data another way.

The opening proof bench.py times (eval_commitment, final_poly, prove_openings over the headline batch) is checked the same
way: every opening, the 2^20-coefficient final polynomial, its 2^23-point LDE and the whole proof against fri_ref, on a
resident and on an on-demand batch, each after a decoy proof over other data with non-canonical coefficients."""
import ctypes as C

import numpy as np
import pytest

import oracle
from helpers import P, as_oracle_proof, assert_same_proof, brev, mem_available_bytes, seeded_polys
from oracle import fri_ref as fr

pytestmark = pytest.mark.gpu

HEADLINE = (135, 20, 3, 4)   # (w, lg_d, rate_bits, cap_height): bench.py's workload
DEEP = (17, 22, 2, 6)        # 2^24 leaves; the NTT of a coset runs a 3-pass plan (7 + 7 + 8 stages); a 1-element final absorb
DECOY_SEED = 0xDEC0_0000
N_SAMPLE = 4096
MIN_FREE_HBM = 24 << 30
MIN_HOST_MEM = 40 << 30      # the oracle's peak at the headline shape, plus the inputs and readbacks of a case


@pytest.fixture(scope="module")
def L():
    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    free_hbm, host = torch.cuda.mem_get_info()[0], mem_available_bytes()
    if free_hbm < MIN_FREE_HBM:
        pytest.skip(f"benchmark-size commits need {MIN_FREE_HBM >> 30} GiB of free HBM ({free_hbm >> 30} GiB free)")
    if host < MIN_HOST_MEM:
        pytest.skip(f"the benchmark-size CPU reference needs {MIN_HOST_MEM >> 30} GiB of host memory ({host >> 30} GiB available)")
    p.init(0)
    yield _ffi.lib()
    p.shutdown()


class Reference:
    """The oracle's commitment of seeded_polys(w, 2^lg_d): cap, every digest, the leaf digests and a fixed sample of rows."""

    def __init__(self, shape):
        self.w, self.lg_d, self.r, self.cap_h = w, lg_d, r, cap_h = shape
        self.d, self.n = 1 << lg_d, 1 << (lg_d + r)
        self.coeffs = seeded_polys(w, self.d)
        self.decoy = seeded_polys(w, self.d, base_seed=DECOY_SEED)
        oracle.use_all_cores()
        ref = oracle.commit_from_coeffs(self.coeffs, r, cap_h)
        self.cap, self.digests = ref["cap"], ref["digests"]
        d, n = self.d, self.n
        edges = [0, 1, d - 1, d, n // 2 - 1, n // 2, n - 2, n - 1] + [c * d + o for c in range(1 << r) for o in (0, d - 1)]
        rng = np.random.default_rng(lg_d)
        self.idx = np.unique(np.concatenate([edges, rng.integers(0, n, size=N_SAMPLE - len(edges))]).astype(np.uint64))
        self.rows = ref["leaves"][self.idx.astype(np.int64)]
        del ref                                                     # the 9 GB of leaves
        # leaf q of cap subtree s sits at s * sub_len + 2q - (q & 1) (the level-0 case of k_prove's index formula)
        sub = self.n >> cap_h
        q = np.arange(sub)
        pos = (np.arange(1 << cap_h)[:, None] * (2 * (sub - 1)) + (2 * q - (q & 1))[None, :]).ravel()
        self.leaf_digests = np.ascontiguousarray(self.digests[pos])

    def at_cap_height(self, cap_h):
        """(digests, cap) of the same leaves for another cap height: rows of 4 elements are copied by hash_or_noop, not
        hashed, so the tree over the leaf digests is the tree over the leaves."""
        if cap_h == self.cap_h:
            return self.digests, self.cap
        return oracle.merkle_build(self.leaf_digests, cap_h)


@pytest.fixture(scope="module")
def headline():
    return Reference(HEADLINE)


@pytest.fixture(scope="module")
def deep():
    return Reference(DEEP)


def _to_device(x):
    import torch

    return torch.from_numpy(x.view(np.int64)).cuda()


def _dev_ptrs(t, first, count, d):
    from plonky2_demo_b200 import _ffi

    return _ffi.dev_ptr_array(t.data_ptr() + 8 * first * d, count, d)


def _decoy(L, ref, dev_decoy, streamed, cap_h=None, coset_first=0, lg_cosets=None):
    """Commit ref.decoy (on the device) over the given coset range and free it in stream order, without a host sync.
    streamed: through pcs_shard_begin / extend / finish in two groups (the streaming sponge); otherwise in one call with
    the coefficients kept (the whole-leaf hash kernel, and a staging buffer the size of a commit's coefficients)."""
    from plonky2_demo_b200 import _ffi

    w, lg_d, r, d = ref.w, ref.lg_d, ref.r, ref.d
    cap_h = ref.cap_h if cap_h is None else cap_h
    lg_cosets = r if lg_cosets is None else lg_cosets
    h = C.c_void_p()
    if streamed:
        _ffi.check(L.pcs_shard_begin(w, 0, lg_d, r, coset_first, lg_cosets, cap_h, C.byref(h)))
        for j0, j1 in ((0, 8), (8, w)):
            _ffi.check(L.pcs_shard_extend(h, j0, j1 - j0, _dev_ptrs(dev_decoy, j0, j1 - j0, d)))
        _ffi.check(L.pcs_shard_finish(h, None))
    else:
        _ffi.check(L.pcs_commit_shard_from_coeffs(_dev_ptrs(dev_decoy, 0, w, d), w, lg_d, r, coset_first, lg_cosets, cap_h,
                                                  None, 0, _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS, None, C.byref(h)))
    L.pcs_batch_free(h)


def _assert_rows_equal(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero((got != want).any(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} of {len(want)} differ, the first at {bad[:8].tolist()}"


def _check(L, h, digests, cap, idx, rows, cap_out=None):
    """The batch's cap, every digest and the sampled rows (leaf indices relative to the batch) against the reference."""
    from plonky2_demo_b200 import _ffi

    got_cap = np.empty_like(cap)
    _ffi.check(L.pcs_batch_cap(h, _ffi.ptr(got_cap)))
    _assert_rows_equal(got_cap, cap, "cap")
    if cap_out is not None:
        _assert_rows_equal(cap_out, cap, "cap_out")
    got = np.empty_like(digests)
    _ffi.check(L.pcs_batch_digests(h, _ffi.ptr(got)))
    _assert_rows_equal(got, digests, "digests")
    del got
    got_rows = np.empty_like(rows)
    _ffi.check(L.pcs_batch_get_rows(h, _ffi.ptr(idx), idx.size, _ffi.ptr(got_rows)))
    _assert_rows_equal(got_rows, rows, "sampled LDE rows")
    return got_rows


def _commit_device(L, ref, cap_h):
    """Device-resident contiguous coefficients, asynchronous (bench.py's timed commit); the cap is read afterwards."""
    from plonky2_demo_b200 import _ffi

    dev, dev_decoy = _to_device(ref.coeffs), _to_device(ref.decoy)
    _decoy(L, ref, dev_decoy, streamed=True, cap_h=cap_h)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(_dev_ptrs(dev, 0, ref.w, ref.d), ref.w, ref.lg_d, ref.r, cap_h, None, 0,
                                        _ffi.PCS_DEVICE_PTRS, None, C.byref(h)))
    return h, [dev, dev_decoy]


def _commit_pageable(L, ref):
    """Pageable host coefficients through the C ABI with cap_out: the pinned ring and the streaming sponge."""
    from plonky2_demo_b200 import _ffi

    dev_decoy = _to_device(ref.decoy)
    cap_out = np.empty_like(ref.cap)
    _decoy(L, ref, dev_decoy, streamed=False)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(_ffi.ptr_array([ref.coeffs[j] for j in range(ref.w)]), ref.w, ref.lg_d, ref.r,
                                        ref.cap_h, None, 0, 0, _ffi.ptr(cap_out), C.byref(h)))
    return h, cap_out


def test_headline_device_resident(L, headline):
    """The benchmarked path; sampled rows also equal direct evaluation at 7 w_N^brev(leaf) and Merkle paths the oracle's."""
    from plonky2_demo_b200 import _ffi

    ref = headline
    h, owners = _commit_device(L, ref, ref.cap_h)
    try:
        rows = _check(L, h, ref.digests, ref.cap, ref.idx, ref.rows)
        lg_n = ref.lg_d + ref.r
        w_n = oracle.primitive_root_of_unity(lg_n)
        for k in np.linspace(0, ref.idx.size - 1, 8).astype(int):
            x = 7 * pow(w_n, brev(int(ref.idx[k]), lg_n), P) % P
            assert rows[k].tolist() == [oracle.poly_eval(ref.coeffs[j], x) for j in range(ref.w)], int(ref.idx[k])
        some = np.ascontiguousarray(ref.idx[::64])
        paths = np.empty((some.size, lg_n - ref.cap_h, 4), dtype=np.uint64)
        _ffi.check(L.pcs_batch_prove_many(h, _ffi.ptr(some), some.size, _ffi.ptr(paths)))
        for k, leaf in enumerate(some.tolist()):
            assert np.array_equal(paths[k], oracle.merkle_prove(ref.digests, ref.n, ref.cap_h, leaf)), leaf
    finally:
        L.pcs_batch_free(h)
    del owners


def test_headline_pinned_host(L, headline):
    """Pinned host coefficients (bench.py's end-to-end arm): chunks [0, 8, 48, 135) on the copy stream."""
    import torch

    from plonky2_demo_b200 import _ffi

    ref = headline
    pinned = torch.from_numpy(ref.coeffs.view(np.int64)).pin_memory()
    base = pinned.data_ptr()
    polys = (_ffi.u64p * ref.w)(*[C.cast(C.c_void_p(base + 8 * j * ref.d), _ffi.u64p) for j in range(ref.w)])
    dev_decoy = _to_device(ref.decoy)
    cap_out = np.empty_like(ref.cap)
    _decoy(L, ref, dev_decoy, streamed=False)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(polys, ref.w, ref.lg_d, ref.r, ref.cap_h, None, 0, 0, _ffi.ptr(cap_out), C.byref(h)))
    try:
        _check(L, h, ref.digests, ref.cap, ref.idx, ref.rows, cap_out)
    finally:
        L.pcs_batch_free(h)
    del pinned, dev_decoy


def test_headline_pageable_host(L, headline):
    """68 pieces of 16 MB through the 3-slot pinned ring."""
    h, cap_out = _commit_pageable(L, headline)
    try:
        _check(L, h, headline.digests, headline.cap, headline.idx, headline.rows, cap_out)
    finally:
        L.pcs_batch_free(h)


def test_headline_from_values_device(L, headline):
    """from_values on device values = fft(coeffs): the commitment is from_coeffs', the kept coefficients are coeffs."""
    from plonky2_demo_b200 import _ffi

    ref = headline
    dev, dev_decoy = _to_device(oracle.fft(ref.coeffs)), _to_device(ref.decoy)
    _decoy(L, ref, dev_decoy, streamed=True)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_values(_dev_ptrs(dev, 0, ref.w, ref.d), ref.w, ref.lg_d, ref.r, ref.cap_h, None, 0,
                                        _ffi.PCS_DEVICE_PTRS, None, None, C.byref(h)))
    try:
        _check(L, h, ref.digests, ref.cap, ref.idx, ref.rows)
        kept = np.empty_like(ref.coeffs)
        _ffi.check(L.pcs_batch_all_coeffs(h, _ffi.ptr(kept)))
        _assert_rows_equal(kept, ref.coeffs, "kept coefficients")
    finally:
        L.pcs_batch_free(h)
    del dev, dev_decoy


def test_headline_from_values_pageable_coeffs_out(L, headline):
    """from_values from pageable host values with coeffs_out: 1080 MB of coefficients go back one polynomial at a time on
    the main stream (what a Rust caller gets, since it always asks for them)."""
    from plonky2_demo_b200 import _ffi

    ref = headline
    values = oracle.fft(ref.coeffs)
    dev_decoy = _to_device(ref.decoy)
    coeffs_out = np.zeros_like(ref.coeffs)
    cap_out = np.empty_like(ref.cap)
    _decoy(L, ref, dev_decoy, streamed=False)
    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_values(_ffi.ptr_array([values[j] for j in range(ref.w)]), ref.w, ref.lg_d, ref.r, ref.cap_h,
                                        None, 0, 0, _ffi.ptr_array([coeffs_out[j] for j in range(ref.w)]), _ffi.ptr(cap_out),
                                        C.byref(h)))
    try:
        _assert_rows_equal(coeffs_out, ref.coeffs, "coeffs_out")
        _check(L, h, ref.digests, ref.cap, ref.idx, ref.rows, cap_out)
    finally:
        L.pcs_batch_free(h)
    del dev_decoy


SHARD_GROUPS = [(0, 5), (5, 16), (16, 76), (76, 135)]   # boundaries off the sponge rate of 8


def test_headline_streaming_shards(L, headline):
    """Two shards of 4 cosets, local cap height 3, polynomials in groups of 5, 11, 60 and 59; the second shard gets
    [76, 135) before [16, 76), so its sponge may only absorb the columns that arrived in order."""
    from plonky2_demo_b200 import _ffi

    ref = headline
    world, lg_cosets = 2, ref.r - 1
    local_cap = ref.cap_h - 1
    dev, dev_decoy = _to_device(ref.coeffs), _to_device(ref.decoy)
    per_leaves, per_dig, per_cap = ref.n // world, ref.digests.shape[0] // world, ref.cap.shape[0] // world
    for k in range(world):
        coset_first = k << lg_cosets
        groups = SHARD_GROUPS if k == 0 else [SHARD_GROUPS[i] for i in (0, 1, 3, 2)]
        _decoy(L, ref, dev_decoy, streamed=False, cap_h=local_cap, coset_first=coset_first, lg_cosets=lg_cosets)
        h = C.c_void_p()
        _ffi.check(L.pcs_shard_begin(ref.w, 0, ref.lg_d, ref.r, coset_first, lg_cosets, local_cap, C.byref(h)))
        try:
            for j0, j1 in groups:
                _ffi.check(L.pcs_shard_extend(h, j0, j1 - j0, _dev_ptrs(dev, j0, j1 - j0, ref.d)))
            cap_out = np.empty((per_cap, 4), dtype=np.uint64)
            _ffi.check(L.pcs_shard_finish(h, _ffi.ptr(cap_out)))
            mine = (ref.idx >= np.uint64(k * per_leaves)) & (ref.idx < np.uint64((k + 1) * per_leaves))
            _check(L, h, ref.digests[k * per_dig:(k + 1) * per_dig], ref.cap[k * per_cap:(k + 1) * per_cap],
                   np.ascontiguousarray(ref.idx[mine] - np.uint64(k * per_leaves)), ref.rows[mine], cap_out)
        finally:
            L.pcs_batch_free(h)
    del dev, dev_decoy


@pytest.mark.parametrize("cap_h", [0, 16, 23])
def test_headline_cap_height(L, headline, cap_h):
    """One subtree (the deepest tree top), 2^16 subtrees, and cap_height == log2 N (no digests: the cap is the leaf
    digests)."""
    ref = headline
    digests, cap = ref.at_cap_height(cap_h)
    h, owners = _commit_device(L, ref, cap_h)
    try:
        _check(L, h, digests, cap, ref.idx, ref.rows)
    finally:
        L.pcs_batch_free(h)
    del owners


def test_deep_device_resident(L, deep):
    h, owners = _commit_device(L, deep, deep.cap_h)
    try:
        _check(L, h, deep.digests, deep.cap, deep.idx, deep.rows)
    finally:
        L.pcs_batch_free(h)
    del owners


def test_deep_pageable_host(L, deep):
    h, cap_out = _commit_pageable(L, deep)
    try:
        _check(L, h, deep.digests, deep.cap, deep.idx, deep.rows, cap_out)
    finally:
        L.pcs_batch_free(h)


# ---------------------------------------------------------------------------------------------
# the opening proof bench.py times (kernels.fri_opening)
# ---------------------------------------------------------------------------------------------
ZETA = (0x0123456789ABCDEF % P, 0x0FEDCBA987654321 % P)   # bench.py's opening point
N_NEXT = 20                                             # polynomials also opened at g * zeta
FRI_ARITIES, POW_BITS, N_QUERIES = [4, 4, 4, 4], 16, 28  # standard_recursion_config at degree 2^20
DECOY_ZETA, DECOY_ALPHA = (0x1DEC0, 0x2DEC0), (P - 5, 0xDEC0DEC0)


def _opening_batches(zeta, w, lg_d):
    zeta_next = fr.ext_mul((fr.primitive_root_of_unity(lg_d), 0), zeta)
    return [(zeta, [(0, j) for j in range(w)]), (zeta_next, [(0, j) for j in range(min(N_NEXT, w))])]


def _openings(coeffs, batches):
    return [[tuple(int(x) for x in v) for v in fr.eval_base_polys_ext(coeffs[:len(polys)], pt)] for pt, polys in batches]


class OpeningReference:
    """fri_ref's opening proof over the headline batch, with bench.py's instance and transcript (the cap, then every
    opening), and the decoy's openings and final polynomial.  The oracle holds no leaves: query rows are evaluated at
    7 w_N^brev(i) and paths come from the digests.  The decoy's coefficients are non-canonical: every 7th is
    presented as value + p (value < 2^31), and each polynomial starts with 2^64 - 1, p, p + 1."""

    def __init__(self, ref):
        self.batches = _opening_batches(ZETA, ref.w, ref.lg_d)
        self.openings = _openings(ref.coeffs, self.batches)
        och = fr.Challenger()
        och.observe_cap(ref.cap)
        for vals in self.openings:
            och.observe_extension_elements(vals)
        self.challenger = och.clone()
        lg_n, w_n = ref.lg_d + ref.r, fr.primitive_root_of_unity(ref.lg_d + ref.r)

        def rows(i):
            x = fr.COSET_SHIFT * pow(w_n, brev(i, lg_n), P) % P
            return fr.eval_base_polys_ext(ref.coeffs, (x, 0))[:, 0]

        entry = {"coeffs": ref.coeffs, "cap_height": ref.cap_h, "rows": rows,
                 "path": lambda i: oracle.merkle_prove(ref.digests, ref.n, ref.cap_h, i)}
        self.proof = fr.prove_openings([entry], self.batches, och, ref.r, ref.cap_h, FRI_ARITIES, POW_BITS, N_QUERIES)
        self.next_challenge = och.get_challenge()
        nc = ref.decoy.copy()
        flat = nc.reshape(-1)
        flat[3::7] = (flat[3::7] & np.uint64((1 << 31) - 1)) + np.uint64(P)
        nc[:, :3] = np.array([(1 << 64) - 1, P, P + 1], dtype=np.uint64)
        self.decoy_nc = nc
        canon = nc % np.uint64(P)
        self.decoy_batches = _opening_batches(DECOY_ZETA, ref.w, ref.lg_d)
        self.decoy_openings = _openings(canon, self.decoy_batches)
        self.decoy_final = fr.final_poly([canon], self.decoy_batches, DECOY_ALPHA)


@pytest.fixture(scope="module")
def headline_opening(headline):
    return OpeningReference(headline)


def _commit_batch(L, pcs, dev, ref, flags):
    """A PolynomialBatch over a commit of device coefficients with the coefficients kept, built as bench.py builds it."""
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.fri import _DeviceMerkleTree

    h = C.c_void_p()
    _ffi.check(L.pcs_commit_from_coeffs(_dev_ptrs(dev, 0, ref.w, ref.d), ref.w, ref.lg_d, ref.r, ref.cap_h, None, 0,
                                        _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS | flags, None, C.byref(h)))
    b = pcs.PolynomialBatch()
    b._h, b._coeffs_host = h, []
    b.degree_log, b.rate_bits, b.blinding, b.cap_height = ref.lg_d, ref.r, False, ref.cap_h
    b.n_polys, b.salt_w, b.n_leaves = ref.w, 0, ref.n
    b.n_digests = 2 * (ref.n - (1 << ref.cap_h))
    b._cap = np.empty((1 << ref.cap_h, 4), dtype=np.uint64)
    _ffi.check(L.pcs_batch_cap(h, _ffi.ptr(b._cap)))
    b.merkle_tree = _DeviceMerkleTree(b)
    return b


def _instance(batches, w):
    from plonky2_demo_b200.fri_prover import FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo

    return FriInstanceInfo([FriOracleInfo(w, False)],
                           [FriBatchInfo(pt, [FriPolynomialInfo(o, j) for o, j in polys]) for pt, polys in batches])


def _device_openings(b, batches):
    from plonky2_demo_b200.fri_prover import eval_commitment

    return [[tuple(int(x) for x in v) for v in eval_commitment(pt, b)[:len(polys)]] for pt, polys in batches]


@pytest.mark.parametrize("on_demand", [False, True], ids=["resident", "on_demand"])
def test_headline_opening_proof(L, headline, headline_opening, on_demand):
    """bench.py's opening proof, exact: 155 openings, the final polynomial (2^20 coefficients) and its LDE (2^23 values),
    and the proof field by field (4 commit-phase caps, final polynomial, PoW witness, 28 indices, initial rows and paths,
    every step's evals and path); both transcripts end in the same state and the restated verifier accepts.

    First a decoy: an on-demand batch over the decoy's non-canonical coefficients, whose openings and final polynomial are
    checked, and a proof over it with other challenges, freed in stream order; whatever the checked proof fails to write
    then holds the decoy's values, not the other arm's."""
    import plonky2_demo_b200 as pcs
    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.fri_prover import Challenger, final_poly, prove_openings

    ref, want = headline, headline_opening
    cfg = pcs.CircuitConfig.standard_recursion_config().fri_config
    cfg = pcs.FriConfig(ref.r, ref.cap_h, cfg.proof_of_work_bits, cfg.reduction_strategy, cfg.num_query_rounds)
    params = cfg.fri_params(ref.lg_d, False)
    assert (params.reduction_arity_bits, cfg.proof_of_work_bits, cfg.num_query_rounds) == (FRI_ARITIES, POW_BITS, N_QUERIES)

    dev_decoy = _to_device(want.decoy_nc)
    db = _commit_batch(L, pcs, dev_decoy, ref, _ffi.PCS_LDE_ON_DEMAND)
    del dev_decoy
    try:
        assert _device_openings(db, want.decoy_batches) == want.decoy_openings
        fin = final_poly(_instance(want.decoy_batches, ref.w), [db], DECOY_ALPHA)
        try:
            _assert_rows_equal(fin.coeffs, want.decoy_final, "decoy final polynomial")
        finally:
            fin.free()
        ch = Challenger()
        ch.observe_cap(db.merkle_tree.cap)
        prove_openings(_instance(want.decoy_batches, ref.w), [db], ch, params)
    finally:
        db.free()

    dev = _to_device(ref.coeffs)
    b = _commit_batch(L, pcs, dev, ref, _ffi.PCS_LDE_ON_DEMAND if on_demand else 0)
    del dev
    try:
        _assert_rows_equal(b.merkle_tree.cap.hashes, ref.cap, "cap")
        openings = _device_openings(b, want.batches)
        assert openings == want.openings
        inst = _instance(want.batches, ref.w)
        ch = Challenger()
        ch.observe_cap(b.merkle_tree.cap)
        for vals in openings:
            ch.observe_extension_elements(vals)
        got = prove_openings(inst, [b], ch, params)
        assert_same_proof(got, want.proof)
        assert ch.get_challenge() == want.next_challenge
        assert fr.verify_fri_proof(want.batches, openings, want.challenger.clone(), [ref.cap], as_oracle_proof(got), ref.r,
                                   ref.cap_h, FRI_ARITIES, POW_BITS, N_QUERIES, ref.lg_d)
        fin = final_poly(inst, [b], want.proof["_alpha"])
        try:
            _assert_rows_equal(fin.coeffs, want.proof["_final_poly_full"], "final polynomial")
            _assert_rows_equal(fin.lde_coset_fft(ref.r), want.proof["_lde_values"], "final polynomial LDE")
        finally:
            fin.free()
    finally:
        b.free()
