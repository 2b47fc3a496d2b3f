"""GPU parity tests (-m gpu): every CUDA path is called through the C ABI (libpcs.so via the
plonky2_demo_b200 host mirror) and compared bit-exactly with the CPU oracle and with the
reference's golden vectors.  Integer work => the bar is exact equality."""
import numpy as np
import pytest

import oracle
from helpers import P, field_grid, seeded_polys, splitmix64_stream

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcs():
    import plonky2_demo_b200 as p

    p.init(0)
    yield p
    p.shutdown()


def test_extension_loaded(pcs):
    import ctypes

    assert isinstance(pcs.lib(), ctypes.CDLL)
    assert pcs.stream() is not None


# ---------------------------------------------------------------------------------------------
# Poseidon (reference KATs: poseidon_goldilocks.rs:461-482)
# ---------------------------------------------------------------------------------------------
def test_poseidon_reference_kats(pcs, golden):
    from plonky2_demo_b200.hashing import poseidon

    kats = golden["kats"]["poseidon12_kats"] + golden["kats"]["poseidon12_extra_bigint"]
    x = np.array([k["input"] for k in kats], dtype=np.uint64)
    y = np.array([k["output"] for k in kats], dtype=np.uint64)
    assert np.array_equal(poseidon(x), y)


def test_poseidon_random_and_edge_states(pcs):
    from plonky2_demo_b200.hashing import poseidon

    rng = np.random.default_rng(11)
    x = rng.integers(0, 1 << 64, size=(100_000, 12), dtype=np.uint64)  # includes non-canonical values
    g = np.array(field_grid(), dtype=np.uint64)
    edge = g[rng.integers(0, g.size, size=(20_000, 12))]
    nc = np.array([P, P + 1, (1 << 64) - 1, (1 << 64) - 2, 0xFFFFFFFF, 0xFFFFFFFF00000000], dtype=np.uint64)
    edge2 = nc[rng.integers(0, nc.size, size=(5_000, 12))]
    x = np.concatenate([x, edge, edge2])
    got = poseidon(x)
    assert np.array_equal(got, oracle.poseidon(x))
    assert (got < np.uint64(P)).all()


def test_poseidon_permutation_object(pcs, golden):
    perm = pcs.PoseidonPermutation(range(12))
    perm.permute()
    assert perm.state.tolist() == golden["kats"]["poseidon12_kats"][1]["output"]
    assert perm.squeeze().shape == (8,)


@pytest.mark.parametrize("ln", [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 32, 135, 139])
def test_hash_or_noop(pcs, ln):
    rng = np.random.default_rng(ln)
    rows = rng.integers(0, 1 << 64, size=(777, ln), dtype=np.uint64)
    assert np.array_equal(pcs.PoseidonHash.hash_or_noop_batch(rows), oracle.hash_or_noop(rows))


def test_hash_no_pad_short_inputs_are_hashed(pcs):
    for ln in [0, 1, 4]:
        x = np.arange(1, ln + 1, dtype=np.uint64)
        st = np.zeros(12, dtype=np.uint64)
        st[:ln] = x
        exp = oracle.poseidon(st)[0][:4] if ln else np.zeros(4, dtype=np.uint64)
        assert np.array_equal(pcs.PoseidonHash.hash_no_pad(x).elements, exp)


def test_two_to_one(pcs):
    rng = np.random.default_rng(3)
    l = rng.integers(0, 1 << 64, size=(3000, 4), dtype=np.uint64)
    r = rng.integers(0, 1 << 64, size=(3000, 4), dtype=np.uint64)
    assert np.array_equal(pcs.PoseidonHash.two_to_one_batch(l, r), oracle.two_to_one(l, r))


# ---------------------------------------------------------------------------------------------
# NTT / LDE (reference properties: fft.rs:219-253, polynomial/mod.rs:478-518)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_n", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24])
def test_ntt_forward_inverse(pcs, lg_n):
    # every pass-kernel instantiation (1..10 stages per pass) and the 1-, 2- and 3-pass plans (lg 23: [7, 8, 8], 24: [8, 8, 8])
    from plonky2_demo_b200.polynomial import ntt_batch

    w = 2 if lg_n > 16 else 3 if lg_n > 12 else 9
    rng = np.random.default_rng(lg_n)
    x = rng.integers(0, 1 << 64, size=(w, 1 << lg_n), dtype=np.uint64)  # non-canonical inputs allowed
    f = ntt_batch(x, inverse=False)
    assert np.array_equal(f, oracle.fft(x))
    i = ntt_batch(x, inverse=True)
    assert np.array_equal(i, oracle.fft(x, inverse=True))
    assert np.array_equal(ntt_batch(f, inverse=True), x % np.uint64(P))


def test_fft_is_naive_evaluation(pcs):
    # fft.rs:219-243 fft_and_ifft: degree 200 -> 256 points
    import random

    rnd = random.Random(3)
    coeffs = np.array([rnd.randrange(P) for _ in range(200)] + [0] * 56, dtype=np.uint64)
    vals = pcs.PolynomialCoeffs(coeffs).fft().values
    w = oracle.primitive_root_of_unity(8)
    assert vals.tolist() == [oracle.poly_eval(coeffs, pow(w, i, P)) for i in range(256)]
    assert np.array_equal(pcs.PolynomialValues(vals).ifft().coeffs, coeffs)
    # zero_factor equivalence (fft.rs:245-252)
    for r in range(4):
        padded = pcs.PolynomialCoeffs(coeffs).lde(r)
        a = pcs.fft_with_options(padded, None, None).values
        b = pcs.fft_with_options(padded, r, None).values
        assert np.array_equal(a, b)
        assert np.array_equal(a, oracle.fft(padded.coeffs[None, :])[0])


def test_coset_fft_and_lde_onto_coset(pcs):
    # polynomial/mod.rs:478-497
    c = splitmix64_stream(5, 64)
    shift = 7
    got = pcs.PolynomialCoeffs(c).coset_fft(shift).values
    w = oracle.primitive_root_of_unity(6)
    assert got.tolist() == [oracle.poly_eval(c, shift * pow(w, i, P) % P) for i in range(64)]
    vals = oracle.fft(c[None, :])[0]
    lde = pcs.PolynomialValues(vals).lde_onto_coset(3).values
    assert np.array_equal(lde, oracle.coset_lde(c[None, :], 3)[0])
    lde1 = pcs.PolynomialValues(vals).lde(2).values
    assert np.array_equal(lde1, oracle.coset_lde(c[None, :], 2, shift=1)[0])


def test_coset_ifft_roundtrip_and_batch(pcs):
    # polynomial/mod.rs:499-518 test_coset_ifft: coset_ifft(coset_fft(p)) == p; quotient-poly shape 16 x 2^12, shift 7
    import ctypes as C

    from plonky2_demo_b200 import _ffi

    c = splitmix64_stream(9, 256)
    for shift in (7, 3, P - 1):
        vals = pcs.PolynomialCoeffs(c).coset_fft(shift)
        assert np.array_equal(pcs.PolynomialValues(vals.values).coset_ifft(shift).coeffs, c)
    coeffs = seeded_polys(16, 1 << 12, base_seed=44)
    vals = oracle.coset_lde(coeffs, 0)            # evaluations on 7*H, natural order
    got = vals.copy()
    _ffi.check(_ffi.lib().pcs_coset_intt(_ffi.ptr(got), 16, 12, 7))
    assert np.array_equal(got, coeffs)


@pytest.mark.parametrize("lg_d,rate_bits,w", [(0, 3, 5), (1, 0, 4), (2, 2, 3), (3, 3, 135), (4, 0, 33), (5, 1, 7), (6, 3, 129), (7, 2, 70), (8, 1, 65), (9, 3, 20), (10, 3, 9), (11, 2, 16), (12, 4, 3), (13, 3, 17), (14, 1, 9), (15, 3, 6), (17, 2, 3), (18, 0, 2)])
def test_coset_lde_layouts(pcs, lg_d, rate_bits, w):
    import ctypes as C

    from plonky2_demo_b200 import _ffi

    d, n = 1 << lg_d, 1 << (lg_d + rate_bits)
    polys = seeded_polys(w, d, base_seed=1000 * lg_d)
    ref = oracle.coset_lde(polys, rate_bits)
    rows = [polys[j] for j in range(w)]
    out = np.empty((w, n), dtype=np.uint64)
    _ffi.check(_ffi.lib().pcs_coset_lde(_ffi.ptr_array(rows), w, lg_d, rate_bits, 7, _ffi.ptr(out), 0))
    assert np.array_equal(out, ref)
    out1 = np.empty((n, w), dtype=np.uint64)
    _ffi.check(_ffi.lib().pcs_coset_lde(_ffi.ptr_array(rows), w, lg_d, rate_bits, 7, _ffi.ptr(out1), 1))
    assert np.array_equal(out1, oracle.transpose_bitrev(ref))


# ---------------------------------------------------------------------------------------------
# Merkle trees (merkle_tree.rs:239-281)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("log_n,leaf_len,cap_height", [(8, 7, 1), (8, 7, 8), (8, 7, 0), (6, 135, 4), (3, 3, 2), (0, 5, 0), (1, 9, 0), (12, 32, 4), (14, 135, 4), (10, 4, 3), (10, 5, 10)])
def test_merkle_tree_new(pcs, log_n, leaf_len, cap_height):
    n = 1 << log_n
    leaves = splitmix64_stream(99 + log_n, n * leaf_len).reshape(n, leaf_len)
    tree = pcs.MerkleTree.new(leaves, cap_height)
    digests, cap = oracle.merkle_build(leaves, cap_height)
    assert np.array_equal(tree.digests, digests)
    assert np.array_equal(tree.cap.hashes, cap)
    rng = np.random.default_rng(log_n)
    for i in set([0, n - 1] + rng.integers(0, n, size=8).tolist()):
        proof = tree.prove(i)
        assert np.array_equal(proof.siblings, oracle.merkle_prove(digests, n, cap_height, i))
        pcs.verify_merkle_proof_to_cap(tree.get(i), i, tree.cap, proof)
    if n > 1 and cap_height < log_n:
        bad = tree.prove(0)
        bad.siblings[0, 0] ^= np.uint64(1)
        with pytest.raises(ValueError):
            pcs.verify_merkle_proof_to_cap(tree.get(0), 0, tree.cap, bad)


def test_merkle_panics(pcs):
    leaves = splitmix64_stream(1, 8 * 5).reshape(8, 5)
    with pytest.raises(ValueError, match="cap_height=4 should be at most"):
        pcs.MerkleTree.new(leaves, 4)
    with pytest.raises(ValueError, match="Not a power of two"):
        pcs.MerkleTree.new(leaves[:6], 0)
    from plonky2_demo_b200 import _ffi

    dg = np.empty((16, 4), dtype=np.uint64)
    cp = np.empty((16, 4), dtype=np.uint64)
    assert _ffi.lib().pcs_merkle_build(_ffi.ptr(leaves), 8, 5, 4, _ffi.ptr(dg), _ffi.ptr(cp)) == -3
    assert b"cap_height=4" in _ffi.lib().pcs_last_error()
    assert _ffi.lib().pcs_merkle_build(_ffi.ptr(leaves), 6, 5, 0, _ffi.ptr(dg), _ffi.ptr(cp)) == -2


# ---------------------------------------------------------------------------------------------
# The fused hot path: PolynomialBatch::from_coeffs / from_values
# ---------------------------------------------------------------------------------------------
COMMIT_SHAPES = [
    # (w, lg_d, rate_bits, cap_height)
    (135, 3, 3, 4),    # m = 2 demo wires commit: degree 2^3, 16 subtrees of 4 leaves
    (84, 3, 3, 4),     # m = 2 constants/sigmas
    (20, 3, 3, 4),
    (16, 3, 3, 4),
    (1, 0, 0, 0),
    (3, 0, 3, 3),      # cap_height == log2(N): digests empty
    (2, 1, 1, 2),
    (4, 5, 3, 0),      # leaf_len == 4 -> hash_or_noop copies
    (5, 5, 2, 4),
    (9, 10, 3, 4),
    (8, 11, 3, 4),     # two passes
    (135, 12, 3, 4),
    (3, 14, 3, 4),
    (33, 13, 3, 4),    # host polynomials > 32 KB, 3 H2D chunks: pipelined copy / LDE path
]


@pytest.mark.parametrize("w,lg_d,rate_bits,cap_height", COMMIT_SHAPES)
def test_from_coeffs(pcs, w, lg_d, rate_bits, cap_height):
    d, n = 1 << lg_d, 1 << (lg_d + rate_bits)
    coeffs = seeded_polys(w, d)
    ref = oracle.commit_from_coeffs(coeffs, rate_bits, cap_height)
    timing = {}
    b = pcs.PolynomialBatch.from_coeffs([pcs.PolynomialCoeffs(c) for c in coeffs], rate_bits, False, cap_height, timing)
    assert set(timing) == {"FFT + blinding", "transpose LDEs", "build Merkle tree"}
    assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b.merkle_tree.digests, ref["digests"])
    assert np.array_equal(b.merkle_tree.leaves[:], ref["leaves"])
    assert (b.degree_log, b.rate_bits, b.blinding) == (lg_d, rate_bits, False)
    rng = np.random.default_rng(w)
    for i in set([0, n - 1] + rng.integers(0, n, size=4).tolist()):
        assert np.array_equal(b.merkle_tree.get(i), ref["leaves"][i])
        proof = b.merkle_tree.prove(i)
        assert np.array_equal(proof.siblings, oracle.merkle_prove(ref["digests"], n, cap_height, i))
        assert oracle.merkle_verify(ref["leaves"][i], i, ref["cap"], proof.siblings)
    # get_lde_values(index, step): natural-order LDE column (oracle.rs:128-133)
    lde = oracle.coset_lde(coeffs, rate_bits)
    step = 1 << rate_bits
    for idx in range(min(d, 4)):
        assert np.array_equal(b.get_lde_values(idx, step), lde[:, idx * step])
    # get_lde_values_packed(index_start, step): `width` consecutive points, one column per point (oracle.rs:137-159)
    width = min(d, 4)
    packed = b.get_lde_values_packed(0, step, width)
    assert np.array_equal(packed, lde[:, [i * step for i in range(width)]])
    b.free()


@pytest.mark.parametrize("w,lg_d,rate_bits,cap_height", [(135, 3, 3, 4), (7, 6, 3, 2), (20, 10, 3, 4), (5, 12, 2, 4), (1, 0, 2, 1), (40, 14, 3, 4)])
def test_from_values(pcs, w, lg_d, rate_bits, cap_height):
    d = 1 << lg_d
    rng = np.random.default_rng(lg_d)
    values = rng.integers(0, 1 << 64, size=(w, d), dtype=np.uint64)  # non-canonical allowed
    ref = oracle.commit_from_values(values, rate_bits, cap_height)
    timing = {}
    b = pcs.PolynomialBatch.from_values([pcs.PolynomialValues(v) for v in values], rate_bits, False, cap_height, timing)
    assert "IFFT" in timing
    assert np.array_equal(np.stack([p.coeffs for p in b.polynomials]), ref["coeffs"])
    assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b.merkle_tree.digests, ref["digests"])
    assert np.array_equal(b.merkle_tree.leaves[:], ref["leaves"])
    b.free()


def test_from_coeffs_blinding_salts(pcs):
    w, lg_d, r, cap = 6, 5, 3, 4
    n = 1 << (lg_d + r)
    coeffs = seeded_polys(w, 1 << lg_d)
    salts = splitmix64_stream(42, 4 * n).reshape(4, n)
    ref = oracle.commit_from_coeffs(coeffs, r, cap, salts=salts)
    b = pcs.PolynomialBatch.from_coeffs(coeffs, r, True, cap, salts=salts)
    assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b.merkle_tree.leaves[:], ref["leaves"])
    assert b.get_lde_values(3, 1).shape == (w,)  # salt columns are stripped
    # OsRng salts: only shape/consistency can be checked
    b2 = pcs.PolynomialBatch.from_coeffs(coeffs, r, True, cap)
    rows = b2.merkle_tree.leaves[:]
    assert rows.shape == (n, w + 4) and np.array_equal(rows[:, :w], ref["leaves"][:, :w])
    d2, c2 = oracle.merkle_build(rows, cap)
    assert np.array_equal(b2.merkle_tree.cap.hashes, c2) and np.array_equal(b2.merkle_tree.digests, d2)


def test_from_coeffs_error_behaviour(pcs):
    coeffs = seeded_polys(3, 8)
    with pytest.raises(ValueError, match="cap_height=7 should be at most"):
        pcs.PolynomialBatch.from_coeffs(coeffs, 3, False, 7)
    with pytest.raises(IndexError):
        pcs.PolynomialBatch.from_coeffs([], 3, False, 0)
    with pytest.raises(ValueError, match="Not a power of two"):
        pcs.PolynomialBatch.from_coeffs([np.zeros(6, dtype=np.uint64)], 3, False, 0)
    with pytest.raises(ValueError, match="same length"):
        pcs.PolynomialBatch.from_coeffs([np.zeros(8, dtype=np.uint64), np.zeros(4, dtype=np.uint64)], 3, False, 0)


def test_fri_commit_phase_tree_shapes(pcs):
    # fri/prover.rs:81-87: per folding layer, leaves of arity*D = 32 base elements, cap_height 4
    for log_n in (14, 10, 6):
        n = 1 << log_n
        leaves = splitmix64_stream(log_n, n * 32).reshape(n, 32)
        t = pcs.MerkleTree.new(leaves, 4)
        dg, cp = oracle.merkle_build(leaves, 4)
        assert np.array_equal(t.cap.hashes, cp) and np.array_equal(t.digests, dg)


def test_m64_demo_shape_sampled(pcs):
    """m = 64 demo commit shape (d = 2^15, N = 2^18, 135 wires): full cap/digest parity."""
    w, lg_d, r, cap = 135, 15, 3, 4
    coeffs = seeded_polys(w, 1 << lg_d)
    ref = oracle.commit_from_coeffs(coeffs, r, cap)
    b = pcs.PolynomialBatch.from_coeffs(coeffs, r, False, cap)
    assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b.merkle_tree.digests, ref["digests"])
    idx = np.random.default_rng(0).integers(0, 1 << 18, size=512)
    assert np.array_equal(b.get_rows(idx), ref["leaves"][idx])
    b.free()


@pytest.mark.parametrize("fill", ["zero", "p_minus_1", "u64_max", "non_canonical_mix"])
def test_from_coeffs_adversarial_values(pcs, fill):
    """SURVEY 8d edge distributions: all-zero, all p-1, non-canonical inputs (>= p) -- outputs canonical, parity exact."""
    w, lg_d, r, cap = 9, 6, 3, 2
    d = 1 << lg_d
    if fill == "zero":
        coeffs = np.zeros((w, d), dtype=np.uint64)
    elif fill == "p_minus_1":
        coeffs = np.full((w, d), P - 1, dtype=np.uint64)
    elif fill == "u64_max":
        coeffs = np.full((w, d), (1 << 64) - 1, dtype=np.uint64)
    else:
        nc = np.array([P, P + 1, (1 << 64) - 1, (1 << 64) - 2, 0xFFFFFFFF, 0xFFFFFFFF00000000, 0, 1, P - 1], dtype=np.uint64)
        coeffs = nc[np.random.default_rng(5).integers(0, nc.size, size=(w, d))]
    ref = oracle.commit_from_coeffs(coeffs, r, cap)
    b = pcs.PolynomialBatch.from_coeffs(coeffs, r, False, cap)
    leaves = b.merkle_tree.leaves[:]
    assert (leaves < np.uint64(P)).all()
    assert np.array_equal(leaves, ref["leaves"])
    assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"])
    assert np.array_equal(b.merkle_tree.digests, ref["digests"])
    b2 = pcs.PolynomialBatch.from_values(coeffs, r, False, cap)
    ref2 = oracle.commit_from_values(coeffs, r, cap)
    assert np.array_equal(b2.merkle_tree.cap.hashes, ref2["cap"])
    assert np.array_equal(np.stack([p.coeffs for p in b2.polynomials]), ref2["coeffs"])


@pytest.mark.parametrize("bits,buffered", [(8, 3), (12, 0), (16, 7)])
def test_fri_proof_of_work(pcs, bits, buffered):
    """fri/prover.rs:115-160: the witness is the smallest candidate whose response has enough leading zeros."""
    rng = np.random.default_rng(bits)
    state = rng.integers(0, P, size=12, dtype=np.uint64)
    buf = rng.integers(0, P, size=buffered, dtype=np.uint64)
    cfg = pcs.FriConfig(3, 4, bits, pcs.FriReductionStrategy.ConstantArityBits(4, 5), 28)
    w = pcs.fri_proof_of_work(state, buf, cfg)
    st = state.copy()
    st[:buffered] = buf
    cand = np.arange(0, w + 1, dtype=np.uint64)
    states = np.tile(st, (cand.size, 1))
    states[:, buffered] = cand
    resp = oracle.poseidon(states)[:, 7]
    ok = resp < np.uint64(1 << (64 - bits))            # >= bits leading zeros
    assert ok[-1] and not ok[:-1].any(), "not the smallest valid witness"


def test_commit_random_shapes(pcs):
    """40 seeded random (w, degree, rate_bits, cap_height, blinding, from_values) shapes incl. non-canonical inputs:
    cap, digests and leaves equal the oracle's (SURVEY 8d edge grid: d in 2^0..2^11, W in 1..139, rate_bits 0..4)."""
    rng = np.random.default_rng(2024)
    for case in range(40):
        lg_d = int(rng.integers(0, 12))
        r = int(rng.integers(0, 5))
        w = int(rng.choice([1, 2, 3, 4, 5, 8, 9, 17, 33, 135, 139])) if lg_d <= 8 else int(rng.integers(1, 24))
        cap = int(rng.integers(0, lg_d + r + 1))
        blinding = bool(rng.integers(0, 2))
        from_values = bool(rng.integers(0, 2))
        d, n = 1 << lg_d, 1 << (lg_d + r)
        x = rng.integers(0, 1 << 64, size=(w, d), dtype=np.uint64)           # non-canonical values allowed
        salts = rng.integers(0, 1 << 64, size=(4, n), dtype=np.uint64) if blinding else None
        if from_values:
            ref = oracle.commit_from_values(x, r, cap, salts=salts)
            b = pcs.PolynomialBatch.from_values(x, r, blinding, cap, salts=salts)
        else:
            ref = oracle.commit_from_coeffs(x, r, cap, salts=salts)
            b = pcs.PolynomialBatch.from_coeffs(x, r, blinding, cap, salts=salts)
        tag = (case, w, lg_d, r, cap, blinding, from_values)
        assert np.array_equal(b.merkle_tree.cap.hashes, ref["cap"]), tag
        assert np.array_equal(b.merkle_tree.digests, ref["digests"]), tag
        assert np.array_equal(b.merkle_tree.leaves[:], ref["leaves"]), tag
        b.free()


def test_coset_lde_dev_is_the_leaf_order_lde(pcs):
    """pcs_coset_lde_dev (BASELINE configs[2]): device in, device out, leaf order; contiguous and scattered inputs."""
    import ctypes as C

    import torch

    from plonky2_demo_b200 import _ffi

    for w, lg_d, r in [(9, 11, 3), (135, 6, 3), (3, 14, 1), (4, 0, 2)]:
        d, n = 1 << lg_d, 1 << (lg_d + r)
        coeffs = seeded_polys(w, d, base_seed=7 * lg_d)
        ref = oracle.transpose_bitrev(oracle.coset_lde(coeffs, r)).T          # [w][N] in leaf order
        t = torch.from_numpy(coeffs.view(np.int64).copy()).cuda()
        out = torch.empty((w, n), dtype=torch.int64, device="cuda")
        _ffi.check(_ffi.lib().pcs_coset_lde_dev(_ffi.dev_ptr_array(t.data_ptr(), w, d), w, lg_d, r, 7, C.c_void_p(out.data_ptr())))
        pcs.synchronize()
        assert np.array_equal(out.cpu().numpy().view(np.uint64), ref)
        rows = [torch.from_numpy(coeffs[j].view(np.int64).copy()).cuda() for j in range(w)]
        ptrs = (_ffi.u64p * w)(*[C.cast(C.c_void_p(x.data_ptr()), _ffi.u64p) for x in rows])
        out.zero_()
        _ffi.check(_ffi.lib().pcs_coset_lde_dev(ptrs, w, lg_d, r, 7, C.c_void_p(out.data_ptr())))
        pcs.synchronize()
        assert np.array_equal(out.cpu().numpy().view(np.uint64), ref)


def test_bench_dump_outputs_hold_the_last_timed_commit(tmp_path):
    """bench.py --dump-outputs at a small shape: the files hold the commitment of the benchmark's seeded inputs bit for bit
    (cap, the sampled LDE rows and their Merkle paths, every element as float64 low / high 32-bit halves)."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    w, lg_d, r, cap_h = 9, 10, 3, 4
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "0", "--width", str(w),
                          "--lg-d", str(lg_d), "--rate-bits", str(r), "--cap-height", str(cap_h), "--no-fri", "--no-e2e",
                          "--no-from-values", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    files = {f: np.load(tmp_path / f"{f}.npy") for f in ("cap", "leaf_indices", "leaves", "merkle_paths")}
    assert all(a.dtype == np.float64 for a in files.values())
    assert sum(a.nbytes for a in files.values()) <= 64 << 20

    def join(a):
        assert np.all(a >= 0) and np.all(a < 2.0 ** 32) and np.all(a == np.floor(a))
        return a[..., 0].astype(np.uint64) | (a[..., 1].astype(np.uint64) << np.uint64(32))

    n = 1 << (lg_d + r)
    ref = oracle.commit_from_coeffs(seeded_polys(w, 1 << lg_d), r, cap_h)
    idx = files["leaf_indices"].astype(np.int64)
    assert idx.size == 4096 and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(join(files["cap"]), ref["cap"])
    assert np.array_equal(join(files["leaves"]), ref["leaves"][idx])
    paths = join(files["merkle_paths"])
    assert paths.shape == (idx.size, lg_d + r - cap_h, 4)
    for k in range(0, idx.size, 97):
        assert np.array_equal(paths[k], oracle.merkle_prove(ref["digests"], n, cap_h, int(idx[k])))
