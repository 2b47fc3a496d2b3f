"""GPU parity tests (-m gpu) of the FRI opening proof on the device (SURVEY 8f N2 / N3): every entry point of the
"FRI opening proof" section of include/pcs.h is called through the C ABI (plonky2_demo_b200.fri_prover) and compared
bit-exactly with the CPU oracle (oracle/fri.c, oracle/fri_ref.py); whole proofs are compared field by field and
checked by the restated verifier (fri/verifier.rs)."""
import random

import numpy as np
import pytest

import oracle
from oracle import fri_ref as fr
from helpers import P, as_oracle_proof, assert_same_proof, seeded_polys, splitmix64_stream

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcs():
    import plonky2_demo_b200 as p

    p.init(0)
    yield p
    p.shutdown()


def rand_ext(rng):
    return (rng.randrange(P), rng.randrange(P))


def with_noncanonical(a, rng):
    """(canonical, non-canonical) views of the same field elements: a tenth of the entries are made small (< 2^31) and
    presented as value + p, which still fits a u64."""
    a = np.array(a, dtype=np.uint64, copy=True)
    mask = rng.random(a.shape) < 0.1
    a[mask] &= np.uint64((1 << 31) - 1)
    nc = a.copy()
    nc[mask] += np.uint64(P)
    return a, nc


# ---------------------------------------------------------------------------------------------
# eval_commitment (proof.rs:316-322)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,lg_d", [(1, 0), (3, 1), (5, 7), (4, 12), (7, 13), (135, 15), (2, 17),
                                    (3, 20), (1, 24)])   # 64 and 1024 chunks per polynomial (bench.py: 2^20; configs[4]: 2^24)
def test_eval_commitment(pcs, w, lg_d):
    from plonky2_demo_b200.fri_prover import eval_commitment

    rng = random.Random(w * 100 + lg_d)
    nrng = np.random.default_rng(w)
    c, nc = with_noncanonical(seeded_polys(w, 1 << lg_d, 0xE0A1), nrng)
    b = pcs.PolynomialBatch.from_coeffs(nc, 1, False, 0, keep_coeffs=True)
    for z in [rand_ext(rng), (rng.randrange(P), 0), (0, 0), (1, 0), (P - 1, P - 1), (P + 3, (1 << 64) - 1)]:
        got = eval_commitment(z, b)
        assert np.array_equal(got, fr.eval_base_polys_ext(c, z)), z
        assert (got < np.uint64(P)).all()
    b.free()


def test_eval_commitment_needs_coefficients(pcs):
    from plonky2_demo_b200.fri_prover import eval_commitment

    b = pcs.PolynomialBatch.from_coeffs(seeded_polys(2, 16), 1, False, 0)
    with pytest.raises(pcs.PcsError, match="PCS_KEEP_COEFFS"):
        eval_commitment((1, 2), b)
    b.free()
    # from_values keeps them (the reference's `polynomials`)
    v = seeded_polys(3, 64, 5)
    b = pcs.PolynomialBatch.from_values(v, 1, False, 0)
    co = oracle.fft(v, inverse=True)
    assert np.array_equal(eval_commitment((5, 9), b), fr.eval_base_polys_ext(co, (5, 9)))
    b.free()


# ---------------------------------------------------------------------------------------------
# extension polynomials: round trip, LDE, fold
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_d,rate_bits", [(0, 0), (0, 3), (1, 1), (5, 3), (10, 2), (11, 3), (15, 3), (16, 1),
                                            # the benchmark proof's final-poly LDE (plan [10, 10] at rate 3), then 2^24 outputs
                                            # at rate 1 and 0 (3-pass plans)
                                            (20, 3), (23, 1), (24, 0)])
def test_ext_poly_lde(pcs, lg_d, rate_bits):
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial

    d = 1 << lg_d
    c, nc = with_noncanonical(splitmix64_stream(0xF00 + lg_d, 2 * d).reshape(d, 2), np.random.default_rng(lg_d))
    p = ExtensionPolynomial.from_coeffs(nc)
    assert len(p) == d
    assert np.array_equal(p.coeffs, c)                       # canonical on the way out
    for shift in (7, pow(7, 16, P), P - 2):
        got = p.lde_coset_fft(rate_bits, shift)
        assert np.array_equal(got, fr.ext_coset_lde(c, rate_bits, shift)), (lg_d, rate_bits, shift)
    p.free()


@pytest.mark.parametrize("lg_d,arity_bits", [(4, 4), (4, 1), (8, 3), (12, 4), (15, 4), (13, 0),
                                             (16, 4), (20, 4), (24, 4)])   # outputs past 2^15: the benchmark's folds
def test_fri_fold(pcs, lg_d, arity_bits):
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial

    rng = random.Random(lg_d * 7 + arity_bits)
    d = 1 << lg_d
    c = splitmix64_stream(0xF01D + lg_d, 2 * d).reshape(d, 2)
    p = ExtensionPolynomial.from_coeffs(c)
    beta = rand_ext(rng)
    p.fold(arity_bits, beta)
    assert len(p) == d >> arity_bits
    assert np.array_equal(p.coeffs, fr.fri_fold(c, 1 << arity_bits, beta))
    # folding again keeps working on the shortened polynomial
    if (d >> arity_bits) >= 2:
        beta2 = (P + 1, (1 << 64) - 1)                      # non-canonical challenge
        p.fold(1, beta2)
        assert np.array_equal(p.coeffs, fr.fri_fold(fr.fri_fold(c, 1 << arity_bits, beta), 2, beta2))
    p.free()


def test_fold_rejects_ragged_length(pcs):
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial

    p = ExtensionPolynomial.from_coeffs(np.zeros((4, 2), dtype=np.uint64))
    with pytest.raises(pcs.PcsError):
        p.fold(3, (1, 1))
    p.free()


# ---------------------------------------------------------------------------------------------
# commit-phase trees (prover.rs:81-87)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_d,rate_bits,arity_bits,cap_height,shift", [
    (4, 3, 4, 0, 7), (4, 3, 4, 3, 7), (6, 1, 2, 1, 49), (10, 3, 4, 4, 7), (12, 3, 4, 4, pow(7, 16, P)), (3, 2, 1, 4, 7),
    (15, 3, 4, 4, 7),
    (20, 3, 4, 4, 7), (16, 3, 4, 4, pow(7, 16, P)),    # the benchmark proof's first two trees: 2^19 and 2^15 leaves of 32
])
def test_fri_commit_layer(pcs, lg_d, rate_bits, arity_bits, cap_height, shift):
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial

    d = 1 << lg_d
    c = splitmix64_stream(0xC0DE + lg_d, 2 * d).reshape(d, 2)
    p = ExtensionPolynomial.from_coeffs(c)
    tree = p.commit_layer(rate_bits, shift, arity_bits, cap_height)
    vals = fr.ext_coset_lde(c, rate_bits, shift)
    n = vals.shape[0]
    idx = oracle.reverse_index_bits(np.arange(n, dtype=np.uint64)).astype(np.int64)
    leaves = vals[idx].reshape(n >> arity_bits, 2 << arity_bits)
    digests, cap = oracle.merkle_build(leaves, cap_height)
    assert np.array_equal(tree.merkle_tree.cap.hashes, cap)
    assert np.array_equal(tree.merkle_tree.digests.reshape(-1, 4), digests)
    rng = random.Random(lg_d)
    for i in {0, leaves.shape[0] - 1, rng.randrange(leaves.shape[0])}:
        assert np.array_equal(tree.merkle_tree.get(i), leaves[i])
        sib = tree.merkle_tree.prove(i).siblings
        assert np.array_equal(sib, oracle.merkle_prove(digests, leaves.shape[0], cap_height, i))
        assert oracle.merkle_verify(leaves[i], i, cap, sib)
    tree.free()
    p.free()


def test_fri_commit_layer_cap_too_high(pcs):
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial

    p = ExtensionPolynomial.from_coeffs(np.ones((4, 2), dtype=np.uint64))
    with pytest.raises(ValueError, match="cap_height=3 should be at most"):
        p.commit_layer(1, 7, 1, 3)       # 8 values / arity 2 = 4 leaves
    p.free()


# ---------------------------------------------------------------------------------------------
# prove_openings (oracle.rs:162-219): final polynomial, then whole proofs
# ---------------------------------------------------------------------------------------------
def build_instance(pcs, lg_d, rate_bits, cap_height, widths, seed=0, from_values=False):
    """The reference's four-oracle PLONK instance in miniature (circuit_data.rs:461-481): everything opened at zeta,
    a prefix of oracle [-2] also at g * zeta.  Returns GPU batches, the oracle-side commits and both instance forms."""
    from plonky2_demo_b200.fri_prover import FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo

    d = 1 << lg_d
    gpu, cpu = [], []
    for k, w in enumerate(widths):
        coeffs = seeded_polys(w, d, 0xABC000 + 97 * k + seed)
        if from_values and k == 1:
            values = oracle.fft(coeffs)
            gpu.append(pcs.PolynomialBatch.from_values(values, rate_bits, False, cap_height))
        else:
            gpu.append(pcs.PolynomialBatch.from_coeffs(coeffs, rate_bits, False, cap_height, keep_coeffs=True))
        o = oracle.commit_from_coeffs(coeffs, rate_bits, cap_height)
        o["coeffs"], o["cap_height"] = coeffs, cap_height
        cpu.append(o)
    rng = random.Random(1000 + seed)
    zeta = rand_ext(rng)
    g = fr.primitive_root_of_unity(lg_d)
    zeta_next = fr.ext_mul((g, 0), zeta)
    all_polys = [(k, j) for k, w in enumerate(widths) for j in range(w)]
    k2 = max(len(widths) - 2, 0)
    next_polys = [(k2, j) for j in range(min(2, widths[k2]))]
    batches = [(zeta, all_polys), (zeta_next, next_polys)]
    inst = FriInstanceInfo(
        oracles=[FriOracleInfo(w, False) for w in widths],
        batches=[FriBatchInfo(pt, [FriPolynomialInfo(o, j) for o, j in polys]) for pt, polys in batches],
    )
    return gpu, cpu, inst, batches


@pytest.mark.parametrize("lg_d,widths", [(0, [1]), (1, [2, 1]), (6, [3, 5, 4, 2]), (9, [70, 3]), (13, [5, 2, 3]),
                                         (15, [84, 135, 20, 16]),
                                         # more than 256 polynomials in one FRI batch: several carry-free runs per block,
                                         # odd and even numbers of 8-polynomial groups (mbarrier phase bookkeeping)
                                         (8, [257]), (9, [300, 3]), (8, [520, 9, 1]), (10, [248, 8]), (5, [1100])])
def test_fri_final_poly(pcs, lg_d, widths):
    from plonky2_demo_b200.fri_prover import final_poly

    gpu, cpu, inst, batches = build_instance(pcs, lg_d, 1, 0, widths, seed=lg_d)
    rng = random.Random(lg_d)
    for alpha in (rand_ext(rng), (P + 2, (1 << 64) - 1)):
        p = final_poly(inst, gpu, alpha)
        want = fr.final_poly([o["coeffs"] for o in cpu], batches, (alpha[0] % P, alpha[1] % P))
        assert np.array_equal(p.coeffs, want), (lg_d, widths)
        p.free()
    for b in gpu:
        b.free()


@pytest.mark.parametrize("lg_d", range(25))
def test_fri_final_poly_single_polynomial(pcs, lg_d):
    """One polynomial opened at two points, through pcs_fri_final_poly_dev on a torch tensor (no commit), for every degree
    up to configs[4]'s 2^24: every recursion depth of the divide_by_linear suffix scan (segments of 16), including a level
    of exactly 16 coefficients and levels of one or two segments.  Coefficients include 2^64 - 1, p and p + 1."""
    import ctypes as C

    import torch

    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial, _ext_arg, _poly_ptr_array

    d = 1 << lg_d
    c = splitmix64_stream(0xF1A1 + lg_d, d)
    edge = np.array([(1 << 64) - 1, P, P + 1], dtype=np.uint64)
    c[: min(3, d)] = edge[: min(3, d)]
    c[-min(3, d):] = edge[::-1][-min(3, d):]
    c[d // 2::5] = edge[np.arange(c[d // 2::5].size) % 3]
    rng = random.Random(lg_d)
    batches = [(rand_ext(rng), [(0, 0)]), (rand_ext(rng), [(0, 0)])]
    alpha = rand_ext(rng)
    want = fr.final_poly([(c % np.uint64(P))[None, :]], batches, alpha)
    t = torch.from_numpy(c.view(np.int64)).cuda()
    torch.cuda.synchronize()
    pts =np.array([pt for pt, _ in batches], dtype=np.uint64)
    h = C.c_void_p()
    _ffi.check(_ffi.lib().pcs_fri_final_poly_dev(_poly_ptr_array([t.data_ptr()] * 2), lg_d, 2, _ffi.ptr(pts),
                                                 (C.c_size_t * 2)(1, 1), _ext_arg(alpha), C.byref(h)))
    p = ExtensionPolynomial(h)
    try:
        got = p.coeffs
    finally:
        p.free()
    bad = np.flatnonzero((got != want).any(axis=1))
    assert bad.size == 0, f"{bad.size} of {d} coefficients differ, the first at {bad[:8].tolist()}"


def test_fri_final_poly_errors(pcs):
    from plonky2_demo_b200.fri_prover import FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo, final_poly

    a = pcs.PolynomialBatch.from_coeffs(seeded_polys(2, 16), 1, False, 0, keep_coeffs=True)
    b = pcs.PolynomialBatch.from_coeffs(seeded_polys(2, 32), 1, False, 0, keep_coeffs=True)
    nokeep = pcs.PolynomialBatch.from_coeffs(seeded_polys(2, 16), 1, False, 0)
    info = [FriOracleInfo(2, False)]
    with pytest.raises(pcs.PcsError, match="different degrees"):
        final_poly(FriInstanceInfo(info * 2, [FriBatchInfo((1, 1), [FriPolynomialInfo(0, 0)])]), [a, b], (3, 4))
    with pytest.raises(pcs.PcsError, match="PCS_KEEP_COEFFS"):
        final_poly(FriInstanceInfo(info, [FriBatchInfo((1, 1), [FriPolynomialInfo(0, 0)])]), [nokeep], (3, 4))
    with pytest.raises(pcs.PcsError, match="out of bounds"):
        final_poly(FriInstanceInfo(info, [FriBatchInfo((1, 1), [FriPolynomialInfo(0, 2)])]), [a], (3, 4))
    with pytest.raises(pcs.PcsError, match="out of bounds"):
        final_poly(FriInstanceInfo(info, [FriBatchInfo((1, 1), [FriPolynomialInfo(1, 0)])]), [a], (3, 4))
    with pytest.raises(pcs.PcsError, match="empty"):
        final_poly(FriInstanceInfo(info, [FriBatchInfo((1, 1), [])]), [a], (3, 4))
    for x in (a, b, nokeep):
        x.free()


@pytest.mark.parametrize("lg_d,rate_bits,cap_height,arities,widths,pow_bits,n_queries,from_values", [
    (6, 3, 2, [2, 2], [3, 5, 4, 2], 5, 6, False),
    (8, 1, 0, [4], [2, 1], 8, 4, True),
    (5, 2, 1, [], [4], 3, 3, False),
    (7, 3, 4, [4], [6, 9, 3, 2], 10, 5, True),
    (3, 3, 4, [], [2, 3, 2, 2], 4, 4, False),                     # the m = 2 demo's degree (SURVEY 8a)
])
def test_prove_openings_matches_oracle_and_verifies(pcs, lg_d, rate_bits, cap_height, arities, widths, pow_bits,
                                                    n_queries, from_values):
    from plonky2_demo_b200.fri_prover import Challenger, eval_commitment, prove_openings

    gpu, cpu, inst, batches = build_instance(pcs, lg_d, rate_bits, cap_height, widths, from_values=from_values)
    # OpeningSet::new on the device, FriOpenings order = the batches' polynomial order
    per_oracle = {pt: [eval_commitment(pt, b) for b in gpu] for pt, _ in batches}
    openings = [[tuple(int(x) for x in per_oracle[pt][o][j]) for o, j in polys] for pt, polys in batches]
    for (pt, polys), vals in zip(batches, openings):
        for (o, j), v in zip(polys, vals):
            assert v == tuple(int(x) for x in fr.eval_base_polys_ext(cpu[o]["coeffs"][j:j + 1], pt)[0])

    ch, och = Challenger(), fr.Challenger()
    for c in (ch, och):
        for o in cpu:
            c.observe_cap(o["cap"])
        for vals in openings:
            c.observe_extension_elements(vals)
    cfg = pcs.FriConfig(rate_bits, cap_height, pow_bits, pcs.FriReductionStrategy.Fixed(arities), n_queries)
    params = cfg.fri_params(lg_d, False)
    verifier_ch = och.clone()
    got = prove_openings(inst, gpu, ch, params)
    want = fr.prove_openings(cpu, batches, och, rate_bits, cap_height, arities, pow_bits, n_queries)
    assert_same_proof(got, want)
    # both transcripts end in the same state
    assert ch.get_challenge() == och.get_challenge()
    # and the restated verifier accepts the GPU proof
    assert fr.verify_fri_proof(batches, openings, verifier_ch, [o["cap"] for o in cpu], as_oracle_proof(got), rate_bits,
                               cap_height, arities, pow_bits, n_queries, lg_d)
    for b in gpu:
        b.free()


def test_prove_openings_m64_demo_shape(pcs):
    """The m = 64 demo's opening proof in shape (SURVEY 8a): degree 2^15, oracles of 84 / 135 / 20 / 16 polynomials,
    standard_recursion_config (rate 3, cap 4, arity 16 x 3, 28 queries; 16 PoW bits).  The GPU proof is checked by the
    restated verifier and its commit-phase caps / final polynomial against the oracle's prover."""
    from plonky2_demo_b200.fri_prover import Challenger, eval_commitment, prove_openings

    lg_d, widths = 15, [84, 135, 20, 16]
    cfg = pcs.CircuitConfig.standard_recursion_config().fri_config
    params = cfg.fri_params(lg_d, False)
    assert params.reduction_arity_bits == [4, 4, 4]
    gpu, cpu, inst, batches = build_instance(pcs, lg_d, cfg.rate_bits, cfg.cap_height, widths, seed=64)
    per_oracle = {pt: [eval_commitment(pt, b) for b in gpu] for pt, _ in batches}
    openings = [[tuple(int(x) for x in per_oracle[pt][o][j]) for o, j in polys] for pt, polys in batches]
    ch = Challenger()
    for o, b in zip(cpu, gpu):
        assert np.array_equal(b.merkle_tree.cap.hashes, o["cap"])
        ch.observe_cap(b.merkle_tree.cap)
    for vals in openings:
        ch.observe_extension_elements(vals)
    och = fr.Challenger()
    och.sponge_state = [int(x) for x in ch.sponge_state.state]
    och.input_buffer, och.output_buffer = list(ch.input_buffer), list(ch.output_buffer)
    verifier_ch = och.clone()
    got = prove_openings(inst, gpu, ch, params)
    want = fr.prove_openings(cpu, batches, och, cfg.rate_bits, cfg.cap_height, params.reduction_arity_bits,
                             cfg.proof_of_work_bits, cfg.num_query_rounds)
    assert_same_proof(got, want)
    assert fr.verify_fri_proof(batches, openings, verifier_ch, [o["cap"] for o in cpu], as_oracle_proof(got),
                               cfg.rate_bits, cfg.cap_height, params.reduction_arity_bits, cfg.proof_of_work_bits,
                               cfg.num_query_rounds, lg_d)
    for b in gpu:
        b.free()


# ---------------------------------------------------------------------------------------------
# on-wire formats of device-resident data (util/serialization/mod.rs; SURVEY 8f N4)
# ---------------------------------------------------------------------------------------------
def test_serialize_device_batch_and_proof(pcs):
    from plonky2_demo_b200.fri_prover import Challenger, prove_openings
    from plonky2_demo_b200.serialization import Buffer, fri_proof_to_bytes, polynomial_batch_to_bytes

    lg_d, rate_bits, cap_height, widths = 6, 2, 2, [3, 4]
    gpu, cpu, inst, batches = build_instance(pcs, lg_d, rate_bits, cap_height, widths, seed=5, from_values=True)
    for b, o in zip(gpu, cpu):
        data = polynomial_batch_to_bytes(b)
        r = Buffer(data).read_polynomial_batch()
        assert np.array_equal(np.stack([p.coeffs for p in r.polynomials]), o["coeffs"])
        assert np.array_equal(r.merkle_tree.leaves, o["leaves"])
        assert np.array_equal(r.merkle_tree.digests, o["digests"])
        assert np.array_equal(r.merkle_tree.cap.hashes, o["cap"])
        assert (r.degree_log, r.rate_bits, r.blinding) == (lg_d, rate_bits, False)
        # polynomials (len + coeffs each), tree (leaves with lengths, digests with length, cap height, cap), 2 usize, 1 bool
        w, d, n = o["coeffs"].shape[0], 1 << lg_d, (1 << lg_d) << rate_bits
        assert len(data) == 8 + w * (d + 1) * 8 + 8 + n * (w + 1) * 8 + 8 + o["digests"].shape[0] * 32 + 8 + (32 << cap_height) + 17
    cfg = pcs.FriConfig(rate_bits, cap_height, 4, pcs.FriReductionStrategy.Fixed([2, 1]), 3)
    params = cfg.fri_params(lg_d, False)
    ch = Challenger()
    for o in cpu:
        ch.observe_cap(o["cap"])
    proof = prove_openings(inst, gpu, ch, params)
    data = fri_proof_to_bytes(proof)
    back = Buffer(data).read_fri_proof(widths, params.reduction_arity_bits, cap_height, 3, params.final_poly_len())
    assert fri_proof_to_bytes(back) == data
    assert back.pow_witness == proof.pow_witness and np.array_equal(back.final_poly, proof.final_poly)
    for b in gpu:
        b.free()


def test_opening_set_and_plonk_instance(pcs):
    """OpeningSet::new + get_fri_instance + prove_openings wired the way plonk/prover.rs:283-330 does it, on the m = 64
    demo's oracle widths at a small degree; the restated verifier accepts."""
    from plonky2_demo_b200.fri_prover import Challenger, OpeningSet, PlonkOpeningShape, prove_openings

    lg_d = 7
    shape = PlonkOpeningShape(degree_bits=lg_d, num_constants=4, num_routed_wires=80, num_wires=135, num_challenges=2,
                              num_partial_products=9, quotient_degree_factor=8)
    assert shape.oracle_widths() == [84, 135, 20, 16]
    cfg = pcs.CircuitConfig.standard_recursion_config().fri_config
    params = cfg.fri_params(lg_d, False)
    coeffs = [seeded_polys(w, 1 << lg_d, 0x0511 + k) for k, w in enumerate(shape.oracle_widths())]
    gpu = [pcs.PolynomialBatch.from_coeffs(c, cfg.rate_bits, False, cfg.cap_height, keep_coeffs=True) for c in coeffs]
    zeta = (0x1234567 % P, 0x7654321 % P)
    g = fr.primitive_root_of_unity(lg_d)
    os_ = OpeningSet.new(zeta, g, *gpu, shape)
    assert os_.constants.shape == (4, 2) and os_.plonk_sigmas.shape == (80, 2) and os_.plonk_zs_next.shape == (2, 2)
    assert os_.partial_products.shape == (18, 2) and os_.quotient_polys.shape == (16, 2)
    assert np.array_equal(os_.plonk_zs_next, fr.eval_base_polys_ext(coeffs[2][:2], fr.ext_mul((g, 0), zeta)))
    inst = shape.get_fri_instance(zeta)
    openings = os_.to_fri_openings()
    assert len(openings[0]) == 255 and len(openings[1]) == 2
    batches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    ch = Challenger()
    for b in gpu:
        ch.observe_cap(b.merkle_tree.cap)
    for vals in openings:
        ch.observe_extension_elements(vals)
    och = fr.Challenger()
    och.sponge_state = [int(x) for x in ch.sponge_state.state]
    och.input_buffer, och.output_buffer = list(ch.input_buffer), list(ch.output_buffer)
    proof = prove_openings(inst, gpu, ch, params)
    assert fr.verify_fri_proof(batches, openings, och, [b.merkle_tree.cap.hashes for b in gpu], as_oracle_proof(proof),
                               cfg.rate_bits, cfg.cap_height, params.reduction_arity_bits, cfg.proof_of_work_bits,
                               cfg.num_query_rounds, lg_d)
    for b in gpu:
        b.free()


def test_prove_openings_random_instances(pcs):
    """30 seeded random instances: oracle counts and widths, degree, rate, cap height, arities (any split that leaves a
    final polynomial), PoW bits, query counts, from_values / from_coeffs oracles.  GPU proof == oracle proof, verifier accepts."""
    from plonky2_demo_b200.fri_prover import Challenger, eval_commitment, prove_openings

    rng = random.Random(20261018)
    for case in range(30):
        lg_d = rng.randrange(0, 11)
        rate_bits = rng.randrange(0, 4) if lg_d else rng.randrange(1, 4)
        n_or = rng.randrange(1, 5)
        widths = [rng.randrange(1, 12) for _ in range(n_or)]
        arities, left = [], lg_d
        while left > 0 and rng.random() < 0.7:
            a = rng.randrange(1, min(4, left) + 1)
            arities.append(a)
            left -= a
        # every tree needs cap_height <= log2(leaves) = lg_d + rate_bits - (arity bits so far) - arity
        min_leaves_log = min([lg_d + rate_bits] + [lg_d + rate_bits - sum(arities[: i + 1]) for i in range(len(arities))])
        cap_height = rng.randrange(0, min(min_leaves_log, 4) + 1)
        pow_bits, n_q = rng.randrange(0, 9), rng.randrange(1, 6)
        gpu, cpu, inst, batches = build_instance(pcs, lg_d, rate_bits, cap_height, widths, seed=1000 + case,
                                                 from_values=bool(case & 1) and n_or > 1)
        per_oracle = {pt: [eval_commitment(pt, b) for b in gpu] for pt, _ in batches}
        openings = [[tuple(int(x) for x in per_oracle[pt][o][j]) for o, j in polys] for pt, polys in batches]
        ch, och = Challenger(), fr.Challenger()
        for c in (ch, och):
            for o in cpu:
                c.observe_cap(o["cap"])
            for vals in openings:
                c.observe_extension_elements(vals)
        vch = och.clone()
        cfg = pcs.FriConfig(rate_bits, cap_height, pow_bits, pcs.FriReductionStrategy.Fixed(arities), n_q)
        params = cfg.fri_params(lg_d, False)
        got = prove_openings(inst, gpu, ch, params)
        want = fr.prove_openings(cpu, batches, och, rate_bits, cap_height, arities, pow_bits, n_q)
        ctx = (case, lg_d, rate_bits, cap_height, arities, widths)
        try:
            assert_same_proof(got, want)
        except AssertionError as e:
            raise AssertionError(f"case {ctx}: {e}")
        assert fr.verify_fri_proof(batches, openings, vch, [o["cap"] for o in cpu], as_oracle_proof(got), rate_bits,
                                   cap_height, arities, pow_bits, n_q, lg_d), ctx
        for b in gpu:
            b.free()


def test_device_pointer_entry_points_alignment_and_errors(pcs):
    """pcs_eval_ext_dev / pcs_fri_final_poly_dev on scattered polynomials: 16-byte aligned rows take the TMA-staged kernels,
    rows at an odd multiple of 8 bytes must fall back to the register-staged ones (bulk copies need 16-byte alignment)."""
    import ctypes as C

    import torch

    from plonky2_demo_b200 import _ffi
    from plonky2_demo_b200.fri_prover import ExtensionPolynomial, _ext_arg, _poly_ptr_array

    L = _ffi.lib()
    w, lg_d = 5, 9
    d = 1 << lg_d
    c = seeded_polys(w, d, 0xA11C)
    z, alpha = (0x1234567, 0x7654321), (0xABCDEF, 0x13579B)
    want_eval = fr.eval_base_polys_ext(c, z)
    batches = [(z, [(0, j) for j in range(w)]), ((3, 4), [(0, 1), (0, 3)])]
    want_fin = fr.final_poly([c], batches, alpha)
    for offset in (0, 1):                                   # in u64 elements: 0 -> aligned, 1 -> base + 8 bytes
        buf = torch.zeros(w * (d + 2) + 2, dtype=torch.int64, device="cuda")
        addrs = []
        for j in range(w):
            start = j * (d + 2) + offset                    # rows 2 elements apart keep every row at the same parity
            buf[start:start + d] = torch.from_numpy(c[j].view(np.int64)).cuda()
            addrs.append(buf.data_ptr() + 8 * start)
        assert all((a % 16 == 0) == (offset == 0) for a in addrs)
        torch.cuda.synchronize()
        out = np.empty((w, 2), dtype=np.uint64)
        _ffi.check(L.pcs_eval_ext_dev(_poly_ptr_array(addrs), w, lg_d, _ext_arg(z), _ffi.ptr(out)))
        assert np.array_equal(out, want_eval), offset
        order = [addrs[j] for _, polys in batches for _, j in polys]
        pts = np.array([[pt[0], pt[1]] for pt, _ in batches], dtype=np.uint64)
        lens = (C.c_size_t * 2)(w, 2)
        h = C.c_void_p()
        _ffi.check(L.pcs_fri_final_poly_dev(_poly_ptr_array(order), lg_d, 2, _ffi.ptr(pts), lens, _ext_arg(alpha), C.byref(h)))
        p = ExtensionPolynomial(h)
        assert np.array_equal(p.coeffs, want_fin), offset
        p.free()
    # errors
    out = np.empty((w, 2), dtype=np.uint64)
    bad = _poly_ptr_array(addrs)
    bad[2] = None
    with pytest.raises(pcs.PcsError, match="NULL polynomial"):
        _ffi.check(L.pcs_eval_ext_dev(bad, w, lg_d, _ext_arg(z), _ffi.ptr(out)))
    h = C.c_void_p()
    with pytest.raises(pcs.PcsError, match="empty FRI batch"):
        _ffi.check(L.pcs_fri_final_poly_dev(_poly_ptr_array(order), lg_d, 2, _ffi.ptr(pts), (C.c_size_t * 2)(w, 0), _ext_arg(alpha), C.byref(h)))
    with pytest.raises(pcs.PcsError, match="TWO_ADICITY"):
        _ffi.check(L.pcs_eval_ext_dev(_poly_ptr_array(addrs), w, 33, _ext_arg(z), _ffi.ptr(out)))

