"""CPU tests of the FRI oracle (oracle/fri.c + oracle/fri_ref.py): the restated arithmetic against Python big-int
algebra, the identities the reference's own tests check (division.rs test_division_by_linear, polynomial/mod.rs coset
FFT == evaluation), and the restated verifier (fri/verifier.rs) accepting the restated prover's proofs and rejecting
tampered ones.  No GPU."""
import random

import numpy as np
import pytest

import oracle
from oracle import fri_ref as fr
from helpers import P, seeded_polys, splitmix64_stream


def rand_ext(rng):
    return (rng.randrange(P), rng.randrange(P))


def test_extension_constants():
    # goldilocks_extensions.rs:19-27: W = 7 is a non-residue, EXT_POWER_OF_TWO_GENERATOR^2 is the base generator
    assert pow(7, (P - 1) // 2, P) == P - 1
    g = (0, 15659105665374529263)
    assert fr.ext_mul(g, g) == (1753635133440165772, 0)
    assert fr.c_ext_mul(g, g) == (1753635133440165772, 0)
    # DTH_ROOT = W^((p-1)/2)
    assert pow(7, (P - 1) // 2, P) == 18446744069414584320
    # EXT_MULTIPLICATIVE_GROUP_GENERATOR has full order p^2 - 1: not killed by any (p^2-1)/q for the small prime factors
    gen = (18081566051660590251, 16121475356294670766)
    order = P * P - 1
    for q in (2, 3, 5, 17, 257, 65537):
        assert order % q == 0
        e = order // q
        # exponent does not fit u64: big-int square and multiply
        acc, b = (1, 0), gen
        while e:
            if e & 1:
                acc = fr.ext_mul(acc, b)
            b = fr.ext_mul(b, b)
            e >>= 1
        assert acc != (1, 0)


def test_ext_arithmetic_vs_bigint():
    rng = random.Random(1)
    edge = [0, 1, 2, P - 1, P - 2, (1 << 32) - 1, 1 << 32, (1 << 63)]
    xs = [(a, b) for a in edge for b in edge[:4]] + [rand_ext(rng) for _ in range(200)]
    for x in xs[:60]:
        for y in xs[-40:]:
            assert fr.c_ext_mul(x, y) == fr.ext_mul(x, y)
    # non-canonical inputs (>= p) are accepted
    assert fr.c_ext_mul((P + 5, 2**64 - 1), (3, P)) == fr.ext_mul((5, (2**64 - 1) % P), (3, 0))
    for x in xs[-20:]:
        e = rng.randrange(1 << 40)
        assert fr.c_ext_pow(x, e) == fr.ext_pow(x, e)
        if x != (0, 0):
            assert fr.ext_mul(x, fr.ext_inv(x)) == (1, 0)


def test_eval_base_polys_ext():
    rng = random.Random(2)
    for w, d in [(1, 1), (3, 2), (5, 64), (2, 300 // 4 * 4)]:
        c = seeded_polys(w, d, 77)
        z = rand_ext(rng)
        got = fr.eval_base_polys_ext(c, z)
        for j in range(w):
            acc = (0, 0)
            for i in reversed(range(d)):
                acc = fr.ext_add(fr.ext_mul(acc, z), (int(c[j, i]), 0))
            assert (int(got[j, 0]), int(got[j, 1])) == acc
    # a base-field point agrees with the base-field Horner evaluation (oracle.poly_eval)
    c = seeded_polys(2, 128, 5)
    got = fr.eval_base_polys_ext(c, (12345, 0))
    for j in range(2):
        assert (int(got[j, 0]), int(got[j, 1])) == (oracle.poly_eval(c[j], 12345), 0)


def test_reduce_polys_base_and_scale_add():
    rng = random.Random(3)
    k, d = 7, 33
    c = seeded_polys(k, d, 9)
    alpha = rand_ext(rng)
    got = fr.reduce_polys_base(c, alpha)
    for i in range(d):
        acc = (0, 0)
        for j in range(k):
            pw = fr.ext_pow(alpha, j)
            acc = fr.ext_add(acc, (pw[0] * int(c[j, i]) % P, pw[1] * int(c[j, i]) % P))
        assert (int(got[i, 0]), int(got[i, 1])) == acc
    s = rand_ext(rng)
    q = splitmix64_stream(11, 2 * d).reshape(d, 2)
    out = fr.ext_scale_add(got, s, q)
    for i in range(d):
        e = fr.ext_add(fr.ext_mul((int(got[i, 0]), int(got[i, 1])), s), (int(q[i, 0]), int(q[i, 1])))
        assert (int(out[i, 0]), int(out[i, 1])) == e


def test_divide_by_linear_is_long_division():
    # division.rs test_division_by_linear: quotient * (X - z) + P(z) == P
    rng = random.Random(4)
    for n in (1, 2, 5, 64, 257):
        c = splitmix64_stream(100 + n, 2 * n).reshape(n, 2)
        z = rand_ext(rng)
        q = fr.ext_divide_by_linear(c, z)
        assert (int(q[n - 1, 0]), int(q[n - 1, 1])) == (0, 0)   # padded back with one zero
        pz = fr.ext_poly_eval(c, z)
        qq = [(int(a), int(b)) for a, b in q]
        # (X - z) * q + pz
        for i in range(n):
            lower = qq[i - 1] if i > 0 else (0, 0)
            term = fr.ext_sub(lower, fr.ext_mul(z, qq[i]))
            if i == 0:
                term = fr.ext_add(term, pz)
            assert term == (int(c[i, 0]), int(c[i, 1])), (n, i)


def test_ext_coset_lde_is_evaluation():
    # polynomial/mod.rs:478-497 test_coset_fft restated over the extension: values[i] = P(shift * w^i)
    rng = random.Random(5)
    for lg_d, rate_bits, shift in [(0, 0, 7), (0, 3, 7), (3, 0, 7), (3, 2, 7), (5, 1, 49), (4, 3, pow(7, 16, P))]:
        d = 1 << lg_d
        c = splitmix64_stream(lg_d * 10 + rate_bits, 2 * d).reshape(d, 2)
        vals = fr.ext_coset_lde(c, rate_bits, shift)
        n = d << rate_bits
        w = fr.primitive_root_of_unity(lg_d + rate_bits)
        for i in rng.sample(range(n), min(n, 12)):
            x = shift * pow(w, i, P) % P
            assert (int(vals[i, 0]), int(vals[i, 1])) == fr.ext_poly_eval(c, (x, 0))


def test_fold_matches_definition_and_verifier_interpolation():
    # P(x) = sum_{i<r} x^i P_i(x^r)  ->  folded(y) = sum_i beta^i P_i(y)   (prover.rs:92)
    rng = random.Random(6)
    arity_bits, n = 2, 32
    arity = 1 << arity_bits
    c = splitmix64_stream(21, 2 * n).reshape(n, 2)
    beta = rand_ext(rng)
    folded = fr.fri_fold(c, arity, beta)
    assert folded.shape == (n // arity, 2)
    for i in range(n // arity):
        acc = (0, 0)
        for j in range(arity):
            acc = fr.ext_add(acc, fr.ext_mul(fr.ext_pow(beta, j), (int(c[i * arity + j, 0]), int(c[i * arity + j, 1]))))
        assert (int(folded[i, 0]), int(folded[i, 1])) == acc
    # compute_evaluation (verifier.rs:20-46) recovers folded(x^arity) from the arity values on the coset of x
    lg_n = 5
    w = fr.primitive_root_of_unity(lg_n)
    for x_index in (0, 5, 31):
        x = 7 * pow(w, fr.reverse_bits(x_index, lg_n), P) % P
        coset_index, within = x_index >> arity_bits, x_index & (arity - 1)
        # the committed leaf: values in bit-reversed order, chunk `coset_index`
        evals = []
        for m in range(arity):
            pos = coset_index * arity + m
            xm = 7 * pow(w, fr.reverse_bits(pos, lg_n), P) % P
            evals.append(fr.ext_poly_eval(c, (xm, 0)))
        got = fr.compute_evaluation(x, within, arity_bits, evals, beta)
        assert got == fr.ext_poly_eval(folded, (pow(x, arity, P), 0))


def test_challenger_duplex_semantics():
    # challenger.rs: outputs are popped from the END of the squeezed rate portion; observing clears pending outputs
    ch = fr.Challenger()
    ch.observe_elements([1, 2, 3])
    st = np.zeros(12, dtype=np.uint64)
    st[:3] = [1, 2, 3]
    out = oracle.poseidon(st)[0]
    assert ch.get_challenge() == int(out[7])
    assert ch.get_challenge() == int(out[6])
    ch.observe_element(9)
    st2 = out.copy()
    st2[0] = 9
    out2 = oracle.poseidon(st2)[0]
    assert ch.get_challenge() == int(out2[7])
    # a full rate block triggers the permutation immediately
    ch2 = fr.Challenger()
    ch2.observe_elements(list(range(8)))
    assert ch2.input_buffer == [] and len(ch2.output_buffer) == 8


def make_instance(lg_d, rate_bits, cap_height, widths, seed=0):
    """Four-oracle shape of the reference's PLONK instance in miniature: every polynomial opened at zeta, the
    polynomials of oracle 2 also at g * zeta (circuit_data.rs:461-481)."""
    d = 1 << lg_d
    oracles = []
    for k, w in enumerate(widths):
        coeffs = seeded_polys(w, d, 0xABC000 + 97 * k + seed)
        o = oracle.commit_from_coeffs(coeffs, rate_bits, cap_height)
        o["coeffs"] = coeffs
        o["cap_height"] = cap_height
        oracles.append(o)
    rng = random.Random(1000 + seed)
    zeta = rand_ext(rng)
    g = fr.primitive_root_of_unity(lg_d)
    zeta_next = fr.ext_mul((g, 0), zeta)
    all_polys = [(k, j) for k, w in enumerate(widths) for j in range(w)]
    next_polys = [(len(widths) - 2, j) for j in range(min(2, widths[-2]))] if len(widths) >= 2 else []
    batches = [(zeta, all_polys)]
    if next_polys:
        batches.append((zeta_next, next_polys))
    return oracles, batches


def openings_of(oracles, batches):
    out = []
    for point, polys in batches:
        vals = []
        for o, j in polys:
            v = fr.eval_base_polys_ext(oracles[o]["coeffs"][j:j + 1], point)[0]
            vals.append((int(v[0]), int(v[1])))
        out.append(vals)
    return out


def seeded_challenger(oracles, openings):
    ch = fr.Challenger()
    for o in oracles:
        ch.observe_cap(o["cap"])
    for vals in openings:
        ch.observe_extension_elements(vals)
    return ch


@pytest.mark.parametrize("lg_d,rate_bits,cap_height,arities,widths", [
    (6, 3, 2, [2, 2], [3, 5, 4, 2]),
    (8, 1, 0, [4], [2, 1]),
    (5, 2, 1, [], [4]),
    (7, 3, 4, [4], [6, 9, 3, 2]),
])
def test_fri_prover_verifier_roundtrip(lg_d, rate_bits, cap_height, arities, widths):
    pow_bits, n_queries = 5, 6
    oracles, batches = make_instance(lg_d, rate_bits, cap_height, widths)
    openings = openings_of(oracles, batches)
    ch = seeded_challenger(oracles, openings)
    proof = fr.prove_openings(oracles, batches, ch.clone(), rate_bits, cap_height, arities, pow_bits, n_queries)
    assert np.asarray(proof["final_poly"]).shape[0] == (1 << lg_d) >> sum(arities)
    caps = [o["cap"] for o in oracles]
    args = (rate_bits, cap_height, arities, pow_bits, n_queries, lg_d)
    assert fr.verify_fri_proof(batches, openings, ch.clone(), caps, proof, *args)

    # the final polynomial has the claimed degree: its LDE coefficients beyond d are zero by construction, and the
    # quotient really is (F - F(z)) / (X - z): spot-check the identity on the LDE values
    fin = proof["_final_poly_full"]
    alpha = proof["_alpha"]
    w = fr.primitive_root_of_unity(lg_d + rate_bits)
    x = 7 * pow(w, 3, P) % P
    expect = (0, 0)
    for (point, polys), vals in zip(batches, openings):
        acc, red = (0, 0), (0, 0)
        for (o, j), v in zip(reversed(polys), reversed(vals)):
            acc = fr.ext_add(fr.ext_mul(acc, alpha), (oracle.poly_eval(oracles[o]["coeffs"][j], x), 0))
            red = fr.ext_add(fr.ext_mul(red, alpha), v)
        q = fr.ext_mul(fr.ext_sub(acc, red), fr.ext_inv(fr.ext_sub((x, 0), point)))
        expect = fr.ext_add(fr.ext_mul(expect, fr.ext_pow(alpha, len(polys))), q)
    assert fr.ext_poly_eval(fin, (x, 0)) == expect
    assert (int(proof["_lde_values"][3, 0]), int(proof["_lde_values"][3, 1])) == expect

    # tampering is rejected
    import copy
    bad = copy.deepcopy(proof)
    bad["final_poly"] = np.array(bad["final_poly"], copy=True)
    bad["final_poly"][0, 0] = (int(bad["final_poly"][0, 0]) + 1) % P
    with pytest.raises(AssertionError):
        fr.verify_fri_proof(batches, openings, ch.clone(), caps, bad, *args)
    bad = copy.deepcopy(proof)
    ev = bad["query_round_proofs"][0]["initial_trees_proof"][0][0]
    ev[0] = (int(ev[0]) + 1) % P
    with pytest.raises(AssertionError):
        fr.verify_fri_proof(batches, openings, ch.clone(), caps, bad, *args)
    bad_open = [list(v) for v in openings]
    bad_open[0][0] = ((bad_open[0][0][0] + 1) % P, bad_open[0][0][1])
    with pytest.raises(AssertionError):
        # a wrong opening changes the transcript AND the quotient check
        fr.verify_fri_proof(batches, bad_open, seeded_challenger(oracles, bad_open), caps, proof, *args)
    if arities:
        bad = copy.deepcopy(proof)
        st = bad["query_round_proofs"][1]["steps"][0]["evals"]
        st[1, 1] = (int(st[1, 1]) + 1) % P
        with pytest.raises(AssertionError):
            fr.verify_fri_proof(batches, openings, ch.clone(), caps, bad, *args)


def test_fri_roundtrip_random_shapes_and_more_tampering():
    """Ten seeded random shapes through the restated prover and verifier, then the tamper classes the parametrised test does
    not cover: proof-of-work witness, a commit-phase cap, a Merkle path, a proof transplanted onto another transcript."""
    import copy

    rng = random.Random(424242)
    for case in range(10):
        lg_d = rng.randrange(1, 8)
        rate_bits = rng.randrange(1, 4)
        widths = [rng.randrange(1, 6) for _ in range(rng.randrange(1, 4))]
        arities, left = [], lg_d
        while left > 0 and rng.random() < 0.7:
            a = rng.randrange(1, min(3, left) + 1)
            arities.append(a)
            left -= a
        min_leaves_log = min([lg_d + rate_bits] + [lg_d + rate_bits - sum(arities[: i + 1]) for i in range(len(arities))])
        cap_height = rng.randrange(0, min(min_leaves_log, 3) + 1)
        pow_bits, n_q = rng.randrange(0, 7), rng.randrange(1, 5)
        oracles, batches = make_instance(lg_d, rate_bits, cap_height, widths, seed=case)
        openings = openings_of(oracles, batches)
        ch = seeded_challenger(oracles, openings)
        proof = fr.prove_openings(oracles, batches, ch.clone(), rate_bits, cap_height, arities, pow_bits, n_q)
        caps = [o["cap"] for o in oracles]
        args = (rate_bits, cap_height, arities, pow_bits, n_q, lg_d)
        assert fr.verify_fri_proof(batches, openings, ch.clone(), caps, proof, *args), (case, lg_d, rate_bits, arities)
        if case % 3 == 0:
            # a different transcript (one more observed element) must not accept the same proof
            other = ch.clone()
            other.observe_element(1)
            with pytest.raises(AssertionError):
                fr.verify_fri_proof(batches, openings, other, caps, proof, *args)
            # wrong initial cap
            bad_caps = [c.copy() for c in caps]
            bad_caps[0][0, 0] = (int(bad_caps[0][0, 0]) + 1) % P
            with pytest.raises(AssertionError):
                fr.verify_fri_proof(batches, openings, ch.clone(), bad_caps, proof, *args)
            if cap_height < lg_d + rate_bits:
                bad = copy.deepcopy(proof)
                path = bad["query_round_proofs"][0]["initial_trees_proof"][0][1]
                path[0, 0] = (int(path[0, 0]) + 1) % P
                with pytest.raises(AssertionError):
                    fr.verify_fri_proof(batches, openings, ch.clone(), caps, bad, *args)
            if arities:
                bad = copy.deepcopy(proof)
                bad["commit_phase_merkle_caps"][0] = bad["commit_phase_merkle_caps"][0].copy()
                bad["commit_phase_merkle_caps"][0][0, 1] = (int(bad["commit_phase_merkle_caps"][0][0, 1]) + 1) % P
                with pytest.raises(AssertionError):
                    fr.verify_fri_proof(batches, openings, ch.clone(), caps, bad, *args)
    # proof of work: with 12 bits a random witness almost surely fails
    oracles, batches = make_instance(5, 2, 1, [3, 2], seed=99)
    openings = openings_of(oracles, batches)
    ch = seeded_challenger(oracles, openings)
    proof = fr.prove_openings(oracles, batches, ch.clone(), 2, 1, [2], 12, 3)
    args = (2, 1, [2], 12, 3, 5)
    assert fr.verify_fri_proof(batches, openings, ch.clone(), [o["cap"] for o in oracles], proof, *args)
    bad = dict(proof)
    bad["pow_witness"] = proof["pow_witness"] + 1
    with pytest.raises(AssertionError):
        fr.verify_fri_proof(batches, openings, ch.clone(), [o["cap"] for o in oracles], bad, *args)


def test_prove_openings_with_row_and_path_callables():
    """An oracle entry may give rows(i) / path(i) instead of leaves / digests (the benchmark-size tests hold no leaves):
    rows by direct evaluation at 7 w_N^brev(i), paths from the digests, give the same proof as the leaves."""
    lg_d, rate_bits, cap_height, arities, widths = 6, 3, 2, [2, 2], [3, 5, 4, 2]
    oracles, batches = make_instance(lg_d, rate_bits, cap_height, widths, seed=7)
    openings = openings_of(oracles, batches)
    ch = seeded_challenger(oracles, openings)
    want = fr.prove_openings(oracles, batches, ch.clone(), rate_bits, cap_height, arities, 4, 5)
    lg_n = lg_d + rate_bits
    w_n = fr.primitive_root_of_unity(lg_n)

    def lean(o):
        def rows(i):
            x = fr.COSET_SHIFT * pow(w_n, fr.reverse_bits(i, lg_n), P) % P
            return fr.eval_base_polys_ext(o["coeffs"], (x, 0))[:, 0]

        return {"coeffs": o["coeffs"], "cap_height": cap_height, "rows": rows,
                "path": lambda i: oracle.merkle_prove(o["digests"], 1 << lg_n, cap_height, i)}

    got = fr.prove_openings([lean(o) for o in oracles], batches, ch.clone(), rate_bits, cap_height, arities, 4, 5)
    assert got["_indices"] == want["_indices"]
    for r, wr in zip(got["query_round_proofs"], want["query_round_proofs"]):
        for (ev, mp), (wev, wmp) in zip(r["initial_trees_proof"], wr["initial_trees_proof"]):
            assert np.array_equal(ev, wev) and np.array_equal(mp, wmp)
