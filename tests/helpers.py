"""Shared test helpers: seeded inputs (SURVEY 8d generator) and big-int field arithmetic."""
import numpy as np

P = 0xFFFFFFFF00000001
MASK = (1 << 64) - 1


def splitmix64_stream(seed, n):
    """splitmix64(seed) stream with rejection < p => canonical uniform elements (vectorised)."""
    out = np.empty(0, dtype=np.uint64)
    state = np.uint64(seed)
    with np.errstate(over="ignore"):
        while out.size < n:
            m = n - out.size + 16
            idx = np.arange(1, m + 1, dtype=np.uint64)
            z = state + idx * np.uint64(0x9E3779B97F4A7C15)
            state = z[-1]
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
            out = np.concatenate([out, z[z < np.uint64(P)]])
    return out[:n]


def seeded_polys(w, d, base_seed=0x5EED0000):
    return np.stack([splitmix64_stream(base_seed + j, d) for j in range(w)])


def field_grid():
    """field/src/prime_field_testing.rs:7-17 test_inputs(p) (restated)."""
    vals = list(range(0, 10))
    for k in (31, 32, 63):
        vals += list(range((1 << k) - 10, (1 << k) + 11))
    vals += list(range(P - 10, P))
    return sorted(set(v for v in vals if v < P))


def brev(i, bits):
    return int(format(i, f"0{bits}b")[::-1], 2) if bits else 0


def canon(a):
    a = np.asarray(a, dtype=np.uint64)
    return np.where(a >= np.uint64(P), a - np.uint64(P), a)


def assert_same_proof(got, want):
    """A device FriProof against fri_ref.prove_openings' dict, field by field."""
    assert len(got.commit_phase_merkle_caps) == len(want["commit_phase_merkle_caps"])
    for c, wc in zip(got.commit_phase_merkle_caps, want["commit_phase_merkle_caps"]):
        assert np.array_equal(c.hashes, wc)
    assert np.array_equal(got.final_poly, want["final_poly"])
    assert got.pow_witness == want["pow_witness"]
    assert got.fri_query_indices == want["_indices"]
    assert len(got.query_round_proofs) == len(want["query_round_proofs"])
    for r, wr in zip(got.query_round_proofs, want["query_round_proofs"]):
        for (ev, mp), (wev, wmp) in zip(r.initial_trees_proof.evals_proofs, wr["initial_trees_proof"]):
            assert np.array_equal(ev, wev)
            assert np.array_equal(np.asarray(mp.siblings).reshape(-1, 4), wmp)
        assert len(r.steps) == len(wr["steps"])
        for s, ws in zip(r.steps, wr["steps"]):
            assert np.array_equal(s.evals, ws["evals"])
            assert np.array_equal(np.asarray(s.merkle_proof.siblings).reshape(-1, 4), ws["merkle_proof"])


def as_oracle_proof(proof):
    """A device FriProof in the dict form fri_ref.verify_fri_proof reads."""
    return {
        "commit_phase_merkle_caps": [c.hashes for c in proof.commit_phase_merkle_caps],
        "final_poly": proof.final_poly,
        "pow_witness": proof.pow_witness,
        "query_round_proofs": [
            {"initial_trees_proof": [(ev, np.asarray(mp.siblings).reshape(-1, 4)) for ev, mp in r.initial_trees_proof.evals_proofs],
             "steps": [{"evals": s.evals, "merkle_proof": np.asarray(s.merkle_proof.siblings).reshape(-1, 4)} for s in r.steps]}
            for r in proof.query_round_proofs
        ],
    }
