"""Shared test helpers: seeded inputs (SURVEY 8d generator), big-int field arithmetic and device buffers for the GPU tests."""
import ctypes as C

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


def noncanonical(rng, shape):
    """uniform u64 with a share of values in [p, 2^64) (the reference's loose representation)"""
    a = rng.integers(0, 1 << 64, size=shape, dtype=np.uint64, endpoint=False)
    hi = rng.random(shape) < 0.25
    a[hi] = np.uint64(P) + (a[hi] % np.uint64((1 << 64) - P))
    return a


class Ext:
    """a + b X in F[X] / (X^2 - 7), the reference's quadratic extension; % P is a no-op (values stay reduced)"""

    def __init__(self, a, b=0):
        self.a, self.b = int(a) % P, int(b) % P

    def _c(self, o):
        return o if isinstance(o, Ext) else Ext(o)

    def __add__(self, o):
        o = self._c(o)
        return Ext(self.a + o.a, self.b + o.b)

    __radd__ = __add__

    def __sub__(self, o):
        o = self._c(o)
        return Ext(self.a - o.a, self.b - o.b)

    def __rsub__(self, o):
        return self._c(o) - self

    def __mul__(self, o):
        o = self._c(o)
        return Ext(self.a * o.a + 7 * self.b * o.b, self.a * o.b + self.b * o.a)

    __rmul__ = __mul__

    def __mod__(self, _):
        return self

    def __eq__(self, o):
        o = self._c(o)
        return (self.a, self.b) == (o.a, o.b)

    def __repr__(self):
        return f"Ext({self.a}, {self.b})"

    def pow(self, e):
        r, x = Ext(1), self
        while e:
            if e & 1:
                r = r * x
            x = x * x
            e >>= 1
        return r

    def inv(self):
        ni = pow((self.a * self.a - 7 * self.b * self.b) % P, P - 2, P)
        return Ext(self.a * ni, (P - self.b) * ni)


def mem_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def torch_u64(a):
    """a u64 array as a device tensor of the same bits"""
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def dev_table(tensors):
    """a host table of the tensors' device pointers"""
    from plonky2_demo_b200 import _ffi

    return (_ffi.u64p * len(tensors))(*[C.cast(C.c_void_p(t.data_ptr()), _ffi.u64p) for t in tensors])


def free(*batches):
    """free the batches now: a failing test's traceback would otherwise keep them alive past pcs_shutdown"""
    for b in batches:
        b.free()
