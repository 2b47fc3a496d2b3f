"""The gate-constraint CPU oracle (tests/harness/gate_oracle.c), no GPU needed:

- it equals a literal big-integer restatement of evaluate_gate_constraints_base_batch (compute_filter, the five gates'
  constraints, reduce_with_powers) on small shapes with non-canonical inputs, with one selector and with two or three groups, for
  one to five challenges, with each gate alone and all gates together;
- PoseidonGate's partial rounds in the reference's fast form (the oracle) and in the naive form (constant layer, S-box on lane 0,
  full MDS: the restatement here, and the device's form) give equal constraints for random states and random S-box wires;
- on a satisfied instance built from the gates' generators (Poseidon rows from the naive permutation, whose output is the
  permutation the KATs pin), committed through the oracle with the oracle's gate terms as the tail of quotient_oracle, the trim
  succeeds and the plonk verifier's identity vanishing(z) = Z_H(z) sum_k z^(k n) chunk_k(z) holds at random points with the gate
  constraints recomputed from the polynomials' values at z; one changed partial S-box wire, full-round wire or arithmetic
  output, swap = 2 or another public-inputs hash makes the trim fail.  This pins the gates' meaning to the permutation
  independently of any restatement.

The trim is checked at D = 7: the gates' filtered constraints have degree 8, so a satisfied instance's quotient has degree below
7 n, and the size-8n quotient domain (q = 3) leaves coefficients [7 n, 8 n) to check.  At D = 8 = 2^q there is nothing to trim,
and the identity is what fails."""
import json
import os
import sys
import zlib

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))

import gate_oracle as go  # noqa: E402
import permutation_oracle as po  # noqa: E402
import quotient_oracle as qo  # noqa: E402
from helpers import Ext, noncanonical  # noqa: E402
from test_quotient_oracle import vanishing_at  # noqa: E402

P = 0xFFFFFFFF00000001
GEN = 1753635133440165772
UNUSED_SELECTOR = (1 << 32) - 1
NOOP, CONSTANT, PUBLIC_INPUT, ARITHMETIC, POSEIDON = range(5)

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "poseidon_params.json")) as _f:
    PARAMS = json.load(_f)
RC = [int(v) for v in PARAMS["all_round_constants"]]
CIRC, DIAG = [int(v) for v in PARAMS["mds_circ"]], [int(v) for v in PARAMS["mds_diag"]]


def omega(lg):
    return pow(GEN, 1 << (32 - lg), P)


# ---- literal big-int restatement of the reference ------------------------------------------------------------------------
# Written with + - * and % P only, so that it evaluates base-field ints and Ext elements (the verifier's openings) alike.
def _el(v):
    return v if isinstance(v, Ext) else int(v) % P


def sbox(x):
    x2 = x * x % P
    return x2 * x2 % P * x2 % P * x % P


def mds(s):
    return [(sum(s[(i + r) % 12] * CIRC[i] for i in range(12)) + s[r] * DIAG[r]) % P for r in range(12)]


def poseidon_gate_naive(w):
    """PoseidonGate::eval_unfiltered with the partial rounds in the naive form -> 123 constraints"""
    w = [_el(v) for v in w]
    out = []
    swap = w[24]
    out.append(swap * (swap - 1) % P)
    for i in range(4):
        out.append((swap * (w[i + 4] - w[i]) - w[25 + i]) % P)
    s = [0] * 12
    for i in range(4):
        s[i] = (w[i] + w[25 + i]) % P
        s[i + 4] = (w[i + 4] - w[25 + i]) % P
    s[8:12] = w[8:12]
    for rnd in range(30):
        s = [(v + RC[12 * rnd + i]) % P for i, v in enumerate(s)]
        if rnd < 4 or rnd >= 26:
            if rnd != 0:
                w0 = 29 + 12 * (rnd - 1) if rnd < 4 else 87 + 12 * (rnd - 26)
                for i in range(12):
                    out.append((s[i] - w[w0 + i]) % P)
                    s[i] = w[w0 + i]
            s = [sbox(v) for v in s]
        else:
            out.append((s[0] - w[65 + rnd - 4]) % P)
            s[0] = sbox(w[65 + rnd - 4])
        s = mds(s)
    for i in range(12):
        out.append((s[i] - w[12 + i]) % P)
    assert len(out) == 123
    return out


def gate_constraints(kind, param, w, c, pih):
    """eval_unfiltered: w = local wires, c = local constants after the selector prefix"""
    w, c = [_el(v) for v in w], [_el(v) for v in c]
    if kind == NOOP:
        return []
    if kind == CONSTANT:
        return [(c[k] - w[k]) % P for k in range(param)]
    if kind == PUBLIC_INPUT:
        return [(w[k] - int(pih[k])) % P for k in range(4)]
    if kind == ARITHMETIC:
        c0, c1 = c[0], c[1]
        return [(w[4 * i + 3] - (w[4 * i] * w[4 * i + 1] * c0 + w[4 * i + 2] * c1)) % P for i in range(param)]
    return poseidon_gate_naive(w)


def compute_filter(row, group, s, many):
    f = 1
    for i in list(range(*group)) + ([UNUSED_SELECTOR] if many else []):
        if i != row:
            f = f * (i - s) % P
    return f


def gate_slots(gates, groups, local_wires, local_constants, pih):
    """evaluate_gate_constraints_base: the num_gate_constraints slots"""
    S = len(groups)
    slots = []
    for g, (kind, param, sel) in enumerate(gates):
        f = compute_filter(g, groups[sel], _el(local_constants[sel]), S > 1)
        for k, v in enumerate(gate_constraints(kind, param, local_wires, local_constants[S:], pih)):
            if k == len(slots):
                slots.append(0)
            slots[k] = (slots[k] + f * v) % P
    return slots


def reduce_with_powers(terms, alpha):
    acc = 0
    for t in reversed(terms):
        acc = (acc * alpha + t) % P
    return acc


def big_gate_terms(cs, wires, rate_bits, gates, groups, pih, alphas, D):
    N = cs.shape[1]
    n = N >> rate_bits
    q = (D - 1).bit_length()
    M, step = n << q, 1 << (rate_bits - q)
    out = np.empty((len(alphas), M), dtype=np.uint64)
    for i in range(M):
        m = i * step
        slots = gate_slots(gates, groups, wires[:, m], cs[:, m], pih)
        for a, al in enumerate(alphas):
            out[a, i] = reduce_with_powers(slots, int(al) % P)
    return out


# ---- oracle == restatement -----------------------------------------------------------------------------------------------
DEMO_GATES = [(NOOP, 0, 0), (CONSTANT, 2, 0), (PUBLIC_INPUT, 0, 0), (ARITHMETIC, 20, 0), (POSEIDON, 0, 1)]
DEMO_GROUPS = [(0, 4), (4, 5)]
GATE_SETS = {   # name -> (gates, groups, constants after the selectors)
    "demo": (DEMO_GATES, DEMO_GROUPS, 2),
    "one_selector": ([(NOOP, 0, 0), (ARITHMETIC, 3, 0), (CONSTANT, 2, 0)], [(0, 3)], 2),
    "three_groups": ([(PUBLIC_INPUT, 0, 0), (CONSTANT, 3, 1), (ARITHMETIC, 2, 1), (POSEIDON, 0, 2), (NOOP, 0, 2)],
                     [(0, 1), (1, 3), (3, 5)], 3),
    "noop": ([(NOOP, 0, 0)], [(0, 1)], 0),
    "constant": ([(CONSTANT, 3, 0)], [(0, 1)], 3),
    "public_input": ([(PUBLIC_INPUT, 0, 0)], [(0, 1)], 0),
    "arithmetic": ([(ARITHMETIC, 4, 0)], [(0, 1)], 2),
    "poseidon": ([(POSEIDON, 0, 0)], [(0, 1)], 0),
}
SHAPES = [   # (gate set, lg_n, C, D, rate_bits)
    ("demo", 2, 2, 8, 3),
    ("demo", 1, 5, 4, 3),
    ("one_selector", 2, 1, 8, 3),
    ("three_groups", 1, 3, 5, 3),
    ("noop", 2, 1, 2, 1),
    ("constant", 2, 4, 3, 2),
    ("public_input", 1, 2, 8, 3),
    ("arithmetic", 2, 3, 4, 3),
    ("poseidon", 1, 5, 8, 4),
]


@pytest.mark.parametrize("name,lg_n,C,D,rate_bits", SHAPES)
def test_oracle_equals_big_int_restatement(name, lg_n, C, D, rate_bits):
    gates, groups, nc_gate = GATE_SETS[name]
    rng = np.random.default_rng([zlib.crc32(name.encode()), lg_n, C, D])
    N = (1 << lg_n) << rate_bits
    S = len(groups)
    cs = noncanonical(rng, (S + nc_gate + 3, N))      # constants, then some sigma columns the gates do not read
    # selector columns holding gate indices and UNUSED_SELECTOR too, so that filters are zero, nonzero and mixed
    for s in range(S):
        picks = rng.integers(0, len(gates) + 1, N)
        cs[s] = np.where(picks < len(gates), picks, UNUSED_SELECTOR).astype(np.uint64)
        cs[s][rng.random(N) < 0.3] = noncanonical(rng, 1)[0]
    wires = noncanonical(rng, (135, N))
    pih, alphas = noncanonical(rng, 4), noncanonical(rng, C)
    got = go.gate_terms(cs, wires, rate_bits, gates, groups, S + nc_gate, pih, alphas, D)
    want = big_gate_terms(cs, wires, rate_bits, gates, groups, pih, alphas, D)
    assert got.shape == (C, (1 << lg_n) << (D - 1).bit_length())
    assert np.array_equal(got, want)


def test_fast_and_naive_partial_rounds_give_equal_constraints():
    """random states and random S-box wires: no witness relation at all"""
    rng = np.random.default_rng(11)
    for _ in range(40):
        w = noncanonical(rng, 135)
        if rng.random() < 0.5:
            w[24] = rng.integers(0, 2)   # a binary swap too
        assert [int(v) for v in go.poseidon_gate_constraints(w)] == poseidon_gate_naive(w)


# ---- a satisfied instance ------------------------------------------------------------------------------------------------
def poseidon_row(inputs, swap):
    """PoseidonGate's generator: the 135 wires of one row, from the naive permutation"""
    w = [0] * 135
    inp = [int(v) % P for v in inputs]
    w[:12] = inp
    w[24] = swap
    for i in range(4):
        w[25 + i] = swap * (inp[i + 4] - inp[i]) % P
    s = inp[:]
    if swap:
        s[0:4], s[4:8] = inp[4:8], inp[0:4]
    state_in = s[:]
    for rnd in range(30):
        s = [(v + RC[12 * rnd + i]) % P for i, v in enumerate(s)]
        if rnd < 4 or rnd >= 26:
            if rnd != 0:
                w0 = 29 + 12 * (rnd - 1) if rnd < 4 else 87 + 12 * (rnd - 26)
                w[w0:w0 + 12] = s
            s = [sbox(v) for v in s]
        else:
            w[65 + rnd - 4] = s[0]
            s[0] = sbox(s[0])
        s = mds(s)
    w[12:24] = s
    assert [int(v) for v in oracle.poseidon(np.array([state_in], dtype=np.uint64))[0]] == s
    return w


def satisfied_instance(rng, lg_n, R=80, tamper=None):
    """wires [135][n], constants [4][n] (2 selectors, 2 gate constants), the public-inputs hash; DEMO_GATES layout:
    row 0 PublicInputGate, row 1 ConstantGate, rows 2..3 ArithmeticGate, rows 4..5 PoseidonGate (swap 0, 1), the rest NoopGate"""
    n = 1 << lg_n
    wires = rng.integers(0, P, (135, n), dtype=np.uint64)
    consts = np.zeros((4, n), dtype=np.uint64)
    consts[0] = 0   # NoopGate's selector value (gate 0), unless a row below says otherwise
    consts[1] = UNUSED_SELECTOR
    pih = rng.integers(0, P, 4, dtype=np.uint64)
    wires[:4, 0] = pih
    consts[0, 0] = 2
    consts[0, 1] = 1
    consts[2:4, 1] = rng.integers(0, P, 2, dtype=np.uint64)
    wires[:2, 1] = consts[2:4, 1]
    for r in (2, 3):
        consts[0, r] = 3
        c0, c1 = (int(v) for v in rng.integers(0, P, 2, dtype=np.uint64))
        consts[2, r], consts[3, r] = c0, c1
        for i in range(20):
            a, b, d = (int(wires[4 * i + j, r]) for j in range(3))
            wires[4 * i + 3, r] = (a * b * c0 + d * c1) % P
    for r, swap in ((4, 0), (5, 1)):
        consts[0, r], consts[1, r] = UNUSED_SELECTOR, 4
        wires[:, r] = poseidon_row(rng.integers(0, P, 12, dtype=np.uint64), swap)
    if tamper == "partial_sbox":
        wires[65 + 7, 4] = (int(wires[65 + 7, 4]) + 1) % P
    elif tamper == "full_sbox":
        wires[87 + 12 * 2 + 5, 5] = (int(wires[87 + 12 * 2 + 5, 5]) + 1) % P
    elif tamper == "arithmetic_output":
        wires[4 * 9 + 3, 3] = (int(wires[4 * 9 + 3, 3]) + 1) % P
    elif tamper == "swap":   # swap = 2, with the deltas it implies
        wires[24, 4] = 2
        for i in range(4):
            wires[25 + i, 4] = 2 * (int(wires[i + 4, 4]) - int(wires[i, 4])) % P
    elif tamper == "public_inputs_hash":
        pih = pih.copy()
        pih[2] = (int(pih[2]) + 1) % P
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    x = [pow(omega(lg_n), i, P) for i in range(n)]
    sigmas = np.array([[int(k_is[j]) * x[i] % P for i in range(n)] for j in range(R)], dtype=np.uint64)   # the identity
    return dict(wires=wires, consts=consts, sigmas=sigmas, k_is=k_is, pih=pih, R=R)


def _commit(values, rate_bits):
    coeffs = oracle.fft(values, inverse=True)
    return coeffs, oracle.coset_lde(coeffs, rate_bits)


def _quotient(inst, D, rate_bits, alphas, betas, gammas):
    R, nc = inst["R"], 4
    n = inst["wires"].shape[1]
    cs_c, cs_lde = _commit(np.vstack([inst["consts"], inst["sigmas"]]), rate_bits)
    w_c, w_lde = _commit(inst["wires"], rate_bits)
    zs = po.prove_order(po.all_wires_permutation_partial_products(inst["wires"][:R], inst["sigmas"], inst["k_is"], betas, gammas,
                                                                  D))
    zs_c, zs_lde = _commit(zs, rate_bits)
    tail = go.gate_terms(cs_lde, w_lde, rate_bits, DEMO_GATES, DEMO_GROUPS, nc, inst["pih"], alphas, D)
    qp = qo.compute_quotient_polys(cs_lde, w_lde, zs_lde, rate_bits, nc, R, inst["k_is"], betas, gammas, alphas, D, tail)
    parts = dict(k_is=inst["k_is"], betas=betas, gammas=gammas, cs=(cs_c, cs_lde), w=(w_c, w_lde))
    return qo.quotient_poly_chunks(qp, n, D), parts, zs_c


def _challenges(rng, C=2):
    return (rng.integers(1, P, C, dtype=np.uint64) for _ in range(3))


def test_satisfied_instance_trims_and_meets_the_verifier_identity():
    rng = np.random.default_rng(2025)
    lg_n, rate_bits, C = 4, 3, 2
    n = 1 << lg_n
    inst = satisfied_instance(rng, lg_n)
    alphas, betas, gammas = _challenges(rng, C)
    _quotient(inst, 7, rate_bits, alphas, betas, gammas)   # the trim of coefficients [7 n, 8 n) succeeds
    chunks, parts, zs_c = _quotient(inst, 8, rate_bits, alphas, betas, gammas)
    R, K = inst["R"], -(-inst["R"] // 8)
    T = C * (K + 1)
    for z in (int(v) for v in rng.integers(2, P, 3, dtype=np.uint64)):
        van = vanishing_at(parts, zs_c, R, 4, 8, alphas, z)
        wz = [oracle.poly_eval(c, z) for c in parts["w"][0]]
        cz = [oracle.poly_eval(c, z) for c in parts["cs"][0][:4]]
        slots = gate_slots(DEMO_GATES, DEMO_GROUPS, wz, cz, inst["pih"])
        for a in range(C):
            al = int(alphas[a])
            v = (van[a] + pow(al, T, P) * reduce_with_powers(slots, al)) % P
            t = sum(pow(z, k * n, P) * oracle.poly_eval(chunks[a * 8 + k], z) for k in range(8)) % P
            assert v == (pow(z, n, P) - 1) * t % P, (a, z)


@pytest.mark.parametrize("tamper", ["partial_sbox", "full_sbox", "arithmetic_output", "swap", "public_inputs_hash"])
def test_a_broken_witness_fails_the_trim(tamper):
    rng = np.random.default_rng(2025)
    inst = satisfied_instance(rng, 4, tamper=tamper)
    alphas, betas, gammas = _challenges(rng)
    with pytest.raises(ValueError, match=qo.QUOTIENT_FAILED):
        _quotient(inst, 7, 3, alphas, betas, gammas)
