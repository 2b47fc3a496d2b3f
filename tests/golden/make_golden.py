#!/usr/bin/env python3
"""Generate the golden fixtures and the generated constant headers.

Run in the BUILD container only (it reads /root/reference, which does not exist
on the GPU box):

    python tests/golden/make_golden.py

Outputs (all committed):
  tests/golden/poseidon_params.json   parameters scraped from the reference
      (ALL_ROUND_CONSTANTS  plonky2/src/hash/poseidon.rs:58-156,
       MDS circ/diag + FAST_PARTIAL_* tables plonky2/src/hash/poseidon_goldilocks.rs:24-215)
  tests/golden/reference_kats.json    every golden number the reference's own tests
      hold for the hot path:
       - Poseidon-12 permutation KATs      poseidon_goldilocks.rs:461-482
       - 256-entry bit-reversal table      plonky2/src/util/mod.rs:59-76
       - field constants                   field/src/goldilocks_field.rs:76-87,152
       - field-op input grid               field/src/prime_field_testing.rs:7-17,78-125 (rule, restated)
  oracle/poseidon_constants.h                         C arrays for the CPU oracle
  plonky2_demo_b200/csrc/poseidon_constants.cuh       __constant__ arrays for the CUDA kernels

Poseidon parameters are data, not code: they cannot be re-derived (round constants
come from a seeded RNG run, plonky2/src/bin/generate_constants.rs). The FAST_PARTIAL_*
tables CAN be re-derived from (ALL_ROUND_CONSTANTS, MDS); this script does so with
big-int Python and asserts equality with the scraped tables, which pins our
understanding of the fast form before any kernel uses it.
"""
import json
import os
import re
import sys

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

P = 0xFFFFFFFF00000001
W = 12
N_FULL_HALF = 4
N_PARTIAL = 22
N_ROUNDS = 30


def read(path):
    with open(os.path.join(REF, path)) as f:
        return f.read()


def strip_comments(src):
    return re.sub(r"//[^\n]*", "", src)


def scrape_array(src, name):
    """All integer literals in the initialiser of `const NAME ... = [ ... ];`."""
    m = re.search(r"const\s+" + name + r"\s*:[^=]*=\s*\[", src)
    assert m, name
    i = m.end()
    depth = 1
    j = i
    while depth:
        c = src[j]
        if c == "[":
            depth += 1
        elif c == "]":
            depth -= 1
        j += 1
    body = strip_comments(src[i : j - 1])
    return [int(x, 0) for x in re.findall(r"0x[0-9a-fA-F]+|\b\d+\b", body)]


def scrape():
    pos = read("plonky2/src/hash/poseidon.rs")
    gl = read("plonky2/src/hash/poseidon_goldilocks.rs")
    rc = scrape_array(pos, "ALL_ROUND_CONSTANTS")
    assert len(rc) == W * N_ROUNDS, len(rc)
    params = {
        "width": W,
        "half_n_full_rounds": N_FULL_HALF,
        "n_partial_rounds": N_PARTIAL,
        "all_round_constants": rc,
        "mds_circ": scrape_array(gl, "MDS_MATRIX_CIRC"),
        "mds_diag": scrape_array(gl, "MDS_MATRIX_DIAG"),
        "fast_partial_first_round_constant": scrape_array(gl, "FAST_PARTIAL_FIRST_ROUND_CONSTANT"),
        "fast_partial_round_constants": scrape_array(gl, "FAST_PARTIAL_ROUND_CONSTANTS"),
        "fast_partial_round_vs": scrape_array(gl, "FAST_PARTIAL_ROUND_VS"),
        "fast_partial_round_w_hats": scrape_array(gl, "FAST_PARTIAL_ROUND_W_HATS"),
        "fast_partial_round_initial_matrix": scrape_array(gl, "FAST_PARTIAL_ROUND_INITIAL_MATRIX"),
    }
    assert len(params["mds_circ"]) == 12 and len(params["mds_diag"]) == 12
    assert len(params["fast_partial_first_round_constant"]) == 12
    assert len(params["fast_partial_round_constants"]) == 22
    assert len(params["fast_partial_round_vs"]) == 22 * 11
    assert len(params["fast_partial_round_w_hats"]) == 22 * 11
    assert len(params["fast_partial_round_initial_matrix"]) == 11 * 11

    # KATs: poseidon_goldilocks.rs test_vectors
    t = gl[gl.index("fn test_vectors") : gl.index("check_test_vectors::<F>(test_vectors12)")]
    t = strip_comments(t)
    neg_one = P - 1
    t = t.replace("neg_one: u64", "").replace("neg_one", hex(neg_one))
    body = t[t.index("vec![") :]
    nums = [int(x, 0) for x in re.findall(r"0x[0-9a-fA-F]+|\b\d+\b", body)]
    assert len(nums) == 4 * 24, len(nums)
    kats = []
    for k in range(4):
        kats.append({"input": nums[24 * k : 24 * k + 12], "output": nums[24 * k + 12 : 24 * k + 24]})

    util = read("plonky2/src/util/mod.rs")
    u = util[util.index("let output256") :]
    u = u[: u.index("];")]
    br = [int(x, 16) for x in re.findall(r"0x[0-9a-fA-F]+", u)]
    assert len(br) == 256

    fld = read("field/src/goldilocks_field.rs")
    two_adicity = int(re.search(r"const TWO_ADICITY: usize = (\d+)", fld).group(1))
    gen = int(re.search(r"MULTIPLICATIVE_GROUP_GENERATOR: Self = Self\((\d+)\)", fld).group(1))
    p2gen = int(re.search(r"POWER_OF_TWO_GENERATOR: Self = Self\((\d+)\)", fld).group(1))
    order = int(re.search(r"const ORDER: u64 = (0x[0-9A-Fa-f]+)", fld).group(1), 16)
    assert order == P

    # prime_field_testing.rs:7-17 test_inputs(modulus): 0..9, 2^31+-10, 2^32+-10, 2^63+-10, p-10..p-1
    # restated as a rule; the grid itself is regenerated in tests.
    kat = {
        "poseidon12_kats": kats,
        "reverse_index_bits_256": br,
        "field": {
            "order": order,
            "two_adicity": two_adicity,
            "multiplicative_group_generator": gen,
            "power_of_two_generator": p2gen,
            "coset_shift": gen,
        },
        "field_grid_rule": "smalls 0..9 ; 2^k-10..2^k+10 for k in (31,32,63) clipped to < p ; p-10..p-1",
        "sources": {
            "poseidon12_kats": "plonky2/src/hash/poseidon_goldilocks.rs:449-485",
            "reverse_index_bits_256": "plonky2/src/util/mod.rs:59-76",
            "field": "field/src/goldilocks_field.rs:76-87,152",
            "field_grid_rule": "field/src/prime_field_testing.rs:7-17",
        },
    }
    return params, kat


# --------------------------------------------------------------------------------------
# Big-int restatement used ONLY to validate/derive tables at generation time.
# --------------------------------------------------------------------------------------
def mds_matrix(params):
    circ, diag = params["mds_circ"], params["mds_diag"]
    # out_r = sum_i s[(i+r)%12]*circ[i] + s[r]*diag[r]   (poseidon.rs:178-198)
    M = [[0] * W for _ in range(W)]
    for r in range(W):
        for i in range(W):
            M[r][(i + r) % W] = (M[r][(i + r) % W] + circ[i]) % P
        M[r][r] = (M[r][r] + diag[r]) % P
    return M


def mat_vec(M, v):
    return [sum(M[r][c] * v[c] for c in range(len(v))) % P for r in range(len(M))]


def mat_mul(A, B):
    n, m, k = len(A), len(B[0]), len(B)
    return [[sum(A[i][t] * B[t][j] for t in range(k)) % P for j in range(m)] for i in range(n)]


def mat_inv(A):
    n = len(A)
    M = [row[:] + [int(i == j) for j in range(n)] for i, row in enumerate(A)]
    for c in range(n):
        piv = next(r for r in range(c, n) if M[r][c] % P)
        M[c], M[piv] = M[piv], M[c]
        inv = pow(M[c][c], P - 2, P)
        M[c] = [x * inv % P for x in M[c]]
        for r in range(n):
            if r != c and M[r][c]:
                f = M[r][c]
                M[r] = [(x - f * y) % P for x, y in zip(M[r], M[c])]
    return [row[n:] for row in M]


def poseidon_naive(params, state):
    """poseidon.rs:613-633 poseidon_naive."""
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    s = [x % P for x in state]
    for r in range(N_ROUNDS):
        s = [(s[i] + rc[12 * r + i]) % P for i in range(W)]
        if r < N_FULL_HALF or r >= N_FULL_HALF + N_PARTIAL:
            s = [pow(x, 7, P) for x in s]
        else:
            s[0] = pow(s[0], 7, P)
        s = mat_vec(M, s)
    return s


def derive_fast_tables(params):
    """Re-derive FAST_PARTIAL_* from (round constants, MDS), following the construction in
    the Poseidon paper (appendix B, 'optimised partial rounds') in the row-vector convention
    the reference uses in mds_partial_layer_fast (poseidon.rs:401-431): the state is a ROW
    vector, new_state = state * A, A = [[M00, v],[w_hat, I]].
    Returns dict with the same keys/shape as the scraped tables."""
    M = mds_matrix(params)  # column convention: new = M * s
    rc = params["all_round_constants"]
    # MDS is symmetric?  Work in the column convention with M, then transpose where needed.
    # Partial round r (naive): s <- M * sbox0(s + c_r).
    # Step 1: push constants through: only the constant on lane 0 must be added before the
    # s-box; the rest can be moved after the linear layer of the previous round.
    Minv = mat_inv(M)
    first = N_FULL_HALF
    consts = [rc[12 * (first + r) : 12 * (first + r) + 12] for r in range(N_PARTIAL)]
    # Work backwards: c'_{last} = c_last ; for r = last-1..0 : move the non-lane-0 part of
    # c'_{r+1} through M^{-1} into round r.
    acc = consts[N_PARTIAL - 1][:]
    fast_rc = [0] * N_PARTIAL
    for r in range(N_PARTIAL - 1, 0, -1):
        inv = mat_vec(Minv, acc)
        fast_rc[r] = inv[0]
        inv0 = inv[:]
        inv0[0] = 0
        acc = [(consts[r - 1][i] + inv0[i]) % P for i in range(W)]
    first_round_constant = acc
    # Step 2: factor M = M' * M'' repeatedly so that all but the first partial round use a sparse matrix.
    # Column convention here; the reference stores the transposed (row-vector) variant.
    Mt = [[M[c][r] for c in range(W)] for r in range(W)]  # transpose
    m_mul = [row[:] for row in Mt]
    vs, w_hats = [None] * N_PARTIAL, [None] * N_PARTIAL
    for r in range(N_PARTIAL - 1, -1, -1):
        m_hat = [row[1:] for row in m_mul[1:]]
        w = [m_mul[i][0] for i in range(1, W)]
        v = m_mul[0][1:]
        m_hat_inv = mat_inv(m_hat)
        w_hat = mat_vec(m_hat_inv, w)
        vs[r] = v
        w_hats[r] = w_hat
        m_prime = [[0] * W for _ in range(W)]
        m_prime[0][0] = 1
        for i in range(1, W):
            for j in range(1, W):
                m_prime[i][j] = m_hat[i - 1][j - 1]
        m_mul = mat_mul(Mt, m_prime)
    init = [row[1:] for row in m_prime[1:]]
    # shift the round constants by one: the reference stores the constant used AFTER s-box r,
    # i.e. fast_rc[r+1], and 0 for the last.
    fast_round_constants = fast_rc[1:] + [0]
    return {
        "fast_partial_first_round_constant": first_round_constant,
        "fast_partial_round_constants": fast_round_constants,
        "fast_partial_round_vs": [x for row in vs for x in row],
        "fast_partial_round_w_hats": [x for row in w_hats for x in row],
        "fast_partial_round_initial_matrix": [x for row in init for x in row],
    }


def poseidon_fast(params, state):
    """poseidon.rs:599-609 poseidon (fast partial rounds)."""
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    s = [x % P for x in state]
    r = 0
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    s = [(s[i] + params["fast_partial_first_round_constant"][i]) % P for i in range(W)]
    im = params["fast_partial_round_initial_matrix"]
    res = [0] * W
    res[0] = s[0]
    for rr in range(1, W):
        for c in range(1, W):
            res[c] = (res[c] + s[rr] * im[(rr - 1) * 11 + (c - 1)]) % P
    s = res
    for i in range(N_PARTIAL):
        s[0] = (pow(s[0], 7, P) + params["fast_partial_round_constants"][i]) % P
        wh = params["fast_partial_round_w_hats"][11 * i : 11 * i + 11]
        vv = params["fast_partial_round_vs"][11 * i : 11 * i + 11]
        d = (s[0] * (params["mds_circ"][0] + params["mds_diag"][0]) + sum(s[j] * wh[j - 1] for j in range(1, W))) % P
        s = [d] + [(s[j] + s[0] * vv[j - 1]) % P for j in range(1, W)]
    r += N_PARTIAL
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    return s


def derive_lazy_tables(params):
    """Tables for the GPU's 'lazy' partial rounds (see csrc/poseidon.cuh).

    In the fast form (poseidon.rs:584-596) lanes 1..11 only ever receive s0 * v_i:
        s_i^(k+1) = s_i^(k) + x_k * v_i^(k),   x_k = sbox(s_0^(k)) + rc_k
        s_0^(k+1) = M00 * x_k + sum_i what_i^(k) * s_i^(k)
    Unrolling, with t = state after mds_partial_layer_init:
        s_0^(k+1) = M00*x_k + sum_i what_i^(k) t_i + sum_{r<k} x_r * C[k][r],
        C[k][r]   = sum_i what_i^(k) * v_i^(r)
        s_i^(22)  = t_i + sum_r x_r v_i^(r)
    so every product has one operand that is a compile-time constant and sums can be
    accumulated unreduced. Returns C as a dense 22x22 lower-triangular list (row k, col r<k).
    """
    vs = params["fast_partial_round_vs"]
    wh = params["fast_partial_round_w_hats"]
    C = [[0] * N_PARTIAL for _ in range(N_PARTIAL)]
    for k in range(N_PARTIAL):
        for r in range(k):
            C[k][r] = sum(wh[11 * k + i] * vs[11 * r + i] for i in range(11)) % P
    return C


def poseidon_lazy(params, C, state):
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    s = [x % P for x in state]
    r = 0
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    s = [(s[i] + params["fast_partial_first_round_constant"][i]) % P for i in range(W)]
    im = params["fast_partial_round_initial_matrix"]
    t = [0] * W
    t[0] = s[0]
    for rr in range(1, W):
        for c in range(1, W):
            t[c] = (t[c] + s[rr] * im[(rr - 1) * 11 + (c - 1)]) % P
    m00 = params["mds_circ"][0] + params["mds_diag"][0]
    xs = []
    s0 = t[0]
    for k in range(N_PARTIAL):
        x = (pow(s0, 7, P) + params["fast_partial_round_constants"][k]) % P
        wh = params["fast_partial_round_w_hats"][11 * k : 11 * k + 11]
        s0 = (m00 * x + sum(wh[i - 1] * t[i] for i in range(1, W)) + sum(xs[q] * C[k][q] for q in range(k))) % P
        xs.append(x)
    out = [s0]
    for i in range(1, W):
        out.append((t[i] + sum(xs[q] * params["fast_partial_round_vs"][11 * q + i - 1] for q in range(N_PARTIAL))) % P)
    s = out
    r += N_PARTIAL
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    return s


def poseidon_dense_partial(params, state):
    """The form the GPU kernel uses (csrc/poseidon.cuh): full rounds as in the reference, partial
    rounds with the DENSE MDS but with the round constants pushed through the linear layer
    (first half of the fast-form derivation only): s += FIRST_RC ; 22 x { s0 = sbox(s0) + c_r ; s = M s }."""
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    s = [x % P for x in state]
    r = 0
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    s = [(s[i] + params["fast_partial_first_round_constant"][i]) % P for i in range(W)]
    for k in range(N_PARTIAL):
        s[0] = (pow(s[0], 7, P) + params["fast_partial_round_constants"][k]) % P
        s = mat_vec(M, s)
    r += N_PARTIAL
    for _ in range(4):
        s = [pow((s[i] + rc[12 * r + i]) % P, 7, P) for i in range(W)]
        s = mat_vec(M, s)
        r += 1
    return s


def round_addends(params):
    """Unified per-round additive constants (csrc/poseidon.cuh: full_round, and the exit of the partial rounds):
        s += RC[0]; for r in 0..29: { s-box (all lanes if full round else lane 0); s = M s + ADD[r] }
    ADD[r] is the constant the NEXT s-box layer needs, moved behind the linear layer:
      r = 0..2   : RC[r+1]
      r = 3      : FAST_PARTIAL_FIRST_ROUND_CONSTANT
      r = 4..25  : PARTIAL_RC[r-4] * M[:,0]   (the scalar added to lane 0 after the s-box, pushed through M)
                   (+ RC[26] for r = 25)
      r = 26..28 : RC[r+1]
      r = 29     : 0
    """
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    col0 = [M[r][0] for r in range(W)]
    add = []
    for r in range(N_ROUNDS):
        if r < 3:
            v = rc[12 * (r + 1) : 12 * (r + 2)]
        elif r == 3:
            v = params["fast_partial_first_round_constant"][:]
        elif r < 26:
            c = params["fast_partial_round_constants"][r - 4]
            v = [c * col0[i] % P for i in range(W)]
            if r == 25:
                v = [(v[i] + rc[12 * 26 + i]) % P for i in range(W)]
        elif r < 29:
            v = rc[12 * (r + 1) : 12 * (r + 2)]
        else:
            v = [0] * W
        add.append([x % P for x in v])
    return add


def poseidon_unified(params, add, state):
    rc = params["all_round_constants"]
    M = mds_matrix(params)
    s = [(state[i] + rc[i]) % P for i in range(W)]
    for r in range(N_ROUNDS):
        if r < 4 or r >= 26:
            s = [pow(x, 7, P) for x in s]
        else:
            s[0] = pow(s[0], 7, P)
        s = mat_vec(M, s)
        s = [(s[i] + add[r][i]) % P for i in range(W)]
    return s


def mds_network(circ, s):
    """Add/shift network for y_r = sum_i circ[i] * s[(r+i) % 12] on integers (csrc/poseidon.cuh:mds_half_fp64).
    x^12 - 1 = prod_{zeta^4=1} (x^3 - zeta): 4-point DFTs of the three stride-3 subsequences, one
    zeta-twisted 3x3 product per frequency, inverse DFTs.  The frequency-domain constants are
    derived here from `circ` (not copied): K = DFT4(c')(1)/4, N = DFT4(c')(-1)/4, Z = DFT4(c')(i)/2."""
    cp = [circ[(-m) % 12] for m in range(12)]  # correlation -> convolution kernel
    K, N, Z = [], [], []
    for b in range(3):
        x0, x1, x2, x3 = (cp[3 * k + b] for k in range(4))
        assert (x0 + x1 + x2 + x3) % 4 == 0 and (x0 - x1 + x2 - x3) % 4 == 0 and (x0 - x2) % 2 == 0 and (x1 - x3) % 2 == 0
        K.append((x0 + x1 + x2 + x3) // 4)
        N.append((x0 - x1 + x2 - x3) // 4)
        Z.append(complex((x0 - x2) // 2, (x1 - x3) // 2))
    assert K == [16, 32, 16] and N == [-1, -8, 2] and Z == [2 + 1j, -4 - 1j, 16 - 1j], (K, N, Z)
    A, B, Pq = [0] * 3, [0] * 3, [0] * 3
    for j in range(3):
        u, v = s[j] + s[j + 6], s[j + 3] + s[j + 9]
        A[j], B[j], Pq[j] = u + v, u - v, complex(s[j] - s[j + 6], s[j + 3] - s[j + 9])
    y = [0] * 12
    for j in range(3):
        ya = sum(A[a] * K[(j - a) % 3] for a in range(3))
        yb = sum((1 if a + b == j else -1) * B[a] * N[b] for a in range(3) for b in range(3) if (a + b) % 3 == j)
        yc = sum((1 if a + b == j else 1j) * Pq[a] * Z[b] for a in range(3) for b in range(3) if (a + b) % 3 == j)
        re, im = int(yc.real), int(yc.imag)
        y[j], y[j + 3], y[j + 6], y[j + 9] = ya + yb + re, ya - yb + im, ya + yb - re, ya - yb - im
    return y


def mds_network_check(params):
    import random

    rnd = random.Random(7)
    circ = params["mds_circ"]
    for _ in range(200):
        s = [rnd.randrange(1 << 32) for _ in range(12)]
        direct = [sum(circ[i] * s[(r + i) % 12] for i in range(12)) for r in range(12)]
        assert mds_network(circ, s) == direct


def c_array(name, vals, per_line=4, ctype="uint64_t", qual="static const"):
    out = [f"{qual} {ctype} {name}[{len(vals)}] = {{"]
    for i in range(0, len(vals), per_line):
        out.append("    " + " ".join(f"0x{v:016x}ULL," for v in vals[i : i + per_line]))
    out.append("};")
    return "\n".join(out)


def write_headers(params, add, root=ROOT):
    banner = (
        "// GENERATED by tests/golden/make_golden.py from tests/golden/poseidon_params.json -- do not edit.\n"
        "// Poseidon-12 / Goldilocks parameters (data, scraped from the reference:\n"
        "//   plonky2/src/hash/poseidon.rs:58-156, plonky2/src/hash/poseidon_goldilocks.rs:24-215).\n"
    )
    # --- oracle header (plain C) ---
    h = [banner, "#pragma once", "#include <stdint.h>", ""]
    h.append(c_array("ALL_ROUND_CONSTANTS", params["all_round_constants"]))
    h.append(c_array("MDS_MATRIX_CIRC", params["mds_circ"]))
    h.append(c_array("MDS_MATRIX_DIAG", params["mds_diag"]))
    h.append(c_array("FAST_PARTIAL_FIRST_ROUND_CONSTANT", params["fast_partial_first_round_constant"]))
    h.append(c_array("FAST_PARTIAL_ROUND_CONSTANTS", params["fast_partial_round_constants"]))
    h.append(c_array("FAST_PARTIAL_ROUND_VS", params["fast_partial_round_vs"]))
    h.append(c_array("FAST_PARTIAL_ROUND_W_HATS", params["fast_partial_round_w_hats"]))
    h.append(c_array("FAST_PARTIAL_ROUND_INITIAL_MATRIX", params["fast_partial_round_initial_matrix"]))
    with open(os.path.join(root, "oracle", "poseidon_constants.h"), "w") as f:
        f.write("\n".join(h) + "\n")

    # --- CUDA header ---
    q = "static __device__ __constant__"
    h = [banner, "#pragma once", "#include <stdint.h>", ""]
    h.append("namespace pcs { namespace pconst {")
    h.append(c_array("RC", params["all_round_constants"], qual=q))
    # the round addends (round_addends: constants moved behind the linear layer), split in 32-bit halves and
    # pre-biased as doubles 2^52 + half (bit pattern 0x43300000_hhhhhhhh): the FP64 MDS network adds them last,
    # which also converts its exact integer result back to "integer in the mantissa" form for free.
    biased = []
    for row in add:
        for x in row:
            biased.append((0x43300000 << 32) | (x & 0xFFFFFFFF))
            biased.append((0x43300000 << 32) | (x >> 32))
    h.append("// ROUND_ADD_D[24*r + 2*i + {0,1}] = bits of the double 2^52 + {low, high} 32-bit half of make_golden.round_addends[r][i]")
    h.append(c_array("ROUND_ADD_D", biased, qual=q))
    h.append(c_array("PARTIAL_RC", params["fast_partial_round_constants"], qual=q))
    h.append("}}  // namespace pcs::pconst")
    with open(os.path.join(root, "plonky2_demo_b200", "csrc", "poseidon_constants.cuh"), "w") as f:
        f.write("\n".join(h) + "\n")


def main():
    if not os.path.isdir(REF):
        sys.exit("needs /root/reference (build container only)")
    params, kat = scrape()

    # 1. the naive big-int restatement reproduces every reference KAT
    for kv in kat["poseidon12_kats"]:
        assert poseidon_naive(params, kv["input"]) == kv["output"], "naive KAT mismatch"
        assert poseidon_fast(params, kv["input"]) == kv["output"], "fast KAT mismatch"
    # 2. the FAST_* tables re-derive from (RC, MDS)
    derived = derive_fast_tables(params)
    for k, v in derived.items():
        assert v == params[k], f"derived table {k} differs from the reference's"
    # 2b. the forms the CUDA kernels use: dense partial rounds with pushed constants; MDS add network
    mds_network_check(params)
    for kv in kat["poseidon12_kats"]:
        assert poseidon_dense_partial(params, kv["input"]) == kv["output"], "dense-partial KAT mismatch"
    add = round_addends(params)
    for kv in kat["poseidon12_kats"]:
        assert poseidon_unified(params, add, kv["input"]) == kv["output"], "unified-loop KAT mismatch"
    # 3. lazy partial-round tables agree too
    C = derive_lazy_tables(params)
    import random

    rnd = random.Random(1)
    for kv in kat["poseidon12_kats"]:
        assert poseidon_lazy(params, C, kv["input"]) == kv["output"], "lazy KAT mismatch"
    extra = []
    for _ in range(16):
        x = [rnd.randrange(P) for _ in range(12)]
        y = poseidon_naive(params, x)
        assert poseidon_fast(params, x) == y and poseidon_lazy(params, C, x) == y
        extra.append({"input": x, "output": y})
    # non-reference vectors produced by the big-int restatement (itself pinned by the 4 KATs above)
    kat["poseidon12_extra_bigint"] = extra

    with open(os.path.join(HERE, "poseidon_params.json"), "w") as f:
        json.dump(params, f, indent=0)
    with open(os.path.join(HERE, "reference_kats.json"), "w") as f:
        json.dump(kat, f, indent=0)
    write_headers(params, add)
    print("golden fixtures + headers written; derived FAST_* tables match the reference")


if __name__ == "__main__":
    main()
