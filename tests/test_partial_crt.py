"""Exactness of Poseidon's transform-domain partial rounds (csrc/poseidon.cuh: crt_forward_d, crt_mid_half,
crt_scale_half, crt_lanes_half, lane0_crt, renorm_d, fold_signed_d).

The state of the 22 partial rounds is U = F(circ part of the state) per 32-bit half, 12 signed integers held in doubles.
The mirrors below repeat the kernel's double operations one for one (nested FMAs included) on two kinds of value:
  * Form: linear forms over the inputs of two rounds between renormalisations, with every input's full SIGNED range;
    each intermediate's exact range follows from its coefficients, so the magnitude checks hold for every input.
  * Exact: Python integers; every operation asserts that its exact result is an integer below 2^53 in magnitude (so the
    double holds it), and the round-down FMA / biased folds assert the window they rely on.
The big-integer tests check the algebra the kernel rests on, and the replay runs the whole permutation through the
Exact mirror against the oracle, including states built backwards so that the partial rounds start from chosen values."""
import importlib.util
import json
import os
import random
from fractions import Fraction

import numpy as np

from test_mds_network_bounds import CIRC, DIAG0, P

HERE = os.path.dirname(os.path.abspath(__file__))
TWO52, LIM = 1 << 52, 1 << 53
C_RD = 3 << 51                                   # 1.5 * 2^52, renorm_d's round-down target
BIAS_LO, BIAS_HI = (1 << 51) + (1 << 19), (1 << 51) - (1 << 20)
M32 = (1 << 32) - 1

_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)
with open(os.path.join(HERE, "golden", "poseidon_params.json")) as _f:
    PARAMS = json.load(_f)
ADD = MG.round_addends(PARAMS)                   # add[r] (ROUND_ADD_D holds its halves as 2^52 + half)
RC0 = PARAMS["all_round_constants"][:12]
PARTIAL_RC = PARAMS["fast_partial_round_constants"]
M = MG.mds_matrix(PARAMS)


class Exact:
    def chk(self, v):
        assert abs(v) < LIM, v
        return v

    def add(self, a, b):
        return self.chk(a + b)

    def sub(self, a, b):
        return self.chk(a - b)

    def scale(self, a, c):
        if isinstance(c, Fraction):
            assert a * c.numerator % c.denominator == 0, (a, c)   # the result stays an integer
            return a * c.numerator // c.denominator
        return a * c

    def mul(self, a, c):
        return self.chk(self.scale(a, c))

    def fma(self, a, c, b):
        return self.chk(self.scale(a, c) + b)


class Form:
    """linear forms over NV variables with per-variable ranges [lo, hi]; records the widest intermediate"""

    def __init__(self, lo, hi):
        self.lo, self.hi = np.array(lo, dtype=object), np.array(hi, dtype=object)
        self.widest = 0

    def var(self, k):
        v = np.zeros(len(self.lo), dtype=object)
        v[k] = Fraction(1)
        return v

    def range(self, v):
        a, b = v * self.lo, v * self.hi
        return sum(np.minimum(a, b)), sum(np.maximum(a, b))

    def chk(self, v):
        assert all(Fraction(c).denominator == 1 for c in v), "non-integer coefficient"   # every value stays an integer
        lo, hi = self.range(v)
        self.widest = max(self.widest, abs(lo), abs(hi))
        assert abs(lo) < LIM and abs(hi) < LIM
        return v

    def add(self, a, b):
        return self.chk(a + b)

    def sub(self, a, b):
        return self.chk(a - b)

    def mul(self, a, c):
        return self.chk(a * Fraction(c))

    def fma(self, a, c, b):
        return self.chk(a * Fraction(c) + b)


# ---- mirrors of the kernel's functions (same operations, same order) ----
def crt_mid(D, u, g):
    """crt_mid_half: w = (4 Ya, Yb, re, im) of u + g tau"""
    A0, A1, A2 = D.add(u[0], g), u[1], u[2]
    B0, B1, B2 = D.add(u[3], g), u[4], u[5]
    P0, P1, P2 = D.add(u[6], g), u[7], u[8]
    Q0, Q1, Q2 = u[9], u[10], u[11]
    T = D.mul(D.add(D.add(A1, A2), A0), 64)
    fma, add, sub = D.fma, D.add, D.sub
    return [fma(A2, 64, T), fma(A0, 64, T), fma(A1, 64, T),
            fma(B1, -2, fma(B2, 8, -B0)), fma(B2, -2, fma(B0, -8, -B1)), fma(B1, -8, fma(B0, 2, -B2)),
            fma(Q2, 4, add(fma(Q1, -16, add(fma(P0, 2, -Q0), P1)), P2)),
            fma(Q2, -16, add(fma(P1, 2, sub(fma(P0, -4, Q0), Q1)), P2)),
            fma(P2, 2, sub(fma(P1, -4, add(fma(P0, 16, Q0), Q1)), Q2)),
            fma(P2, -4, add(fma(P1, 16, add(fma(Q0, 2, P0), Q1)), Q2)),
            fma(P2, 16, add(fma(Q1, 2, add(fma(Q0, -4, -P0), P1)), Q2)),
            fma(Q2, 2, add(fma(Q1, -4, sub(fma(Q0, 16, -P0), P1)), P2))]


def crt_scale(D, w):
    """crt_scale_half: u = S G, ext"""
    u = w[0:3] + [D.mul(v, 4) for v in w[3:6]] + [D.mul(v, 2) for v in w[6:12]]
    return u, D.fma(w[0], Fraction(1, 4), D.add(w[3], w[6]))


def crt_round_half(D, u, g):
    return crt_scale(D, crt_mid(D, u, g))


def crt_lanes(D, w, bias, rc):
    """crt_lanes_half: H w + bias + rc[i], rc[i] = 2^52 + constant half as the double ROUND_ADD_D holds"""
    y = [None] * 12
    for j in range(3):
        e1 = D.fma(w[j], Fraction(1, 4), D.add(w[j + 3], bias))
        e2 = D.fma(w[j], Fraction(1, 4), D.sub(bias, w[j + 3]))
        y[j], y[j + 6] = D.add(D.add(e1, w[j + 6]), rc[j]), D.add(D.sub(e1, w[j + 6]), rc[j + 6])
        y[j + 3], y[j + 9] = D.add(D.add(e2, w[j + 9]), rc[j + 3]), D.add(D.sub(e2, w[j + 9]), rc[j + 9])
    return y


def crt_forward(D, s):
    """s: 12 u32 halves; v = 2^52 + s is the double the kernel builds from the bit pattern"""
    u = [None] * 12
    for j in range(3):
        v0, v3, v6, v9 = (TWO52 + s[j + k] for k in (0, 3, 6, 9))
        Pj, Qj = D.sub(v0, v6), D.sub(v3, v9)
        a, b = D.fma(D.sub(v6, TWO52), 2, Pj), D.fma(D.sub(v9, TWO52), 2, Qj)
        u[j], u[j + 3], u[j + 6], u[j + 9] = D.add(a, b), D.sub(a, b), Pj, Qj
    return u


def floor_rd(x):
    """__fma_rd(x, 2^-32, 1.5 * 2^52) - 1.5 * 2^52: exact floor while the sum lies where doubles are spaced 1 apart"""
    t = Fraction(x, 1 << 32) + C_RD
    assert TWO52 <= t < LIM
    return int(t // 1) - C_RD


def renorm(D, lo, hi):
    l1, h1 = floor_rd(lo), floor_rd(hi)
    return D.sub(D.fma(l1, -(1 << 32), lo), h1), D.add(D.fma(h1, -M32, hi), l1)


def biased_half(D, v, add):
    """2^52 + v + add as fold_halves_biased reads it: a double in [2^52, 2^53) whose high word - 0x43300000 < 2^20"""
    b = D.add(v, TWO52 + add)
    assert TWO52 <= b < LIM and (b - TWO52) >> 32 < 1 << 20
    return b - TWO52


def fold_signed(D, lo, hi):
    return (biased_half(D, lo, BIAS_LO) + (biased_half(D, hi, BIAS_HI) << 32)) % P


def halves(x):
    return x & M32, x >> 32


def lane0(D, el, eh, xl, xh, rc):
    """lane0_crt: returns x's halves and the injected (gl, gh)"""
    s0 = fold_signed(D, D.fma(xl, 8, el), D.fma(xh, 8, eh))
    x = (pow(s0, 7, P) + rc) % P
    (x0, x1), (s00, s01) = halves(x), halves(s0)
    return x0, x1, D.fma(xl, 8, D.sub(TWO52 + x0, TWO52 + s00)), D.fma(xh, 8, D.sub(TWO52 + x1, TWO52 + s01))


def partial_rounds(s):
    """rounds 4..25 of poseidon12 on the 12 (loose u64) lanes entering round 4; returns the lanes after + RC[26]"""
    D = Exact()
    lo, hi = zip(*(halves(v) for v in s))
    ul, uh = crt_forward(D, lo), crt_forward(D, hi)
    (el, eh), (xl, xh) = halves(s[0]), (0, 0)
    rcl, rch = zip(*(halves(v) for v in ADD[25]))
    rcl, rch = [TWO52 + v for v in rcl], [TWO52 + v for v in rch]
    for k in range(11):
        xl, xh, gl, gh = lane0(D, el, eh, xl, xh, PARTIAL_RC[2 * k])
        (ul, el), (uh, eh) = crt_scale(D, crt_mid(D, ul, gl)), crt_scale(D, crt_mid(D, uh, gh))
        xl, xh, gl, gh = lane0(D, el, eh, xl, xh, PARTIAL_RC[2 * k + 1])
        wl, wh = crt_mid(D, ul, gl), crt_mid(D, uh, gh)
        if k < 10:
            (ul, el), (uh, eh) = crt_scale(D, wl), crt_scale(D, wh)
            ul, uh = map(list, zip(*(renorm(D, a, b) for a, b in zip(ul, uh))))
        else:
            ul, uh = crt_lanes(D, wl, BIAS_LO, rcl), crt_lanes(D, wh, BIAS_HI, rch)
            ul[0], uh[0] = D.fma(xl, 8, ul[0]), D.fma(xh, 8, uh[0])
    return [(biased(bl) + (biased(bh) << 32)) % P for bl, bh in zip(ul, uh)]


def biased(b):
    """the half fold_halves_biased reads from the double b = 2^52 + half: b in [2^52, 2^53), high word - 0x43300000 < 2^20"""
    assert TWO52 <= b < LIM and (b - TWO52) >> 32 < 1 << 20
    return b - TWO52


def full_round(s, r):
    return [(v + a) % P for v, a in zip(MG.mat_vec(M, [pow(v, 7, P) for v in s]), ADD[r])]


def poseidon_mirror(state):
    s = [(v + c) % P for v, c in zip(state, RC0)]
    for r in range(4):
        s = full_round(s, r)
    s = partial_rounds(s)
    for r in range(26, 30):
        s = full_round(s, r)
    return s


# ---- the bounds, over the full signed input ranges ----
U_LO, U_HI = -2 * M32, 4 * M32                   # entry: A in [0, 4 M32], B in [-2 M32, 2 M32], P, Q in [-M32, M32]
G_LO, G_HI = -M32, 9 * M32                       # (x - s_0) + 8 x_prev
RN = (1 << 20)                                   # renorm_d outputs lie in [-RN, 2^32 + RN]


def test_two_rounds_between_renormalisations_are_exact():
    # variables: U_0..11, g_A, g_B, x_A, x_B, 1, rc (2^52 + a constant half)
    lo = [U_LO] * 12 + [G_LO, G_LO, 0, 0, 1, TWO52]
    hi = [U_HI] * 12 + [G_HI, G_HI, M32, M32, 1, TWO52 + M32]
    D = Form(lo, hi)
    U = [D.var(i) for i in range(12)]
    gA, gB, xA, xB, one = (D.var(12 + k) for k in range(5))
    uA, extA = crt_round_half(D, U, gA)
    uB, extB = crt_round_half(D, uA, gB)
    # lane-0 folds of the next two rounds (round B, and the next pair's round A or the exit)
    for ext, x in ((extA, xA), (extB, xB)):
        for bias in (BIAS_LO, BIAS_HI):
            a, b = D.range(D.fma(x, 8, ext) + bias * one)
            assert 0 <= a and b < TWO52
    # renorm_d inputs: |v| < 2^51 keeps the round-down target in [2^52, 2^53)
    for v in uB:
        a, b = D.range(v)
        assert -(1 << 51) <= a and b < 1 << 51
    assert D.widest < 1 << 51, D.widest       # every transform-domain intermediate (2^50.9)
    # last round: G on round A's outputs, then H + bias + the next round's biased constant half (2^52 + [0, 2^32)) + 8 x_last
    for bias in (BIAS_LO, BIAS_HI):
        rc = D.var(17)
        y = crt_lanes(D, crt_mid(D, uA, gB), bias * one, [rc] * 12)
        y[0] = D.fma(xB, 8, y[0])
        for v in y:
            a, b = D.range(v)
            assert TWO52 <= a and b < LIM                # the biased double fold_halves_biased reads


def test_renormalisation_signed_ranges_and_value():
    D = Exact()
    lim = (1 << 51) - 1
    edge = [0, 1, -1, M32, M32 + 1, -M32, -(1 << 32), lim, -lim, lim - M32, -lim + M32]
    rnd = random.Random(4)
    cases = [(a, b) for a in edge for b in edge] + [(rnd.randint(-lim, lim), rnd.randint(-lim, lim)) for _ in range(3000)]
    for lo, hi in cases:
        lo2, hi2 = renorm(D, lo, hi)
        assert (lo2 + (hi2 << 32) - lo - (hi << 32)) % P == 0
        assert -RN <= lo2 <= (1 << 32) + RN and -RN <= hi2 <= (1 << 32) + RN
        assert U_LO <= lo2 and hi2 <= U_HI and U_LO <= hi2 and lo2 <= U_HI


def test_fold_bias_is_a_multiple_of_p():
    assert (BIAS_LO + (BIAS_HI << 32)) % P == 0
    rnd = random.Random(6)
    D = Exact()
    for _ in range(2000):
        lo, hi = rnd.randint(-BIAS_HI, BIAS_HI), rnd.randint(-BIAS_HI, BIAS_HI)
        assert fold_signed(D, lo, hi) == (lo + (hi << 32)) % P


# ---- big-integer algebra ----
def mds(s):
    return [sum(CIRC[(j - i) % 12] * s[j] for j in range(12)) + (DIAG0 * s[0] if i == 0 else 0) for i in range(12)]


def circ(s):
    return [sum(CIRC[(j - i) % 12] * s[j] for j in range(12)) for i in range(12)]


def test_mds_matches_the_reference_matrix():
    rnd = random.Random(8)
    for _ in range(20):
        s = [rnd.randrange(P) for _ in range(12)]
        assert [v % P for v in mds(s)] == MG.mat_vec(M, s)


def test_transform_domain_identities():
    """F(circ s) = S G(F s) (crt_mid + crt_scale with g = 0) and H G(F s) = circ s (crt_lanes), on integers"""
    D = Exact()
    rnd = random.Random(9)
    for _ in range(200):
        s = [rnd.randrange(1 << 32) for _ in range(12)]
        w = crt_mid(D, crt_forward(D, s), 0)
        n, ext = crt_scale(D, w)
        c = circ(s)
        assert n == crt_forward_int(c)
        assert ext == c[0]
        assert crt_lanes(D, w, 0, [0] * 12) == c


def crt_forward_int(s):
    return ([s[j] + s[j + 3] + s[j + 6] + s[j + 9] for j in range(3)] + [s[j] - s[j + 3] + s[j + 6] - s[j + 9] for j in range(3)]
            + [s[j] - s[j + 6] for j in range(3)] + [s[j + 3] - s[j + 9] for j in range(3)])


def test_beta_recurrence_matches_direct_partial_rounds():
    """22 transform-domain rounds with the kernel's constants (PARTIAL_RC after the S-box, ADD[25] at the exit)
    against s_0 = sbox(s_0) + PARTIAL_RC[r]; s = M s, mod p, without the double arithmetic"""
    rnd = random.Random(10)
    inv4 = pow(4, -1, P)
    for _ in range(50):
        s = [rnd.randrange(P) for _ in range(12)]
        d = list(s)
        for r in range(22):
            d[0] = (pow(d[0], 7, P) + PARTIAL_RC[r]) % P
            d = [v % P for v in mds(d)]
        d = [(v + a) % P for v, a in zip(d, ADD[25])]
        U, xprev = [v % P for v in crt_forward_int(s)], 0
        for r in range(22):
            ext = (U[0] + U[3] + 2 * U[6]) * inv4 % P
            x = (pow((ext + 8 * xprev) % P, 7, P) + PARTIAL_RC[r]) % P
            U = _sg(U, (x - ext) % P)
            xprev = x
        out = [(v * inv4 * inv4) % P for v in crt_inverse_int(U)]
        out[0] = (out[0] + 8 * xprev) % P
        assert [(v + a) % P for v, a in zip(out, ADD[25])] == d


def _sg(U, beta):
    """S G(U + beta tau) on big integers, reduced mod p"""
    u = list(U)
    for k in (0, 3, 6):
        u[k] += beta
    A, B, Pp, Q = u[0:3], u[3:6], u[6:9], u[9:12]
    t = sum(A)
    Ya = [64 * (t + A[2]), 64 * (t + A[0]), 64 * (t + A[1])]
    Yb = [4 * (8 * B[2] - 2 * B[1] - B[0]), 4 * (-8 * B[0] - B[1] - 2 * B[2]), 4 * (2 * B[0] - 8 * B[1] - B[2])]
    re = [2 * Pp[0] - Q[0] + Pp[1] - 16 * Q[1] + Pp[2] + 4 * Q[2], -4 * Pp[0] + Q[0] + 2 * Pp[1] - Q[1] + Pp[2] - 16 * Q[2],
          16 * Pp[0] + Q[0] - 4 * Pp[1] + Q[1] + 2 * Pp[2] - Q[2]]
    im = [Pp[0] + 2 * Q[0] + 16 * Pp[1] + Q[1] - 4 * Pp[2] + Q[2], -Pp[0] - 4 * Q[0] + Pp[1] + 2 * Q[1] + 16 * Pp[2] + Q[2],
          -Pp[0] + 16 * Q[0] - Pp[1] - 4 * Q[1] + Pp[2] + 2 * Q[2]]
    return [v % P for v in Ya + Yb + [2 * v for v in re] + [2 * v for v in im]]


def crt_inverse_int(U):
    """16 * H(S^-1 U) on integers (scaled so that no division is needed; the caller divides by 16 mod p)"""
    y = [0] * 12
    for j in range(3):
        e1, e2 = 4 * (U[j] + U[j + 3]), 4 * (U[j] - U[j + 3])
        y[j], y[j + 6], y[j + 3], y[j + 9] = e1 + 8 * U[j + 6], e1 - 8 * U[j + 6], e2 + 8 * U[j + 9], e2 - 8 * U[j + 9]
    return y


# ---- replay of the whole permutation ----
def _oracle(states):
    import oracle

    return oracle.poseidon(np.array(states, dtype=np.uint64)).tolist()


def _edge_states():
    from helpers import field_grid

    rng = np.random.default_rng(11)
    g = np.array(field_grid(), dtype=np.uint64)
    nc = np.array([P, P + 1, (1 << 64) - 1, (1 << 64) - 2, 0xFFFFFFFF, 0xFFFFFFFF00000000], dtype=np.uint64)
    return g[rng.integers(0, g.size, size=(300, 12))].tolist() + nc[rng.integers(0, nc.size, size=(200, 12))].tolist()


INV7 = pow(7, -1, P - 1)
MINV = MG.mat_inv(M)


def state_entering_partial_rounds(target):
    """an input whose state entering round 4 is `target` (rounds 0..3 run backwards; x^7 is a bijection, gcd(7, p-1) = 1)"""
    s = [v % P for v in target]
    for r in range(3, -1, -1):
        s = MG.mat_vec(MINV, [(v - a) % P for v, a in zip(s, ADD[r])])
        s = [pow(v, INV7, P) for v in s]
    return [(v - c) % P for v, c in zip(s, RC0)]


def chosen_partial_entry_states():
    """the chosen entry states (canonical lane values); the loose representations v + p < 2^64 are replayed as well"""
    alt = [P - 1 if i % 2 == 0 else 0 for i in range(12)]
    return [[P - 1] * 12, [0] * 12, [M32] * 12, [1 << 32] * 12, alt, alt[::-1], [M32 if i % 2 else P - 1 for i in range(12)],
            [P - 1] + [0] * 11, [0] + [P - 1] * 11, [(1 << 63) + i for i in range(12)]]


def test_chosen_entry_states_reach_round_4():
    for t in chosen_partial_entry_states():
        x = state_entering_partial_rounds(t)
        s = [(v + c) % P for v, c in zip(x, RC0)]
        for r in range(4):
            s = full_round(s, r)
        assert s == [v % P for v in t]


def test_replay_matches_oracle_on_chosen_partial_entry_states():
    for t in chosen_partial_entry_states():
        x = state_entering_partial_rounds(t)
        assert poseidon_mirror(x) == _oracle([x])[0]
        # the same permutation entered with the loose representative v + p of every lane that has one
        loose = [v + P if v + P < 1 << 64 else v for v in t]
        ref = [v % P for v in partial_rounds(t)]
        assert [v % P for v in partial_rounds(loose)] == ref


def test_replay_matches_oracle_on_edge_states():
    states = _edge_states()
    assert [poseidon_mirror(s) for s in states] == _oracle(states)


def test_replay_matches_oracle_on_random_states():
    rnd = random.Random(12)
    states = [[rnd.getrandbits(64) for _ in range(12)] for _ in range(10_000)]
    assert [poseidon_mirror(s) for s in states] == _oracle(states)


def test_constant_headers_regenerate_from_params(tmp_path):
    """Both generated headers (the kernels' __constant__ tables and the oracle's) come out of poseidon_params.json byte
    for byte, so the constants the kernels and the oracle read are the parameters the golden tests pin."""
    rels = [("oracle", "poseidon_constants.h"), ("plonky2_demo_b200", "csrc", "poseidon_constants.cuh")]
    for rel in rels:
        os.makedirs(os.path.join(tmp_path, *rel[:-1]))
    MG.write_headers(PARAMS, ADD, root=str(tmp_path))
    for rel in rels:
        with open(os.path.join(tmp_path, *rel), "rb") as f, open(os.path.join(HERE, "..", *rel), "rb") as g:
            assert f.read() == g.read(), os.path.join(*rel)
