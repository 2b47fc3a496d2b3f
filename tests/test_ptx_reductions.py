"""CPU check of the device field reductions' ALGORITHMS (csrc/gl64.cuh inline PTX) against big-int
arithmetic, through the PTX-subset interpreter in tests/ptx_emu.py.  The reference's reduce128 / reduce96 / add / sub
(field/src/goldilocks_field.rs:199-274,347-369) and its input grid (prime_field_testing.rs:7-17) are the model; ptxas and the
hardware are covered by the `-m gpu` tests (test_device_field_grid_vs_bigint, Poseidon KATs)."""
import os
import random

import pytest

import ptx_emu as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "plonky2_demo_b200", "csrc", "gl64.cuh")
P = (1 << 64) - (1 << 32) + 1
M32, M64 = E.M32, E.M64
BIAS = 0x43300000


def _src(tmp_dir):
    text = "".join(l for l in open(HDR) if not l.startswith(("#include", "#pragma once")))
    tmp = os.path.join(tmp_dir, "gl64.h")
    with open(tmp, "w") as f:
        f.write(text)
    return E.preprocess(tmp, {})


def _grid64():
    # the reference's test inputs (prime_field_testing.rs:7-17): small values, values around powers of two, around p and 2^64
    g = set()
    for k in range(0, 65):
        for dlt in (-2, -1, 0, 1, 2):
            g.add(((1 << k) + dlt) & M64)
    for dlt in range(-3, 4):
        g.add((P + dlt) & M64)
        g.add((M64 + dlt) & M64)
        g.add(((1 << 32) - 1 + dlt) & M64)
    g |= {0, 1, 2, M32, M32 << 32, P - 1, P, M64}
    return sorted(g)


def _rand64(rng, n):
    out = []
    for _ in range(n):
        k = rng.choice((64, 64, 64, 33, 32, 31, 8))
        v = rng.getrandbits(k)
        if rng.random() < 0.25:
            v = (M64 - v) & M64          # close to 2^64
        out.append(v)
    return out


@pytest.fixture(scope="module")
def src(tmp_path_factory):
    return _src(str(tmp_path_factory.mktemp("ptx")))


def test_reduce128(src):
    red = E.extract_asm(src, "reduce128")

    def reduce128(lo, hi):
        return E.run_asm(*red, {"lo": lo, "r2": hi & M32, "r3": hi >> 32})["z"]

    rng = random.Random(0xC0FFEE)
    grid = _grid64()
    pairs = [(a, b) for a in grid for b in grid[::37]] + [(a, b) for a in grid[::53] for b in grid]
    pairs += list(zip(_rand64(rng, 2500), _rand64(rng, 2500)))
    for a, b in pairs:                               # every 128-bit value a product of two u64 can take ...
        q = a * b
        r = reduce128(q & M64, q >> 64)
        assert 0 <= r <= M64 and r % P == q % P, (hex(a), hex(b), hex(r))
    for lo, hi in [(0, M64), (M64, M64), (0, M32 << 32), (M32, M32), (0, M32), (M64, 0), (1, 1 << 32), (M64, M32)] + \
                  list(zip(_rand64(rng, 1000), _rand64(rng, 1000))):     # ... and arbitrary limbs (the reduction accepts any)
        r = reduce128(lo, hi)
        assert 0 <= r <= M64 and r % P == (lo + (hi << 64)) % P, (hex(lo), hex(hi), hex(r))


def test_reduce96(src):
    rng = random.Random(7)
    b = E.extract_asm(src, "reduce96")
    for x, y in [(u, v) for u in _grid64()[::5] for v in _grid64()[::17]] + list(zip(_rand64(rng, 2000), _rand64(rng, 2000))):
        top = y & M32
        env = E.run_asm(*b, {"r0": x & M32, "r1": x >> 32, "top": top})
        r = env["r0"] | (env["r1"] << 32)
        assert r % P == (x + (top << 64)) % P


def test_fold_halves(src):
    rng = random.Random(99)
    a = E.extract_asm(src, "fold_halves_biased")
    c = E.extract_asm(src, "fold_halves")
    # full rounds: L, H < 2^45 (high words < 2^13); partial rounds (fold_d): < 2^52 (high words < 2^20)
    lim = [0, 1, (1 << 13) - 1, 1 << 13, (1 << 20) - 1]
    lows = [0, 1, M32, M32 - 1, 1 << 31, (1 << 13), (1 << 20) - 1]
    cases = [(l0, l1, h0, h1) for l0 in lows for l1 in lim for h0 in lows for h1 in lim]
    cases += [(rng.getrandbits(32), rng.getrandbits(rng.choice((1, 13, 20))), rng.getrandbits(32),
               rng.getrandbits(rng.choice((1, 13, 20)))) for _ in range(2500)]
    for l0, l1, h0, h1 in cases:
        want = (l0 + (l1 << 32) + ((h0 + (h1 << 32)) << 32)) % P          # L + H * 2^32
        env = E.run_asm(*a, {"l0": l0, "l1b": BIAS + l1, "h0": h0, "h1b": BIAS + h1})
        r = env["w0"] | (env["w1"] << 32)
        assert 0 <= r <= M64 and r % P == want, (l0, l1, h0, h1)
        if l1 + h1 < (1 << 13):                                            # the integer network's fold: (L >> 32) + (H >> 32) < 2^13
            env = E.run_asm(*c, {"l0": l0, "l1": l1, "h0": h0, "h1": h1})
            r = env["w0"] | (env["w1"] << 32)
            assert r % P == want


def test_add_sub_canon(src):
    rng = random.Random(5)
    add = E.extract_asm(src, "add_lc")
    sub = E.extract_asm(src, "sub_lc")
    addw = E.extract_asm(src, "add_lc_wide")
    can = E.extract_asm(src, "canon")
    canon_vals = [v for v in _grid64() if v < P] + [rng.randrange(P) for _ in range(1000)]
    loose = _grid64() + _rand64(rng, 1000)
    for x, b in zip(loose, canon_vals[::-1] + canon_vals):
        env = E.run_asm(*add, {"a0": x & M32, "a1": x >> 32, "(uint32_t)b": b & M32, "(uint32_t)(b >> 32)": b >> 32})
        assert (env["a0"] | (env["a1"] << 32)) % P == (x + b) % P
        env = E.run_asm(*sub, {"a0": x & M32, "a1": x >> 32, "(uint32_t)b": b & M32, "(uint32_t)(b >> 32)": b >> 32})
        assert (env["a0"] | (env["a1"] << 32)) % P == (x - b) % P
        env = E.run_asm(*addw, {"a": x, "b": b})
        assert 0 <= env["z"] <= M64 and env["z"] % P == (x + b) % P, (hex(x), hex(b))
        env = E.run_asm(*can, {"lo": x & M32, "hi": x >> 32})
        got = env["s0"] if env["c"] else x
        assert got == x % P
