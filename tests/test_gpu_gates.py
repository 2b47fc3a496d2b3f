"""pcs_gate_constraint_terms (-m gpu): the gate-constraint tail of the quotient step on the device against the CPU oracle
(tests/harness/gate_oracle.c) element by element, on shapes up to the standard one (135 wires x 2^20, 2 challenges, D = 8,
rate 3), into host and device outputs; the device-resident chain wires -> Zs -> commitment #2 -> gate terms -> quotient chunks
-> commitment #3 on a satisfied instance, with the verifier's identity (gate constraints included) at an extension-field point
from the batches' openings and a changed wire failing the trim; every argument error.

Every checked call follows a decoy call over the same batches with other alphas and another public-inputs hash into the same
outputs, its temporaries freed in stream order: whatever the checked call fails to write then holds the decoy's values."""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))
import gate_oracle as go  # noqa: E402
import quotient_oracle as qo  # noqa: E402
from helpers import Ext, dev_table, free, mem_available_bytes, noncanonical, torch_u64  # noqa: E402
from test_gate_oracle import (  # noqa: E402
    ARITHMETIC, CONSTANT, DEMO_GATES, DEMO_GROUPS, NOOP, gate_slots, reduce_with_powers, satisfied_instance)

pytestmark = pytest.mark.gpu

P = 0xFFFFFFFF00000001
MIN_HOST_MEM = 48 << 30   # the oracle's natural-order LDEs at the standard shape (14.7 GB) and the case's arrays
MIN_FREE_HBM = 24 << 30
ONE_SELECTOR = ([(NOOP, 0, 0), (ARITHMETIC, 20, 0), (CONSTANT, 2, 0)], [(0, 3)])

SHAPES = [   # (lg_n, C, D, rate_bits, gate set, wires salt_w)
    (3, 2, 8, 3, "demo", 0),       # m = 2 demo shape
    (15, 2, 8, 3, "demo", 4),      # m = 64 demo shape: salts on the wires batch
    (6, 2, 4, 3, "demo", 0),       # q = 2 < rate_bits
    (8, 5, 8, 3, "demo", 4),       # five challenges: two passes over the alphas
    (7, 3, 5, 4, "one", 0),        # a single selector (no UNUSED_SELECTOR factor), q = 3 < rate_bits
    (20, 2, 8, 3, "demo", 0),      # the standard shape
]
OUT_MODES = ["host", "device"]


def _gate_set(name):
    return (DEMO_GATES, DEMO_GROUPS) if name == "demo" else ONE_SELECTOR


def _tables(gates, groups):
    return (np.ascontiguousarray(np.array(gates, dtype=np.uint32).reshape(-1, 3)),
            np.ascontiguousarray(np.array(groups, dtype=np.uintp).reshape(-1, 2)))


class Case:
    """Coefficients of the constants_sigmas (2 gate constants after the selectors, 80 sigmas) and wires (135) batches, the
    scalars, and the oracle's gate terms"""

    def __init__(self, lg_n, C_, D, rate_bits, gset, salt_w):
        rng = np.random.default_rng(lg_n * 131 + C_ * 17 + D)
        n, N = 1 << lg_n, (1 << lg_n) << rate_bits
        self.shape = (lg_n, C_, D, rate_bits, gset, salt_w)
        self.gates, self.groups = _gate_set(gset)
        self.nc = len(self.groups) + 2
        self.cs = rng.integers(0, P, (self.nc + 80, n), dtype=np.uint64)
        self.wires = rng.integers(0, P, (135, n), dtype=np.uint64)
        self.salts = rng.integers(0, P, (salt_w, N), dtype=np.uint64) if salt_w else None
        self.pih, self.alphas = noncanonical(rng, 4), noncanonical(rng, C_)
        go.use_all_cores()
        oracle.use_all_cores()
        lde = [oracle.coset_lde(c, rate_bits) for c in (self.cs, self.wires)]
        self.want = go.gate_terms(*lde, rate_bits, self.gates, self.groups, self.nc, self.pih, self.alphas, D)


@functools.lru_cache(maxsize=1)
def _case(shape):
    return Case(*shape)


@pytest.fixture(scope="module")
def L():
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    p.init(0)
    yield _ffi.lib()
    p.shutdown()


def _batches(case):
    import plonky2_demo_b200 as p

    rate_bits = case.shape[3]
    cap_h = min(4, case.shape[0] + rate_bits)
    return [p.PolynomialBatch.from_coeffs(case.cs, rate_bits, False, cap_h),
            p.PolynomialBatch.from_coeffs(case.wires, rate_bits, case.salts is not None, cap_h, salts=case.salts)]


def _call(L, cs, w, gates, groups, nc, pih, alphas, D, flags, outs, lookups=0):
    from plonky2_demo_b200 import _ffi

    return L.pcs_gate_constraint_terms(cs, w, gates.ctypes.data_as(C.POINTER(C.c_uint32)), gates.shape[0],
                                       groups.ctypes.data_as(C.POINTER(_ffi.sz)), groups.shape[0], lookups, nc, _ffi.ptr(pih),
                                       _ffi.ptr(alphas), alphas.shape[0], D, flags, outs)


def _run(L, case, batches, out_mode):
    """decoy call, then the checked call into the same outputs -> (rc, [C][M])"""
    import torch

    from plonky2_demo_b200 import _ffi

    C_, M = case.want.shape
    D = case.shape[2]
    rng = np.random.default_rng(0xDEC0 + case.shape[0])
    gates, groups = _tables(case.gates, case.groups)
    flags = _ffi.PCS_DEVICE_PTRS if out_mode == "device" else 0
    if out_mode == "device":
        o = torch.zeros((C_, M), dtype=torch.int64, device="cuda")
        outs = dev_table(list(o))
    else:
        o = np.full((C_, M), 0xDEAD, dtype=np.uint64)
        outs = _ffi.ptr_array(list(o))
    h = [b._h for b in batches]
    assert _call(L, *h, gates, groups, case.nc, noncanonical(rng, 4), noncanonical(rng, C_), D, flags, outs) == 0
    rc = _call(L, *h, gates, groups, case.nc, case.pih, case.alphas, D, flags, outs)
    if out_mode == "device":
        torch.cuda.synchronize()
        return rc, o.cpu().numpy().view(np.uint64)
    return rc, o


def _skip_if_short(shape):
    if shape[0] >= 20:
        if mem_available_bytes() < MIN_HOST_MEM:
            pytest.skip("not enough host memory for the oracle at the standard shape")
        import torch

        if torch.cuda.mem_get_info()[0] < MIN_FREE_HBM:
            pytest.skip("not enough free HBM")


@pytest.mark.parametrize("shape,out_mode", [(s, m) for s in SHAPES for m in OUT_MODES],
                         ids=[f"{'-'.join(map(str, s))}-{m}" for s in SHAPES for m in OUT_MODES])
def test_equals_oracle(L, shape, out_mode):
    _skip_if_short(shape)
    case = _case(shape)
    batches = _batches(case)
    try:
        rc, got = _run(L, case, batches, out_mode)
    finally:
        free(*batches)
    assert rc == 0, L.pcs_last_error()
    assert got.shape == case.want.shape
    assert (got < np.uint64(P)).all()
    assert np.array_equal(got, case.want)


def test_python_api(L):
    import plonky2_demo_b200 as p

    case = _case(SHAPES[2])
    batches = _batches(case)
    gates = [p.NoopGate(), p.ConstantGate(2), p.PublicInputGate(), p.ArithmeticGate(20), p.PoseidonGate()]
    info = p.SelectorsInfo(selector_indices=(0, 0, 0, 0, 1), groups=((0, 4), (4, 5)))
    try:
        got = p.gate_constraint_terms(*batches, gates, info, case.nc, case.pih, case.alphas, case.shape[2])
    finally:
        free(*batches)
    assert np.array_equal(got, case.want)


# ---- the device-resident chain on a satisfied instance ---------------------------------------------------------------------
def _openings(L, h, w, z):
    from plonky2_demo_b200 import _ffi

    out = np.empty((w, 2), dtype=np.uint64)
    _ffi.check(L.pcs_batch_eval_ext(h, _ffi.ptr(np.array([z.a, z.b], dtype=np.uint64)), _ffi.ptr(out)))
    return [Ext(int(a), int(b)) for a, b in out]


@pytest.mark.parametrize("lg_n", [12, 15])
def test_device_resident_chain(L, lg_n):
    """commitment #1 of the wires, the Zs from device wire values, commitment #2, the gate terms into a device buffer, the
    quotient chunks from that device tail (the trim at D = 7 succeeds), commitment #3; the verifier's identity with the gate
    constraints holds at an extension-field point with every value an opening of a committed batch; one changed wire makes the
    quotient's trim fail"""
    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    R, C_, D, rate_bits, cap_h, nc = 80, 2, 7, 3, 4, 4
    n, K = 1 << lg_n, -(-R // D)
    rng = np.random.default_rng(4040 + lg_n)
    inst = satisfied_instance(rng, lg_n, R)
    wires, sigmas, k_is = inst["wires"], inst["sigmas"], inst["k_is"]
    betas, gammas, alphas = (rng.integers(1, P, C_, dtype=np.uint64) for _ in range(3))
    gates, groups = _tables(DEMO_GATES, DEMO_GROUPS)
    M = n << 3
    b_cs = p.PolynomialBatch.from_values(np.vstack([inst["consts"], sigmas]), rate_bits, False, cap_h)
    b_w = p.PolynomialBatch.from_values(wires, rate_bits, False, cap_h)   # commitment #1
    bad_wires = wires.copy()
    bad_wires[65 + 3, 5] = (int(bad_wires[65 + 3, 5]) + 1) % P   # a partial S-box wire of the second Poseidon row
    b_bad = p.PolynomialBatch.from_values(bad_wires, rate_bits, False, cap_h)
    h2, h3 = C.c_void_p(), C.c_void_p()
    try:
        W = C_ * K
        w_dev = torch_u64(wires)
        zs_dev = torch.zeros((W, n), dtype=torch.int64, device="cuda")
        _ffi.check(L.pcs_permutation_partial_products(_ffi.dev_ptr_array(w_dev.data_ptr(), R, n),
                                                      _ffi.dev_ptr_array(torch_u64(sigmas).data_ptr(), R, n), R, lg_n,
                                                      _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas), C_, D,
                                                      _ffi.PCS_DEVICE_PTRS, _ffi.dev_ptr_array(zs_dev.data_ptr(), W, n)))
        _ffi.check(L.pcs_commit_from_values(_ffi.dev_ptr_array(zs_dev.data_ptr(), W, n), W, lg_n, rate_bits, cap_h, None, 0,
                                            _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS, None, None, C.byref(h2)))
        gt = torch.zeros((C_, M), dtype=torch.int64, device="cuda")
        _ffi.check(_call(L, b_cs._h, b_w._h, gates, groups, nc, inst["pih"], alphas, D, _ffi.PCS_DEVICE_PTRS, dev_table(list(gt))))
        q_dev = torch.zeros((C_ * D, n), dtype=torch.int64, device="cuda")
        _ffi.check(L.pcs_quotient_polys(b_cs._h, b_w._h, h2, nc, R, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas),
                                        _ffi.ptr(alphas), C_, D, dev_table(list(gt)), _ffi.PCS_DEVICE_PTRS,
                                        _ffi.dev_ptr_array(q_dev.data_ptr(), C_ * D, n)))
        _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(q_dev.data_ptr(), C_ * D, n), C_ * D, lg_n, rate_bits, cap_h, None,
                                            0, _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS, None, C.byref(h3)))
        go.use_all_cores()
        oracle.use_all_cores()
        cs_lde, w_lde = (oracle.coset_lde(oracle.fft(v, inverse=True), rate_bits) for v in (np.vstack([inst["consts"], sigmas]), wires))
        want_gt = go.gate_terms(cs_lde, w_lde, rate_bits, DEMO_GATES, DEMO_GROUPS, nc, inst["pih"], alphas, D)
        assert np.array_equal(gt.cpu().numpy().view(np.uint64), want_gt)

        # vanishing(zeta) = Z_H(zeta) sum_k zeta^(k n) chunk_k(zeta), every value an opening of a committed batch
        zeta = Ext(int(rng.integers(2, P, dtype=np.uint64)), int(rng.integers(1, P, dtype=np.uint64)))
        g = pow(1753635133440165772, 1 << (32 - lg_n), P)
        w_o, cs_o = _openings(L, b_w._h, 135, zeta), _openings(L, b_cs._h, nc + R, zeta)
        z_o, z_go = _openings(L, h2, W, zeta), _openings(L, h2, W, zeta * g)
        q_o = _openings(L, h3, C_ * D, zeta)
        zn = zeta.pow(n)
        zh = zn - 1
        l_0 = zh * (Ext(n) * (zeta - 1)).inv()
        Pn = K - 1
        terms = [l_0 * (z_o[c] - 1) for c in range(C_)]
        for c in range(C_):
            b, gm = int(betas[c]), int(gammas[c])
            num = [w_o[j] + zeta * (b * int(k_is[j])) + gm for j in range(R)]
            den = [w_o[j] + cs_o[nc + j] * b + gm for j in range(R)]
            acc, chain = z_o[c], z_o[C_ + c * Pn:C_ + (c + 1) * Pn] + [z_go[c]]
            for k in range(K):
                nk, dk = Ext(1), Ext(1)
                for v in num[k * D:(k + 1) * D]:
                    nk = nk * v
                for v in den[k * D:(k + 1) * D]:
                    dk = dk * v
                terms.append(acc * nk - chain[k] * dk)
                acc = chain[k]
        slots = gate_slots(DEMO_GATES, DEMO_GROUPS, w_o, cs_o[:nc], inst["pih"])
        for a in range(C_):
            al = int(alphas[a])
            van = reduce_with_powers(terms, al) + pow(al, len(terms), P) * reduce_with_powers(slots, al)
            tq, zk = Ext(0), Ext(1)
            for k in range(D):
                tq = tq + zk * q_o[a * D + k]
                zk = zk * zn
            assert van == zh * tq, a

        # one changed wire: the gate terms no longer vanish on H, and the quotient's trim fails
        _ffi.check(_call(L, b_cs._h, b_bad._h, gates, groups, nc, inst["pih"], alphas, D, _ffi.PCS_DEVICE_PTRS,
                         dev_table(list(gt))))
        rc = L.pcs_quotient_polys(b_cs._h, b_bad._h, h2, nc, R, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas),
                                  _ffi.ptr(alphas), C_, D, dev_table(list(gt)), _ffi.PCS_DEVICE_PTRS,
                                  _ffi.dev_ptr_array(q_dev.data_ptr(), C_ * D, n))
        assert rc == -5
        assert L.pcs_last_error() == qo.QUOTIENT_FAILED.encode()
    finally:
        L.pcs_batch_free(h2)
        L.pcs_batch_free(h3)
        free(b_cs, b_w, b_bad)


# ---- argument errors ---------------------------------------------------------------------------------------------------------
def _normal_call_works(L):
    case = _case(SHAPES[2])
    batches = _batches(case)
    try:
        rc, got = _run(L, case, batches, "host")
    finally:
        free(*batches)
    assert rc == 0, L.pcs_last_error()
    assert np.array_equal(got, case.want)


def test_argument_errors(L):
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    case = _case(SHAPES[2])
    lg_n, C_, D, rate_bits, _, _ = case.shape
    n = 1 << lg_n
    bs = _batches(case)
    h = [b._h for b in bs]
    out = np.empty((C_, n << 3), dtype=np.uint64)
    outs = _ffi.ptr_array(list(out))
    gates, groups = _tables(case.gates, case.groups)

    def with_gate(g, entry):
        t = gates.copy()
        t[g] = entry
        return t

    narrow = p.PolynomialBatch.from_coeffs(case.wires[:80], rate_bits, False, 0)
    other_degree = p.PolynomialBatch.from_coeffs(np.ones((135, n * 2), dtype=np.uint64), rate_bits, False, 0)
    other_rate = p.PolynomialBatch.from_coeffs(np.ones((135, n), dtype=np.uint64), rate_bits + 1, False, 0)
    on_demand = p.PolynomialBatch.from_coeffs(case.wires, rate_bits, False, 0, lde_on_demand=True)
    shard = C.c_void_p()
    _ffi.check(L.pcs_commit_shard_from_coeffs(_ffi.ptr_array(list(case.wires)), 135, lg_n, rate_bits, 0, rate_bits - 1, 0,
                                              None, 0, 0, None, C.byref(shard)))
    rows_only = C.c_void_p()
    _ffi.check(L.pcs_shard_begin_rows(135, 0, lg_n + rate_bits, 0, C.byref(rows_only)))
    null_out = _ffi.ptr_array(list(out))
    null_out[1] = None
    pih, al = _ffi.ptr(case.pih), _ffi.ptr(case.alphas)
    u32p, szp = C.POINTER(C.c_uint32), C.POINTER(_ffi.sz)

    def args(**kw):
        d = dict(cs=h[0], w=h[1], gates=gates, groups=groups, S=None, lookups=0, nc=case.nc, pih=pih, a=al, C=C_, D=D, f=0,
                 o=outs)
        d.update(kw)
        g, gr = d.pop("gates"), d.pop("groups")
        S = d.pop("S")
        gp = g.ctypes.data_as(u32p) if g is not None else None
        grp = gr.ctypes.data_as(szp) if gr is not None else None
        return (d["cs"], d["w"], gp, gates.shape[0], grp, groups.shape[0] if S is None else S, d["lookups"], d["nc"], d["pih"],
                d["a"], d["C"], d["D"], d["f"], d["o"])

    cases = [
        args(cs=None), args(w=None), args(gates=None), args(groups=None), args(pih=None), args(a=None), args(o=None),
        args(o=null_out),
        args(gates=with_gate(1, (7, 0, 0))),                          # unknown gate kind
        args(gates=with_gate(1, (1, 2, 2))),                          # selector_index >= num_selectors
        args(gates=with_gate(4, (4, 0, 0))),                          # PoseidonGate outside its group
        args(groups=np.array([[0, 4], [4, 6]], dtype=np.uintp)),      # a group past num_gates
        args(groups=np.array([[0, 4], [4, 4]], dtype=np.uintp)),      # an empty group
        args(groups=np.array([[3, 1], [4, 5]], dtype=np.uintp)),      # not a range
        args(lookups=1),
        args(w=narrow._h),                                            # PoseidonGate with 80 wires
        args(nc=3),                                                   # ConstantGate / ArithmeticGate without their constants
        args(nc=case.cs.shape[0] + 1),                                # more constants than the batch holds
        args(D=16),                                                   # q = 4 > rate_bits
        args(D=1), args(C=0),
        args(w=other_degree._h), args(w=other_rate._h), args(w=on_demand._h), args(w=shard), args(w=rows_only),
        args(cs=on_demand._h),
    ]
    try:
        for i, c in enumerate(cases):
            assert L.pcs_gate_constraint_terms(*c) == -5, (i, L.pcs_last_error())
            _normal_call_works(L)
        assert L.pcs_gate_constraint_terms(*args(D=16)) == -5
        assert L.pcs_last_error().startswith(b"Having constraints of degree higher than the rate is not supported yet")
        assert L.pcs_gate_constraint_terms(*args(lookups=1)) == -5
        assert b"lookups" in L.pcs_last_error()
    finally:
        L.pcs_batch_free(shard)
        L.pcs_batch_free(rows_only)
        free(*bs, narrow, other_degree, other_rate, on_demand)
