"""pcs_permutation_partial_products (-m gpu): the permutation argument's Zs and partial products on the device against the CPU
oracle (tests/harness/permutation_oracle.c), element by element, for host inputs, contiguous device columns and scattered
device columns, all with non-canonical inputs; the device-resident chain wires -> Zs -> commitment #2; the error cases."""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))
import permutation_oracle as po  # noqa: E402
from helpers import dev_table, noncanonical, torch_u64  # noqa: E402

pytestmark = pytest.mark.gpu

P = 0xFFFFFFFF00000001

SHAPES = [   # (R, lg_n, C, D)
    (80, 3, 2, 8),     # m = 2 demo shape
    (80, 15, 2, 8),    # m = 64 demo shape
    (3, 0, 1, 2),      # n = 1
    (5, 3, 1, 8),      # P = 0
    (7, 3, 3, 3),      # short last chunk, three challenges
    (9, 4, 1, 2),      # D = 2, odd R
    (10, 13, 5, 4),    # five challenges: two passes over the inputs
    (4, 24, 1, 2),     # 4096 scan tiles
    (80, 20, 2, 8),    # the benchmark shape
]
MODES = ["host", "device", "scattered"]


@functools.lru_cache(maxsize=2)
def _case(R, lg_n, C, D):
    rng = np.random.default_rng(R * 100003 + lg_n * 101 + C)
    wires, sigmas = noncanonical(rng, (R, 1 << lg_n)), noncanonical(rng, (R, 1 << lg_n))
    k_is, betas, gammas = noncanonical(rng, R), noncanonical(rng, C), noncanonical(rng, C)
    po.use_all_cores()
    want = po.prove_order(po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D))
    return wires, sigmas, k_is, betas, gammas, want


@pytest.fixture(scope="module")
def L():
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    p.init(0)
    yield _ffi.lib()
    p.shutdown()


def _run(L, mode, wires, sigmas, k_is, betas, gammas, D, W):
    """-> (rc, [W][n] result as numpy)"""
    from plonky2_demo_b200 import _ffi

    R, n = wires.shape
    lg_n = n.bit_length() - 1
    scalars = (_ffi.ptr(np.ascontiguousarray(k_is)), _ffi.ptr(np.ascontiguousarray(betas)), _ffi.ptr(np.ascontiguousarray(gammas)),
               len(betas), D)
    if mode == "host":
        out = np.full((W, n), 0xDEAD, dtype=np.uint64)
        rc = L.pcs_permutation_partial_products(_ffi.ptr_array(list(wires)), _ffi.ptr_array(list(sigmas)), R, lg_n, *scalars, 0,
                                                _ffi.ptr_array(list(out)))
        return rc, out
    import torch

    if mode == "device":
        w, s = torch_u64(wires), torch_u64(sigmas)
        o = torch.zeros((W, n), dtype=torch.int64, device="cuda")
        tw, ts, to = dev_table(list(w)), dev_table(list(s)), dev_table(list(o))
    else:   # every column its own allocation
        w, s = [torch_u64(c) for c in wires], [torch_u64(c) for c in sigmas]
        o = [torch.zeros(n, dtype=torch.int64, device="cuda") for _ in range(W)]
        tw, ts, to = dev_table(w), dev_table(s), dev_table(o)
    rc = L.pcs_permutation_partial_products(tw, ts, R, lg_n, *scalars, _ffi.PCS_DEVICE_PTRS, to)
    torch.cuda.synchronize()
    res = (o if mode == "device" else torch.stack(o)).cpu().numpy().view(np.uint64)
    if mode == "device":   # inputs are read, not written
        assert np.array_equal(w.cpu().numpy().view(np.uint64), wires) and np.array_equal(s.cpu().numpy().view(np.uint64), sigmas)
    return rc, res


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("R,lg_n,C_,D", SHAPES)
def test_equals_oracle(L, R, lg_n, C_, D, mode):
    wires, sigmas, k_is, betas, gammas, want = _case(R, lg_n, C_, D)
    rc, got = _run(L, mode, wires, sigmas, k_is, betas, gammas, D, want.shape[0])
    assert rc == 0, L.pcs_last_error()
    assert (got < np.uint64(P)).all()
    assert np.array_equal(got, want)


def test_python_api_orders(L):
    """the package's three entry points are the same engine call in the reference's per-challenge order and prove()'s order"""
    import plonky2_demo_b200 as p

    R, lg_n, C_, D = 7, 3, 3, 3
    wires, sigmas, k_is, betas, gammas, want = _case(R, lg_n, C_, D)
    per = po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D)
    extra = np.vstack([wires, noncanonical(np.random.default_rng(1), (4, 1 << lg_n))])   # unrouted wires are not read
    assert np.array_equal(p.zs_partial_products_values(extra, sigmas, k_is, betas, gammas, D, num_routed_wires=R), want)
    assert np.array_equal(p.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D), per)
    assert np.array_equal(p.wires_permutation_partial_products_and_zs(wires, sigmas, k_is, betas[1], gammas[1], D), per[1])


def test_device_resident_chain(L):
    """commitment #1 from device wire values, the Zs into a device [20][n] buffer, commitment #2 from that buffer: equal to the
    oracle's commitment of the oracle's Zs; the device wire values are unchanged."""
    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    num_wires, R, lg_n, C_, D, rate_bits, cap_height = 135, 80, 12, 2, 8, 3, 4
    n = 1 << lg_n
    rng = np.random.default_rng(77)
    wires = noncanonical(rng, (num_wires, n))
    sigmas = noncanonical(rng, (R, n))
    k_is = p.get_unique_coset_shifts(n, R)
    betas, gammas = noncanonical(rng, C_), noncanonical(rng, C_)
    w_dev = torch_u64(wires)
    s_dev = torch_u64(sigmas)
    b1 = C.c_void_p()
    cap1 = np.empty((1 << cap_height, 4), dtype=np.uint64)
    _ffi.check(L.pcs_commit_from_values(_ffi.dev_ptr_array(w_dev.data_ptr(), num_wires, n), num_wires, lg_n, rate_bits, cap_height,
                                        None, 0, _ffi.PCS_DEVICE_PTRS, None, _ffi.ptr(cap1), C.byref(b1)))
    W = C_ * (1 + (-(-R // D) - 1))
    zs_dev = torch.zeros((W, n), dtype=torch.int64, device="cuda")
    _ffi.check(L.pcs_permutation_partial_products(_ffi.dev_ptr_array(w_dev.data_ptr(), R, n), _ffi.dev_ptr_array(s_dev.data_ptr(), R, n),
                                                  R, lg_n, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas), C_, D,
                                                  _ffi.PCS_DEVICE_PTRS, _ffi.dev_ptr_array(zs_dev.data_ptr(), W, n)))
    b2 = C.c_void_p()
    cap2 = np.empty((1 << cap_height, 4), dtype=np.uint64)
    _ffi.check(L.pcs_commit_from_values(_ffi.dev_ptr_array(zs_dev.data_ptr(), W, n), W, lg_n, rate_bits, cap_height, None, 0,
                                        _ffi.PCS_DEVICE_PTRS, None, _ffi.ptr(cap2), C.byref(b2)))
    try:
        zs = po.prove_order(po.all_wires_permutation_partial_products(wires[:R], sigmas, k_is, betas, gammas, D))
        assert W == 20 and np.array_equal(zs_dev.cpu().numpy().view(np.uint64), zs)
        ref = oracle.commit_from_values(zs, rate_bits, cap_height)
        assert np.array_equal(cap2, ref["cap"])
        N = n << rate_bits
        idx = np.unique(np.concatenate([[0, 1, N - 1], rng.integers(0, N, 29)])).astype(np.uint64)
        rows = np.empty((idx.size, W), dtype=np.uint64)
        _ffi.check(L.pcs_batch_get_rows(b2, _ffi.ptr(idx), idx.size, _ffi.ptr(rows)))
        assert np.array_equal(rows, ref["leaves"][idx.astype(np.int64)])
        depth = lg_n + rate_bits - cap_height
        for i in idx[:8]:
            sib = np.empty((depth, 4), dtype=np.uint64)
            _ffi.check(L.pcs_batch_prove(b2, int(i), _ffi.ptr(sib)))
            assert np.array_equal(sib, oracle.merkle_prove(ref["digests"], N, cap_height, int(i)))
        assert np.array_equal(cap1, oracle.commit_from_values(wires, rate_bits, cap_height)["cap"])
        assert np.array_equal(w_dev.cpu().numpy().view(np.uint64), wires)   # commitment #1's inputs are not consumed
    finally:
        L.pcs_batch_free(b1)
        L.pcs_batch_free(b2)


def _normal_call_works(L):
    wires, sigmas, k_is, betas, gammas, want = _case(7, 3, 3, 3)
    rc, got = _run(L, "host", wires, sigmas, k_is, betas, gammas, 3, want.shape[0])
    assert rc == 0 and np.array_equal(got, want)


@pytest.mark.parametrize("mode", ["host", "device"])
def test_zero_denominator(L, mode):
    rng = np.random.default_rng(3)
    R, lg_n, D = 9, 5, 4
    wires, sigmas = noncanonical(rng, (R, 1 << lg_n)), noncanonical(rng, (R, 1 << lg_n))
    k_is, beta = noncanonical(rng, R), 12345
    gamma = (P - (int(wires[6][17]) + beta * int(sigmas[6][17])) % P) % P   # den_6(x_17) = 0
    rc, _ = _run(L, mode, wires, sigmas, k_is, np.array([beta], dtype=np.uint64), np.array([gamma], dtype=np.uint64), D, 3)
    assert rc == -5   # PCS_ERR_ARG
    assert L.pcs_last_error() == b"Tried to invert zero"
    with pytest.raises(ZeroDivisionError):
        po.all_wires_permutation_partial_products(wires, sigmas, k_is, [beta], [gamma], D)
    _normal_call_works(L)


def test_zero_numerator_is_not_an_error(L):
    rng = np.random.default_rng(4)
    R, lg_n, D = 9, 5, 4
    wires, sigmas = noncanonical(rng, (R, 1 << lg_n)), noncanonical(rng, (R, 1 << lg_n))
    k_is, beta = noncanonical(rng, R), 999
    x = pow(pow(1753635133440165772, 1 << (32 - lg_n), P), 5, P)
    gamma = (P - (int(wires[2][5]) + beta * (int(k_is[2]) * x)) % P) % P   # num_2(x_5) = 0
    want = po.prove_order(po.all_wires_permutation_partial_products(wires, sigmas, k_is, [beta], [gamma], D))
    assert want[0, 6] == 0   # Z is zero from the next row on
    for mode in MODES:
        rc, got = _run(L, mode, wires, sigmas, k_is, np.array([beta], dtype=np.uint64), np.array([gamma], dtype=np.uint64), D, 3)
        assert rc == 0 and np.array_equal(got, want)


def test_argument_errors(L):
    from plonky2_demo_b200 import _ffi

    wires, sigmas, k_is, betas, gammas, want = _case(7, 3, 3, 3)
    W, n = want.shape
    out = np.empty((W, n), dtype=np.uint64)
    pw, ps, po_ = _ffi.ptr_array(list(wires)), _ffi.ptr_array(list(sigmas)), _ffi.ptr_array(list(out))
    k, b, g = _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas)
    cases = [
        ((pw, ps, 7, 3, k, b, g, 3, 1, 0, po_), -5),      # quotient_degree_factor < 2
        ((pw, ps, 0, 3, k, b, g, 3, 3, 0, po_), -5),      # no routed wires
        ((pw, ps, 7, 3, k, b, g, 0, 3, 0, po_), -5),      # no challenges
        ((None, ps, 7, 3, k, b, g, 3, 3, 0, po_), -5),    # NULL wires
        ((pw, None, 7, 3, k, b, g, 3, 3, 0, po_), -5),
        ((pw, ps, 7, 3, None, b, g, 3, 3, 0, po_), -5),
        ((pw, ps, 7, 3, k, None, g, 3, 3, 0, po_), -5),
        ((pw, ps, 7, 3, k, b, None, 3, 3, 0, po_), -5),
        ((pw, ps, 7, 3, k, b, g, 3, 3, 0, None), -5),
        ((pw, ps, 7, 33, k, b, g, 3, 3, 0, po_), -6),     # lg_n > TWO_ADICITY
    ]
    nul = _ffi.ptr_array(list(wires))
    nul[3] = None
    cases.append(((nul, ps, 7, 3, k, b, g, 3, 3, 0, po_), -5))   # a NULL column
    for args, code in cases:
        assert L.pcs_permutation_partial_products(*args) == code, L.pcs_last_error()
        _normal_call_works(L)
