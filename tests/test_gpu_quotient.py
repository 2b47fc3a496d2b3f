"""pcs_quotient_polys (-m gpu): the quotient polynomials' chunks on the device against the CPU oracle
(tests/harness/quotient_oracle.c) element by element, on shapes up to the standard one (n = 2^20, 80 routed wires, 2 challenges,
D = 8, rate 3), with and without the caller's tail, from host and device tails into host and device outputs; the
device-resident chain wires -> Zs -> commitment #2 -> quotient chunks -> commitment #3 and the verifier's identity at an
extension-field point from the batches' openings; every argument error and the failed trim.

Every checked call follows a decoy call over the same batches with other challenges and another tail into the same outputs,
its temporaries freed in stream order: whatever the checked call fails to write then holds the decoy's values."""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness"))
import permutation_oracle as po  # noqa: E402
import quotient_oracle as qo  # noqa: E402
from helpers import Ext, dev_table, free, mem_available_bytes, noncanonical, torch_u64  # noqa: E402

pytestmark = pytest.mark.gpu

P = 0xFFFFFFFF00000001
MIN_HOST_MEM = 40 << 30   # the oracle's natural-order LDEs at the standard shape (12 GB) and the case's arrays
MIN_FREE_HBM = 24 << 30

SHAPES = [   # (R, lg_n, C, D, rate_bits, num_constants, wires_w, salt_w)
    (80, 3, 2, 8, 3, 0, 80, 0),      # m = 2 demo shape
    (80, 15, 2, 8, 3, 2, 135, 4),    # m = 64 demo shape: constants, a wider wires batch, salts
    (5, 2, 1, 8, 3, 0, 5, 0),        # P = 0
    (7, 4, 3, 4, 3, 1, 9, 4),        # q = 2 < rate_bits, short last chunk, salts
    (10, 10, 5, 4, 2, 0, 10, 0),     # five challenges: two passes over the inputs
    (9, 6, 2, 2, 2, 3, 12, 4),       # D = 2, q < rate_bits
    (20, 12, 6, 8, 4, 0, 20, 4),     # six challenges, q = 3 < rate_bits
    (80, 20, 2, 8, 3, 0, 80, 0),     # the standard shape
]
MODES = [("none", "host"), ("host", "host"), ("device", "device"), ("none", "device")]   # (tail, outputs)


def _m(lg_n, D):
    return (1 << lg_n) << (D - 1).bit_length()


class Case:
    """Coefficients of the three batches, the scalars and a tail, with the oracle's chunks with and without the tail."""

    def __init__(self, R, lg_n, C_, D, rate_bits, nc, wires_w, salt_w):
        rng = np.random.default_rng(R * 7919 + lg_n * 131 + C_ * 17 + D)
        n, N, M = 1 << lg_n, (1 << lg_n) << rate_bits, _m(lg_n, D)
        K = -(-R // D)
        self.shape = (R, lg_n, C_, D, rate_bits, nc, wires_w, salt_w)
        self.cs = rng.integers(0, P, (nc + R, n), dtype=np.uint64)
        self.wires = rng.integers(0, P, (wires_w, n), dtype=np.uint64)
        self.zs = rng.integers(0, P, (C_ * K, n), dtype=np.uint64)
        self.salts = [rng.integers(0, P, (salt_w, N), dtype=np.uint64) if salt_w else None for _ in range(3)]
        self.k_is, self.betas, self.gammas, self.alphas = (noncanonical(rng, s) for s in (R, C_, C_, C_))
        self.tail = noncanonical(rng, (C_, M))
        qo.use_all_cores()
        oracle.use_all_cores()
        lde = [oracle.coset_lde(c, rate_bits) for c in (self.cs, self.wires[:R], self.zs)]
        args = (rate_bits, nc, R, self.k_is, self.betas, self.gammas, self.alphas, D)
        self.want = {t: qo.quotient_poly_chunks(qo.compute_quotient_polys(*lde, *args, gate_terms=self.tail if t else None), n, D)
                     for t in (False, True)}


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

    rate_bits = case.shape[4]
    cap_h = min(4, case.shape[1] + rate_bits)
    return [p.PolynomialBatch.from_coeffs(c, rate_bits, s is not None, cap_h, salts=s)
            for c, s in zip((case.cs, case.wires, case.zs), case.salts)]


def _call(L, batches, case, betas, gammas, alphas, tail, out_tables, flags, D=None):
    from plonky2_demo_b200 import _ffi

    R, _, C_, D0, _, nc, _, _ = case.shape
    return L.pcs_quotient_polys(batches[0]._h, batches[1]._h, batches[2]._h, nc, R, _ffi.ptr(case.k_is), _ffi.ptr(betas),
                                _ffi.ptr(gammas), _ffi.ptr(alphas), C_, D0 if D is None else D, tail, flags, out_tables)


def _run(L, case, batches, tail_mode, out_mode):
    """decoy call, then the checked call into the same outputs -> (rc, [C D][n])"""
    import torch

    from plonky2_demo_b200 import _ffi

    R, lg_n, C_, D, _, _, _, _ = case.shape
    n, W = 1 << lg_n, C_ * D
    rng = np.random.default_rng(0xDEC0 + lg_n)
    decoy = [noncanonical(rng, C_) for _ in range(3)]
    decoy_tail = noncanonical(rng, case.tail.shape)
    flags = _ffi.PCS_DEVICE_PTRS if out_mode == "device" else 0
    if out_mode == "device":
        o = torch.zeros((W, n), dtype=torch.int64, device="cuda")
        outs = dev_table(list(o))
    else:
        o = np.full((W, n), 0xDEAD, dtype=np.uint64)
        outs = _ffi.ptr_array(list(o))
    if tail_mode == "device":
        t_dev, d_dev = torch_u64(case.tail), torch_u64(decoy_tail)
        tails, dtails = dev_table(list(t_dev)), dev_table(list(d_dev))
    elif tail_mode == "host":
        tails, dtails = _ffi.ptr_array(list(case.tail)), _ffi.ptr_array(list(decoy_tail))
    else:
        tails = dtails = None
    _call(L, batches, case, *decoy, dtails, outs, flags)   # may fail its trim: the outputs then hold whatever it left
    rc = _call(L, batches, case, case.betas, case.gammas, case.alphas, tails, outs, flags)
    if out_mode == "device":
        torch.cuda.synchronize()
        return rc, o.cpu().numpy().view(np.uint64)
    return rc, o


def _skip_if_short(shape):
    if shape[1] >= 20:
        if mem_available_bytes() < MIN_HOST_MEM:
            pytest.skip("not enough host memory for the oracle at the standard shape")
        import torch

        if torch.cuda.mem_get_info()[0] < MIN_FREE_HBM:
            pytest.skip("not enough free HBM")


@pytest.mark.parametrize("shape,mode", [(s, m) for s in SHAPES for m in MODES],
                         ids=[f"{'-'.join(map(str, s))}-{m[0]}-{m[1]}" for s in SHAPES for m in MODES])
def test_equals_oracle(L, shape, mode):
    _skip_if_short(shape)
    case = _case(shape)
    batches = _batches(case)
    try:
        rc, got = _run(L, case, batches, *mode)
    finally:
        free(*batches)
    assert rc == 0, L.pcs_last_error()
    want = case.want[mode[0] != "none"]
    assert got.shape == want.shape
    assert (got < np.uint64(P)).all()
    assert np.array_equal(got, want)


def test_python_api(L):
    import plonky2_demo_b200 as p

    case = _case(SHAPES[3])
    R, lg_n, C_, D, _, nc, _, _ = case.shape
    batches = _batches(case)
    args = (nc, R, case.k_is, case.betas, case.gammas, case.alphas, D)
    try:
        chunks = p.quotient_poly_chunks(*batches, *args, gate_terms=case.tail)
        full = p.compute_quotient_polys(*batches, *args)
    finally:
        free(*batches)
    assert np.array_equal(chunks, case.want[True])
    assert full.shape == (C_, _m(lg_n, D))
    assert np.array_equal(full[:, :D << lg_n].reshape(C_ * D, -1), case.want[False])
    assert not full[:, D << lg_n:].any()


# ---- extension-field arithmetic for the verifier's identity: F[X] / (X^2 - 7) ---------------------------------------------
def _openings(L, batch, z):
    from plonky2_demo_b200 import _ffi

    out = np.empty((batch.n_polys, 2), dtype=np.uint64)
    _ffi.check(L.pcs_batch_eval_ext(batch._h, _ffi.ptr(np.array([z.a, z.b], dtype=np.uint64)), _ffi.ptr(out)))
    return [Ext(int(a), int(b)) for a, b in out]


def test_device_resident_chain(L):
    """commitment #1 of the wire values, the Zs from device wire values into a device buffer, commitment #2 from it, the quotient chunks into a
    device buffer, commitment #3 from it with PCS_DEVICE_PTRS: its cap equals the oracle's commitment of the oracle's chunks,
    and the verifier's identity holds at an extension-field point with every opening taken from the batches."""
    import torch

    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi
    from test_permutation_oracle import copy_constrained_witness

    R, lg_n, C_, D, rate_bits, nc, cap_h = 20, 10, 2, 8, 3, 2, 4
    n, K = 1 << lg_n, -(-R // D)
    rng = np.random.default_rng(2024)
    wires, sigmas, k_is, _, _ = copy_constrained_witness(rng, R, lg_n, n_cycles=60)
    betas, gammas, alphas = (rng.integers(1, P, C_, dtype=np.uint64) for _ in range(3))
    consts = rng.integers(0, P, (nc, n), dtype=np.uint64)
    b_cs = p.PolynomialBatch.from_values(np.vstack([consts, sigmas]), rate_bits, False, cap_h)
    w_dev = torch_u64(wires)
    b_w = p.PolynomialBatch.from_values(wires, rate_bits, False, cap_h)   # commitment #1
    h2, h3 = C.c_void_p(), C.c_void_p()
    try:
        W = C_ * K
        zs_dev = torch.zeros((W, n), dtype=torch.int64, device="cuda")
        _ffi.check(L.pcs_permutation_partial_products(_ffi.dev_ptr_array(w_dev.data_ptr(), R, n),
                                                      _ffi.dev_ptr_array(torch_u64(sigmas).data_ptr(), R, n), R, lg_n,
                                                      _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas), C_, D,
                                                      _ffi.PCS_DEVICE_PTRS, _ffi.dev_ptr_array(zs_dev.data_ptr(), W, n)))
        _ffi.check(L.pcs_commit_from_values(_ffi.dev_ptr_array(zs_dev.data_ptr(), W, n), W, lg_n, rate_bits, cap_h, None, 0,
                                            _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS, None, None, C.byref(h2)))
        q_dev = torch.zeros((C_ * D, n), dtype=torch.int64, device="cuda")
        _ffi.check(L.pcs_quotient_polys(b_cs._h, b_w._h, h2, nc, R, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas),
                                        _ffi.ptr(alphas), C_, D, None, _ffi.PCS_DEVICE_PTRS,
                                        _ffi.dev_ptr_array(q_dev.data_ptr(), C_ * D, n)))
        cap3 = np.empty((1 << cap_h, 4), dtype=np.uint64)
        _ffi.check(L.pcs_commit_from_coeffs(_ffi.dev_ptr_array(q_dev.data_ptr(), C_ * D, n), C_ * D, lg_n, rate_bits, cap_h, None, 0,
                                            _ffi.PCS_DEVICE_PTRS | _ffi.PCS_KEEP_COEFFS, _ffi.ptr(cap3), C.byref(h3)))
        zs = po.prove_order(po.all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, D))
        lde = [oracle.coset_lde(oracle.fft(v, inverse=True), rate_bits) for v in (np.vstack([consts, sigmas]), wires, zs)]
        chunks = qo.quotient_poly_chunks(qo.compute_quotient_polys(*lde, rate_bits, nc, R, k_is, betas, gammas, alphas, D), n, D)
        assert np.array_equal(q_dev.cpu().numpy().view(np.uint64), chunks)
        assert np.array_equal(cap3, oracle.commit_from_coeffs(chunks, rate_bits, cap_h)["cap"])

        # vanishing(zeta) = Z_H(zeta) sum_k zeta^(k n) chunk_k(zeta), every value an opening of a committed batch
        zeta = Ext(int(rng.integers(2, P, dtype=np.uint64)), int(rng.integers(1, P, dtype=np.uint64)))
        g = pow(1753635133440165772, 1 << (32 - lg_n), P)
        zeta_g = zeta * g
        w_o, s_o = _openings(L, b_w, zeta)[:R], _openings(L, b_cs, zeta)[nc:nc + R]

        class _B:   # the raw commitment #2 / #3 handles
            def __init__(self, h, w):
                self._h, self.n_polys = h, w

        z_o, z_go = _openings(L, _B(h2, W), zeta), _openings(L, _B(h2, W), zeta_g)
        q_o = _openings(L, _B(h3, C_ * D), zeta)
        zn = zeta.pow(n)
        zh = zn - 1
        l_0 = zh * (Ext(n) * (zeta - 1)).inv()
        Pn = K - 1
        terms = [l_0 * (z_o[c] - 1) for c in range(C_)]
        for c in range(C_):
            b, gm = int(betas[c]), int(gammas[c])
            num = [w_o[j] + b * (int(k_is[j]) * zeta) + gm for j in range(R)]
            den = [w_o[j] + b * s_o[j] + gm for j in range(R)]
            acc, chain = z_o[c], z_o[C_ + c * Pn:C_ + (c + 1) * Pn] + [z_go[c]]
            for k in range(K):
                nk, dk = Ext(1), Ext(1)
                for v in num[k * D:(k + 1) * D]:
                    nk = nk * v
                for v in den[k * D:(k + 1) * D]:
                    dk = dk * v
                terms.append(acc * nk - chain[k] * dk)
                acc = chain[k]
        for a in range(C_):
            al = int(alphas[a])
            van = Ext(0)
            for t in reversed(terms):
                van = van * al + t
            tq, zk = Ext(0), Ext(1)
            for k in range(D):
                tq = tq + zk * q_o[a * D + k]
                zk = zk * zn
            assert van == zh * tq, a
        assert np.array_equal(w_dev.cpu().numpy().view(np.uint64), wires)
    finally:
        L.pcs_batch_free(h2)
        L.pcs_batch_free(h3)
        free(b_cs, b_w)


def _normal_call_works(L):
    case = _case(SHAPES[3])
    batches = _batches(case)
    try:
        rc, got = _run(L, case, batches, "host", "host")
    finally:
        free(*batches)
    assert rc == 0, L.pcs_last_error()
    assert np.array_equal(got, case.want[True])


def test_argument_errors(L):
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    case = _case(SHAPES[3])
    R, lg_n, C_, D, rate_bits, nc, wires_w, _ = case.shape
    n = 1 << lg_n
    bs = _batches(case)
    out = np.empty((C_ * 16, n), dtype=np.uint64)
    po_ = _ffi.ptr_array(list(out))
    k, b, g, a = (_ffi.ptr(v) for v in (case.k_is, case.betas, case.gammas, case.alphas))
    h = [x._h for x in bs]
    other_degree = p.PolynomialBatch.from_coeffs(np.ones((40, n * 2), dtype=np.uint64), rate_bits, False, 0)
    other_rate = p.PolynomialBatch.from_coeffs(np.ones((40, n), dtype=np.uint64), rate_bits + 1, False, 0)
    on_demand = p.PolynomialBatch.from_coeffs(case.wires, rate_bits, False, 0, lde_on_demand=True)
    shard = C.c_void_p()
    _ffi.check(L.pcs_commit_shard_from_coeffs(_ffi.ptr_array(list(case.wires)), wires_w, lg_n, rate_bits, 0, rate_bits - 1, 0,
                                              None, 0, 0, None, C.byref(shard)))
    rows_only = C.c_void_p()
    _ffi.check(L.pcs_shard_begin_rows(wires_w, 0, lg_n + rate_bits, 0, C.byref(rows_only)))
    null_out = _ffi.ptr_array(list(out))
    null_out[2] = None
    null_tail = _ffi.ptr_array(list(case.tail))
    null_tail[1] = None

    def args(**kw):
        d = dict(cs=h[0], w=h[1], z=h[2], nc=nc, R=R, k=k, b=b, g=g, a=a, C=C_, D=D, t=None, f=0, o=po_)
        d.update(kw)
        return tuple(d.values())

    cases = [
        args(D=1), args(R=0), args(C=0),
        args(cs=None), args(w=None), args(z=None), args(k=None), args(b=None), args(g=None), args(a=None), args(o=None),
        args(o=null_out), args(t=null_tail),
        args(D=16),                                  # q = 4 > rate_bits
        args(w=other_degree._h), args(z=other_rate._h),
        args(nc=nc + 2),                             # the sigmas would end past constants_sigmas
        args(R=wires_w + 1, k=_ffi.ptr(np.zeros(wires_w + 1, dtype=np.uint64))),
        args(C=C_ + 1, b=_ffi.ptr(np.zeros(C_ + 1, dtype=np.uint64)), g=_ffi.ptr(np.zeros(C_ + 1, dtype=np.uint64)),
             a=_ffi.ptr(np.zeros(C_ + 1, dtype=np.uint64))),   # zs_partial_products too narrow
        args(w=on_demand._h), args(w=shard), args(w=rows_only),
    ]
    try:
        for i, c in enumerate(cases):
            assert L.pcs_quotient_polys(*c) == -5, (i, L.pcs_last_error())
            _normal_call_works(L)
        assert L.pcs_quotient_polys(*args(D=16)) == -5
        assert L.pcs_last_error().startswith(b"Having constraints of degree higher than the rate is not supported yet")
    finally:
        L.pcs_batch_free(shard)
        L.pcs_batch_free(rows_only)
        free(*bs, other_degree, other_rate, on_demand)


@pytest.mark.parametrize("out_mode", ["host", "device"])
def test_trim_failure(L, out_mode):
    """random LDE rows at D = 5 (q = 3): the vanishing polynomial is not divisible by Z_H"""
    import plonky2_demo_b200 as p
    from plonky2_demo_b200 import _ffi

    R, lg_n, C_, D, rate_bits = 7, 6, 2, 5, 3
    n = 1 << lg_n
    rng = np.random.default_rng(55)
    coeffs = [rng.integers(0, P, (w, n), dtype=np.uint64) for w in (R, R, C_ * 2)]
    bs = [p.PolynomialBatch.from_coeffs(c, rate_bits, False, 0) for c in coeffs]
    k_is, betas, gammas, alphas = (rng.integers(0, P, s, dtype=np.uint64) for s in (R, C_, C_, C_))
    lde = [oracle.coset_lde(c, rate_bits) for c in coeffs]
    with pytest.raises(ValueError, match=qo.QUOTIENT_FAILED):
        qo.quotient_poly_chunks(qo.compute_quotient_polys(*lde, rate_bits, 0, R, k_is, betas, gammas, alphas, D), n, D)
    if out_mode == "device":
        import torch

        o = torch.zeros((C_ * D, n), dtype=torch.int64, device="cuda")
        outs, flags = dev_table(list(o)), _ffi.PCS_DEVICE_PTRS
    else:
        o = np.empty((C_ * D, n), dtype=np.uint64)
        outs, flags = _ffi.ptr_array(list(o)), 0
    try:
        rc = L.pcs_quotient_polys(bs[0]._h, bs[1]._h, bs[2]._h, 0, R, _ffi.ptr(k_is), _ffi.ptr(betas), _ffi.ptr(gammas),
                                  _ffi.ptr(alphas), C_, D, None, flags, outs)
    finally:
        free(*bs)
    assert rc == -5
    assert L.pcs_last_error() == b"Quotient has failed, the vanishing polynomial is not divisible by Z_H"
    _normal_call_works(L)
