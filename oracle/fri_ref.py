"""ORACLE -- test infrastructure, NOT the product.

CPU restatement of the reference's FRI opening proof around a committed batch (SURVEY 8f N2 / N3): the protocol glue
in Python on top of the C arithmetic in oracle/fri.c.  Allowed importers: tests/, __graft_entry__.smoke(), bench.py.

Follows
  plonky2/src/iop/challenger.rs:16-160          Challenger (duplex sponge, overwrite mode)
  plonky2/src/plonk/proof.rs:316-322            eval_commitment
  plonky2/src/fri/oracle.rs:162-219             PolynomialBatch::prove_openings
  plonky2/src/fri/prover.rs:20-216              fri_proof, fri_committed_trees, fri_proof_of_work, query rounds
  plonky2/src/fri/challenges.rs:24-68           Challenger::fri_challenges
  plonky2/src/fri/verifier.rs:20-250            verify_fri_proof (compute_evaluation, fri_combine_initial, ...)
  field/src/interpolation.rs                    interpolate (restated as plain Lagrange interpolation: same value)

Parity: the reference holds no golden FRI proofs; this restatement is pinned by its own verifier accepting the
prover's output and rejecting tampered proofs (tests/test_fri_oracle.py), on top of the KAT-pinned Poseidon.
"""
import ctypes as C

import numpy as np

from . import P, _arr, _p, lib, merkle_build, merkle_prove, merkle_verify, poseidon, reverse_index_bits

u64p = C.POINTER(C.c_uint64)
COSET_SHIFT = 7           # F::MULTIPLICATIVE_GROUP_GENERATOR (goldilocks_field.rs:76)
RATE, WIDTH = 8, 12       # PoseidonPermutation (poseidon.rs:690-702)


def _fri_lib():
    L = lib()
    if not getattr(L, "_fri_ready", False):
        sz, u32, u64 = C.c_size_t, C.c_uint, C.c_uint64
        L.ref_ext_mul.argtypes = [u64p, u64p, u64p]
        L.ref_ext_mul.restype = None
        L.ref_ext_pow.argtypes = [u64p, u64, u64p]
        L.ref_ext_pow.restype = None
        L.ref_eval_base_polys_ext.argtypes = [u64p, sz, sz, u64p, u64p]
        L.ref_eval_base_polys_ext.restype = None
        L.ref_ext_poly_eval.argtypes = [u64p, sz, u64p, u64p]
        L.ref_ext_poly_eval.restype = None
        L.ref_reduce_polys_base.argtypes = [u64p, sz, sz, u64p, u64p]
        L.ref_reduce_polys_base.restype = None
        L.ref_ext_divide_by_linear.argtypes = [u64p, sz, u64p, u64p]
        L.ref_ext_divide_by_linear.restype = None
        L.ref_ext_scale_add.argtypes = [u64p, u64p, u64p, sz]
        L.ref_ext_scale_add.restype = None
        L.ref_ext_coset_lde.argtypes = [u64p, u32, u32, u64, u64p]
        L.ref_fri_fold.argtypes = [u64p, sz, sz, u64p, u64p]
        L.ref_fri_fold.restype = None
        L._fri_ready = True
    return L


def _e(x):
    return np.array([int(x[0]) % (1 << 64), int(x[1]) % (1 << 64)], dtype=np.uint64)


# ---- extension-field scalars (Python ints; quadratic.rs) ----------------------------------------------------------
def ext_mul(x, y):
    return ((x[0] * y[0] + 7 * x[1] * y[1]) % P, (x[0] * y[1] + x[1] * y[0]) % P)


def ext_add(x, y):
    return ((x[0] + y[0]) % P, (x[1] + y[1]) % P)


def ext_sub(x, y):
    return ((x[0] - y[0]) % P, (x[1] - y[1]) % P)


def ext_pow(x, e):
    acc, b = (1, 0), (x[0] % P, x[1] % P)
    while e:
        if e & 1:
            acc = ext_mul(acc, b)
        b = ext_mul(b, b)
        e >>= 1
    return acc


def ext_inv(x):
    """quadratic.rs:86-96 try_inverse: conjugate over the norm a^2 - 7 b^2."""
    norm = (x[0] * x[0] - 7 * x[1] * x[1]) % P
    ninv = pow(norm, P - 2, P)
    return (x[0] * ninv % P, (-x[1]) * ninv % P)


def c_ext_mul(x, y):
    out = np.empty(2, dtype=np.uint64)
    xx, yy = _e(x), _e(y)
    _fri_lib().ref_ext_mul(_p(xx), _p(yy), _p(out))
    return int(out[0]), int(out[1])


def c_ext_pow(x, e):
    out = np.empty(2, dtype=np.uint64)
    xx = _e(x)
    _fri_lib().ref_ext_pow(_p(xx), e, _p(out))
    return int(out[0]), int(out[1])


# ---- polynomial arithmetic (oracle/fri.c) ---------------------------------------------------------------------------
def eval_base_polys_ext(coeffs, z):
    """eval_commitment: [w][d] base coefficients at the extension point z -> [w][2]."""
    c = _arr(coeffs)
    w, d = c.shape
    out = np.empty((w, 2), dtype=np.uint64)
    zz = _e(z)
    _fri_lib().ref_eval_base_polys_ext(_p(c), w, d, _p(zz), _p(out))
    return out


def ext_poly_eval(coeffs, z):
    c = _arr(coeffs).reshape(-1, 2)
    out = np.empty(2, dtype=np.uint64)
    zz = _e(z)
    _fri_lib().ref_ext_poly_eval(_p(c), c.shape[0], _p(zz), _p(out))
    return int(out[0]), int(out[1])


def reduce_polys_base(polys, alpha):
    c = _arr(polys)
    k, d = c.shape
    out = np.empty((d, 2), dtype=np.uint64)
    a = _e(alpha)
    _fri_lib().ref_reduce_polys_base(_p(c), k, d, _p(a), _p(out))
    return out


def ext_divide_by_linear(coeffs, z):
    """divide_by_linear(z) padded back with one zero coefficient: [n][2] -> [n][2]."""
    c = _arr(coeffs).reshape(-1, 2)
    out = np.empty_like(c)
    zz = _e(z)
    _fri_lib().ref_ext_divide_by_linear(_p(c), c.shape[0], _p(zz), _p(out))
    return out


def ext_scale_add(acc, s, q):
    a = _arr(acc, copy=True).reshape(-1, 2)
    qq = _arr(q).reshape(-1, 2)
    ss = _e(s)
    _fri_lib().ref_ext_scale_add(_p(a), _p(ss), _p(qq), a.shape[0])
    return a


def ext_coset_lde(coeffs, rate_bits, shift=COSET_SHIFT):
    """p.lde(rate_bits).coset_fft(shift): [d][2] -> [d << rate_bits][2], natural order."""
    c = _arr(coeffs).reshape(-1, 2)
    d = c.shape[0]
    lg_d = d.bit_length() - 1
    assert 1 << lg_d == d
    out = np.empty((d << rate_bits, 2), dtype=np.uint64)
    assert _fri_lib().ref_ext_coset_lde(_p(c), lg_d, rate_bits, shift, _p(out)) == 0
    return out


def fri_fold(coeffs, arity, beta):
    c = _arr(coeffs).reshape(-1, 2)
    out = np.empty((c.shape[0] // arity, 2), dtype=np.uint64)
    b = _e(beta)
    _fri_lib().ref_fri_fold(_p(c), c.shape[0], arity, _p(b), _p(out))
    return out


def final_poly(oracle_coeffs, batches, alpha):
    """oracle.rs:171-200.  oracle_coeffs: list of [w_o][d] arrays; batches: [(point, [(oracle_index, poly_index)])]."""
    d = oracle_coeffs[0].shape[1]
    fin = np.zeros((d, 2), dtype=np.uint64)
    for point, polys in batches:
        o0, j0 = polys[0]
        if all(o == o0 and j == j0 + k for k, (o, j) in enumerate(polys)):
            rows = oracle_coeffs[o0][j0:j0 + len(polys)]     # a run of one oracle: a view, not a copy (18 GB at 135 x 2^24)
        else:
            rows = np.stack([oracle_coeffs[o][j] for o, j in polys])
        comp = reduce_polys_base(rows, alpha)
        quotient = ext_divide_by_linear(comp, point)
        fin = ext_scale_add(fin, ext_pow(alpha, len(polys)), quotient)
    return fin


# ---- Challenger (challenger.rs) -------------------------------------------------------------------------------------
class Challenger:
    def __init__(self):
        self.sponge_state = [0] * WIDTH
        self.input_buffer = []
        self.output_buffer = []

    def observe_element(self, e):
        self.output_buffer = []
        self.input_buffer.append(int(e) % P)
        if len(self.input_buffer) == RATE:
            self.duplexing()

    def observe_elements(self, es):
        for e in es:
            self.observe_element(e)

    def observe_extension_element(self, e):
        self.observe_elements([e[0], e[1]])

    def observe_extension_elements(self, es):
        for e in es:
            self.observe_extension_element(e)

    def observe_cap(self, cap):
        for h in np.asarray(cap).reshape(-1, 4):
            self.observe_elements([int(x) for x in h])

    def get_challenge(self):
        if self.input_buffer or not self.output_buffer:
            self.duplexing()
        return self.output_buffer.pop()

    def get_n_challenges(self, n):
        return [self.get_challenge() for _ in range(n)]

    def get_extension_challenge(self):
        a, b = self.get_n_challenges(2)
        return (a, b)

    def duplexing(self):
        assert len(self.input_buffer) <= RATE
        for i, v in enumerate(self.input_buffer):
            self.sponge_state[i] = v
        self.input_buffer = []
        st = poseidon(np.array(self.sponge_state, dtype=np.uint64))[0]
        self.sponge_state = [int(x) for x in st]
        self.output_buffer = self.sponge_state[:RATE]   # squeeze()

    def clone(self):
        c = Challenger()
        c.sponge_state = list(self.sponge_state)
        c.input_buffer = list(self.input_buffer)
        c.output_buffer = list(self.output_buffer)
        return c


# ---- prover (fri/prover.rs) ---------------------------------------------------------------------------------------
def fri_committed_trees(coeffs, values, challenger, reduction_arity_bits, rate_bits, cap_height):
    """prover.rs:69-112.  coeffs [N][2] (zero beyond N >> rate_bits), values [N][2] natural order."""
    trees = []
    shift = COSET_SHIFT
    coeffs = np.array(coeffs, dtype=np.uint64)
    values = np.array(values, dtype=np.uint64)
    betas = []
    for arity_bits in reduction_arity_bits:
        arity = 1 << arity_bits
        n = values.shape[0]
        idx = reverse_index_bits(np.arange(n, dtype=np.uint64)).astype(np.int64)
        rev = values[idx]                                  # reverse_index_bits_in_place (an involution)
        leaves = rev.reshape(n // arity, 2 * arity)       # chunks of `arity`, flatten()
        digests, cap = merkle_build(leaves, cap_height)
        challenger.observe_cap(cap)
        trees.append({"leaves": leaves, "digests": digests, "cap": cap, "cap_height": cap_height})
        beta = challenger.get_extension_challenge()
        betas.append(beta)
        coeffs = fri_fold(coeffs, arity, beta)
        shift = pow(shift, arity, P)
        values = ext_coset_lde(coeffs, 0, shift)           # coeffs.coset_fft(shift.into())
    final = coeffs[: coeffs.shape[0] >> rate_bits]
    challenger.observe_extension_elements([(int(a), int(b)) for a, b in final])
    return trees, final, betas


def fri_proof_of_work(challenger, proof_of_work_bits, limit=1 << 24):
    """prover.rs:115-160 with a single thread: the smallest witness."""
    min_lz = proof_of_work_bits + (64 - P.bit_length())
    state = list(challenger.sponge_state)
    for i, v in enumerate(challenger.input_buffer):
        state[i] = v
    pos = len(challenger.input_buffer)
    batch = 1 << 12
    witness = None
    for base in range(0, limit, batch):
        st = np.tile(np.array(state, dtype=np.uint64), (batch, 1))
        st[:, pos] = np.arange(base, base + batch, dtype=np.uint64)
        out = poseidon(st)
        resp = out[:, RATE - 1]                                 # squeeze().last()
        ok = np.nonzero(resp < (1 << (64 - min_lz)))[0] if min_lz else np.arange(batch)
        if ok.size:
            witness = base + int(ok[0])
            break
    assert witness is not None, "Proof of work failed. This is highly unlikely!"
    challenger.observe_element(witness)
    resp = challenger.get_challenge()
    assert resp < (1 << (64 - min_lz)) or min_lz == 0
    return witness


def prove_openings(oracles, batches, challenger, rate_bits, cap_height, reduction_arity_bits, proof_of_work_bits,
                   num_query_rounds):
    """oracle.rs:162-219 + prover.rs:20-67.  oracles: list of dicts (coeffs [w][d], leaves [N][w+s], digests, cap,
    cap_height) as the commit oracle returns them.  An oracle whose leaves are too large to hold may give callables
    instead: rows(i) -> leaf i, path(i) -> its Merkle path ([depth][4]); its leaves / digests are then not read.
    Returns the FriProof as a dict."""
    alpha = challenger.get_extension_challenge()
    fin = final_poly([o["coeffs"] for o in oracles], batches, alpha)
    d = fin.shape[0]
    n = d << rate_bits
    lde_coeffs = np.zeros((n, 2), dtype=np.uint64)
    lde_coeffs[:d] = fin                                        # final_poly.lde(rate_bits)
    lde_values = ext_coset_lde(fin, rate_bits, COSET_SHIFT)
    trees, final_coeffs, betas = fri_committed_trees(lde_coeffs, lde_values, challenger, reduction_arity_bits, rate_bits,
                                                     cap_height)
    pow_witness = fri_proof_of_work(challenger, proof_of_work_bits)
    lg_n = n.bit_length() - 1
    rounds = []
    indices = []
    for rand in challenger.get_n_challenges(num_query_rounds):
        x_index = rand % n
        indices.append(x_index)
        initial = []
        for o in oracles:
            if "rows" in o:
                initial.append((np.asarray(o["rows"](x_index), dtype=np.uint64), np.asarray(o["path"](x_index))))
                continue
            lv = np.asarray(o["leaves"])
            initial.append((lv[x_index].copy(), merkle_prove(o["digests"], lv.shape[0], o["cap_height"], x_index)))
        steps = []
        xi = x_index
        for i, t in enumerate(trees):
            ab = reduction_arity_bits[i]
            steps.append({"evals": t["leaves"][xi >> ab].reshape(-1, 2).copy(),
                          "merkle_proof": merkle_prove(t["digests"], t["leaves"].shape[0], t["cap_height"], xi >> ab)})
            xi >>= ab
        rounds.append({"initial_trees_proof": initial, "steps": steps})
    return {
        "commit_phase_merkle_caps": [t["cap"] for t in trees],
        "query_round_proofs": rounds,
        "final_poly": final_coeffs,
        "pow_witness": pow_witness,
        # not part of FriProof: exposed for parity checks of the intermediate values
        "_alpha": alpha, "_betas": betas, "_final_poly_full": fin, "_lde_values": lde_values, "_indices": indices,
        "_lg_n": lg_n,
    }


# ---- verifier (fri/verifier.rs, fri/challenges.rs) --------------------------------------------------------------------
def reverse_bits(x, bits):
    return int(format(x, f"0{bits}b")[::-1], 2) if bits else 0


def primitive_root_of_unity(lg):
    g = 1753635133440165772
    for _ in range(lg, 32):
        g = g * g % P
    return g


def compute_evaluation(x, x_index_within_coset, arity_bits, evals, beta):
    """verifier.rs:20-46: P'(x^arity) by interpolating {(x g^i, P(x g^i))} and evaluating at beta."""
    arity = 1 << arity_bits
    g = primitive_root_of_unity(arity_bits)
    ev = [evals[reverse_bits(i, arity_bits)] for i in range(arity)]
    rev = reverse_bits(x_index_within_coset, arity_bits)
    coset_start = x * pow(g, arity - rev, P) % P
    pts = [(coset_start * pow(g, i, P) % P, 0) for i in range(arity)]
    # Lagrange interpolation at beta (interpolation.rs computes the same value with barycentric weights)
    total = (0, 0)
    for i in range(arity):
        num, den = (1, 0), (1, 0)
        for j in range(arity):
            if j != i:
                num = ext_mul(num, ext_sub(beta, pts[j]))
                den = ext_mul(den, ext_sub(pts[i], pts[j]))
        total = ext_add(total, ext_mul(ev[i], ext_mul(num, ext_inv(den))))
    return total


def verify_fri_proof(batches, openings, challenger, initial_caps, proof, rate_bits, cap_height, reduction_arity_bits,
                     proof_of_work_bits, num_query_rounds, degree_bits):
    """verifier.rs:61-250 with the challenges re-derived as challenges.rs:24-68 does.
    openings: per batch, the list of opened extension values (FriOpenings).  The challenger must be in the state the
    prover's was in when prove_openings started.  Raises AssertionError when the proof does not verify."""
    n = 1 << (degree_bits + rate_bits)
    lg_n = degree_bits + rate_bits
    alpha = challenger.get_extension_challenge()
    betas = []
    for cap in proof["commit_phase_merkle_caps"]:
        challenger.observe_cap(cap)
        betas.append(challenger.get_extension_challenge())
    challenger.observe_extension_elements([(int(a), int(b)) for a, b in np.asarray(proof["final_poly"]).reshape(-1, 2)])
    challenger.observe_element(proof["pow_witness"])
    pow_response = challenger.get_challenge()
    indices = [challenger.get_challenge() % n for _ in range(num_query_rounds)]
    # validate_fri_proof_shape (the parts that matter here)
    assert len(proof["commit_phase_merkle_caps"]) == len(reduction_arity_bits)
    assert np.asarray(proof["final_poly"]).reshape(-1, 2).shape[0] == (1 << degree_bits) >> sum(reduction_arity_bits)
    assert len(proof["query_round_proofs"]) == num_query_rounds, "Number of query rounds does not match config."
    min_lz = proof_of_work_bits + (64 - P.bit_length())
    assert min_lz == 0 or pow_response < (1 << (64 - min_lz)), "Invalid proof of work witness."
    # PrecomputedReducedOpenings::from_os_and_alpha: ReducingFactor::reduce = sum_j alpha^j v_j
    reduced_openings = []
    for vals in openings:
        acc = (0, 0)
        for v in reversed(vals):
            acc = ext_add(ext_mul(acc, alpha), (int(v[0]), int(v[1])))
        reduced_openings.append(acc)
    for x_index, rp in zip(indices, proof["query_round_proofs"]):
        for (evals, mp), cap in zip(rp["initial_trees_proof"], initial_caps):
            assert merkle_verify(evals, x_index, cap, mp), "initial Merkle proof"
        subgroup_x = COSET_SHIFT * pow(primitive_root_of_unity(lg_n), reverse_bits(x_index, lg_n), P) % P
        # fri_combine_initial
        total = (0, 0)
        for (point, polys), red in zip(batches, reduced_openings):
            acc = (0, 0)
            for o, j in reversed(polys):
                acc = ext_add(ext_mul(acc, alpha), (int(rp["initial_trees_proof"][o][0][j]), 0))
            numerator = ext_sub(acc, red)
            denominator = ext_sub((subgroup_x, 0), (point[0] % P, point[1] % P))
            total = ext_mul(total, ext_pow(alpha, len(polys)))      # alpha.shift(sum)
            total = ext_add(total, ext_mul(numerator, ext_inv(denominator)))
        old_eval = total
        xi = x_index
        for i, ab in enumerate(reduction_arity_bits):
            arity = 1 << ab
            evals = [(int(a), int(b)) for a, b in np.asarray(rp["steps"][i]["evals"]).reshape(-1, 2)]
            coset_index, within = xi >> ab, xi & (arity - 1)
            assert evals[within] == old_eval, "fold consistency"
            old_eval = compute_evaluation(subgroup_x, within, ab, evals, betas[i])
            flat = np.asarray(rp["steps"][i]["evals"], dtype=np.uint64).reshape(-1)
            assert merkle_verify(flat, coset_index, proof["commit_phase_merkle_caps"][i], rp["steps"][i]["merkle_proof"]), \
                "commit-phase Merkle proof"
            subgroup_x = pow(subgroup_x, arity, P)
            xi = coset_index
        assert ext_poly_eval(proof["final_poly"], (subgroup_x, 0)) == old_eval, "Final polynomial evaluation is invalid."
    return True
