"""The per-thread permutation kernel (k_permute: more than COOP_MAX_PERMS = 8192 states per call) on the reference KATs
and on states whose partial rounds start from chosen values (built backwards in test_partial_crt), against the
reference's outputs and the oracle.  Fewer states than that take the half-warp form, which does not run poseidon12."""
import numpy as np
import pytest

import oracle
from test_partial_crt import chosen_partial_entry_states, state_entering_partial_rounds

pytestmark = pytest.mark.gpu

N = 8192 + 1000


@pytest.fixture(scope="module")
def pcs():
    import plonky2_demo_b200 as p

    p.init(0)
    yield p
    p.shutdown()


def _tile(x):
    return np.tile(x, (N // len(x) + 1, 1))[:N]


def test_reference_kats_on_the_per_thread_kernel(pcs, golden):
    from plonky2_demo_b200.hashing import poseidon

    kats = golden["kats"]["poseidon12_kats"] + golden["kats"]["poseidon12_extra_bigint"]
    x = _tile(np.array([k["input"] for k in kats], dtype=np.uint64))
    y = _tile(np.array([k["output"] for k in kats], dtype=np.uint64))
    assert np.array_equal(poseidon(x), y)


def test_chosen_partial_entry_states_on_the_per_thread_kernel(pcs):
    from plonky2_demo_b200.hashing import poseidon

    x = _tile(np.array([state_entering_partial_rounds(t) for t in chosen_partial_entry_states()], dtype=np.uint64))
    assert np.array_equal(poseidon(x), oracle.poseidon(x))
