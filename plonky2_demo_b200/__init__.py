"""B200-native polynomial-commitment engine for the Plonky2 matmul demo's prover hot path.

Host-side mirror (Python over the C ABI in include/pcs.h) of the reference's Rust interface for
ONE path: PolynomialBatch::from_values / from_coeffs (plonky2/src/fri/oracle.rs:43-98).
Names, argument meaning and error behaviour follow the reference:

    PolynomialValues / PolynomialCoeffs   field/src/polynomial/mod.rs:23,118
    fft_with_options / ifft_with_options  field/src/fft.rs:57,72
    PoseidonHash / PoseidonPermutation    plonky2/src/hash/poseidon.rs:637-719
    MerkleTree / MerkleCap / MerkleProof  plonky2/src/hash/merkle_tree.rs:18,39 ; merkle_proofs.rs:17
    FriConfig / FriParams                 plonky2/src/fri/mod.rs:19-103
    PolynomialBatch                       plonky2/src/fri/oracle.rs:30-159 (+ prove_openings :162-219)
    Challenger                            plonky2/src/iop/challenger.rs:16-160
    permutation Zs / partial products     plonky2/src/plonk/prover.rs (all_wires_permutation_partial_products)
    quotient polynomials / chunks         plonky2/src/plonk/prover.rs:576-744 (compute_quotient_polys, no gate constraints)
    gate constraints of the quotient step plonk/vanishing_poly.rs (evaluate_gate_constraints_base_batch), gates/*.rs
    FriInstanceInfo / FriProof            plonky2/src/fri/structure.rs, fri/proof.rs
    Buffer (write_/read_polynomial_batch, _merkle_tree, _fri_proof)   plonky2/src/util/serialization/mod.rs
    PoseidonGoldilocksConfig              plonky2/src/plonk/config.rs:101-108

All arithmetic runs in hand-written CUDA kernels (libpcs.so).  There is no CPU fallback: importing
works without a GPU (so that CPU-only checks can load the library and inspect its symbols), but
every compute call raises PcsError when no CUDA device is present.
"""
from ._ffi import LIB_PATH, SIGNATURES, PcsError, lib  # noqa: F401
from .config import CircuitConfig, PoseidonGoldilocksConfig  # noqa: F401
from .fri import FriConfig, FriParams, FriReductionStrategy, PolynomialBatch, SALT_SIZE, fri_proof_of_work  # noqa: F401
from .fri_prover import (  # noqa: F401
    Challenger,
    ExtensionPolynomial,
    FriBatchInfo,
    FriInstanceInfo,
    FriOracleInfo,
    FriPolynomialInfo,
    FriProof,
    OpeningSet,
    PlonkOpeningShape,
    eval_commitment,
    prove_openings,
)
from .hashing import (  # noqa: F401
    HashOut,
    MerkleCap,
    MerkleProof,
    MerkleTree,
    PoseidonHash,
    PoseidonPermutation,
    verify_merkle_proof_to_cap,
)
from .permutation import (  # noqa: F401
    all_wires_permutation_partial_products,
    get_unique_coset_shifts,
    wires_permutation_partial_products_and_zs,
    zs_partial_products_values,
)
from .gates import (  # noqa: F401
    ArithmeticGate,
    ConstantGate,
    NoopGate,
    PoseidonGate,
    PublicInputGate,
    SelectorsInfo,
    gate_constraint_terms,
)
from .quotient import compute_quotient_polys, quotient_poly_chunks  # noqa: F401
from .polynomial import (  # noqa: F401
    GOLDILOCKS_ORDER,
    PolynomialCoeffs,
    PolynomialValues,
    fft_with_options,
    ifft_with_options,
    log2_strict,
    reverse_bits,
    reverse_index_bits,
)
from .runtime import init, shutdown, stream, synchronize  # noqa: F401
from .serialization import Buffer, fri_proof_to_bytes, polynomial_batch_to_bytes  # noqa: F401

__all__ = [
    "PolynomialBatch", "PolynomialValues", "PolynomialCoeffs", "MerkleTree", "MerkleCap", "MerkleProof",
    "FriConfig", "FriParams", "FriReductionStrategy", "PoseidonGoldilocksConfig", "PoseidonHash",
    "PoseidonPermutation", "HashOut", "CircuitConfig", "fft_with_options", "ifft_with_options",
    "verify_merkle_proof_to_cap", "Challenger", "FriInstanceInfo", "FriBatchInfo", "FriPolynomialInfo", "FriOracleInfo",
    "FriProof", "OpeningSet", "PlonkOpeningShape", "ExtensionPolynomial", "eval_commitment", "prove_openings",
    "get_unique_coset_shifts", "wires_permutation_partial_products_and_zs", "all_wires_permutation_partial_products",
    "zs_partial_products_values", "compute_quotient_polys", "quotient_poly_chunks", "NoopGate", "ConstantGate", "PublicInputGate", "ArithmeticGate", "PoseidonGate",
    "SelectorsInfo", "gate_constraint_terms", "init", "shutdown", "synchronize", "PcsError",
]
