/*
 * pcs.h -- C ABI of the B200 polynomial-commitment engine (libpcs.so).
 *
 * Drop-in boundary for ONE hot path of Lain-Iwakuro/Plonky2-Demo:
 *     PolynomialBatch::from_values / from_coeffs      plonky2/src/fri/oracle.rs:43-98
 *       = batched Goldilocks coset LDE                field/src/fft.rs:57-206, field/src/polynomial/mod.rs:201-295
 *       + transpose / reverse_index_bits              plonky2/src/util/mod.rs:22-28, util/src/lib.rs:188-237
 *       + MerkleTree::new (Poseidon)                  plonky2/src/hash/merkle_tree.rs:135-166
 * The reference has no FFI: its boundary is the generic Rust API.  These entry points are what
 * a Rust `-sys` crate binds so that the shim's from_values / from_coeffs / MerkleTree::new / get /
 * prove (INTEGRATION.md) forward here for F = GoldilocksField, H = PoseidonHash.
 *
 * Conventions
 *   - Field elements are uint64_t.  GoldilocksField is #[repr(transparent)] over u64
 *     (field/src/goldilocks_field.rs:23-25) so Vec<GoldilocksField> == const uint64_t*.
 *     Inputs may be non-canonical (any u64); every output is canonical (< p).
 *   - HashOut<F> == uint64_t[4] (plonky2/src/hash/hash_types.rs:22-24), Vec<HashOut> == flat u64[4n].
 *   - All pointers are HOST pointers unless the PCS_DEVICE_PTRS flag is given or the name ends in _dev.
 *   - Every function returns 0 on success or a negative pcs_status; pcs_last_error() has the text.
 *     The reference panics on invalid input; the Rust shim turns non-zero into panic!() with the
 *     reference's message (INTEGRATION.md).
 *   - There is NO CPU fallback: without a CUDA device every compute entry point fails with PCS_ERR_CUDA.
 *   - Contexts: the engine keeps one context (stream, staging buffers, twiddle tables) per CUDA device.  The
 *     single-device entry points act on the calling thread's CURRENT context = the device of its last pcs_init
 *     (device 0 by default); a batch remembers the context that made it, so its accessors and pcs_batch_free run on the
 *     right device whatever is current.  One call in flight per context (the reference's call sites are sequential:
 *     plonk/prover.rs:145,212,260; circuit_builder.rs:1021); different contexts may be driven from different host
 *     threads at the same time (that is how pcs_multi_* uses a whole box).
 */
#ifndef PCS_H
#define PCS_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define PCS_API __attribute__((visibility("default")))
#else
#define PCS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    PCS_OK = 0,
    PCS_ERR_CUDA = -1,         /* CUDA runtime error (incl. "no device")                                  */
    PCS_ERR_NOT_POW2 = -2,     /* "Not a power of two: {n}"                       util/src/lib.rs:37      */
    PCS_ERR_CAP_HEIGHT = -3,   /* "cap_height={} should be at most log2(leaves.len())={}" merkle_tree.rs:136-142 */
    PCS_ERR_ALLOC = -4,
    PCS_ERR_ARG = -5,          /* empty batch (oracle.rs:76 polynomials[0]), unequal lengths (oracle.rs:114), NULL */
    PCS_ERR_TWO_ADICITY = -6,  /* log2(N) > 32                                    field/src/types.rs:269  */
    PCS_ERR_NOT_INIT = -7
} pcs_status;

enum {
    PCS_DEVICE_PTRS = 1u << 0,   /* input polynomial pointers are device pointers (no H2D copy)         */
    PCS_KEEP_COEFFS = 1u << 1,   /* keep the coefficient vectors on the device (PolynomialBatch.polynomials) */
    PCS_MULTI_CE_GATHER = 1u << 2,   /* pcs_multi_*: exchange by copy-engine gathers instead of peer loads inside the first NTT pass (slower; kept for A/B) */
    PCS_LDE_ON_DEMAND = 1u << 3      /* pcs_commit_from_coeffs / _from_values: keep no LDE rows in HBM.  The LDE is extended and
                                      * hashed a few columns at a time through a reused scratch buffer; the batch keeps the
                                      * coefficients (implies PCS_KEEP_COEFFS: device inputs are copied), salts, digests and
                                      * cap, about 1 / (2^rate_bits + 1) of a resident batch's HBM plus the salt rows.  The
                                      * commitment is bit-identical.  pcs_batch_get_rows, pcs_batch_leaves and
                                      * pcs_batch_lde_natural recompute the rows they return (few rows: evaluated from the
                                      * coefficients; many: the LDE regenerated group by group); pcs_batch_lde_dev returns NULL.
                                      * Refused (PCS_ERR_ARG) by the shard and pcs_multi_* commits. */
};

/* ---- lifetime ------------------------------------------------------------------------------- */
/* Select the CUDA device this process commits on and create the engine's stream.
 * `stream` may be NULL (the engine creates its own) or an existing cudaStream_t the caller owns
 * (e.g. torch's current stream) so that caller-side CUDA events time the engine's kernels. */
PCS_API int pcs_init(int device, void* stream);
/* The CUDA device of the calling thread's current context, or -1 before pcs_init. */
PCS_API int pcs_device(void);
/* Destroys every context (all devices) and the multi-GPU state; batches must have been freed. */
PCS_API void pcs_shutdown(void);
PCS_API const char* pcs_last_error(void);
/* The cudaStream_t all engine work is enqueued on. */
PCS_API void* pcs_stream(void);
PCS_API int pcs_synchronize(void);

/* ---- primitives (unit-testable against the reference's own tests) ------------------------------ */
/* Element-wise GoldilocksField arithmetic on the device: out[i] = a[i] (op) b[i], any u64 in, canonical out -- the
 * device counterpart of the field grid test, field/src/prime_field_testing.rs:78-125.  b may be NULL for unary ops.  */
typedef enum {
    PCS_OP_ADD = 0,       /* goldilocks_field.rs:199-221                                              */
    PCS_OP_SUB = 1,       /* :223-243                                                                 */
    PCS_OP_MUL = 2,       /* :267-274, reduce128 :356-369 (the kernels' reduction); 3 is unused       */
    PCS_OP_SQUARE = 4,
    PCS_OP_CANON = 5,     /* to_canonical_u64 :171-178                                                */
    PCS_OP_NEG = 6,       /* :245-255                                                                 */
    PCS_OP_REDUCE96 = 7,  /* a + (b mod 2^32) * 2^64, reduce96 :347-354                               */
    PCS_OP_MUL_2EXP = 8   /* a * 2^b                                                                  */
} pcs_field_op_kind;
PCS_API int pcs_field_op(int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out);
/* Poseidon::poseidon on n states, in place.                      plonky2/src/hash/poseidon.rs:599-609 */
PCS_API int pcs_poseidon_permute(uint64_t* states /*[n][12]*/, size_t n);
/* fri_proof_of_work: smallest witness w in 0..p-1 such that, with w written to lane `witness_pos` of the duplex
 * intermediate `state` (sponge state overwritten with the pending challenger inputs), the permuted state's last rate
 * lane has >= min_leading_zeros leading zeros.  The reference searches with rayon find_any (any hit; the smallest one
 * with a single thread, which is how the demo runs).                plonky2/src/fri/prover.rs:115-160        */
PCS_API int pcs_pow_grind(const uint64_t* state /*[12]*/, unsigned witness_pos, unsigned min_leading_zeros, uint64_t* witness);
/* Hasher::hash_or_noop on n rows of `len` elements.               plonky2/src/plonk/config.rs:55-66   */
PCS_API int pcs_hash_or_noop(const uint64_t* rows /*[n][len]*/, size_t n, size_t len, uint64_t* out /*[n][4]*/);
/* PoseidonHash::two_to_one = compress.                            plonky2/src/hash/hashing.rs:98-115  */
PCS_API int pcs_two_to_one(const uint64_t* left /*[n][4]*/, const uint64_t* right /*[n][4]*/, size_t n, uint64_t* out);
/* fft_with_options(.., None, ..) / ifft_with_options on w polynomials, natural order in and out.
 *                                                                 field/src/fft.rs:57-65, 72-95       */
PCS_API int pcs_ntt(uint64_t* polys /*[w][n] in/out*/, size_t w, unsigned lg_n, int inverse);
/* PolynomialValues::coset_ifft(shift) on w value vectors (natural order): coefficients of the polynomial whose
 * evaluations on shift*<w_n> are given -- what compute_quotient_polys ends with (plonk/prover.rs:739-743).
 *                                                                 field/src/polynomial/mod.rs:63-73   */
PCS_API int pcs_coset_intt(uint64_t* values /*[w][n] in/out*/, size_t w, unsigned lg_n, uint64_t shift);
/* The same transform in place on a DEVICE matrix [w][n] (natural order in and out), asynchronous on
 * pcs_stream(): the per-GPU IFFT of a polynomial-partitioned from_values (SURVEY 8e).                */
PCS_API int pcs_ntt_dev(uint64_t* polys_dev, size_t w, unsigned lg_n, int inverse);
/* pcs_coset_intt in place on a DEVICE matrix [w][n], asynchronous on pcs_stream(): the quotient polynomials'
 * coset_ifft (plonk/prover.rs:739-743) when their values were computed on, or already copied to, the device.  */
PCS_API int pcs_coset_intt_dev(uint64_t* values_dev, size_t w, unsigned lg_n, uint64_t shift);
/* PolynomialBatch::lde_values (no salts): p.lde(rate_bits).coset_fft_with_options(shift, Some(rate_bits), ..)
 * for every polynomial.                                           plonky2/src/fri/oracle.rs:100-118
 * layout 0: out[w][N] natural order (== the reference's Vec<Vec<F>>);
 * layout 1: out[N][w] leaf order (== transpose + reverse_index_bits_in_place, oracle.rs:83-84).       */
PCS_API int pcs_coset_lde(const uint64_t* const* coeffs /*w pointers, d elements each*/, size_t w, unsigned lg_d,
                  unsigned rate_bits, uint64_t shift, uint64_t* out, int layout);
/* The same LDE entirely on the device (BASELINE configs[2], "standalone batched coset LDE"): w DEVICE pointers to d
 * coefficients each -> out_dev [w][N] poly-major in LEAF order (coset block c = evaluations on shift*w_N^brev(c)*<w_d>
 * in bit-reversed order at [c*d, (c+1)*d)), asynchronous on pcs_stream().                              */
PCS_API int pcs_coset_lde_dev(const uint64_t* const* coeffs_dev, size_t w, unsigned lg_d, unsigned rate_bits,
                      uint64_t shift, uint64_t* out_dev);
/* MerkleTree::new(leaves, cap_height).                            plonky2/src/hash/merkle_tree.rs:135-166
 * leaves row-major [n][len]; digests [2(n - 2^cap_height)][4] in the reference's interleaved layout
 * (merkle_tree.rs:43-51); cap [2^cap_height][4].                                                      */
PCS_API int pcs_merkle_build(const uint64_t* leaves, size_t n, size_t len, unsigned cap_height, uint64_t* digests,
                     uint64_t* cap);

/* ---- the fused hot path ------------------------------------------------------------------------- */
/* Opaque device-resident PolynomialBatch: coefficients (optional), LDE in leaf order (poly-major),
 * digests and cap all stay in HBM; the accessors below serve the reference's consumers. */
typedef struct pcs_batch pcs_batch;

/* PolynomialBatch::from_coeffs(polynomials, rate_bits, blinding, cap_height, ..)  oracle.rs:68-98.
 *   polys   : w pointers to d = 2^lg_d coefficients each (all the same length, oracle.rs:114)
 *   salts   : NULL, or salt_w pointers to N = d << rate_bits elements each -- the reference draws
 *             SALT_SIZE = 4 columns from OsRng when `blinding` (oracle.rs:26,119-123); the caller
 *             supplies them so that the commitment is reproducible.
 *   cap_out : NULL or [2^cap_height][4] host buffer, filled before return (the only D2H copy).
 * With PCS_DEVICE_PTRS the call is asynchronous on pcs_stream() unless cap_out != NULL.           */
PCS_API int pcs_commit_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits,
                           unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                           uint64_t* cap_out, pcs_batch** out);
/* One SHARD of from_coeffs for a commitment spread over several GPUs (one process per GPU; SURVEY 8e).
 * In leaf order the LDE is 2^rate_bits coset blocks of d leaves each (block c = evaluations on the coset
 * 7 * w_N^{brev(c)} <w_d>), so a contiguous leaf range [coset_first*d, (coset_first + 2^lg_cosets)*d) needs
 * only the coefficients: this call extends exactly those cosets and builds the Merkle subtrees over them.
 *   local_cap_height : cap height of the LOCAL tree = cap_height - log2(n_shards); the local cap is the
 *                      slice cap[shard*2^local_cap_height ..] of the reference's cap, the local digests the
 *                      matching contiguous slice of the reference's digests (merkle_tree.rs:43-46).
 *   salts            : NULL, or salt_w pointers to the shard's d << lg_cosets salt values in LEAF order.
 * The batch accessors then address leaves relative to the shard.                                     */
PCS_API int pcs_commit_shard_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits,
                                 unsigned coset_first, unsigned lg_cosets, unsigned local_cap_height,
                                 const uint64_t* const* salts, size_t salt_w, unsigned flags, uint64_t* cap_out,
                                 pcs_batch** out);
/* The same shard commit with the polynomials arriving in groups (DEVICE pointers, contiguous or scattered, possibly in
 * peer memory): begin allocates the shard, every extend runs the coset LDE of polynomials [poly_first, poly_first+count)
 * asynchronously on pcs_stream() -- e.g. while the next chunk of an all-gather or H2D copy is still in flight -- and
 * finish hashes the leaves, builds the subtrees and returns the local cap.  Every polynomial must be supplied once. */
PCS_API int pcs_shard_begin(size_t w, size_t salt_w, unsigned lg_d, unsigned rate_bits, unsigned coset_first, unsigned lg_cosets,
                    unsigned local_cap_height, pcs_batch** out);
PCS_API int pcs_shard_extend(pcs_batch* b, size_t poly_first, size_t count, const uint64_t* const* polys_dev);
PCS_API int pcs_shard_finish(pcs_batch* b, uint64_t* cap_out /*NULL or [2^local_cap_height][4]*/);
/* A shard whose LDE rows are computed ELSEWHERE -- the north-star's other partition: every GPU extends its own block of
 * polynomials over all cosets and the rows travel (all-to-all over NVLink) to the GPU that hashes their leaf range.
 * `width` columns (the last salt_w of them salts) of 2^lg_n leaves; fill them with pcs_shard_set_rows or write them in
 * place at pcs_batch_lde_dev(b) + row * 2^lg_n, then pcs_shard_finish.  Leaf ranges need not be whole cosets, so this
 * form also serves more GPUs than 2^rate_bits.                                                                     */
PCS_API int pcs_shard_begin_rows(size_t width, size_t salt_w, unsigned lg_n, unsigned local_cap_height, pcs_batch** out);
/* Rows [row_first, row_first + count) of a begun shard <- count DEVICE pointers to 2^lg_n values each, already in LEAF
 * order (salt columns of a shard: row_first = w; received LDE rows).  canonical != 0: the values are known to be < p
 * (the engine's own LDE output) and are not canonicalised again.  Asynchronous on pcs_stream().                    */
PCS_API int pcs_shard_set_rows(pcs_batch* b, size_t row_first, size_t count, const uint64_t* const* rows_dev, int canonical);
/* PolynomialBatch::from_values: IFFT every column first.                         oracle.rs:43-65
 *   coeffs_out : NULL, or w host pointers receiving the d coefficients of each polynomial
 *                (the reference keeps them as `polynomials`).                                      */
PCS_API int pcs_commit_from_values(const uint64_t* const* values, size_t w, unsigned lg_d, unsigned rate_bits,
                           unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                           uint64_t* const* coeffs_out, uint64_t* cap_out, pcs_batch** out);

/* Shape of a batch: n_leaves = N, leaf_len = w + salt_w, n_digests = 2 (N - 2^cap_height). */
PCS_API int pcs_batch_shape(const pcs_batch* b, size_t* n_leaves, size_t* leaf_len, size_t* n_digests, unsigned* cap_height);
/* merkle_tree.cap                                                                                   */
PCS_API int pcs_batch_cap(const pcs_batch* b, uint64_t* cap /*[2^cap_height][4]*/);
/* merkle_tree.digests (reference layout)                                                            */
PCS_API int pcs_batch_digests(const pcs_batch* b, uint64_t* digests /*[n_digests][4]*/);
/* merkle_tree.leaves[first .. first+count) as row-major [count][leaf_len] (transposed on the device). */
PCS_API int pcs_batch_leaves(const pcs_batch* b, size_t first, size_t count, uint64_t* rows);
/* MerkleTree::get for many indices at once (merkle_tree.rs:168); get_lde_values(i, step) is
 * leaf index reverse_bits(i*step, log2 N) minus the salt columns (oracle.rs:128-133).              */
PCS_API int pcs_batch_get_rows(const pcs_batch* b, const uint64_t* leaf_indices, size_t n, uint64_t* rows /*[n][leaf_len]*/);
/* get_lde_values(index_start + k, step) for k = 0 .. count-1 in ONE call: rows[k][0..w) = the LDE values of every
 * polynomial at the (index_start + k) * step -th point of the NATURAL-order domain, salt columns dropped
 * (oracle.rs:128-133: leaf reverse_bits(index * step, log2 N)); step is a power of two.  This is the access pattern of
 * compute_quotient_polys (plonk/prover.rs:576-744: batches of 32 consecutive points through get_lde_values_packed,
 * oracle.rs:137-159) -- one call per oracle can serve the whole loop, or a window of it.  Rows are gathered on the device
 * and streamed to the host in 16 MB pieces through pinned double buffering.                                        */
PCS_API int pcs_batch_lde_natural(const pcs_batch* b, size_t index_start, size_t step, size_t count, uint64_t* rows /*[count][w]*/);
/* MerkleTree::prove(leaf_index): siblings bottom-up, [log2 N - cap_height][4].  merkle_tree.rs:173-207 */
PCS_API int pcs_batch_prove(const pcs_batch* b, size_t leaf_index, uint64_t* siblings);
/* The same for n leaves in one call: siblings [n][log2 N - cap_height][4] (the FRI query phase asks every tree for
 * num_query_rounds paths, fri/prover.rs:162-216).                                                    */
PCS_API int pcs_batch_prove_many(const pcs_batch* b, const uint64_t* leaf_indices, size_t n, uint64_t* siblings);
/* polynomials[i].coeffs (needs PCS_KEEP_COEFFS or from_values).                                     */
PCS_API int pcs_batch_coeffs(const pcs_batch* b, size_t poly, uint64_t* coeffs /*[d]*/);
/* All of `polynomials` at once as one [w][d] matrix.                                                  */
PCS_API int pcs_batch_all_coeffs(const pcs_batch* b, uint64_t* coeffs /*[w][d]*/);
/* Device views (valid until pcs_batch_free): LDE is [leaf_len][N] poly-major in leaf order, NULL for a batch committed
 * with PCS_LDE_ON_DEMAND (it keeps no LDE rows).                                                    */
PCS_API const uint64_t* pcs_batch_lde_dev(const pcs_batch* b);
PCS_API const uint64_t* pcs_batch_coeffs_dev(const pcs_batch* b);   /* [w][d], or NULL when the coefficients were not kept */
PCS_API const uint64_t* pcs_batch_digests_dev(const pcs_batch* b);
PCS_API const uint64_t* pcs_batch_cap_dev(const pcs_batch* b);
/* Wall-clock of the last commit's phases in ms, measured with CUDA events on pcs_stream():
 * [0] "IFFT"  [1] "FFT + blinding"  [2] "transpose LDEs" (always 0: fused away)
 * [3] leaf hashing  [4] node levels   ([3]+[4] = "build Merkle tree")   -- TimingTree scopes, oracle.rs:51-89.
 * Synchronises the stream.                                                                         */
PCS_API int pcs_batch_timings(const pcs_batch* b, float ms[5]);
PCS_API void pcs_batch_free(pcs_batch* b);
/* Phase times (same five slots as pcs_batch_timings) summed over every batch freed since the last
 * reset, and how many batches that was; lets a caller free each batch immediately (so the next
 * commit reuses its HBM) and still read per-kernel times afterwards.  Synchronises the stream. */
PCS_API int pcs_timing_totals(float ms[5], unsigned* n_commits, int reset);

/* ---- one commitment over several GPUs of this box from ONE host process (SURVEY 5 / 8e) -----------------------------
 * The reference's caller is a single Rust thread (prove(), plonk/prover.rs:145,212,260); these entry points let it use a
 * whole 8 x B200 box without a process per GPU: the library keeps a context and a worker thread per device, device g
 * extends and hashes the coset blocks [g 2^r / G, (g+1) 2^r / G) (= a contiguous leaf range = whole cap subtrees).  The
 * coefficient exchange is fused into the first NTT pass, which reads the other devices' blocks over NVLink in place
 * (PCS_MULTI_CE_GATHER: copy-engine gathers of polynomial group c+1 under the compute of group c instead -- measured slower).
 * With more devices than coset blocks (n_devices > 2^rate_bits) the other partition is used: every device extends its own
 * polynomials over all cosets and every device pulls its leaf range of every polynomial out of the owner's LDE (peer copies)
 * into a row shard.  Results are bit-identical to pcs_commit_from_* on one GPU.  n_devices: a power of two, <= the leaf count. */
typedef struct pcs_multi_batch pcs_multi_batch;
/* devices == NULL: the first n_devices visible devices (all of them, rounded down to a power of two, when n_devices <= 0). */
PCS_API int pcs_multi_init(const int* devices, int n_devices);
/* Number of devices of the multi-GPU state (0 before pcs_multi_init); fills `devices` when not NULL.                  */
PCS_API int pcs_multi_devices(int* devices);
/* PolynomialBatch::from_coeffs over the devices of pcs_multi_init.  polys: HOST pointers (pageable or pinned; every
 * device copies its share of each chunk over its own PCIe link while the previous chunk is being extended), or with
 * PCS_DEVICE_PTRS device pointers on ANY of the devices (read in place, over NVLink where remote).  salts: NULL or salt_w
 * pointers to N values each in natural LDE order, as in pcs_commit_from_coeffs.  Synchronous.                         */
PCS_API int pcs_multi_commit_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits,
                                 unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                                 uint64_t* cap_out, pcs_multi_batch** out);
/* PolynomialBatch::from_values: every device IFFTs its own block of the polynomials first (oracle.rs:51-55).          */
PCS_API int pcs_multi_commit_from_values(const uint64_t* const* values, size_t w, unsigned lg_d, unsigned rate_bits,
                                 unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                                 uint64_t* const* coeffs_out, uint64_t* cap_out, pcs_multi_batch** out);
PCS_API int pcs_multi_batch_shape(const pcs_multi_batch* b, size_t* n_leaves, size_t* leaf_len, int* n_shards, unsigned* cap_height);
PCS_API int pcs_multi_batch_cap(const pcs_multi_batch* b, uint64_t* cap /*[2^cap_height][4]*/);
/* merkle_tree.leaves[i] / MerkleTree::prove(i) for GLOBAL leaf indices, served by the device that owns the leaf; above a
 * device's root (n_devices > 2^cap_height) the path continues through the other devices' roots.                      */
PCS_API int pcs_multi_batch_get_rows(const pcs_multi_batch* b, const uint64_t* leaf_indices, size_t n, uint64_t* rows);
PCS_API int pcs_multi_batch_prove(const pcs_multi_batch* b, size_t leaf_index, uint64_t* siblings /*[log2 N - cap_height][4]*/);
/* The shard of device i as a plain batch (leaf indices relative to the shard; its digests are the contiguous slice
 * [i * n_digests / G ..] of the reference's `digests` when G <= 2^cap_height).  Owned by the multi batch.             */
PCS_API pcs_batch* pcs_multi_batch_shard(const pcs_multi_batch* b, int i);
/* Device address of every polynomial's coefficient vector (needs PCS_KEEP_COEFFS, from_values or PCS_DEVICE_PTRS inputs):
 * what pcs_eval_ext_dev / pcs_fri_final_poly_dev read, from any device of the group.                                  */
PCS_API int pcs_multi_batch_poly_ptrs(const pcs_multi_batch* b, const uint64_t** ptrs /*[w]*/);
/* Phase times as in pcs_batch_timings, maximum over the devices.                                                      */
PCS_API int pcs_multi_batch_timings(const pcs_multi_batch* b, float ms[5]);
PCS_API void pcs_multi_batch_free(pcs_multi_batch* b);

/* ---- FRI opening proof on the device (SURVEY 8f N2 / N3): the consumers of a committed batch's coefficients ------------
 * Extension elements are F::Extension = QuadraticExtension<GoldilocksField> = [u64; 2] = a + b*X, X^2 = 7
 * (field/src/goldilocks_extensions.rs:14-28); Vec<F::Extension> == flat u64[2n], the layout every ext pointer below uses.
 * All of these need batches committed with PCS_KEEP_COEFFS (or from_values): the reference keeps `polynomials` too.   */

/* OpeningSet::new's eval_commitment(z, c): c.polynomials[j].to_extension().eval(z) for every j.
 *                                                                  plonky2/src/plonk/proof.rs:316-322          */
PCS_API int pcs_batch_eval_ext(const pcs_batch* b, const uint64_t point[2], uint64_t* out /*[w][2]*/);

/* The same for w polynomials given as DEVICE pointers (d = 2^lg_d coefficients each, anywhere in this GPU's memory):
 * what a sharded commitment holds after its coefficient exchange (SURVEY 8e), where no single batch owns them.        */
PCS_API int pcs_eval_ext_dev(const uint64_t* const* polys_dev, size_t w, unsigned lg_d, const uint64_t point[2],
                     uint64_t* out /*[w][2]*/);

/* Device-resident PolynomialCoeffs<F::Extension> (coefficients of the polynomial FRI runs on).                       */
typedef struct pcs_ext_poly pcs_ext_poly;
PCS_API int pcs_ext_poly_new(const uint64_t* coeffs /*[len][2]*/, size_t len, pcs_ext_poly** out);
PCS_API int pcs_ext_poly_len(const pcs_ext_poly* p, size_t* len);
PCS_API int pcs_ext_poly_read(const pcs_ext_poly* p, uint64_t* coeffs /*[len][2]*/);
PCS_API void pcs_ext_poly_free(pcs_ext_poly* p);

/* The final polynomial of PolynomialBatch::prove_openings (plonky2/src/fri/oracle.rs:171-200), for an instance of
 * n_batches FriBatchInfo {point, polynomials}: per batch  F_i = sum_j alpha^j f_ij  (ReducingFactor::reduce_polys_base,
 * util/reducing.rs:84-96),  Q_i = F_i.divide_by_linear(point_i) padded back to d coefficients
 * (field/src/polynomial/division.rs:75-88),  final = final * alpha^{|batch i|} + Q_i  (shift_poly, reducing.rs:104-107).
 *   oracles        : the committed batches the instance indexes (all of the same degree, coefficients kept)
 *   batch_len[i]   : number of polynomials of batch i (>= 1); their (oracle_index, poly_index) pairs follow each other in
 *                    the two index arrays, batch after batch (FriPolynomialInfo, fri/structure.rs)
 * Result: d = 2^lg_d coefficients (before .lde(rate_bits)).                                                            */
PCS_API int pcs_fri_final_poly(const pcs_batch* const* oracles, size_t n_oracles, size_t n_batches,
                       const uint64_t* points /*[n_batches][2]*/, const size_t* batch_len,
                       const uint32_t* oracle_index, const uint32_t* poly_index, const uint64_t alpha[2],
                       pcs_ext_poly** out);

/* The same with the instance's polynomials given directly as DEVICE pointers, batch after batch (sum of batch_len of
 * them, d = 2^lg_d coefficients each).                                                                                */
PCS_API int pcs_fri_final_poly_dev(const uint64_t* const* polys_dev, unsigned lg_d, size_t n_batches,
                           const uint64_t* points /*[n_batches][2]*/, const size_t* batch_len, const uint64_t alpha[2],
                           pcs_ext_poly** out);

/* p.lde(rate_bits).coset_fft(shift.into()) of an extension polynomial: values in natural order, [len << rate_bits][2]
 * (`lde_final_values`, oracle.rs:202-207; the transform is F-linear, so it is the base-field coset LDE of both
 * components -- the extension's root of unity of order <= 2^32 is the base field's, quadratic.rs:70-74).          */
PCS_API int pcs_ext_coset_lde(const pcs_ext_poly* p, unsigned rate_bits, uint64_t shift, uint64_t* values);

/* One round of fri_committed_trees (plonky2/src/fri/prover.rs:81-87): values = p.lde(rate_bits).coset_fft(shift),
 * reverse_index_bits_in_place, chunks of 2^arity_bits flattened to leaves of 2 * 2^arity_bits base elements,
 * MerkleTree::new(leaves, cap_height).  The tree comes back as a batch handle (leaf_len = 2 << arity_bits), so
 * pcs_batch_get_rows / pcs_batch_prove serve the query phase (prover.rs:183-216).
 *   shift : 7^(product of the earlier rounds' arities) (prover.rs:77,102).                                          */
PCS_API int pcs_fri_commit_layer(const pcs_ext_poly* p, unsigned rate_bits, uint64_t shift, unsigned arity_bits,
                         unsigned cap_height, uint64_t* cap_out /*NULL or [2^cap_height][4]*/, pcs_batch** tree);

/* The fold between two rounds (prover.rs:93-101), in place: coeffs[i] <- reduce_with_powers(coeffs[i*arity ..
 * (i+1)*arity], beta) = sum_j beta^j coeffs[i*arity + j] (plonk_common.rs:116-128); len /= 2^arity_bits.            */
PCS_API int pcs_fri_fold(pcs_ext_poly* p, unsigned arity_bits, const uint64_t beta[2]);

/* ---- the permutation argument between commitments #1 and #2 of prove() ---------------------------------------------------
 * all_wires_permutation_partial_products (plonk/prover.rs): for every challenge c, wires_permutation_partial_products_and_zs
 * (plonk/prover.rs) with beta = betas[c], gamma = gammas[c], n = 2^lg_n rows at x_i = w^i (w = primitive_root_of_unity(lg_n)),
 * R = num_routed_wires, D = quotient_degree_factor, K = ceil(R / D) chunks of wires [kD, min((k+1)D, R)), P = K - 1:
 *     q_j(i) = (wires[j][i] + beta k_is[j] x_i + gamma) / (wires[j][i] + beta sigmas[j][i] + gamma)
 *     Q_k(i) = prod of q_j(i) over chunk k                           quotient_chunk_products (util/partial_products.rs)
 *     Z(x_0) = 1,  Z(x_{i+1}) = Z(x_i) Q_0(i) .. Q_{K-1}(i),  pp_k(x_i) = Z(x_i) Q_0(i) .. Q_k(i), k < P
 *                                                                    partial_products_and_z_gx + its swap (prover.rs)
 * k_is = get_unique_coset_shifts(n, R) (field/src/cosets.rs), sigmas[j] = the j-th sigma polynomial's values
 * (prover_data.sigmas[i][j] = sigmas[j][i]).
 *   wires, sigmas : R pointers to n values each; HOST pointers, or with PCS_DEVICE_PTRS device pointers on the current
 *                   context's device (contiguous or scattered; read, never written)
 *   k_is [R], betas [C], gammas [C] : host arrays, always
 *   out           : C (1 + P) pointers to n values each, in the order of prove()'s commitment #2: Z of challenge 0 .. C-1,
 *                   then the partial products challenge-major (out[C + c P + k] = pp_k of challenge c), as
 *                   PlonkOpeningShape zs_range / partial_products_range; host pointers, or device pointers with
 *                   PCS_DEVICE_PTRS
 * Any u64 is accepted as input; every output is canonical.  Synchronous: it reads back one device flag, and a zero
 * denominator returns PCS_ERR_ARG "Tried to invert zero" (batch_multiplicative_inverse; the outputs are then undefined).
 * quotient_degree_factor < 2, num_routed_wires == 0, num_challenges == 0 or a NULL pointer: PCS_ERR_ARG;
 * lg_n > 32: PCS_ERR_TWO_ADICITY.  The context stays usable after every error.                                          */
PCS_API int pcs_permutation_partial_products(const uint64_t* const* wires, const uint64_t* const* sigmas, size_t num_routed_wires,
                                     unsigned lg_n, const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas,
                                     size_t num_challenges, unsigned quotient_degree_factor, unsigned flags,
                                     uint64_t* const* out);

/* ---- the quotient polynomials between commitments #2 and #3 of prove() ------------------------------------------------------
 * compute_quotient_polys (plonk/prover.rs:576-744) without the gate constraints, followed by prove()'s trim_to_len(D n) and
 * chunks(n): the C D polynomials prove() commits as #3 (all_quotient_poly_chunks).  With n = 2^lg_d of the batches,
 * q = log2_ceil(D), D = quotient_degree_factor, R = num_routed_wires, C = num_challenges, K = ceil(R / D), P = K - 1, at every
 * point x_i = 7 w^i of the size-n 2^q domain (w = primitive_root_of_unity(lg_d + q)):
 *     terms = [L_0(x)(Z_c(x) - 1) for c < C]                                    L_0 = ZeroPolyOnCoset::eval_l_0
 *           ++ [check_partial_products(num_c, den_c, pp_c, Z_c(x), Z_c(g x), D) for c < C]   (K terms each, util/partial_products.rs)
 *     num_j = w_j + beta_c k_is[j] x + gamma_c,  den_j = w_j + beta_c sigma_j + gamma_c
 *     quotient_a(x_i) = (sum_t terms_t alpha_a^t + alpha_a^(C (P + 2)) gate_terms[a][i]) / Z_H(x_i)    reduce_with_powers_multi
 * then coset_ifft(7) of each of the C value vectors, coefficients [D n, n 2^q) checked to be zero and the first D n split into
 * D chunks of n.  The LDE rows of the three batches are read in place (leaves [0, n 2^q) = the quotient domain):
 *   constants_sigmas     : prover_data.constants_sigmas_commitment; sigma j = polynomial num_constants + j
 *   wires                : commitment #1; wire j = polynomial j (j < R; wider batches are fine)
 *   zs_partial_products  : commitment #2 in pcs_permutation_partial_products' output order: Z_c = polynomial c,
 *                          pp_{c,k} = polynomial C + c P + k
 * Other polynomials and the salt columns are not read.  All three must be resident, whole batches of the same context, degree
 * and rate (committed without PCS_LDE_ON_DEMAND, not shards or pcs_multi_* shards).
 *   k_is [R], betas [C], gammas [C], alphas [C] : host arrays, always (any u64)
 *   gate_terms : NULL (zero), or C columns of n 2^q values in NATURAL order of the quotient domain: column a holds, at point i,
 *                the alpha_a-reduced remainder of the vanishing terms sum_j constraint_j(x_i) alpha_a^j -- the gate constraints
 *                (evaluate_gate_constraints_base_batch), preceded by any lookup terms the circuit has, i.e. what
 *                reduce_with_powers_multi reduces after the permutation terms, restarted at alpha^0.  Any u64.
 *   out        : C D pointers to n coefficients each, alpha-major (out[a D + k] = chunk k of quotient polynomial a).
 * gate_terms and out are host pointers (pageable or pinned), or device pointers on the batches' device with PCS_DEVICE_PTRS;
 * every output is canonical.  Synchronous: it reads back the trim check.  PCS_ERR_ARG (the context stays usable): NULL
 * pointers, D < 2, R == 0, C == 0, q > rate_bits ("Having constraints of degree higher than the rate is not supported yet"),
 * batches of different contexts, degrees or rates, a column range beyond its batch, an on-demand, shard or rows-only batch,
 * and a failed trim ("Quotient has failed, the vanishing polynomial is not divisible by Z_H"; the outputs are then undefined). */
PCS_API int pcs_quotient_polys(const pcs_batch* constants_sigmas, const pcs_batch* wires, const pcs_batch* zs_partial_products,
                               size_t num_constants, size_t num_routed_wires, const uint64_t* k_is, const uint64_t* betas,
                               const uint64_t* gammas, const uint64_t* alphas, size_t num_challenges,
                               unsigned quotient_degree_factor, const uint64_t* const* gate_terms, unsigned flags,
                               uint64_t* const* out);

/* ---- the gate constraints of the quotient step ------------------------------------------------------------------------------
 * The gate-constraint tail of compute_quotient_polys (plonk/prover.rs:576-744): evaluate_gate_constraints_base_batch
 * (plonk/vanishing_poly.rs) at every point x_i = 7 w^i, i < M = n 2^q, of the quotient domain, reduced with powers of each
 * alpha:  out[a][i] = sum_j constraint_j(x_i) alphas[a]^j.  That is exactly pcs_quotient_polys' gate_terms, so the two chain on
 * the device.  Slot j of the constraints sums constraint j of every gate g times its filter
 *     compute_filter(g, groups[sel_g], s = local_constants[sel_g], num_selectors > 1)
 *       = prod_{i in [start, end), i != g} (i - s) * (num_selectors > 1 ? (2^32 - 1) - s : 1);
 * the gates read local_constants[num_selectors + k] and local_wires[k] (wire k = wires polynomial k).  The gates:
 *     PCS_GATE_NOOP          NoopGate                      no constraint
 *     PCS_GATE_CONSTANT      ConstantGate { num_consts }    c[k] - w[k], k < param
 *     PCS_GATE_PUBLIC_INPUT  PublicInputGate               w[k] - public_inputs_hash[k], k < 4
 *     PCS_GATE_ARITHMETIC    ArithmeticGate { num_ops }     w[4i+3] - (w[4i] w[4i+1] c[0] + w[4i+2] c[1]), i < param
 *     PCS_GATE_POSEIDON      PoseidonGate                  the 123 constraints of gates/poseidon.rs over 135 wires
 *   gates           : [num_gates][3] = { kind, param (num_consts / num_ops, else unused), selector_index }, in common_data.gates
 *                     order
 *   selector_groups : [num_selectors][2] = selectors_info.groups as [start, end) gate ranges
 *   public_inputs_hash [4], alphas [C] : host arrays (any u64)
 *   out             : C columns of M values in NATURAL order of the quotient domain, host pointers or, with PCS_DEVICE_PTRS,
 *                     device pointers on the batches' device; every output is canonical.
 * The LDE rows of constants_sigmas (constant k = polynomial k) and wires are read in place; both must be resident, whole,
 * committed batches of the same context, degree and rate.  Synchronous for host outputs, asynchronous on pcs_stream() for device
 * outputs.  PCS_ERR_ARG (the context stays usable): NULL pointers, C == 0, D < 2, q > rate_bits, an unknown gate kind, a
 * selector_index >= num_selectors, a gate outside its own group, a group that is not a non-empty range in [0, num_gates),
 * num_lookup_selectors > 0 (lookups are not built), batches too narrow for the gates (PoseidonGate needs 135 wires,
 * ArithmeticGate num_selectors + 2 constants), batches of different contexts, degrees or rates, and an on-demand, shard or
 * uncommitted batch. */
enum {
    PCS_GATE_NOOP = 0,
    PCS_GATE_CONSTANT = 1,
    PCS_GATE_PUBLIC_INPUT = 2,
    PCS_GATE_ARITHMETIC = 3,
    PCS_GATE_POSEIDON = 4
};
PCS_API int pcs_gate_constraint_terms(const pcs_batch* constants_sigmas, const pcs_batch* wires, const uint32_t* gates,
                                      size_t num_gates, const size_t* selector_groups, size_t num_selectors,
                                      size_t num_lookup_selectors, size_t num_constants, const uint64_t* public_inputs_hash,
                                      const uint64_t* alphas, size_t num_challenges, unsigned quotient_degree_factor,
                                      unsigned flags, uint64_t* const* out);

#ifdef __cplusplus
}
#endif
#endif /* PCS_H */
