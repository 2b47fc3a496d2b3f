// Shared declarations for the polynomial-commitment engine (libpcs.so).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <memory>
#include <string>
#include <vector>

#include "pcs.h"

// Device-resident PolynomialBatch / MerkleTree (opaque in pcs.h)
struct pcs_batch {
    size_t w = 0, salt_w = 0;
    unsigned lg_d = 0, rate_bits = 0, cap_height = 0;   // rate_bits = log2(coset blocks held) for a shard
    unsigned full_rate_bits = 0, coset_first = 0;       // the LDE this batch is (a shard of)
    size_t n = 0;          // N = d << rate_bits
    size_t n_digests = 0;  // 2 (N - 2^cap)
    uint64_t* coeffs = nullptr;   // [w][d] or null
    uint64_t* lde = nullptr;      // [w + salt_w][N], leaf order; null for an on-demand batch
    uint64_t* salts = nullptr;    // on-demand batch: [salt_w][N], leaf order (blinding cannot be recomputed)
    uint64_t* digests = nullptr;  // [n_digests][4]
    uint64_t* cap = nullptr;      // [2^cap][4]
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool has_ifft = false;
    bool committed = false;  // all six events recorded
    bool rows_only = false;  // pcs_shard_begin_rows: LDE rows are supplied, not computed here
    bool on_demand = false;  // PCS_LDE_ON_DEMAND: no LDE rows in HBM; accessors recompute them from `coeffs`
    uint64_t* scratch = nullptr;     // on-demand commit in flight: [LDE_GROUP + salt_w][N] columns of the current group
    // streaming sponge (leaf hashing group by group while later groups are still in flight)
    uint64_t* sponge = nullptr;      // [12][n] parked states, allocated at the first partial absorb
    size_t absorbed = 0;             // columns [0, absorbed) are in the sponge states
    size_t extended = 0;             // polynomials [0, extended) have their LDE rows in place (contiguous prefix)
    std::vector<cudaEvent_t> absorb_ev;   // start/stop pairs around the absorbs that ran inside the "FFT + blinding" phase
    void* ctx = nullptr;     // the per-device engine context (api.cu) that owns the buffers: accessors and free run there
};

namespace pcs {

void set_error(const std::string& msg);

#define PCS_CUDA(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            pcs::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
            return PCS_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)



int fail(int code, const std::string& msg);   // set_error + return code
// Initialise the engine on first use, else re-select the current context's device (the caller -- torch ... -- may have
// switched this thread's device).  Every entry point that works on the current context starts with it (api.cu).
int need_init();
// argument checks shared by the entry points: PCS_OK, or the reference's panic message and its code
static inline int check_two_adicity(unsigned lg_n) {
    return lg_n > 32 ? fail(PCS_ERR_TWO_ADICITY, "n_log <= TWO_ADICITY violated") : PCS_OK;
}
static inline int check_cap_height(unsigned cap_height, unsigned lg_n) {
    if (cap_height <= lg_n) return PCS_OK;
    return fail(PCS_ERR_CAP_HEIGHT, "cap_height=" + std::to_string(cap_height) +
                                        " should be at most log2(leaves.len())=" + std::to_string(lg_n));
}
static inline int check_shift(uint64_t shift) {   // a coset shift must be a unit
    return shift % 0xFFFFFFFF00000001ULL == 0 ? fail(PCS_ERR_ARG, "shift must be non-zero") : PCS_OK;
}
// host polynomials (pageable memory) -> contiguous device block through the current context's pinned ring (api.cu)
int stage_pageable(const uint64_t* const* polys, size_t count, size_t d, uint64_t* dst, cudaStream_t copy_st);
bool is_pageable_host(const void* p);         // not page-locked or registered: plain copies stage through the driver (api.cu)
void multi_shutdown_locked();                 // multi.cu: release the multi-GPU state (called by pcs_shutdown)
pcs_batch* batch_new();                       // a batch bound to the calling thread's current context (api.cu)
struct BatchFree {
    void operator()(pcs_batch* b) const { pcs_batch_free(b); }
};
using BatchOwner = std::unique_ptr<pcs_batch, BatchFree>;   // frees the batch on every exit until it is released

// One commitment's lifecycle (api.cu), shared by the single-GPU commit, the shard commits and every device of pcs_multi_*.
//   batch_begin:  checks the shape and allocates the batch (LDE rows, digests, cap) of the cosets [coset_first,
//                 coset_first + 2^lg_cosets) of a rate-2^rate_bits LDE of w polynomials of degree 2^lg_d plus salt_w salt
//                 rows, with a Merkle tree of cap height cap_height over its d << lg_cosets leaves.
//   batch_extend: the LDE rows of polynomials [first, first + count), read from src + j * d or from a device table of
//                 pointers; polynomials that arrive in order are leaf-hashed at once (streaming sponge).
//   batch_finish: records phase events 2-5, hashes the remaining columns (or all of them), builds the node levels and marks
//                 the batch committed; with cap_out, copies the cap out and synchronises.
enum BatchKind : unsigned {
    BATCH_LDE = 0,        // polynomials are extended by batch_extend (its twiddle tables are made here)
    BATCH_ROWS = 1,       // the caller writes the LDE rows itself
    BATCH_UNTIMED = 2,    // no phase events
    BATCH_ON_DEMAND = 4,  // no LDE rows: salt rows only; batch_extend writes each group to b->scratch (PCS_LDE_ON_DEMAND)
};
// Columns per group of an on-demand batch: the commit extends and absorbs at most this many polynomials at a time, and the
// row accessors recompute them group by group.  A multiple of the sponge rate (8).  16: the widest group that keeps the
// 135 x 2^20 rate-3 commit under 4 GB of HBM (3.55 GB, 121.3 ms; 32: 4.62 GB, 120.9 ms; profiles/r03_lde_on_demand.md).
#ifndef PCS_LDE_GROUP
#define PCS_LDE_GROUP 16
#endif
constexpr size_t LDE_GROUP = PCS_LDE_GROUP;
static_assert(LDE_GROUP % 8 == 0, "a group must end on the sponge rate");
// pcs_batch_get_rows of an on-demand batch: up to this many rows are evaluated from the coefficients (rows_eval.cu), more are
// gathered from the regenerated LDE.  At 135 x 2^20, rate 3: 128 rows take 19.5 ms evaluated and 21.1 ms regenerated, 512
// rows 77.8 ms and 21.1 ms (profiles/r03_lde_on_demand.md)
#ifndef PCS_ROWS_EVAL_MAX
#define PCS_ROWS_EVAL_MAX 128
#endif
constexpr size_t ROWS_EVAL_MAX = PCS_ROWS_EVAL_MAX;
int batch_begin(size_t w, size_t salt_w, unsigned lg_d, unsigned rate_bits, unsigned coset_first, unsigned lg_cosets,
                unsigned cap_height, unsigned kind, BatchOwner& out);
int batch_extend(pcs_batch* b, const uint64_t* src, const uint64_t* const* ptr_table, size_t first, size_t count);
int batch_finish(pcs_batch* b, uint64_t* cap_out);
// Run on the context (device + stream) that owns `b`, whatever the calling thread's current one is; the caller's
// context is restored on destruction (api.cu).
struct BatchScope {
    void* prev;
    explicit BatchScope(const pcs_batch* b);
    ~BatchScope();
};
// The same for any object that remembers the context it was made on (pcs_ext_poly): cur_ctx() at creation, CtxScope at use.
void* cur_ctx();
struct CtxScope {
    void* prev;
    explicit CtxScope(void* ctx);
    ~CtxScope();
};

// rows_eval.cu: rows [n][w + salt_w] of an on-demand batch at the leaves idx_dev[0 .. n) (device), evaluated from its kept
// coefficients (salt columns gathered from its salt rows), into out_dev; asynchronous on st
int rows_eval(const pcs_batch* b, const uint64_t* idx_dev, size_t n, uint64_t* out_dev, cudaStream_t st);

// stream-ordered temporary buffer
struct DevBuf {
    void* p = nullptr;
    cudaStream_t st = nullptr;
    cudaError_t alloc(size_t bytes, cudaStream_t s) {
        st = s;
        return cudaMallocAsync(&p, bytes ? bytes : 8, s);
    }
    uint64_t* u64() { return (uint64_t*)p; }
    void release() {
        if (p) cudaFreeAsync(p, st);
        p = nullptr;
    }
    ~DevBuf() { release(); }
};

// leaf digests + all node levels of MerkleTree::new over a poly-major matrix cols [width][n] (api.cu)
int build_tree_dev(const uint64_t* cols, size_t n, size_t width, unsigned lg_n, unsigned cap_height, uint64_t* digests,
                   uint64_t* cap, cudaStream_t st, cudaEvent_t after_leaves);

static inline int ilog2_strict(size_t n) {
    if (n == 0 || (n & (n - 1))) return -1;
    int r = 0;
    while ((n >> r) != 1) r++;
    return r;
}

// ------------------------------------------------------------------------------------------------
// hash_kernels.cu
// ------------------------------------------------------------------------------------------------
// In-place Poseidon permutation of n states, row-major [n][12].
cudaError_t launch_permute(uint64_t* states, size_t n, cudaStream_t st);
// FRI proof-of-work: smallest candidate in [base, base + n) whose response has >= min_lz leading zeros -> atomicMin(*best)
cudaError_t launch_pow_search(const uint64_t* state_dev, unsigned pos, unsigned min_lz, uint64_t base, uint64_t n,
                              unsigned long long* best_dev, cudaStream_t st);
// Leaf digests from a column-major (poly-major) matrix: element (leaf i, column j) at
// cols[j*col_stride + i].  Digest of leaf i goes to its slot in the reference digest layout
// (merkle_tree.rs:43-51) or into cap when the subtree is a single leaf.
cudaError_t launch_leaf_hash_cols(const uint64_t* cols, size_t col_stride, uint32_t width, size_t n_leaves,
                                  unsigned lg_sub /*log2 leaves per cap subtree*/, uint64_t* digests,
                                  uint64_t* cap, cudaStream_t st, size_t first_leaf = 0, size_t leaf_count = (size_t)-1);
// One GROUP of columns of a streaming sponge: cols = first column of the group, width = columns in it (a multiple of 8 unless
// it is the last group); state = [12][n_leaves] parked sponge states (unused when first && last).
cudaError_t launch_leaf_hash_group(const uint64_t* cols, size_t col_stride, uint32_t width, size_t n_leaves, bool first, bool last,
                                   uint64_t* state, unsigned lg_sub, uint64_t* digests, uint64_t* cap, cudaStream_t st);
// Plain variant: digest i -> out[i*4..] (pcs_hash_or_noop)
cudaError_t launch_hash_cols_plain(const uint64_t* cols, size_t col_stride, uint32_t width, size_t n,
                                   uint64_t* out, cudaStream_t st);
// One level of two_to_one: nodes of level `level` (1 = parents of leaf digests) for all subtrees.
cudaError_t launch_node_level(uint64_t* digests, uint64_t* cap, unsigned lg_sub, unsigned level,
                              size_t n_nodes /*total at this level*/, cudaStream_t st);
// Levels [level_first, lg_sub] of every cap subtree in one launch (<= 256 nodes per subtree at level_first).
cudaError_t launch_node_top(uint64_t* digests, uint64_t* cap, unsigned lg_sub, unsigned level_first, size_t n_subtrees,
                            cudaStream_t st);
cudaError_t launch_two_to_one(const uint64_t* l, const uint64_t* r, size_t n, uint64_t* out, cudaStream_t st);
// Merkle path gather: siblings of leaf_index, bottom-up ([lg_sub][4]).
cudaError_t launch_prove(const uint64_t* digests, unsigned lg_sub, size_t leaf_index, uint64_t* siblings,
                         cudaStream_t st);
cudaError_t launch_prove_many(const uint64_t* digests, unsigned lg_sub, const uint64_t* leaf_indices_dev, size_t n,
                              uint64_t* siblings, cudaStream_t st);

// field_ops.cu: out[i] = a[i] (op) b[i]
cudaError_t launch_field_op(int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// ntt.cu
// ------------------------------------------------------------------------------------------------
struct NttPlan;  // twiddle tables for one (lg_d, rate_bits, direction, shift)
NttPlan* ntt_plan_get(unsigned lg_d, unsigned rate_bits, bool inverse, uint64_t shift, cudaStream_t st);
void ntt_plans_free();
// Coset LDE: coeffs [w][d] (poly stride in_stride) -> out [w][N] (poly stride out_stride), leaf
// (bit-reversed) order: out[j][c*d + t] = P_j(shift * w_N^{brev_r(c)} * w_d^{brev(t)}).
cudaError_t ntt_lde(const NttPlan* plan, const uint64_t* coeffs, size_t in_stride, uint64_t* out,
                    size_t out_stride, size_t w, cudaStream_t st);
// Same for the coset sub-range [coset_first, coset_first + 2^lg_cosets) in leaf order (shard commits):
// out [w][d << lg_cosets].
// coeff_ptrs_dev (optional, lg_d >= 1): DEVICE array of w per-polynomial pointers read instead of coeffs + j*in_stride;
// the pointers may address peer GPUs' memory (read over NVLink inside the first pass, no staging copy).
cudaError_t ntt_lde_cosets(const NttPlan* plan, const uint64_t* coeffs, size_t in_stride, uint64_t* out,
                           size_t out_stride, size_t w, unsigned coset_first, unsigned lg_cosets, cudaStream_t st,
                           const uint64_t* const* coeff_ptrs_dev = nullptr);
// Inverse NTT WITHOUT the 1/d scaling: values [w][d] natural order -> `out` in BIT-REVERSED order; the
// bit-reversal permutation that always follows applies ntt_plan_scale(plan).
cudaError_t ntt_inverse_bitrev(const NttPlan* plan, const uint64_t* values, size_t in_stride, uint64_t* out,
                               size_t out_stride, size_t w, cudaStream_t st);
// out[j][brev(i)] = in[j][i]
// out[j][brev(i)] = in[j][i] * scale
cudaError_t launch_bitrev_permute(const uint64_t* in, size_t in_stride, uint64_t* out, size_t out_stride,
                                  size_t w, unsigned lg_n, cudaStream_t st, uint64_t scale = 1);
uint64_t ntt_plan_scale(const NttPlan* plan);
// out[i] = canon(in[brev_{lg_n}(first + i)]), i < count
cudaError_t launch_bitrev_gather(const uint64_t* in, unsigned lg_n, size_t first, size_t count, uint64_t* out,
                                 cudaStream_t st);
// out[c][r] = in[r][c] for in [rows][cols] (row pitch in_pitch), out row pitch out_pitch
cudaError_t launch_transpose(const uint64_t* in, size_t in_pitch, uint64_t* out, size_t out_pitch,
                             size_t rows, size_t cols, cudaStream_t st);
// gather rows: out[k][j] = cols[j*col_stride + idx[k]]
cudaError_t launch_gather_rows(const uint64_t* cols, size_t col_stride, uint32_t width, const uint64_t* idx,
                               size_t n_idx, uint64_t* out, cudaStream_t st);
cudaError_t launch_canonicalize(uint64_t* data, size_t n, cudaStream_t st);
// out[k][j] = cols[j][brev_{lg_n}((index_start + k) * step)], k < count, j < width
cudaError_t launch_lde_natural(const uint64_t* cols, size_t col_stride, uint32_t width, unsigned lg_n, size_t index_start,
                               size_t step, size_t count, uint64_t* out, cudaStream_t st);
// data[j][i] *= base^i for j < w, i < n (row stride `stride`)
cudaError_t launch_mul_powers(uint64_t* data, size_t stride, size_t w, size_t n, uint64_t base, cudaStream_t st);

}  // namespace pcs
