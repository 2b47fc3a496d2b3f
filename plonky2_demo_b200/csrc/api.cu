// C ABI (include/pcs.h) of the polynomial-commitment engine: context, the fused
// PolynomialBatch::from_coeffs / from_values path (plonky2/src/fri/oracle.rs:43-98) and the
// accessors the reference's consumers need.  No CPU fallback anywhere in this file.
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace pcs {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

struct PendingEvents { cudaEvent_t ev[6]; std::vector<cudaEvent_t> absorb_ev; };

struct Ctx {
    std::vector<PendingEvents> pending;   // events of freed batches, not yet folded into totals
    float totals[5] = {0, 0, 0, 0, 0};
    unsigned n_totals = 0;
    bool init = false;
    int device = -1;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // host-input pipeline: H2D copies run on their own stream, one event per chunk of polynomials,
    // so that the LDE of chunk k overlaps the PCIe transfer of chunk k+1
    // small host inputs / outputs (polynomials of a few KB): gathered through pinned staging so that W tiny copies
    // become one (a cudaMemcpyAsync call costs more than moving 64 bytes)
    void* pin_in = nullptr;  size_t pin_in_bytes = 0;
    void* pin_out = nullptr; size_t pin_out_bytes = 0;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t d2h_stream = nullptr;    // coefficients going back to the host while the LDE / hashing continue
    std::vector<cudaEvent_t> d2h_ev;
    cudaEvent_t ev_sync = nullptr;
    std::vector<cudaEvent_t> chunk_ev;
    // PAGEABLE host inputs (Rust Vecs, numpy arrays): gathered by a few host threads into a ring of pinned slots and
    // sent with one DMA per slot; a plain cudaMemcpyAsync from pageable memory stages single-threaded inside the driver
    void* ring[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ring_ev[3] = {nullptr, nullptr, nullptr};   // the DMA out of the slot has finished
    bool ring_busy[3] = {false, false, false};
    unsigned next_slot = 0;
};
// One context per CUDA device (created by pcs_init / pcs_multi_init, destroyed by pcs_shutdown).  The single-device
// entry points work on the calling thread's CURRENT context (the device of its last pcs_init, device 0 by default); a
// batch remembers the context that made it, so accessors and pcs_batch_free act on the right device and stream whatever
// is current.  One call in flight per context; different contexts may be driven from different host threads.
constexpr int MAX_DEVICES = 64;
static Ctx g_none;                                   // never initialised: what a thread sees before pcs_init
static Ctx* g_ctxs[MAX_DEVICES] = {nullptr};
static std::mutex g_ctx_mutex;
static thread_local Ctx* g_cur = &g_none;
#define g_ctx (*g_cur)

// make `c` current on this thread (device included); returns the previous one
static Ctx* ctx_enter(Ctx* c) {
    Ctx* prev = g_cur;
    if (c && c != g_cur) {
        g_cur = c;
        cudaSetDevice(c->device);
    }
    return prev;
}
// The five phase times of a committed batch (or of the events a freed one left pending) from its six events.  Leaf hashing
// that ran group by group inside the "FFT + blinding" phase (streaming sponge) is booked as leaf hashing.
template <class Events>
static int phase_times(const Events* b, float ms[5]) {
    for (int i = 0; i < 5; i++) PCS_CUDA(cudaEventElapsedTime(&ms[i], b->ev[i], b->ev[i + 1]));
    for (size_t k = 0; k + 1 < b->absorb_ev.size(); k += 2) {
        float t = 0;
        PCS_CUDA(cudaEventElapsedTime(&t, b->absorb_ev[k], b->absorb_ev[k + 1]));
        ms[1] -= t;
        ms[3] += t;
    }
    return PCS_OK;
}

// fold completed/pending event sets into the running totals (caller has synchronised the stream)
static void drain_pending() {
    for (auto& pe : g_ctx.pending) {
        float ms[5];
        if (phase_times(&pe, ms) == PCS_OK) {
            for (int i = 0; i < 5; i++) g_ctx.totals[i] += ms[i];
            g_ctx.n_totals++;
        }
        for (auto& e : pe.ev) cudaEventDestroy(e);
        for (auto& e : pe.absorb_ev) cudaEventDestroy(e);
    }
    g_ctx.pending.clear();
    cudaGetLastError();
}

int fail(int code, const std::string& msg) {
    set_error(msg);
    return code;
}

BatchScope::BatchScope(const pcs_batch* b) : prev(g_cur) {
    if (b && b->ctx) ctx_enter((Ctx*)b->ctx);
}
BatchScope::~BatchScope() { ctx_enter((Ctx*)prev); }

void* cur_ctx() { return g_cur; }
CtxScope::CtxScope(void* ctx) : prev(g_cur) {
    if (ctx) ctx_enter((Ctx*)ctx);
}
CtxScope::~CtxScope() { ctx_enter((Ctx*)prev); }

pcs_batch* batch_new() {
    pcs_batch* b = new pcs_batch();
    b->ctx = g_cur;
    return b;
}

int need_init() {
    if (!g_ctx.init) return pcs_init(-1, nullptr);
    cudaSetDevice(g_ctx.device);
    return PCS_OK;
}

static int node_levels_dev(size_t n, unsigned lg_sub, uint64_t* digests, uint64_t* cap, cudaStream_t st) {
    // one launch per level while a level still fills the GPU (more than 256 nodes per cap subtree), then the top of every
    // subtree in ONE launch
    // (levels of <= 8192 nodes run in the latency form, one node per half-warp: node_hash.cu; the top launch then starts
    // once a subtree has <= 64 nodes, before that it needs <= 256)
    unsigned level = 1;
    for (; level <= lg_sub; level++) {
        const size_t nodes = n >> level;
        const unsigned left = lg_sub - level;                     // log2(nodes per subtree at this level)
        if (nodes <= 8192 ? left <= 6 : left <= 8) break;
        PCS_CUDA(launch_node_level(digests, cap, lg_sub, level, nodes, st));
    }
    if (level <= lg_sub) PCS_CUDA(launch_node_top(digests, cap, lg_sub, level, n >> lg_sub, st));
    return PCS_OK;
}

// leaf digests + all node levels; cols = [width][n] poly-major
int build_tree_dev(const uint64_t* cols, size_t n, size_t width, unsigned lg_n, unsigned cap_height,
                          uint64_t* digests, uint64_t* cap, cudaStream_t st, cudaEvent_t after_leaves) {
    unsigned lg_sub = lg_n - cap_height;
    PCS_CUDA(launch_leaf_hash_cols(cols, n, (uint32_t)width, n, lg_sub, digests, cap, st));
    if (after_leaves) PCS_CUDA(cudaEventRecord(after_leaves, st));
    return node_levels_dev(n, lg_sub, digests, cap, st);
}

// Streaming sponge: absorb the LDE columns [b->absorbed, upto) of every leaf (upto a multiple of the rate, or all columns
// with last = true, which also emits the digests); an on-demand batch holds them at the start of its group scratch.
// timed: bracket the launch with an event pair (absorbs that run inside the "FFT + blinding" phase are booked as leaf hashing
// by the timing queries).
static int absorb_columns(pcs_batch* b, size_t upto, bool last, cudaStream_t st, bool timed) {
    if (upto < b->absorbed) return fail(PCS_ERR_ARG, "internal: sponge cannot go backwards");
    if (upto == b->absorbed && !last) return PCS_OK;
    const bool first = b->absorbed == 0;
    const unsigned lg_sub = b->lg_d + b->rate_bits - b->cap_height;
    if (!(first && last) && !b->sponge) PCS_CUDA(cudaMallocAsync((void**)&b->sponge, 12 * b->n * 8, st));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (timed) {
        PCS_CUDA(cudaEventCreate(&e0));
        PCS_CUDA(cudaEventCreate(&e1));
        b->absorb_ev.push_back(e0);
        b->absorb_ev.push_back(e1);
        PCS_CUDA(cudaEventRecord(e0, st));
    }
    const uint64_t* cols = b->on_demand ? b->scratch : b->lde + b->absorbed * b->n;
    PCS_CUDA(launch_leaf_hash_group(cols, b->n, (uint32_t)(upto - b->absorbed), b->n, first, last, b->sponge,
                                    lg_sub, b->digests, b->cap, st));
    if (timed) PCS_CUDA(cudaEventRecord(e1, st));
    b->absorbed = upto;
    if (last && b->sponge) {
        cudaFreeAsync(b->sponge, st);
        b->sponge = nullptr;
    }
    return PCS_OK;
}

int batch_begin(size_t w, size_t salt_w, unsigned lg_d, unsigned rate_bits, unsigned coset_first, unsigned lg_cosets,
                unsigned cap_height, unsigned kind, BatchOwner& out) {
    if (int rc = check_two_adicity(lg_d + rate_bits)) return rc;
    if (lg_cosets > rate_bits || ((size_t)coset_first + ((size_t)1 << lg_cosets)) > ((size_t)1 << rate_bits))
        return fail(PCS_ERR_ARG, "coset range outside [0, 2^rate_bits)");
    const unsigned lg_n = lg_d + lg_cosets;   // leaves of this (shard of the) tree
    if (int rc = check_cap_height(cap_height, lg_n)) return rc;
    cudaStream_t st = g_ctx.stream;
    if (!(kind & BATCH_ROWS) && !ntt_plan_get(lg_d, rate_bits, false, 7 /* F::coset_shift(), types.rs:437 */, st))
        return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    const size_t n = (size_t)1 << lg_n, n_cap = (size_t)1 << cap_height;
    BatchOwner b(batch_new());
    b->w = w; b->salt_w = salt_w; b->lg_d = lg_d; b->rate_bits = lg_cosets; b->cap_height = cap_height;
    b->full_rate_bits = rate_bits; b->coset_first = coset_first; b->rows_only = kind & BATCH_ROWS;
    b->on_demand = kind & BATCH_ON_DEMAND;
    b->n = n; b->n_digests = 2 * (n - n_cap);
    if (!(kind & BATCH_UNTIMED))
        for (auto& e : b->ev) PCS_CUDA(cudaEventCreate(&e));
    if (b->on_demand)
        PCS_CUDA(cudaMallocAsync((void**)&b->salts, salt_w * n * 8, st));
    else
        PCS_CUDA(cudaMallocAsync((void**)&b->lde, (w + salt_w) * n * 8, st));
    PCS_CUDA(cudaMallocAsync((void**)&b->digests, b->n_digests ? b->n_digests * 32 : 32, st));
    PCS_CUDA(cudaMallocAsync((void**)&b->cap, n_cap * 32, st));
    out = std::move(b);
    return PCS_OK;
}

int batch_extend(pcs_batch* b, const uint64_t* src, const uint64_t* const* ptr_table, size_t first, size_t count) {
    cudaStream_t st = g_ctx.stream;
    NttPlan* plan = ntt_plan_get(b->lg_d, b->full_rate_bits, false, 7, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    // an on-demand batch gets its polynomials in order, one group of <= LDE_GROUP at a time: each overwrites the scratch
    // once the previous one has been absorbed (stream order)
    uint64_t* const dst = b->on_demand ? b->scratch : b->lde + first * b->n;
    PCS_CUDA(ntt_lde_cosets(plan, src, (size_t)1 << b->lg_d, dst, b->n, count, b->coset_first, b->rate_bits, st, ptr_table));
    // streaming sponge: groups that arrive in order are hashed at once, up to a multiple of the sponge rate, while later
    // groups are still in flight; the last group is absorbed by batch_finish together with the salt columns, and a batch
    // that gets all its polynomials in one call keeps the single hash kernel
    if (b->on_demand && first != b->absorbed) return fail(PCS_ERR_ARG, "internal: on-demand groups must arrive in order");
    if (first == b->extended) b->extended += count;
    const bool whole = first == 0 && count == b->w;
    if (!whole && b->w + b->salt_w > 4 && b->extended < b->w) return absorb_columns(b, (b->extended / 8) * 8, false, st, true);
    // the last group and the salt rows are absorbed together by batch_finish: one sponge chunk may cover both
    if (b->on_demand && b->salt_w && b->extended == b->w)
        PCS_CUDA(cudaMemcpyAsync(b->scratch + count * b->n, b->salts, b->salt_w * b->n * 8, cudaMemcpyDeviceToDevice, st));
    return PCS_OK;
}

int batch_finish(pcs_batch* b, uint64_t* cap_out) {
    cudaStream_t st = g_ctx.stream;
    PCS_CUDA(cudaEventRecord(b->ev[2], st));
    // "transpose LDEs" (oracle.rs:83): fused away -- the hash kernel reads columns directly
    PCS_CUDA(cudaEventRecord(b->ev[3], st));
    // "build Merkle tree" (oracle.rs:85-89)
    const size_t wt = b->w + b->salt_w;
    const unsigned lg_n = b->lg_d + b->rate_bits;
    int rc;
    if (b->absorbed > 0) {
        rc = absorb_columns(b, wt, true, st, false);     // the remaining columns (+ salts) and the digests
        if (rc) return rc;
        PCS_CUDA(cudaEventRecord(b->ev[4], st));
        rc = node_levels_dev(b->n, lg_n - b->cap_height, b->digests, b->cap, st);
    } else {
        rc = build_tree_dev(b->on_demand ? b->scratch : b->lde, b->n, wt, lg_n, b->cap_height, b->digests, b->cap, st, b->ev[4]);
    }
    if (rc) return rc;
    PCS_CUDA(cudaEventRecord(b->ev[5], st));
    b->committed = true;
    if (cap_out) {
        PCS_CUDA(cudaMemcpyAsync(cap_out, b->cap, ((size_t)32) << b->cap_height, cudaMemcpyDeviceToHost, st));
        PCS_CUDA(cudaStreamSynchronize(st));
    }
    return PCS_OK;
}

}  // namespace pcs

using namespace pcs;

extern "C" {

const char* pcs_last_error(void) { return g_err.c_str(); }

static int ctx_create(int device, void* stream, Ctx** out) {
    PCS_CUDA(cudaSetDevice(device));
    Ctx* c = new Ctx();
    c->device = device;
    if (stream) {
        c->stream = (cudaStream_t)stream;
        c->own_stream = false;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete c;
            return fail(PCS_ERR_CUDA, std::string("cudaStreamCreateWithFlags: ") + cudaGetErrorString(e));
        }
        c->own_stream = true;
    }
    // keep freed blocks cached in the pool: commits reuse multi-GB buffers
    cudaMemPool_t pool;
    uint64_t thr = UINT64_MAX;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess)
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    cudaGetLastError();
    c->init = true;
    *out = c;
    return PCS_OK;
}

int pcs_init(int device, void* stream) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(PCS_ERR_CUDA, std::string("no CUDA device: the engine has no CPU fallback (") +
                                      cudaGetErrorString(e) + ")");
    if (device < 0) {
        if (g_ctx.init) return PCS_OK;
        device = 0;
    }
    if (device >= count || device >= MAX_DEVICES)
        return fail(PCS_ERR_ARG, "device " + std::to_string(device) + " out of range (" + std::to_string(count) + " visible)");
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    Ctx* c = g_ctxs[device];
    if (!c) {
        int rc = ctx_create(device, stream, &c);
        if (rc) return rc;
        g_ctxs[device] = c;
    } else if (stream && stream != (void*)c->stream) {
        // re-bind the stream only; work already enqueued on the old stream must be finished first (twiddle tables,
        // batches) because nothing orders the new stream behind it
        cudaSetDevice(device);
        cudaStreamSynchronize(c->stream);
        if (c->own_stream) cudaStreamDestroy(c->stream);
        c->stream = (cudaStream_t)stream;
        c->own_stream = false;
    }
    ctx_enter(c);                      // current for this thread; other devices' contexts (and their batches) stay alive
    PCS_CUDA(cudaSetDevice(device));
    return PCS_OK;
}

int pcs_device(void) { return g_ctx.init ? g_ctx.device : -1; }

static void ctx_destroy(Ctx* c) {
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    g_cur = c;
    drain_pending();
    ntt_plans_free();                  // this device's twiddle tables
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    for (auto& e : c->d2h_ev) cudaEventDestroy(e);
    if (c->pin_in) cudaFreeHost(c->pin_in);
    if (c->pin_out) cudaFreeHost(c->pin_out);
    if (c->ev_sync) cudaEventDestroy(c->ev_sync);
    for (auto& e : c->chunk_ev) cudaEventDestroy(e);
    for (auto& r : c->ring)
        if (r) cudaFreeHost(r);
    for (auto& e : c->ring_ev)
        if (e) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

void pcs_shutdown(void) {
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    multi_shutdown_locked();
    for (auto& c : g_ctxs)
        if (c) {
            ctx_destroy(c);
            c = nullptr;
        }
    g_cur = &g_none;
    cudaGetLastError();
}

void* pcs_stream(void) { return g_ctx.init ? (void*)g_ctx.stream : nullptr; }

int pcs_synchronize(void) {
    if (int rc = need_init()) return rc;
    PCS_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return PCS_OK;
}

// ------------------------------------------------------------------------------------------------
// primitives
// ------------------------------------------------------------------------------------------------
int pcs_field_op(int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out) {
    if (int rc = need_init()) return rc;
    if (n == 0) return PCS_OK;
    if (!a || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (op < PCS_OP_ADD || op > PCS_OP_MUL_2EXP || op == 3 /* no operation has this value */)
        return fail(PCS_ERR_ARG, "unknown field operation");
    const bool binary = op != PCS_OP_SQUARE && op != PCS_OP_CANON && op != PCS_OP_NEG;
    if (binary && !b) return fail(PCS_ERR_ARG, "second operand is NULL");
    cudaStream_t st = g_ctx.stream;
    DevBuf da, db, dout;
    PCS_CUDA(da.alloc(n * 8, st));
    PCS_CUDA(dout.alloc(n * 8, st));
    PCS_CUDA(cudaMemcpyAsync(da.p, a, n * 8, cudaMemcpyHostToDevice, st));
    if (binary) {
        PCS_CUDA(db.alloc(n * 8, st));
        PCS_CUDA(cudaMemcpyAsync(db.p, b, n * 8, cudaMemcpyHostToDevice, st));
    }
    PCS_CUDA(launch_field_op(op, da.u64(), binary ? db.u64() : nullptr, n, dout.u64(), st));
    PCS_CUDA(cudaMemcpyAsync(out, dout.p, n * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_poseidon_permute(uint64_t* states, size_t n) {
    if (int rc = need_init()) return rc;
    if (n == 0) return PCS_OK;
    if (!states) return fail(PCS_ERR_ARG, "states is NULL");
    cudaStream_t st = g_ctx.stream;
    DevBuf d;
    PCS_CUDA(d.alloc(n * 12 * 8, st));
    PCS_CUDA(cudaMemcpyAsync(d.p, states, n * 12 * 8, cudaMemcpyHostToDevice, st));
    PCS_CUDA(launch_permute(d.u64(), n, st));
    PCS_CUDA(cudaMemcpyAsync(states, d.p, n * 12 * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_pow_grind(const uint64_t* state, unsigned witness_pos, unsigned min_leading_zeros, uint64_t* witness) {
    if (int rc = need_init()) return rc;
    if (!state || !witness) return fail(PCS_ERR_ARG, "NULL pointer");
    if (witness_pos >= 12) return fail(PCS_ERR_ARG, "witness position outside the sponge state");
    if (min_leading_zeros > 40) return fail(PCS_ERR_ARG, "proof-of-work difficulty above 40 bits is not supported");
    cudaStream_t st = g_ctx.stream;
    DevBuf d_state, d_best;
    PCS_CUDA(d_state.alloc(12 * 8, st));
    PCS_CUDA(d_best.alloc(8, st));
    PCS_CUDA(cudaMemcpyAsync(d_state.p, state, 12 * 8, cudaMemcpyHostToDevice, st));
    const uint64_t P = 0xFFFFFFFF00000001ULL, none = ~0ULL;
    PCS_CUDA(cudaMemcpyAsync(d_best.p, &none, 8, cudaMemcpyHostToDevice, st));
    // batches of four times the expected number of tries (2^min_lz): one launch finds the witness with probability
    // 1 - e^-4; at least 2^14 and at most 2^26 candidates per launch.  Batches are searched in order and a batch returns its
    // smallest hit, so the result is the smallest witness whatever the batch size.
    const unsigned lg_batch = min_leading_zeros + 2 < 14 ? 14 : (min_leading_zeros + 2 > 26 ? 26 : min_leading_zeros + 2);
    uint64_t batch = (uint64_t)1 << lg_batch;
    for (uint64_t base = 0; base < P; base += batch) {          // candidates 0 ..= p - 1 (prover.rs:141)
        uint64_t n = P - base < batch ? P - base : batch;
        PCS_CUDA(launch_pow_search(d_state.u64(), witness_pos, min_leading_zeros, base, n, (unsigned long long*)d_best.p, st));
        uint64_t best;
        PCS_CUDA(cudaMemcpyAsync(&best, d_best.p, 8, cudaMemcpyDeviceToHost, st));
        PCS_CUDA(cudaStreamSynchronize(st));
        if (best != none) {
            *witness = best;
            return PCS_OK;
        }
    }
    return fail(PCS_ERR_ARG, "Proof of work failed. This is highly unlikely!");
}

int pcs_hash_or_noop(const uint64_t* rows, size_t n, size_t len, uint64_t* out) {
    if (int rc = need_init()) return rc;
    if (n == 0) return PCS_OK;
    if (!rows || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (len == 0) {  // hash_or_noop of an empty slice: all-zero HashOut (config.rs:56-62)
        memset(out, 0, n * 32);
        return PCS_OK;
    }
    cudaStream_t st = g_ctx.stream;
    DevBuf d_rows, d_cols, d_out;
    PCS_CUDA(d_rows.alloc(n * len * 8, st));
    PCS_CUDA(d_cols.alloc(n * len * 8, st));
    PCS_CUDA(d_out.alloc(n * 32, st));
    PCS_CUDA(cudaMemcpyAsync(d_rows.p, rows, n * len * 8, cudaMemcpyHostToDevice, st));
    PCS_CUDA(launch_transpose(d_rows.u64(), len, d_cols.u64(), n, n, len, st));
    PCS_CUDA(launch_hash_cols_plain(d_cols.u64(), n, (uint32_t)len, n, d_out.u64(), st));
    PCS_CUDA(cudaMemcpyAsync(out, d_out.p, n * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_two_to_one(const uint64_t* left, const uint64_t* right, size_t n, uint64_t* out) {
    if (int rc = need_init()) return rc;
    if (n == 0) return PCS_OK;
    if (!left || !right || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    cudaStream_t st = g_ctx.stream;
    DevBuf l, r, o;
    PCS_CUDA(l.alloc(n * 32, st));
    PCS_CUDA(r.alloc(n * 32, st));
    PCS_CUDA(o.alloc(n * 32, st));
    PCS_CUDA(cudaMemcpyAsync(l.p, left, n * 32, cudaMemcpyHostToDevice, st));
    PCS_CUDA(cudaMemcpyAsync(r.p, right, n * 32, cudaMemcpyHostToDevice, st));
    PCS_CUDA(launch_two_to_one(l.u64(), r.u64(), n, o.u64(), st));
    PCS_CUDA(cudaMemcpyAsync(out, o.p, n * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

}  // extern "C"

// In place on the device, natural order in and out: w polynomials [w][2^lg_n], forward NTT or inverse NTT (scaled by 1/n)
static int ntt_dev(uint64_t* polys, size_t w, unsigned lg_n, bool inverse, cudaStream_t st) {
    const size_t n = (size_t)1 << lg_n;
    NttPlan* plan = ntt_plan_get(lg_n, 0, inverse, 1, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    DevBuf b;
    PCS_CUDA(b.alloc(w * n * 8, st));
    PCS_CUDA(ntt_lde(plan, polys, n, b.u64(), n, w, st));                                          // -> bit-reversed
    PCS_CUDA(launch_bitrev_permute(b.u64(), n, polys, n, w, lg_n, st, ntt_plan_scale(plan)));      // -> natural (* 1/n)
    return PCS_OK;
}

static uint64_t host_inverse(uint64_t a) {  // a^(p-2) mod p
    const uint64_t P = 0xFFFFFFFF00000001ULL;
    unsigned __int128 acc = 1, b = a % P;
    for (uint64_t e = P - 2; e; e >>= 1) {
        if (e & 1) acc = acc * b % P;
        b = b * b % P;
    }
    return (uint64_t)acc;
}

// coset_ifft in place on the device: values on shift * <w_n>, natural order -> coefficients
static int coset_intt_dev(uint64_t* values, size_t w, unsigned lg_n, uint64_t shift, cudaStream_t st) {
    const size_t n = (size_t)1 << lg_n;
    if (int rc = ntt_dev(values, w, lg_n, true, st)) return rc;
    PCS_CUDA(launch_mul_powers(values, n, w, n, host_inverse(shift), st));   // c_i *= shift^-i  (mod.rs:68-72)
    return PCS_OK;
}

// host data [w][2^lg_n] -> a device copy -> body(copy) -> back into data; synchronises
template <class Body>
static int through_device(uint64_t* data, size_t w, unsigned lg_n, Body body) {
    cudaStream_t st = g_ctx.stream;
    const size_t bytes = (w * 8) << lg_n;
    DevBuf a;
    PCS_CUDA(a.alloc(bytes, st));
    PCS_CUDA(cudaMemcpyAsync(a.p, data, bytes, cudaMemcpyHostToDevice, st));
    if (int rc = body(a.u64(), st)) return rc;
    PCS_CUDA(cudaMemcpyAsync(data, a.p, bytes, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

extern "C" {

int pcs_ntt(uint64_t* polys, size_t w, unsigned lg_n, int inverse) {
    if (int rc = need_init()) return rc;
    if (w == 0) return PCS_OK;
    if (!polys) return fail(PCS_ERR_ARG, "polys is NULL");
    if (int rc = check_two_adicity(lg_n)) return rc;
    return through_device(polys, w, lg_n, [&](uint64_t* p, cudaStream_t st) { return ntt_dev(p, w, lg_n, inverse != 0, st); });
}

int pcs_coset_intt(uint64_t* values, size_t w, unsigned lg_n, uint64_t shift) {
    if (int rc = need_init()) return rc;
    if (w == 0) return PCS_OK;
    if (!values) return fail(PCS_ERR_ARG, "values is NULL");
    if (int rc = check_two_adicity(lg_n)) return rc;
    if (int rc = check_shift(shift)) return rc;
    return through_device(values, w, lg_n, [&](uint64_t* v, cudaStream_t st) { return coset_intt_dev(v, w, lg_n, shift, st); });
}

int pcs_coset_intt_dev(uint64_t* values_dev, size_t w, unsigned lg_n, uint64_t shift) {
    if (int rc = need_init()) return rc;
    if (w == 0) return PCS_OK;
    if (!values_dev) return fail(PCS_ERR_ARG, "values is NULL");
    if (int rc = check_two_adicity(lg_n)) return rc;
    if (int rc = check_shift(shift)) return rc;
    return coset_intt_dev(values_dev, w, lg_n, shift, g_ctx.stream);   // asynchronous on pcs_stream()
}

int pcs_ntt_dev(uint64_t* polys_dev, size_t w, unsigned lg_n, int inverse) {
    if (int rc = need_init()) return rc;
    if (w == 0) return PCS_OK;
    if (!polys_dev) return fail(PCS_ERR_ARG, "polys is NULL");
    if (int rc = check_two_adicity(lg_n)) return rc;
    return ntt_dev(polys_dev, w, lg_n, inverse != 0, g_ctx.stream);   // asynchronous on pcs_stream()
}

}  // extern "C"

constexpr size_t SMALL_POLY_BYTES = 32 * 1024;     // below this, host polynomials go through pinned staging
constexpr size_t PIN_STAGING_MAX = 64u << 20;

static void* pinned(void*& buf, size_t& cap, size_t bytes) {
    if (bytes > cap) {
        if (buf) cudaFreeHost(buf);
        buf = nullptr;
        cap = 0;
        if (cudaHostAlloc(&buf, bytes, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        cap = bytes;
    }
    return buf;
}

// Device -> pageable host memory: D2H into one of two pinned buffers, then a multi-threaded copy into the caller's memory
// (fresh Vecs / numpy arrays fault their pages on first touch: one thread moves ~5 GB/s, four ~15) while the next piece is
// already crossing PCIe.  Synchronises the stream.
static int d2h_pageable(void* dst, const void* src_dev, size_t bytes, cudaStream_t st);

constexpr size_t RING_SLOT_BYTES = 16u << 20;
constexpr unsigned STAGE_THREADS = 4;

bool pcs::is_pageable_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

// copy stream bytes [off, off + len) of the concatenation polys[0] | polys[1] | ... (bytes_each each) to dst
static void gather_bytes(char* dst, const uint64_t* const* polys, size_t bytes_each, size_t off, size_t len) {
    while (len) {
        size_t j = off / bytes_each, o = off % bytes_each;
        size_t n = bytes_each - o < len ? bytes_each - o : len;
        memcpy(dst, (const char*)polys[j] + o, n);
        dst += n;
        off += n;
        len -= n;
    }
}

// Send `count` pageable host polynomials (d elements each) to the contiguous device block `dst` through the pinned
// ring: pieces of <= RING_SLOT_BYTES are gathered by STAGE_THREADS host threads and leave with one DMA each on the
// copy stream; the gather of piece p + 1 overlaps the DMA of piece p.
int pcs::stage_pageable(const uint64_t* const* polys, size_t count, size_t d, uint64_t* dst, cudaStream_t copy_st) {
    const size_t bytes_each = d * 8, total = count * bytes_each;
    for (size_t off = 0; off < total; off += RING_SLOT_BYTES) {
        const size_t len = total - off < RING_SLOT_BYTES ? total - off : RING_SLOT_BYTES;
        const unsigned sl = g_ctx.next_slot++ % 3;
        if (!g_ctx.ring[sl]) {
            PCS_CUDA(cudaHostAlloc(&g_ctx.ring[sl], RING_SLOT_BYTES, cudaHostAllocDefault));
            PCS_CUDA(cudaEventCreateWithFlags(&g_ctx.ring_ev[sl], cudaEventDisableTiming));
        }
        if (g_ctx.ring_busy[sl]) PCS_CUDA(cudaEventSynchronize(g_ctx.ring_ev[sl]));
        char* slot = (char*)g_ctx.ring[sl];
        const unsigned nt = len >= (1u << 20) ? STAGE_THREADS : 1;
        if (nt == 1) {
            gather_bytes(slot, polys, bytes_each, off, len);
        } else {
            std::thread th[STAGE_THREADS];
            for (unsigned t = 0; t < nt; t++) {
                size_t a = len * t / nt, e = len * (t + 1) / nt;
                th[t] = std::thread(gather_bytes, slot + a, polys, bytes_each, off + a, e - a);
            }
            for (unsigned t = 0; t < nt; t++) th[t].join();
        }
        PCS_CUDA(cudaMemcpyAsync((char*)dst + off, slot, len, cudaMemcpyHostToDevice, copy_st));
        PCS_CUDA(cudaEventRecord(g_ctx.ring_ev[sl], copy_st));
        g_ctx.ring_busy[sl] = true;
    }
    return PCS_OK;
}

// gather w separately allocated host/device polynomials into one [w][d] device matrix
static int stage_polys(const uint64_t* const* polys, size_t w, size_t d, bool device_ptrs, uint64_t* dst,
                       cudaStream_t st) {
    for (size_t j = 0; j < w; j++) {
        if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
        PCS_CUDA(cudaMemcpyAsync(dst + j * d, polys[j], d * 8, device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    }
    return PCS_OK;
}

static bool contiguous(const uint64_t* const* polys, size_t count, size_t d) {
    for (size_t j = 1; j < count; j++)
        if (polys[j] != polys[0] + j * d) return false;
    return true;
}

// Where ntt_lde_cosets reads `count` device polynomials of 2^lg_d coefficients from: the caller's matrix when they are
// contiguous, else a device table of their pointers that the first NTT pass follows (they may live in PEER memory: no
// staging copy), or, for lg_d == 0, which has no such pass, a staged contiguous copy.
struct DevInput {
    const uint64_t* src = nullptr;
    const uint64_t* const* ptrs = nullptr;
    DevBuf table, staged;
};

static int resolve_dev_input(const uint64_t* const* polys, size_t count, unsigned lg_d, cudaStream_t st, DevInput& in) {
    const size_t d = (size_t)1 << lg_d;
    for (size_t j = 0; j < count; j++)
        if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
    in.src = polys[0];
    if (contiguous(polys, count, d)) return PCS_OK;
    if (lg_d >= 1) {
        PCS_CUDA(in.table.alloc(count * sizeof(uint64_t*), st));
        PCS_CUDA(cudaMemcpyAsync(in.table.p, polys, count * sizeof(uint64_t*), cudaMemcpyHostToDevice, st));
        in.ptrs = (const uint64_t* const*)in.table.p;
        return PCS_OK;
    }
    PCS_CUDA(in.staged.alloc(count * d * 8, st));
    in.src = in.staged.u64();
    return stage_polys(polys, count, d, true, in.staged.u64(), st);
}

static void host_copy_mt(char* dst, const char* src, size_t bytes) {
    const unsigned nt = bytes >= (4u << 20) ? STAGE_THREADS : 1;
    if (nt == 1) {
        memcpy(dst, src, bytes);
        return;
    }
    std::thread th[STAGE_THREADS];
    const size_t per = (bytes / nt + 4095) & ~(size_t)4095;
    for (unsigned t = 0; t < nt; t++) {
        const size_t o = (size_t)t * per, l = o >= bytes ? 0 : (bytes - o < per ? bytes - o : per);
        th[t] = std::thread([=]() { if (l) memcpy(dst + o, src + o, l); });
    }
    for (unsigned t = 0; t < nt; t++) th[t].join();
}

static int d2h_pageable(void* dst, const void* src_dev, size_t bytes, cudaStream_t st) {
    const size_t PIECE = 16u << 20;
    if (bytes <= (1u << 20) || !is_pageable_host(dst)) {
        PCS_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDeviceToHost, st));
        PCS_CUDA(cudaStreamSynchronize(st));
        return PCS_OK;
    }
    if (!pinned(g_ctx.pin_out, g_ctx.pin_out_bytes, 2 * PIECE)) return fail(PCS_ERR_ALLOC, "pinned staging allocation failed");
    cudaEvent_t ev[2];
    PCS_CUDA(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
    PCS_CUDA(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } evg{ev};
    size_t prev_off = 0, prev_len = 0;
    int slot = 0;
    for (size_t off = 0; off < bytes; off += PIECE, slot ^= 1) {
        const size_t len = bytes - off < PIECE ? bytes - off : PIECE;
        PCS_CUDA(cudaMemcpyAsync((char*)g_ctx.pin_out + (size_t)slot * PIECE, (const char*)src_dev + off, len, cudaMemcpyDeviceToHost, st));
        PCS_CUDA(cudaEventRecord(ev[slot], st));
        if (prev_len) {
            PCS_CUDA(cudaEventSynchronize(ev[slot ^ 1]));
            host_copy_mt((char*)dst + prev_off, (char*)g_ctx.pin_out + (size_t)(slot ^ 1) * PIECE, prev_len);
        }
        prev_off = off;
        prev_len = len;
    }
    PCS_CUDA(cudaEventSynchronize(ev[slot ^ 1]));
    host_copy_mt((char*)dst + prev_off, (char*)g_ctx.pin_out + (size_t)(slot ^ 1) * PIECE, prev_len);
    return PCS_OK;
}

// Row accessors of an on-demand batch: the leaf columns [0, width) on the cosets [c0, c1), recomputed group by group.
// body(cols, stride, j0, j1) reads leaf c0 * d + l of column j0 + k at cols[k * stride + l]: polynomial columns are
// regenerated from the kept coefficients into scratch ([LDE_GROUP][(c1 - c0) * d]); salt columns (width > w) are read where
// the batch keeps them.
template <class Body>
static int for_each_group(const pcs_batch* b, size_t width, size_t c0, size_t c1, uint64_t* scratch, cudaStream_t st,
                          Body body) {
    const size_t d = (size_t)1 << b->lg_d, stride = (c1 - c0) * d;
    NttPlan* plan = ntt_plan_get(b->lg_d, b->rate_bits, false, 7, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    for (size_t g0 = 0; g0 < b->w; g0 += LDE_GROUP) {
        const size_t g1 = b->w - g0 < LDE_GROUP ? b->w : g0 + LDE_GROUP;
        const uint64_t* src = b->coeffs + g0 * d;
        if (c1 - c0 == ((size_t)1 << b->rate_bits))
            PCS_CUDA(ntt_lde_cosets(plan, src, d, scratch, stride, g1 - g0, 0, b->rate_bits, st));
        else
            for (size_t c = c0; c < c1; c++)
                PCS_CUDA(ntt_lde_cosets(plan, src, d, scratch + (c - c0) * d, stride, g1 - g0, (unsigned)c, 0, st));
        if (int rc = body((const uint64_t*)scratch, stride, g0, g1)) return rc;
    }
    if (width > b->w) return body((const uint64_t*)b->salts + c0 * d, b->n, b->w, width);
    return PCS_OK;
}

extern "C" {

int pcs_coset_lde(const uint64_t* const* coeffs, size_t w, unsigned lg_d, unsigned rate_bits, uint64_t shift,
                  uint64_t* out, int layout) {
    if (int rc = need_init()) return rc;
    if (w == 0) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:103 polynomials[0])");
    if (!coeffs || !out) return fail(PCS_ERR_ARG, "NULL pointer");
    if (int rc = check_two_adicity(lg_d + rate_bits)) return rc;
    cudaStream_t st = g_ctx.stream;
    size_t d = (size_t)1 << lg_d, n = d << rate_bits;
    NttPlan* plan = ntt_plan_get(lg_d, rate_bits, false, shift, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    DevBuf c, lde, o;
    PCS_CUDA(c.alloc(w * d * 8, st));
    PCS_CUDA(lde.alloc(w * n * 8, st));
    PCS_CUDA(o.alloc(w * n * 8, st));
    int rc = stage_polys(coeffs, w, d, false, c.u64(), st);
    if (rc) return rc;
    PCS_CUDA(ntt_lde(plan, c.u64(), d, lde.u64(), n, w, st));
    if (layout == 0)
        PCS_CUDA(launch_bitrev_permute(lde.u64(), n, o.u64(), n, w, lg_d + rate_bits, st));
    else
        PCS_CUDA(launch_transpose(lde.u64(), n, o.u64(), w, w, n, st));
    PCS_CUDA(cudaMemcpyAsync(out, o.p, w * n * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_coset_lde_dev(const uint64_t* const* coeffs_dev, size_t w, unsigned lg_d, unsigned rate_bits, uint64_t shift,
                      uint64_t* out_dev) {
    if (int rc = need_init()) return rc;
    if (w == 0) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:103 polynomials[0])");
    if (!coeffs_dev || !out_dev) return fail(PCS_ERR_ARG, "NULL pointer");
    if (int rc = check_two_adicity(lg_d + rate_bits)) return rc;
    cudaStream_t st = g_ctx.stream;
    const size_t d = (size_t)1 << lg_d, n = d << rate_bits;
    NttPlan* plan = ntt_plan_get(lg_d, rate_bits, false, shift, st);
    if (!plan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    DevInput in;
    if (int rc = resolve_dev_input(coeffs_dev, w, lg_d, st, in)) return rc;
    PCS_CUDA(ntt_lde_cosets(plan, in.src, d, out_dev, n, w, 0, rate_bits, st, in.ptrs));
    return PCS_OK;   // asynchronous on pcs_stream()
}

int pcs_merkle_build(const uint64_t* leaves, size_t n, size_t len, unsigned cap_height, uint64_t* digests,
                     uint64_t* cap) {
    if (int rc = need_init()) return rc;
    int lg_n = ilog2_strict(n);
    if (lg_n < 0) return fail(PCS_ERR_NOT_POW2, "Not a power of two: " + std::to_string(n));
    if (int rc = check_cap_height(cap_height, (unsigned)lg_n)) return rc;
    if (!leaves || !cap || len == 0) return fail(PCS_ERR_ARG, "NULL pointer or empty leaves");
    cudaStream_t st = g_ctx.stream;
    size_t n_cap = (size_t)1 << cap_height, n_dig = 2 * (n - n_cap);
    if (n_dig && !digests) return fail(PCS_ERR_ARG, "digests is NULL");
    DevBuf d_rows, d_cols, d_dig, d_cap;
    PCS_CUDA(d_rows.alloc(n * len * 8, st));
    PCS_CUDA(d_cols.alloc(n * len * 8, st));
    PCS_CUDA(d_dig.alloc(n_dig * 32, st));
    PCS_CUDA(d_cap.alloc(n_cap * 32, st));
    PCS_CUDA(cudaMemcpyAsync(d_rows.p, leaves, n * len * 8, cudaMemcpyHostToDevice, st));
    PCS_CUDA(launch_transpose(d_rows.u64(), len, d_cols.u64(), n, n, len, st));
    int rc = build_tree_dev(d_cols.u64(), n, len, (unsigned)lg_n, cap_height, d_dig.u64(), d_cap.u64(), st, nullptr);
    if (rc) return rc;
    if (n_dig) PCS_CUDA(cudaMemcpyAsync(digests, d_dig.p, n_dig * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaMemcpyAsync(cap, d_cap.p, n_cap * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

// ------------------------------------------------------------------------------------------------
// fused hot path
// ------------------------------------------------------------------------------------------------
void pcs_batch_free(pcs_batch* b) {
    if (!b) return;
    BatchScope scope(b);
    cudaStream_t st = g_ctx.stream;
    if (b->coeffs) cudaFreeAsync(b->coeffs, st);
    if (b->lde) cudaFreeAsync(b->lde, st);
    if (b->salts) cudaFreeAsync(b->salts, st);
    if (b->digests) cudaFreeAsync(b->digests, st);
    if (b->cap) cudaFreeAsync(b->cap, st);
    if (b->sponge) cudaFreeAsync(b->sponge, st);
    if (b->ev[5] && b->committed) {
        PendingEvents pe;
        for (int i = 0; i < 6; i++) pe.ev[i] = b->ev[i];
        pe.absorb_ev.swap(b->absorb_ev);
        g_ctx.pending.push_back(pe);
        if (g_ctx.pending.size() > 256) {
            cudaStreamSynchronize(st);
            drain_pending();
        }
    } else {
        for (auto& e : b->ev)
            if (e) cudaEventDestroy(e);
    }
    for (auto& e : b->absorb_ev) cudaEventDestroy(e);
    delete b;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// the steps of commit_common
// ------------------------------------------------------------------------------------------------
// On every exit taken once H2D copies were enqueued on the copy stream, wait for them before the batch's owner returns their
// destination to the pool (and release the pinned ring slots).  Declared after the owner, so destroyed before it.
struct CopyDrain {
    bool armed = false;
    ~CopyDrain() {
        if (g_ctx.d2h_stream) cudaStreamSynchronize(g_ctx.d2h_stream);   // D2H copies out of a buffer the owner is about to free
        if (!armed || !g_ctx.copy_stream) return;
        cudaStreamSynchronize(g_ctx.copy_stream);
        for (auto& busy : g_ctx.ring_busy) busy = false;
    }
};

// Where the LDE reads a commitment's input (values or coefficients) from, and, for host inputs that arrive chunk by chunk
// on the copy stream, the chunk bounds: chunk k = polynomials [cb[k], cb[k+1]).
struct CommitInput {
    DevInput dev;
    std::vector<size_t> cb;   // empty: the whole input is in place once the main stream gets there
    bool pageable = false;    // chunks go through the pinned ring, each staged right before its compute is enqueued
};

// Device coefficients that are neither kept nor transformed are read in place; every other input is copied into b->coeffs:
// device inputs and small host polynomials at once, larger host polynomials chunk by chunk on the copy stream.
static int stage_inputs(const uint64_t* const* polys, bool from_values, unsigned flags, pcs_batch* b, CommitInput& in,
                        CopyDrain& drain) {
    cudaStream_t st = g_ctx.stream;
    const size_t w = b->w, d = (size_t)1 << b->lg_d;
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    if (dev_ptrs && !from_values && !(flags & PCS_KEEP_COEFFS)) return resolve_dev_input(polys, w, b->lg_d, st, in.dev);
    PCS_CUDA(cudaMallocAsync((void**)&b->coeffs, w * d * 8, st));   // owned by the batch from here on
    uint64_t* const staged = b->coeffs;
    in.dev.src = staged;
    if (dev_ptrs) {
        if (!contiguous(polys, w, d)) return stage_polys(polys, w, d, true, staged, st);
        PCS_CUDA(cudaMemcpyAsync(staged, polys[0], w * d * 8, cudaMemcpyDeviceToDevice, st));
        return PCS_OK;
    }
    if (d * 8 <= SMALL_POLY_BYTES && w * d * 8 <= PIN_STAGING_MAX && pinned(g_ctx.pin_in, g_ctx.pin_in_bytes, w * d * 8)) {
        // small host polynomials: one gather on the host, one H2D copy
        for (size_t j = 0; j < w; j++) {
            if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
            memcpy((char*)g_ctx.pin_in + j * d * 8, polys[j], d * 8);
        }
        PCS_CUDA(cudaMemcpyAsync(staged, g_ctx.pin_in, w * d * 8, cudaMemcpyHostToDevice, st));
        return PCS_OK;
    }
    // host inputs: chunked H2D on the copy stream, one event per chunk
    if (!g_ctx.copy_stream) PCS_CUDA(cudaStreamCreateWithFlags(&g_ctx.copy_stream, cudaStreamNonBlocking));
    if (!g_ctx.ev_sync) PCS_CUDA(cudaEventCreateWithFlags(&g_ctx.ev_sync, cudaEventDisableTiming));
    for (size_t j = 0; j < w; j++)
        if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
    in.pageable = w * d * 8 >= (8u << 20) && is_pageable_host(polys[0]);   // below 8 MB the threads cost more than they save
    // Chunk sizes: the first transfer is the only one nothing hides, so it is small (8 polynomials = one absorb of the
    // sponge, or one 16 MB ring slot's worth for short polynomials); a chunk's compute (LDE + its share of the leaf
    // hashing, ~0.9 ms per polynomial at 2^20) outlasts a transfer 5x its size, so the groups grow 5x and few sponge
    // states have to be parked (each group boundary costs 192 B of HBM traffic per leaf).
    std::vector<size_t>& cb = in.cb;
    size_t first = 8;
    if (first * d * 8 < RING_SLOT_BYTES) first = (RING_SLOT_BYTES / (d * 8) + 7) / 8 * 8;
    cb.assign(1, 0);
    for (size_t sz = first; cb.back() < w; sz *= 5) cb.push_back(cb.back() + sz < w ? cb.back() + sz : w);
    if (cb.size() > 2 && w - cb[cb.size() - 2] < 8) cb.erase(cb.end() - 2);   // no tiny tail group
    const size_t n_chunks = cb.size() - 1;
    while (g_ctx.chunk_ev.size() < n_chunks) {
        cudaEvent_t e;
        PCS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g_ctx.chunk_ev.push_back(e);
    }
    PCS_CUDA(cudaEventRecord(g_ctx.ev_sync, st));               // `staged` exists from here on
    PCS_CUDA(cudaStreamWaitEvent(g_ctx.copy_stream, g_ctx.ev_sync, 0));
    drain.armed = true;
    for (size_t k = 0; k < n_chunks && !in.pageable; k++) {
        if (int rc = stage_polys(polys + cb[k], cb[k + 1] - cb[k], d, false, staged + cb[k] * d, g_ctx.copy_stream)) return rc;
        PCS_CUDA(cudaEventRecord(g_ctx.chunk_ev[k], g_ctx.copy_stream));
    }
    return PCS_OK;
}

// How from_values returns the coefficients to coeffs_out
enum class CoeffsOut {
    none,
    small_pinned,   // one D2H copy into pinned staging after the LDE, scattered to the caller's vectors after the final sync
    big_pinned,     // every chunk's coefficients leave on the D2H stream into pinned staging while the LDE and the hashing go
                    // on, and are scattered into the caller's (pageable, separately allocated) vectors by a few host threads
    direct,         // one D2H copy per polynomial on the main stream
};

static CoeffsOut choose_coeffs_out(bool from_values, uint64_t* const* coeffs_out, size_t w, size_t d) {
    if (!from_values || !coeffs_out) return CoeffsOut::none;
    const size_t bytes = w * d * 8;
    if (d * 8 <= SMALL_POLY_BYTES && bytes <= PIN_STAGING_MAX && pinned(g_ctx.pin_out, g_ctx.pin_out_bytes, bytes))
        return CoeffsOut::small_pinned;
    // larger outputs: the reference keeps `polynomials`, so a Rust caller always asks for them
    if (bytes <= ((size_t)512 << 20) && pinned(g_ctx.pin_out, g_ctx.pin_out_bytes, bytes)) return CoeffsOut::big_pinned;
    return CoeffsOut::direct;
}

// after the commit has been synchronised: the coefficients staged in pinned memory into the caller's vectors
static int hand_back_coeffs(CoeffsOut mode, uint64_t* const* coeffs_out, size_t w, size_t d) {
    const char* srcp = (const char*)g_ctx.pin_out;
    if (mode == CoeffsOut::small_pinned)
        for (size_t j = 0; j < w; j++)
            if (coeffs_out[j]) memcpy(coeffs_out[j], srcp + j * d * 8, d * 8);
    if (mode == CoeffsOut::big_pinned) {
        PCS_CUDA(cudaStreamSynchronize(g_ctx.stream));
        PCS_CUDA(cudaStreamSynchronize(g_ctx.d2h_stream));
        const unsigned nt = STAGE_THREADS;
        std::thread th[STAGE_THREADS];
        for (unsigned t = 0; t < nt; t++)
            th[t] = std::thread([=]() {
                for (size_t j = t; j < w; j += nt)
                    if (coeffs_out[j]) memcpy(coeffs_out[j], srcp + j * d * 8, d * 8);
            });
        for (unsigned t = 0; t < nt; t++) th[t].join();
    }
    return PCS_OK;
}

// Blinding (oracle.rs:119-123): the caller's salt column k is in natural LDE order like lde_values, the leaves are in
// bit-reversed order (oracle.rs:84).  A shard's salt rows are its own leaf range, already in leaf order.
static int write_salts(pcs_batch* b, const uint64_t* const* salts, bool dev_ptrs, bool shard, cudaStream_t st) {
    const size_t n = b->n;
    for (size_t k = 0; k < b->salt_w; k++) {
        if (!salts[k]) return fail(PCS_ERR_ARG, "NULL salt pointer");
        uint64_t* row = b->on_demand ? b->salts + k * n : b->lde + (b->w + k) * n;
        DevBuf tmp;
        PCS_CUDA(tmp.alloc(n * 8, st));
        PCS_CUDA(cudaMemcpyAsync(tmp.p, salts[k], n * 8, dev_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        PCS_CUDA(launch_canonicalize(tmp.u64(), n, st));
        if (shard)
            PCS_CUDA(cudaMemcpyAsync(row, tmp.p, n * 8, cudaMemcpyDeviceToDevice, st));
        else
            PCS_CUDA(launch_bitrev_permute(tmp.u64(), n, row, n, 1, b->lg_d + b->rate_bits, st));
    }
    return PCS_OK;
}

// PolynomialBatch::from_coeffs / from_values (oracle.rs:43-125).
// shard == true: only the cosets [coset_first, coset_first + 2^lg_cosets) (leaf order) are extended and the
// tree is built over those d << lg_cosets leaves with `cap_height` (the caller's LOCAL cap height); salts are
// then the shard's rows, already in leaf order.
static int commit_common(const uint64_t* const* polys, bool from_values, size_t w, unsigned lg_d, unsigned rate_bits,
                         unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                         uint64_t* const* coeffs_out, uint64_t* cap_out, pcs_batch** out, bool shard = false,
                         unsigned coset_first = 0, unsigned lg_cosets = 0) {
    if (int rc = need_init()) return rc;
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (w == 0 || !polys) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:76 polynomials[0])");
    if (salt_w && !salts) return fail(PCS_ERR_ARG, "salts is NULL");
    if (!shard) lg_cosets = rate_bits;
    const bool on_demand = flags & PCS_LDE_ON_DEMAND;
    if (on_demand && shard) return fail(PCS_ERR_ARG, "PCS_LDE_ON_DEMAND is not supported by shard commits");
    if (on_demand) flags |= PCS_KEEP_COEFFS;   // the rows are recomputed from the coefficients: copy device inputs
    BatchOwner b;
    if (int rc = batch_begin(w, salt_w, lg_d, rate_bits, coset_first, lg_cosets, cap_height,
                             on_demand ? BATCH_ON_DEMAND : BATCH_LDE, b))
        return rc;
    cudaStream_t st = g_ctx.stream;
    NttPlan* iplan = from_values ? ntt_plan_get(lg_d, 0, true, 1, st) : nullptr;
    if (from_values && !iplan) return fail(PCS_ERR_ALLOC, "twiddle table allocation failed");
    b->has_ifft = from_values;
    CopyDrain drain;
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    const size_t d = (size_t)1 << lg_d, n = b->n, wt = w + salt_w;

    // ---- inputs ----
    CommitInput in;
    if (int rc = stage_inputs(polys, from_values, flags, b.get(), in, drain)) return rc;
    const uint64_t* const src = in.dev.src;
    const size_t n_chunks = in.cb.empty() ? 0 : in.cb.size() - 1;   // > 0: IFFT and LDE follow each chunk as it lands
    PCS_CUDA(cudaEventRecord(b->ev[0], st));

    // ---- "IFFT" (oracle.rs:51-55) for polynomials [j0, j1): values (natural order) -> coefficients in b->coeffs ----
    // scratch for the bit-reversed intermediate = the TAIL of the LDE buffer (the last w*d elements): LDE rows already
    // written for earlier polynomials end at j0*n <= wt*n - w*d + j0*d, so chunk-by-chunk processing never clobbers them.
    // An on-demand batch has no LDE buffer: it transforms group by group through the group scratch (chunked inputs), or all
    // at once through a [w][d] buffer released before the group scratch is allocated.
    DevBuf ifft_buf, group_scratch;
    if (on_demand && from_values && in.cb.empty()) PCS_CUDA(ifft_buf.alloc(w * d * 8, st));
    uint64_t* const ifft_scratch = on_demand ? ifft_buf.u64() : b->lde + (wt * n - w * d);
    uint64_t* const coeffs = b->coeffs;
    const CoeffsOut mode = choose_coeffs_out(from_values, coeffs_out, w, d);
    if (mode == CoeffsOut::big_pinned && !g_ctx.d2h_stream)
        PCS_CUDA(cudaStreamCreateWithFlags(&g_ctx.d2h_stream, cudaStreamNonBlocking));
    size_t n_d2h = 0;
    auto ifft_range = [&](size_t j0, size_t j1) -> int {
        uint64_t* const scr = on_demand && !ifft_buf.p ? b->scratch : ifft_scratch + j0 * d;
        PCS_CUDA(ntt_inverse_bitrev(iplan, src + j0 * d, d, scr, d, j1 - j0, st));
        PCS_CUDA(launch_bitrev_permute(scr, d, coeffs + j0 * d, d, j1 - j0, lg_d, st, ntt_plan_scale(iplan)));
        if (mode == CoeffsOut::big_pinned) {
            if (g_ctx.d2h_ev.size() <= n_d2h) {
                cudaEvent_t e;
                PCS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                g_ctx.d2h_ev.push_back(e);
            }
            PCS_CUDA(cudaEventRecord(g_ctx.d2h_ev[n_d2h], st));
            PCS_CUDA(cudaStreamWaitEvent(g_ctx.d2h_stream, g_ctx.d2h_ev[n_d2h], 0));
            n_d2h++;
            PCS_CUDA(cudaMemcpyAsync((char*)g_ctx.pin_out + j0 * d * 8, coeffs + j0 * d, (j1 - j0) * d * 8, cudaMemcpyDeviceToHost,
                                     g_ctx.d2h_stream));
        } else if (mode == CoeffsOut::direct) {
            for (size_t j = j0; j < j1; j++)
                if (coeffs_out[j])
                    PCS_CUDA(cudaMemcpyAsync(coeffs_out[j], coeffs + j * d, d * 8, cudaMemcpyDeviceToHost, st));
        }
        return PCS_OK;
    };
    if (from_values && !n_chunks)
        if (int rc = ifft_range(0, w)) return rc;
    PCS_CUDA(cudaEventRecord(b->ev[1], st));

    // ---- "FFT + blinding" (oracle.rs:100-125), output already in leaf order ----
    // On demand: polynomials [j0, j1) are extended and absorbed in groups of <= LDE_GROUP through one scratch of LDE_GROUP
    // columns plus the salt rows, which follow the last group's columns (written first: they cannot be recomputed).
    auto extend = [&](size_t j0, size_t j1, bool ifft) -> int {
        if (!on_demand) {
            if (ifft)
                if (int rc = ifft_range(j0, j1)) return rc;
            return batch_extend(b.get(), src + j0 * d, j0 == 0 && j1 == w ? in.dev.ptrs : nullptr, j0, j1 - j0);
        }
        for (size_t g0 = j0; g0 < j1; g0 += LDE_GROUP) {
            const size_t g1 = j1 - g0 < LDE_GROUP ? j1 : g0 + LDE_GROUP;
            if (ifft)
                if (int rc = ifft_range(g0, g1)) return rc;
            if (int rc = batch_extend(b.get(), src + g0 * d, nullptr, g0, g1 - g0)) return rc;
        }
        return PCS_OK;
    };
    if (on_demand) {
        ifft_buf.release();
        PCS_CUDA(group_scratch.alloc((LDE_GROUP + salt_w) * n * 8, st));
        b->scratch = group_scratch.u64();
        if (int rc = write_salts(b.get(), salts, dev_ptrs, shard, st)) return rc;
    }
    for (size_t k = 0; k < n_chunks; k++) {
        const size_t j0 = in.cb[k], j1 = in.cb[k + 1];
        if (in.pageable) {
            if (int rc = stage_pageable(polys + j0, j1 - j0, d, coeffs + j0 * d, g_ctx.copy_stream)) return rc;
            PCS_CUDA(cudaEventRecord(g_ctx.chunk_ev[k], g_ctx.copy_stream));
        }
        PCS_CUDA(cudaStreamWaitEvent(st, g_ctx.chunk_ev[k], 0));
        if (int rc = extend(j0, j1, from_values)) return rc;
    }
    if (!n_chunks)
        if (int rc = extend(0, w, false)) return rc;
    if (mode == CoeffsOut::small_pinned) PCS_CUDA(cudaMemcpyAsync(g_ctx.pin_out, coeffs, w * d * 8, cudaMemcpyDeviceToHost, st));
    if (!on_demand)
        if (int rc = write_salts(b.get(), salts, dev_ptrs, shard, st)) return rc;

    // ---- "transpose LDEs" (fused away), "build Merkle tree" (oracle.rs:83-89) ----
    if (int rc = batch_finish(b.get(), cap_out)) return rc;
    b->scratch = nullptr;   // group_scratch goes back to the pool, in stream order, on return
    if (b->coeffs && !from_values && !(flags & PCS_KEEP_COEFFS)) {
        cudaFreeAsync(b->coeffs, st);
        b->coeffs = nullptr;
    }
    if (!cap_out && (!dev_ptrs || mode == CoeffsOut::small_pinned))
        PCS_CUDA(cudaStreamSynchronize(st));  // host inputs must not be reused before the copies finish
    if (int rc = hand_back_coeffs(mode, coeffs_out, w, d)) return rc;
    drain.armed = false;   // the main stream waited on every chunk event and has been synchronised (host inputs)
    *out = b.release();
    return PCS_OK;
}

extern "C" {

int pcs_commit_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits,
                           unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                           uint64_t* cap_out, pcs_batch** out) {
    return commit_common(polys, false, w, lg_d, rate_bits, cap_height, salts, salt_w, flags, nullptr, cap_out, out);
}

int pcs_commit_shard_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits,
                                 unsigned coset_first, unsigned lg_cosets, unsigned local_cap_height,
                                 const uint64_t* const* salts, size_t salt_w, unsigned flags, uint64_t* cap_out,
                                 pcs_batch** out) {
    return commit_common(polys, false, w, lg_d, rate_bits, local_cap_height, salts, salt_w, flags, nullptr, cap_out, out,
                         true, coset_first, lg_cosets);
}

// ---- streaming shard commit: the polynomials arrive in groups (e.g. chunks of an all-gather still in flight) ----
// The input and IFFT phases of such a shard are empty.
static int shard_open(BatchOwner& b, pcs_batch** out) {
    PCS_CUDA(cudaEventRecord(b->ev[0], g_ctx.stream));
    PCS_CUDA(cudaEventRecord(b->ev[1], g_ctx.stream));
    *out = b.release();
    return PCS_OK;
}

int pcs_shard_begin(size_t w, size_t salt_w, unsigned lg_d, unsigned rate_bits, unsigned coset_first, unsigned lg_cosets,
                    unsigned local_cap_height, pcs_batch** out) {
    if (int rc = need_init()) return rc;
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (w == 0) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:76 polynomials[0])");
    BatchOwner b;
    if (int rc = batch_begin(w, salt_w, lg_d, rate_bits, coset_first, lg_cosets, local_cap_height, BATCH_LDE, b)) return rc;
    return shard_open(b, out);
}

// A tree shard whose LDE rows are computed elsewhere (another GPU's LDE arriving over NVLink: the north-star's
// polynomial-partitioned LDE + all-to-all): `width` rows of 2^lg_n leaves each, filled through pcs_shard_set_rows or written
// in place at pcs_batch_lde_dev() + row * 2^lg_n, then pcs_shard_finish.
int pcs_shard_begin_rows(size_t width, size_t salt_w, unsigned lg_n, unsigned local_cap_height, pcs_batch** out) {
    if (int rc = need_init()) return rc;
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (width == 0) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:76 polynomials[0])");
    if (salt_w > width) return fail(PCS_ERR_ARG, "more salt columns than columns");
    BatchOwner b;
    if (int rc = batch_begin(width - salt_w, salt_w, lg_n, 0, 0, 0, local_cap_height, BATCH_ROWS, b)) return rc;
    return shard_open(b, out);
}

int pcs_shard_set_rows(pcs_batch* b, size_t row_first, size_t count, const uint64_t* const* rows_dev, int canonical) {
    if (!b || (count && !rows_dev)) return fail(PCS_ERR_ARG, "NULL pointer");
    BatchScope scope(b);
    if (b->committed) return fail(PCS_ERR_ARG, "batch already finished");
    const size_t wt = b->w + b->salt_w;
    if (row_first > wt || count > wt - row_first) return fail(PCS_ERR_ARG, "row range out of bounds");
    cudaStream_t st = g_ctx.stream;
    for (size_t k = 0; k < count; k++) {
        if (!rows_dev[k]) return fail(PCS_ERR_ARG, "NULL row pointer");
        uint64_t* dst = b->lde + (row_first + k) * b->n;
        if (rows_dev[k] != dst)
            PCS_CUDA(cudaMemcpyAsync(dst, rows_dev[k], b->n * 8, cudaMemcpyDeviceToDevice, st));
    }
    if (!canonical && count) PCS_CUDA(launch_canonicalize(b->lde + row_first * b->n, count * b->n, st));
    return PCS_OK;   // asynchronous on pcs_stream()
}

int pcs_shard_extend(pcs_batch* b, size_t poly_first, size_t count, const uint64_t* const* polys) {
    BatchScope scope(b);
    if (!b || !polys) return fail(PCS_ERR_ARG, "NULL pointer");
    if (b->committed) return fail(PCS_ERR_ARG, "batch already finished");
    if (b->rows_only) return fail(PCS_ERR_ARG, "this shard takes LDE rows (pcs_shard_set_rows), not polynomials");
    if (poly_first > b->w || count > b->w - poly_first) return fail(PCS_ERR_ARG, "polynomial range out of bounds");
    if (count == 0) return PCS_OK;
    DevInput in;
    if (int rc = resolve_dev_input(polys, count, b->lg_d, g_ctx.stream, in)) return rc;
    return batch_extend(b, in.src, in.ptrs, poly_first, count);   // asynchronous on pcs_stream()
}

int pcs_shard_finish(pcs_batch* b, uint64_t* cap_out) {
    BatchScope scope(b);
    if (!b) return fail(PCS_ERR_ARG, "NULL pointer");
    if (b->committed) return fail(PCS_ERR_ARG, "batch already finished");
    return batch_finish(b, cap_out);
}

int pcs_commit_from_values(const uint64_t* const* values, size_t w, unsigned lg_d, unsigned rate_bits,
                           unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                           uint64_t* const* coeffs_out, uint64_t* cap_out, pcs_batch** out) {
    return commit_common(values, true, w, lg_d, rate_bits, cap_height, salts, salt_w, flags, coeffs_out, cap_out, out);
}

int pcs_batch_shape(const pcs_batch* b, size_t* n_leaves, size_t* leaf_len, size_t* n_digests, unsigned* cap_height) {
    if (!b) return fail(PCS_ERR_ARG, "batch is NULL");
    if (n_leaves) *n_leaves = b->n;
    if (leaf_len) *leaf_len = b->w + b->salt_w;
    if (n_digests) *n_digests = b->n_digests;
    if (cap_height) *cap_height = b->cap_height;
    return PCS_OK;
}

int pcs_batch_cap(const pcs_batch* b, uint64_t* cap) {
    BatchScope scope(b);
    if (!b || !cap) return fail(PCS_ERR_ARG, "NULL pointer");
    cudaStream_t st = g_ctx.stream;
    PCS_CUDA(cudaMemcpyAsync(cap, b->cap, ((size_t)32) << b->cap_height, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_digests(const pcs_batch* b, uint64_t* digests) {
    BatchScope scope(b);
    if (!b) return fail(PCS_ERR_ARG, "NULL pointer");
    if (b->n_digests == 0) return PCS_OK;
    if (!digests) return fail(PCS_ERR_ARG, "NULL pointer");
    cudaStream_t st = g_ctx.stream;
    PCS_CUDA(cudaMemcpyAsync(digests, b->digests, b->n_digests * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_leaves(const pcs_batch* b, size_t first, size_t count, uint64_t* rows) {
    BatchScope scope(b);
    if (!b || !rows) return fail(PCS_ERR_ARG, "NULL pointer");
    if (first > b->n || count > b->n - first) return fail(PCS_ERR_ARG, "leaf range out of bounds");
    if (count == 0) return PCS_OK;
    cudaStream_t st = g_ctx.stream;
    size_t wt = b->w + b->salt_w;
    // transpose in slabs so that the staging buffer stays small
    size_t slab = (size_t)1 << 18;
    const size_t d = (size_t)1 << b->lg_d;
    // on demand, every slab regenerates the cosets it touches: slabs of up to a coset (and 1 GB) waste less of that work
    while (b->on_demand && slab < d && 2 * slab * wt * 8 <= ((size_t)1 << 30)) slab *= 2;
    DevBuf tmp, scratch;
    PCS_CUDA(tmp.alloc((count < slab ? count : slab) * wt * 8, st));
    if (b->on_demand) {
        size_t span = (slab + d - 1) / d + 1;   // cosets one slab can touch
        if (span > ((size_t)1 << b->rate_bits)) span = (size_t)1 << b->rate_bits;
        PCS_CUDA(scratch.alloc(LDE_GROUP * span * d * 8, st));
    }
    for (size_t off = 0; off < count; off += slab) {
        size_t c = count - off < slab ? count - off : slab;
        if (b->on_demand) {
            const size_t f = first + off, c0 = f / d, c1 = (f + c - 1) / d + 1;
            int rc = for_each_group(b, wt, c0, c1, scratch.u64(), st, [&](const uint64_t* cols, size_t stride, size_t j0, size_t j1) {
                PCS_CUDA(launch_transpose(cols + (f - c0 * d), stride, tmp.u64() + j0, wt, j1 - j0, c, st));
                return PCS_OK;
            });
            if (rc) return rc;
        } else {
            PCS_CUDA(launch_transpose(b->lde + first + off, b->n, tmp.u64(), wt, wt, c, st));
        }
        int rc = d2h_pageable(rows + off * wt, tmp.p, c * wt * 8, st);
        if (rc) return rc;
    }
    return PCS_OK;
}

int pcs_batch_get_rows(const pcs_batch* b, const uint64_t* leaf_indices, size_t n, uint64_t* rows) {
    BatchScope scope(b);
    if (!b || (n && (!leaf_indices || !rows))) return fail(PCS_ERR_ARG, "NULL pointer");
    if (n == 0) return PCS_OK;
    for (size_t k = 0; k < n; k++)
        if (leaf_indices[k] >= b->n) return fail(PCS_ERR_ARG, "leaf index out of bounds");
    cudaStream_t st = g_ctx.stream;
    size_t wt = b->w + b->salt_w;
    DevBuf idx, o;
    PCS_CUDA(idx.alloc(n * 8, st));
    PCS_CUDA(o.alloc(n * wt * 8, st));
    std::vector<uint64_t> rel;   // on demand, many rows: leaf indices relative to the first coset regenerated
    if (b->on_demand && n <= ROWS_EVAL_MAX) {
        PCS_CUDA(cudaMemcpyAsync(idx.p, leaf_indices, n * 8, cudaMemcpyHostToDevice, st));
        if (int rc = rows_eval(b, idx.u64(), n, o.u64(), st)) return rc;
    } else if (b->on_demand) {
        // regenerate the cosets [c0, c1) the leaves fall in, group by group, and gather from each group
        const size_t d = (size_t)1 << b->lg_d;
        size_t lo = leaf_indices[0], hi = leaf_indices[0];
        for (size_t k = 1; k < n; k++) {
            lo = leaf_indices[k] < lo ? leaf_indices[k] : lo;
            hi = leaf_indices[k] > hi ? leaf_indices[k] : hi;
        }
        const size_t c0 = lo / d, c1 = hi / d + 1;
        rel.assign(leaf_indices, leaf_indices + n);
        for (auto& i : rel) i -= c0 * d;
        PCS_CUDA(cudaMemcpyAsync(idx.p, rel.data(), n * 8, cudaMemcpyHostToDevice, st));
        DevBuf scratch, g;
        PCS_CUDA(scratch.alloc(LDE_GROUP * (c1 - c0) * d * 8, st));
        PCS_CUDA(g.alloc(n * (LDE_GROUP > b->salt_w ? LDE_GROUP : b->salt_w) * 8, st));
        int rc = for_each_group(b, wt, c0, c1, scratch.u64(), st, [&](const uint64_t* cols, size_t stride, size_t j0, size_t j1) {
            PCS_CUDA(launch_gather_rows(cols, stride, (uint32_t)(j1 - j0), idx.u64(), n, g.u64(), st));
            PCS_CUDA(cudaMemcpy2DAsync(o.u64() + j0, wt * 8, g.p, (j1 - j0) * 8, (j1 - j0) * 8, n, cudaMemcpyDeviceToDevice, st));
            return PCS_OK;
        });
        if (rc) return rc;
    } else {
        PCS_CUDA(cudaMemcpyAsync(idx.p, leaf_indices, n * 8, cudaMemcpyHostToDevice, st));
        PCS_CUDA(launch_gather_rows(b->lde, b->n, (uint32_t)wt, idx.u64(), n, o.u64(), st));
    }
    PCS_CUDA(cudaMemcpyAsync(rows, o.p, n * wt * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_lde_natural(const pcs_batch* b, size_t index_start, size_t step, size_t count, uint64_t* rows) {
    BatchScope scope(b);
    if (!b || (count && !rows)) return fail(PCS_ERR_ARG, "NULL pointer");
    if (count == 0) return PCS_OK;
    if (step == 0 || (step & (step - 1))) return fail(PCS_ERR_ARG, "step must be a power of two");
    // (index_start + k) * step < N for every k (oracle.rs:129-130 indexes merkle_tree.leaves with the reversed product)
    if (index_start > b->n / step || count > b->n / step - index_start) return fail(PCS_ERR_ARG, "point range out of bounds");
    cudaStream_t st = g_ctx.stream;
    const size_t w = b->w;                       // salt columns are dropped (oracle.rs:131-132)
    const unsigned lg_n = b->lg_d + b->rate_bits;
    // slabs of <= 256 MB: gather on the device, then stream to the caller's (usually pageable) rows.  On demand every slab
    // regenerates the LDE, so slabs are 1 GB.
    const size_t SLAB = (size_t)(b->on_demand ? 1024 : 256) << 20;
    size_t ch = SLAB / (w * 8);
    if (ch < 1) ch = 1;
    if (ch > count) ch = count;
    DevBuf tmp, scratch, g;
    PCS_CUDA(tmp.alloc(ch * w * 8, st));
    // natural points that are multiples of step = 2^s lie on the cosets [0, 2^(rate_bits - s)) of the leaf order
    unsigned s = 0;
    while (((size_t)1 << s) < step) s++;
    const size_t d = (size_t)1 << b->lg_d, c1 = (size_t)1 << (s < b->rate_bits ? b->rate_bits - s : 0);
    if (b->on_demand) {
        PCS_CUDA(scratch.alloc(LDE_GROUP * c1 * d * 8, st));
        PCS_CUDA(g.alloc(ch * LDE_GROUP * 8, st));
    }
    for (size_t off = 0; off < count; off += ch) {
        const size_t c = count - off < ch ? count - off : ch;
        if (b->on_demand) {
            int rc = for_each_group(b, w, 0, c1, scratch.u64(), st, [&](const uint64_t* cols, size_t stride, size_t j0, size_t j1) {
                PCS_CUDA(launch_lde_natural(cols, stride, (uint32_t)(j1 - j0), lg_n, index_start + off, step, c, g.u64(), st));
                PCS_CUDA(cudaMemcpy2DAsync(tmp.u64() + j0, w * 8, g.p, (j1 - j0) * 8, (j1 - j0) * 8, c, cudaMemcpyDeviceToDevice, st));
                return PCS_OK;
            });
            if (rc) return rc;
        } else {
            PCS_CUDA(launch_lde_natural(b->lde, b->n, (uint32_t)w, lg_n, index_start + off, step, c, tmp.u64(), st));
        }
        int rc = d2h_pageable(rows + off * w, tmp.p, c * w * 8, st);
        if (rc) return rc;
    }
    return PCS_OK;
}

int pcs_batch_prove(const pcs_batch* b, size_t leaf_index, uint64_t* siblings) {
    BatchScope scope(b);
    if (!b) return fail(PCS_ERR_ARG, "NULL pointer");
    if (leaf_index >= b->n) return fail(PCS_ERR_ARG, "leaf index out of bounds");
    unsigned lg_sub = b->lg_d + b->rate_bits - b->cap_height;
    if (lg_sub == 0) return PCS_OK;
    if (!siblings) return fail(PCS_ERR_ARG, "NULL pointer");
    cudaStream_t st = g_ctx.stream;
    DevBuf o;
    PCS_CUDA(o.alloc(lg_sub * 32, st));
    PCS_CUDA(launch_prove(b->digests, lg_sub, leaf_index, o.u64(), st));
    PCS_CUDA(cudaMemcpyAsync(siblings, o.p, lg_sub * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_prove_many(const pcs_batch* b, const uint64_t* leaf_indices, size_t n, uint64_t* siblings) {
    BatchScope scope(b);
    if (!b || (n && !leaf_indices)) return fail(PCS_ERR_ARG, "NULL pointer");
    for (size_t k = 0; k < n; k++)
        if (leaf_indices[k] >= b->n) return fail(PCS_ERR_ARG, "leaf index out of bounds");
    unsigned lg_sub = b->lg_d + b->rate_bits - b->cap_height;
    if (lg_sub == 0 || n == 0) return PCS_OK;
    if (!siblings) return fail(PCS_ERR_ARG, "NULL pointer");
    cudaStream_t st = g_ctx.stream;
    DevBuf o, idx;
    PCS_CUDA(o.alloc(n * lg_sub * 32, st));
    PCS_CUDA(idx.alloc(n * 8, st));
    PCS_CUDA(cudaMemcpyAsync(idx.p, leaf_indices, n * 8, cudaMemcpyHostToDevice, st));
    PCS_CUDA(launch_prove_many(b->digests, lg_sub, idx.u64(), n, o.u64(), st));
    PCS_CUDA(cudaMemcpyAsync(siblings, o.p, n * lg_sub * 32, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_coeffs(const pcs_batch* b, size_t poly, uint64_t* coeffs) {
    BatchScope scope(b);
    if (!b || !coeffs) return fail(PCS_ERR_ARG, "NULL pointer");
    if (!b->coeffs) return fail(PCS_ERR_ARG, "coefficients were not kept (PCS_KEEP_COEFFS)");
    if (poly >= b->w) return fail(PCS_ERR_ARG, "polynomial index out of bounds");
    cudaStream_t st = g_ctx.stream;
    size_t d = (size_t)1 << b->lg_d;
    PCS_CUDA(cudaMemcpyAsync(coeffs, b->coeffs + poly * d, d * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_batch_all_coeffs(const pcs_batch* b, uint64_t* coeffs) {
    BatchScope scope(b);
    if (!b || !coeffs) return fail(PCS_ERR_ARG, "NULL pointer");
    if (!b->coeffs) return fail(PCS_ERR_ARG, "coefficients were not kept (PCS_KEEP_COEFFS)");
    cudaStream_t st = g_ctx.stream;
    PCS_CUDA(cudaMemcpyAsync(coeffs, b->coeffs, (b->w << b->lg_d) * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

const uint64_t* pcs_batch_lde_dev(const pcs_batch* b) { return b ? b->lde : nullptr; }   // NULL for an on-demand batch
const uint64_t* pcs_batch_coeffs_dev(const pcs_batch* b) { return b ? b->coeffs : nullptr; }
const uint64_t* pcs_batch_digests_dev(const pcs_batch* b) { return b ? b->digests : nullptr; }
const uint64_t* pcs_batch_cap_dev(const pcs_batch* b) { return b ? b->cap : nullptr; }

int pcs_batch_timings(const pcs_batch* b, float ms[5]) {
    BatchScope scope(b);
    if (!b || !ms) return fail(PCS_ERR_ARG, "NULL pointer");
    PCS_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return phase_times(b, ms);
}

int pcs_timing_totals(float ms[5], unsigned* n_commits, int reset) {
    if (int rc = need_init()) return rc;
    PCS_CUDA(cudaStreamSynchronize(g_ctx.stream));
    drain_pending();
    if (ms)
        for (int i = 0; i < 5; i++) ms[i] = g_ctx.totals[i];
    if (n_commits) *n_commits = g_ctx.n_totals;
    if (reset) {
        for (auto& t : g_ctx.totals) t = 0;
        g_ctx.n_totals = 0;
    }
    return PCS_OK;
}

}  // extern "C"
