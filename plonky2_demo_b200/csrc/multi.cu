// One commitment over several GPUs of one box, driven from ONE host process (include/pcs.h, pcs_multi_*).
//
// The reference has no distributed path (one process, one rayon pool: SURVEY 5, 8e); its caller -- prove() in
// plonky2/src/plonk/prover.rs:145,212,260 -- is a single Rust thread.  This file is what lets that caller use a whole
// 8 x B200 box without Python, torch or a process per GPU: the library owns one engine context per device, one host
// worker thread per device, and the exchange step runs INSIDE the first NTT pass.
//
// Partition (same as plonky2_demo_b200/sharded.py): in leaf order the LDE is 2^rate_bits coset blocks, block c = the
// evaluations of all polynomials on 7 w_N^brev(c) <w_d>.  Device g of G owns the coset blocks [g 2^r / G, (g+1) 2^r / G) =
// a contiguous leaf range = whole cap subtrees = a contiguous slice of the reference's `digests` (merkle_tree.rs:43-46).
// It needs every polynomial's coefficients and nobody's LDE output.
//
// Exchange = peer memory, fused with compute (default): every device holds a block of the polynomials (its share of each H2D chunk);
// the first NTT pass of every device follows a per-polynomial pointer table and loads the other devices' coefficients
// straight from their HBM over NVLink / NVSwitch (k_ntt_pass, PassArgs::in_ptrs) -- no staging copy, no collective, the
// transfer is hidden behind the butterflies.  Cross-device ordering is one cudaStreamWaitEvent per (peer, chunk): inside
// one process an event recorded on device p's copy stream can be waited on by device q's compute stream.
// PCS_MULTI_CE_GATHER selects the other exchange that was built and measured: every device PULLS the other devices' parts of
// polynomial group c+1 into a local copy with peer cudaMemcpyAsync (copy engines, no SMs) while it extends and hashes group c.
// On 8 x B200 it loses clearly (device-resident inputs: 28.8 ms per commitment against 17.1 ms with the fused peer loads; host
// inputs 22.0 against 20.3 ms, profiles/r02_scaling.md): eight devices pulling 118 x 8 MB each through the copy engines reach
// ~70 GB/s per device, while the NTT pass streams the same bytes at NVLink speed behind its butterflies.
// Host inputs are cut into chunks so that the LDE of chunk c runs while chunk c+1 crosses PCIe on every device at once.
//
// More devices than coset blocks (n_devices > 2^rate_bits): the coset partition does not apply, so the other partition of
// SURVEY 8e is used -- every device extends ITS polynomials over all cosets (pcs_coset_lde_dev) and every device pulls, for
// every polynomial, the slice of its own leaf range out of the owner's LDE (peer cudaMemcpyAsync) straight into a row shard
// (pcs_shard_begin_rows), then hashes.  Same results, same accessors; leaf ranges are fractions of a coset block.
#include <atomic>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

struct pcs_multi_batch {
    int n_dev = 0;
    size_t w = 0, salt_w = 0;
    unsigned lg_d = 0, rate_bits = 0, cap_height = 0;
    unsigned lg_dev = 0, lg_cosets = 0, local_cap_height = 0, top_levels = 0;
    unsigned lg_local = 0;                         // log2(leaves per device)
    std::vector<pcs_batch*> shard;                 // per device
    std::vector<const uint64_t*> poly_ptr;         // [w] device address of every polynomial's coefficients (kept blocks or the caller's)
    std::vector<uint64_t*> owned_blocks;           // coefficient blocks this batch owns (PCS_KEEP_COEFFS / from_values)
    std::vector<int> owned_block_dev;
    std::vector<uint64_t> local_caps;              // [n_dev][2^local_cap_height][4]
    std::vector<uint64_t> cap;                     // [2^cap_height][4]
};

namespace pcs {
namespace {

struct FreeBlock { uint64_t* p; size_t bytes; };

struct Multi {
    bool init = false;
    std::vector<int> devices;
    std::vector<cudaStream_t> copy_stream;              // per device
    std::vector<std::vector<FreeBlock>> free_blocks;    // per device: cudaMalloc'ed coefficient blocks kept for reuse
    std::vector<std::vector<cudaEvent_t>> chunk_ev;     // [device][chunk]: "my part of chunk c is in my block"
    std::vector<cudaStream_t> gather_stream;            // per device: copy-engine pulls of the other devices' parts
    std::vector<std::vector<cudaEvent_t>> gather_ev;    // [device][chunk]: "all of chunk c is in my local copy"
};
Multi g_multi;
std::recursive_mutex g_multi_mutex;   // one multi commit at a time (recursive: a failing commit frees its batch under the lock)

constexpr size_t MULTI_MAX_CHUNKS = 16;

uint64_t* block_take(int gi, size_t bytes) {
    auto& fl = g_multi.free_blocks[gi];
    for (size_t i = 0; i < fl.size(); i++)
        if (fl[i].bytes >= bytes && fl[i].bytes <= 2 * bytes) {
            uint64_t* p = fl[i].p;
            fl.erase(fl.begin() + i);
            return p;
        }
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        // give cached blocks back and retry once
        for (auto& b : fl) cudaFree(b.p);
        fl.clear();
        cudaGetLastError();
        if (cudaMalloc(&p, bytes) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
    }
    return (uint64_t*)p;
}

size_t block_bytes(size_t rows, size_t d) { return (rows ? rows : 1) * d * 8; }

struct Plan {
    int G;
    unsigned lg_dev, lg_cosets, local_cap_height, top_levels;
    size_t chunks;
    size_t w;
    std::vector<size_t> bounds;   // chunk c = polynomials [bounds[c], bounds[c+1])
    // Groups for the streaming pipeline.  The H2D copies run back to back on the copy stream; a group boundary only decides
    // when compute may start on what has arrived.  With t = transfer time and c = compute time per polynomial (rho = t / c < 1),
    // group k+1 has landed before group k is finished iff  b[k+2] <= b[1] + b[k+1] / rho  (b = cumulative bounds), so the
    // groups may grow geometrically and only the FIRST transfer (8 polynomials = one sponge absorb) is exposed.  Boundaries are
    // multiples of the sponge rate 8 so that every group is hashed as soon as it is extended.
    void make_chunks(double rho) {
        bounds.assign(1, 0);
        if (rho <= 0 || w <= 16) {
            bounds.push_back(w);
        } else {
            bounds.push_back(8);
            while (bounds.back() < w && bounds.size() < MULTI_MAX_CHUNKS) {
                size_t next = (size_t)(8 + bounds.back() / rho) / 8 * 8;
                if (next <= bounds.back()) next = bounds.back() + 8;
                bounds.push_back(next < w ? next : w);
            }
            if (bounds.back() < w) bounds.back() = w;
            if (bounds.size() > 2 && w - bounds[bounds.size() - 2] < 8) bounds.erase(bounds.end() - 2);
        }
        chunks = bounds.size() - 1;
    }
    // polynomials [lo, hi) of chunk c; device g holds rows [lo + g m, min(lo + (g+1) m, hi)) of it, m = ceil((hi-lo)/G)
    void chunk_range(size_t c, size_t& lo, size_t& hi) const {
        lo = bounds[c];
        hi = bounds[c + 1];
    }
    void part(size_t c, int g, size_t& a, size_t& b) const {
        size_t lo, hi;
        chunk_range(c, lo, hi);
        size_t m = (hi - lo + G - 1) / G;
        a = lo + g * m < hi ? lo + g * m : hi;
        b = a + m < hi ? a + m : hi;
    }
    size_t rows_of(int g) const {
        size_t n = 0;
        for (size_t c = 0; c < chunks; c++) {
            size_t a, b;
            part(c, g, a, b);
            n += b - a;
        }
        return n;
    }
};

// The levels of two_to_one above the devices' local caps (merkle_tree.rs:69-96): `level` (digests in device order) becomes the
// level `levels` above.  With `siblings`, the sibling of node `idx` is collected at every level on the way, bottom-up.
int combine_top_levels(std::vector<uint64_t>& level, unsigned levels, size_t idx, uint64_t* siblings) {
    for (unsigned t = 0; t < levels; t++, idx >>= 1) {
        if (siblings) memcpy(siblings + (size_t)t * 4, level.data() + (idx ^ 1) * 4, 32);
        const size_t m = level.size() / 8;
        std::vector<uint64_t> l(m * 4), r(m * 4), o(m * 4);
        for (size_t i = 0; i < m; i++)
            for (int k = 0; k < 4; k++) {
                l[4 * i + k] = level[8 * i + k];
                r[4 * i + k] = level[8 * i + 4 + k];
            }
        if (int rc = pcs_two_to_one(l.data(), r.data(), m, o.data())) return rc;
        level.swap(o);
    }
    return PCS_OK;
}

}  // namespace

void multi_shutdown_locked() {
    if (!g_multi.init) return;
    for (size_t gi = 0; gi < g_multi.devices.size(); gi++) {
        cudaSetDevice(g_multi.devices[gi]);
        cudaDeviceSynchronize();
        for (auto& b : g_multi.free_blocks[gi]) cudaFree(b.p);
        for (auto& e : g_multi.chunk_ev[gi]) cudaEventDestroy(e);
        for (auto& e : g_multi.gather_ev[gi]) cudaEventDestroy(e);
        if (g_multi.copy_stream[gi]) cudaStreamDestroy(g_multi.copy_stream[gi]);
        if (g_multi.gather_stream[gi]) cudaStreamDestroy(g_multi.gather_stream[gi]);
    }
    g_multi = Multi();
    cudaGetLastError();
}

}  // namespace pcs

using namespace pcs;

extern "C" {

int pcs_multi_init(const int* devices, int n_devices) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(PCS_ERR_CUDA, std::string("no CUDA device: the engine has no CPU fallback (") + cudaGetErrorString(e) + ")");
    std::vector<int> devs;
    if (!devices) {
        if (n_devices <= 0) n_devices = count;   // NULL, 0: every visible device (rounded down to a power of two)
        while (n_devices & (n_devices - 1)) n_devices &= n_devices - 1;
        for (int i = 0; i < n_devices; i++) devs.push_back(i);
    } else {
        for (int i = 0; i < n_devices; i++) devs.push_back(devices[i]);
    }
    const int n = (int)devs.size();
    if (n < 1 || (n & (n - 1)))
        return fail(PCS_ERR_ARG, "the number of devices must be a power of two (cap subtrees are split evenly), got " + std::to_string(n));
    for (int i = 0; i < n; i++) {
        if (devs[i] < 0 || devs[i] >= count) return fail(PCS_ERR_ARG, "device " + std::to_string(devs[i]) + " is not visible");
        for (int k = 0; k < i; k++)
            if (devs[k] == devs[i]) return fail(PCS_ERR_ARG, "device " + std::to_string(devs[i]) + " listed twice");
    }
    std::lock_guard<std::recursive_mutex> lock(g_multi_mutex);
    if (g_multi.init) {
        if (g_multi.devices == devs) return PCS_OK;
        return fail(PCS_ERR_ARG, "pcs_multi_init was already called with another device list (pcs_shutdown first)");
    }
    const int prev = pcs_device();
    for (int i = 0; i < n; i++) {
        int rc = pcs_init(devs[i], nullptr);
        if (rc) return rc;
    }
    // every device reads every other device's coefficient blocks in place
    for (int i = 0; i < n; i++) {
        PCS_CUDA(cudaSetDevice(devs[i]));
        for (int k = 0; k < n; k++) {
            if (k == i) continue;
            int can = 0;
            PCS_CUDA(cudaDeviceCanAccessPeer(&can, devs[i], devs[k]));
            if (!can)
                return fail(PCS_ERR_CUDA, "device " + std::to_string(devs[i]) + " cannot access device " + std::to_string(devs[k]) +
                                              " (no NVLink / PCIe peer path): pcs_multi needs peer access");
            cudaError_t pe = cudaDeviceEnablePeerAccess(devs[k], 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled)
                return fail(PCS_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe));
            cudaGetLastError();
        }
    }
    g_multi.devices = devs;
    g_multi.copy_stream.assign(n, nullptr);
    g_multi.free_blocks.assign(n, {});
    g_multi.chunk_ev.assign(n, {});
    g_multi.gather_stream.assign(n, nullptr);
    g_multi.gather_ev.assign(n, {});
    for (int i = 0; i < n; i++) {
        PCS_CUDA(cudaSetDevice(devs[i]));
        PCS_CUDA(cudaStreamCreateWithFlags(&g_multi.copy_stream[i], cudaStreamNonBlocking));
        PCS_CUDA(cudaStreamCreateWithFlags(&g_multi.gather_stream[i], cudaStreamNonBlocking));
        for (size_t c = 0; c < MULTI_MAX_CHUNKS; c++) {
            cudaEvent_t ev;
            PCS_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            g_multi.chunk_ev[i].push_back(ev);
            PCS_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            g_multi.gather_ev[i].push_back(ev);
        }
    }
    g_multi.init = true;
    return pcs_init(prev >= 0 ? prev : devs[0], nullptr);   // the caller's current device is left as it was
}

int pcs_multi_devices(int* devices) {
    if (!g_multi.init) return 0;
    if (devices)
        for (size_t i = 0; i < g_multi.devices.size(); i++) devices[i] = g_multi.devices[i];
    return (int)g_multi.devices.size();
}

void pcs_multi_batch_free(pcs_multi_batch* mb) {
    if (!mb) return;
    for (auto* s : mb->shard) pcs_batch_free(s);
    if (!mb->owned_blocks.empty()) {
        std::lock_guard<std::recursive_mutex> lock(g_multi_mutex);
        for (size_t i = 0; i < mb->owned_blocks.size(); i++) {
            const int gi = mb->owned_block_dev[i];
            if (g_multi.init && gi < (int)g_multi.devices.size()) {
                // other devices' kernels of THIS batch have long finished (every commit ends synchronised)
                cudaSetDevice(g_multi.devices[gi]);
                cudaFree(mb->owned_blocks[i]);
            }
        }
    }
    delete mb;
}

// from_values == true: `polys` are point values; every device IFFTs its own block in place (pcs_ntt_dev) before the LDE.
static int multi_commit(const uint64_t* const* polys, bool from_values, size_t w, unsigned lg_d, unsigned rate_bits,
                        unsigned cap_height, const uint64_t* const* salts, size_t salt_w, unsigned flags,
                        uint64_t* const* coeffs_out, uint64_t* cap_out, pcs_multi_batch** out) {
    if (!out) return fail(PCS_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (flags & PCS_LDE_ON_DEMAND) return fail(PCS_ERR_ARG, "PCS_LDE_ON_DEMAND is not supported by pcs_multi_* commits");
    if (!g_multi.init) return fail(PCS_ERR_NOT_INIT, "pcs_multi_init has not been called");
    if (w == 0 || !polys) return fail(PCS_ERR_ARG, "empty batch (oracle.rs:76 polynomials[0])");
    if (salt_w && !salts) return fail(PCS_ERR_ARG, "salts is NULL");
    if (int rc = check_two_adicity(lg_d + rate_bits)) return rc;
    if (int rc = check_cap_height(cap_height, lg_d + rate_bits)) return rc;
    for (size_t j = 0; j < w; j++)
        if (!polys[j]) return fail(PCS_ERR_ARG, "NULL polynomial pointer");
    std::lock_guard<std::recursive_mutex> lock(g_multi_mutex);
    const int G = (int)g_multi.devices.size();
    Plan plan;
    plan.G = G;
    plan.w = w;
    plan.lg_dev = 0;
    while ((1 << plan.lg_dev) < G) plan.lg_dev++;
    if (plan.lg_dev > lg_d + rate_bits)
        return fail(PCS_ERR_ARG, "cannot split " + std::to_string((size_t)1 << (lg_d + rate_bits)) + " leaves over " + std::to_string(G) + " devices");
    // more devices than coset blocks: polynomial-partitioned LDE + peer pulls of LDE rows into row shards
    const bool rows_mode = plan.lg_dev > rate_bits;
    plan.lg_cosets = rows_mode ? 0 : rate_bits - plan.lg_dev;
    const unsigned lg_local = lg_d + rate_bits - plan.lg_dev;
    plan.local_cap_height = cap_height > plan.lg_dev ? cap_height - plan.lg_dev : 0;
    plan.top_levels = plan.lg_dev > cap_height ? plan.lg_dev - cap_height : 0;
    if (plan.local_cap_height > lg_local)
        return fail(PCS_ERR_CAP_HEIGHT, "cap_height too large for the per-device leaf range");
    const bool dev_ptrs = flags & PCS_DEVICE_PTRS;
    const bool keep = from_values || (flags & PCS_KEEP_COEFFS);
    const size_t d = (size_t)1 << lg_d, n = d << rate_bits, n_loc = n >> plan.lg_dev;
    // device-resident inputs are read in place; host inputs arrive in chunks (H2D of chunk c+1 under the LDE of chunk c)
    const bool staged = !dev_ptrs || from_values || rows_mode;   // from_values transforms in place: always on engine-owned blocks;
                                                                 // rows mode: every device extends the block it holds
    // host inputs: pipeline the H2D copies under the compute.  rho = transfer / compute time per polynomial: one device moves a
    // polynomial in ~0.15 ms against ~0.9 ms of LDE + hashing (2^20, rate 3); with 8 devices copying at once the host side
    // saturates and the ratio approaches 0.75 (profiles/r02_scaling.md)
    const bool gather = G > 1 && (flags & PCS_MULTI_CE_GATHER) && !rows_mode;
    double rho = 0;
    if (staged && !from_values && !dev_ptrs && !rows_mode && w * d * 8 >= ((size_t)G << 24)) rho = G >= 4 ? 0.75 : (G == 2 ? 0.4 : 0.25);
    // device-resident inputs, gathered by the copy engines: an NVLink pull is ~10x faster than the compute on what it brings
    if (!staged && gather && w * d * 8 >= ((size_t)G << 24)) rho = 0.1;
    plan.make_chunks(rho);
    if (plan.chunks > MULTI_MAX_CHUNKS) return fail(PCS_ERR_ARG, "internal: too many chunks");
    const size_t n_local_cap = (size_t)1 << plan.local_cap_height;

    pcs_multi_batch* mb = new pcs_multi_batch();
    mb->n_dev = G; mb->w = w; mb->salt_w = salt_w; mb->lg_d = lg_d; mb->rate_bits = rate_bits; mb->cap_height = cap_height;
    mb->lg_dev = plan.lg_dev; mb->lg_cosets = plan.lg_cosets; mb->local_cap_height = plan.local_cap_height;
    mb->top_levels = plan.top_levels;
    mb->lg_local = lg_local;
    mb->shard.assign(G, nullptr);
    mb->poly_ptr.assign(w, nullptr);
    mb->local_caps.assign((size_t)G * n_local_cap * 4, 0);
    struct Guard { pcs_multi_batch* mb; bool armed = true; ~Guard() { if (armed) pcs_multi_batch_free(mb); } } guard{mb};

    // ---- coefficient blocks (staged inputs): device g holds its rows of every chunk, chunk after chunk ----
    std::vector<uint64_t*> block(G, nullptr);
    std::vector<uint64_t*> gath(G, nullptr);
    const int prev = pcs_device();
    // on EVERY exit: blocks this call does not hand to the batch go back to the per-device pool, and the calling thread gets its
    // current device / context back (the loops below walk the devices)
    struct Cleanup {
        std::vector<uint64_t*>& block;
        std::vector<uint64_t*>& gath;
        pcs_multi_batch* mb;
        const Plan& plan;
        size_t d, w;
        int prev;
        size_t n = 0;          // rows mode: gath[g] holds rows_of(g) LDE rows of n elements
        bool rows_mode = false;
        ~Cleanup() {
            auto owned = [&](uint64_t* p) {
                for (auto* o : mb->owned_blocks)
                    if (o == p) return true;
                return false;
            };
            for (size_t g = 0; g < block.size(); g++) {
                if (block[g] && !owned(block[g])) g_multi.free_blocks[g].push_back({block[g], block_bytes(plan.rows_of((int)g), d)});
                if (gath[g] && !owned(gath[g]))
                    g_multi.free_blocks[g].push_back({gath[g], rows_mode ? block_bytes(plan.rows_of((int)g), n) : w * d * 8});
            }
            pcs_init(prev >= 0 ? prev : g_multi.devices[0], nullptr);
        }
    } cleanup{block, gath, mb, plan, d, w, prev};
    cleanup.n = n;
    cleanup.rows_mode = rows_mode;
    if (staged) {
        for (int g = 0; g < G; g++) {
            PCS_CUDA(cudaSetDevice(g_multi.devices[g]));
            block[g] = block_take(g, block_bytes(plan.rows_of(g), d));
            if (!block[g]) return fail(PCS_ERR_ALLOC, "coefficient block allocation failed on device " + std::to_string(g_multi.devices[g]));
            if (keep && !(G > 1 && (flags & PCS_MULTI_CE_GATHER))) {   // peer-load form: the blocks ARE `polynomials`
                mb->owned_blocks.push_back(block[g]);
                mb->owned_block_dev.push_back(g);
            }
        }
        for (int g = 0; g < G; g++) {
            size_t row = 0;
            for (size_t c = 0; c < plan.chunks; c++) {
                size_t a, b;
                plan.part(c, g, a, b);
                for (size_t j = a; j < b; j++) mb->poly_ptr[j] = block[g] + (row + (j - a)) * d;
                row += b - a;
            }
        }
    } else {
        for (size_t j = 0; j < w; j++) mb->poly_ptr[j] = polys[j];
    }
    // rows mode: the LDE of a device's own polynomials over all cosets, [rows_of(g)][N]; pulled from by every device
    if (rows_mode)
        for (int g = 0; g < G; g++) {
            PCS_CUDA(cudaSetDevice(g_multi.devices[g]));
            gath[g] = block_take(g, block_bytes(plan.rows_of(g), n));
            if (!gath[g]) return fail(PCS_ERR_ALLOC, "LDE buffer allocation failed on device " + std::to_string(g_multi.devices[g]));
        }
    // copy-engine gather: a local [w][d] copy of all coefficients per device (what the LDE then reads at HBM speed)
    if (gather)
        for (int g = 0; g < G; g++) {
            PCS_CUDA(cudaSetDevice(g_multi.devices[g]));
            gath[g] = block_take(g, w * d * 8);
            if (!gath[g]) return fail(PCS_ERR_ALLOC, "gather buffer allocation failed on device " + std::to_string(g_multi.devices[g]));
        }
    std::vector<const uint64_t*> src_ptr = mb->poly_ptr;    // where every polynomial's coefficients are BEFORE the gather
    if (gather && keep) {
        // PolynomialBatch.polynomials = device 0's gathered copy (one contiguous matrix); the staging blocks go back to the pool
        mb->owned_blocks.assign(1, gath[0]);
        mb->owned_block_dev.assign(1, 0);
        for (size_t j = 0; j < w; j++) mb->poly_ptr[j] = gath[0] + j * d;
    }
    // ---- one worker thread per device ----
    std::vector<std::atomic<int>> recorded(G * MULTI_MAX_CHUNKS);   // chunk_ev[g][c] has been recorded
    for (auto& r : recorded) r.store(0);
    std::atomic<int> abort_flag{0};
    std::vector<int> rcs(G, PCS_OK);
    std::vector<std::string> errs(G);
    auto worker = [&](int g) {
        auto body = [&]() -> int {
            int rc = pcs_init(g_multi.devices[g], nullptr);
            if (rc) return rc;
            cudaStream_t st = (cudaStream_t)pcs_stream(), cst = g_multi.copy_stream[g];
            pcs_batch* sh = nullptr;
            rc = rows_mode ? pcs_shard_begin_rows(w + salt_w, salt_w, lg_local, plan.local_cap_height, &sh)
                           : pcs_shard_begin(w, salt_w, lg_d, rate_bits, (unsigned)g << plan.lg_cosets, plan.lg_cosets, plan.local_cap_height, &sh);
            if (rc) return rc;
            mb->shard[g] = sh;
            cudaStream_t gs = g_multi.gather_stream[g];
            std::vector<const uint64_t*> local_ptr;
            auto extend_chunk = [&](size_t c) -> int {
                size_t lo, hi;
                plan.chunk_range(c, lo, hi);
                if (hi == lo) return PCS_OK;
                cudaStream_t waiter = gather ? gs : st;      // who has to see the other devices' parts of this chunk
                if (staged)
                    for (int q = 0; q < G; q++) {
                        while (!recorded[q * MULTI_MAX_CHUNKS + c].load(std::memory_order_acquire)) {
                            if (abort_flag.load()) return fail(PCS_ERR_CUDA, "another device's worker failed");
                            std::this_thread::yield();
                        }
                        PCS_CUDA(cudaStreamWaitEvent(waiter, g_multi.chunk_ev[q][c], 0));
                    }
                if (!gather) return pcs_shard_extend(sh, lo, hi - lo, src_ptr.data() + lo);
                // pull every part of the chunk into the local copy (peer copies over NVLink on the copy engines)
                if (staged) {
                    for (int q = 0; q < G; q++) {
                        size_t a, b;
                        plan.part(c, q, a, b);
                        if (b > a)
                            PCS_CUDA(cudaMemcpyAsync(gath[g] + a * d, src_ptr[a], (b - a) * d * 8, cudaMemcpyDefault, gs));
                    }
                } else {
                    for (size_t j = lo; j < hi; j++)
                        PCS_CUDA(cudaMemcpyAsync(gath[g] + j * d, src_ptr[j], d * 8, cudaMemcpyDefault, gs));
                }
                PCS_CUDA(cudaEventRecord(g_multi.gather_ev[g][c], gs));
                PCS_CUDA(cudaStreamWaitEvent(st, g_multi.gather_ev[g][c], 0));
                local_ptr.resize(hi - lo);
                for (size_t j = lo; j < hi; j++) local_ptr[j - lo] = gath[g] + j * d;
                return pcs_shard_extend(sh, lo, hi - lo, local_ptr.data());
            };
            if (staged) {
                size_t row = 0;
                for (size_t c = 0; c <= plan.chunks; c++) {
                    if (c < plan.chunks) {
                        size_t a, b;
                        plan.part(c, g, a, b);
                        uint64_t* dst = block[g] + row * d;
                        cudaStream_t prod = cst;   // the stream whose event says "my part of chunk c is in place"
                        if (b > a) {
                            if (dev_ptrs) {
                                for (size_t j = a; j < b; j++)
                                    PCS_CUDA(cudaMemcpyAsync(dst + (j - a) * d, polys[j], d * 8, cudaMemcpyDefault, cst));
                            } else {
                                if (is_pageable_host(polys[a]) && (b - a) * d * 8 >= (1u << 20)) {
                                    rc = stage_pageable(polys + a, b - a, d, dst, cst);
                                    if (rc) return rc;
                                } else {
                                    for (size_t j = a; j < b; j++)
                                        PCS_CUDA(cudaMemcpyAsync(dst + (j - a) * d, polys[j], d * 8, cudaMemcpyHostToDevice, cst));
                                }
                            }
                            if (from_values) {
                                // IFFT of my block on the compute stream, behind the copy (oracle.rs:51-55)
                                PCS_CUDA(cudaEventRecord(g_multi.chunk_ev[g][c], cst));
                                PCS_CUDA(cudaStreamWaitEvent(st, g_multi.chunk_ev[g][c], 0));
                                rc = pcs_ntt_dev(dst, b - a, lg_d, 1);
                                if (rc) return rc;
                                if (coeffs_out)
                                    for (size_t j = a; j < b; j++)
                                        if (coeffs_out[j])
                                            PCS_CUDA(cudaMemcpyAsync(coeffs_out[j], dst + (j - a) * d, d * 8, cudaMemcpyDeviceToHost, st));
                                prod = st;
                            }
                        }
                        PCS_CUDA(cudaEventRecord(g_multi.chunk_ev[g][c], prod));
                        recorded[g * MULTI_MAX_CHUNKS + c].store(1, std::memory_order_release);
                        row += b - a;
                    }
                    if (c >= 1 && !rows_mode) {
                        rc = extend_chunk(c - 1);
                        if (rc) return rc;
                    }
                }
                if (rows_mode) {
                    // (1) the LDE of my block over all cosets, behind my staging copy / IFFT
                    size_t a, b;
                    plan.part(0, g, a, b);
                    PCS_CUDA(cudaStreamWaitEvent(st, g_multi.chunk_ev[g][0], 0));
                    if (b > a) {
                        std::vector<const uint64_t*> mine(b - a);
                        for (size_t j = a; j < b; j++) mine[j - a] = block[g] + (j - a) * d;
                        rc = pcs_coset_lde_dev(mine.data(), b - a, lg_d, rate_bits, 7, gath[g]);
                        if (rc) return rc;
                    }
                    PCS_CUDA(cudaEventRecord(g_multi.chunk_ev[g][1], st));
                    recorded[g * MULTI_MAX_CHUNKS + 1].store(1, std::memory_order_release);
                    // (2) pull my leaf range of every polynomial out of its owner's LDE, straight into the shard's rows
                    uint64_t* rows = const_cast<uint64_t*>(pcs_batch_lde_dev(sh));
                    cudaStream_t gs = g_multi.gather_stream[g];
                    PCS_CUDA(cudaEventRecord(g_multi.gather_ev[g][1], st));          // the shard's buffer exists
                    PCS_CUDA(cudaStreamWaitEvent(gs, g_multi.gather_ev[g][1], 0));
                    for (int q = 0; q < G; q++) {
                        while (!recorded[q * MULTI_MAX_CHUNKS + 1].load(std::memory_order_acquire)) {
                            if (abort_flag.load()) return fail(PCS_ERR_CUDA, "another device's worker failed");
                            std::this_thread::yield();
                        }
                        PCS_CUDA(cudaStreamWaitEvent(gs, g_multi.chunk_ev[q][1], 0));
                        size_t qa, qb;
                        plan.part(0, q, qa, qb);
                        if (qb > qa)      // (qb - qa) rows of n_loc elements, source pitch n, destination pitch n_loc
                            PCS_CUDA(cudaMemcpy2DAsync(rows + qa * n_loc, n_loc * 8, gath[q] + (size_t)g * n_loc, n * 8, n_loc * 8, qb - qa,
                                                       cudaMemcpyDefault, gs));
                    }
                    PCS_CUDA(cudaEventRecord(g_multi.gather_ev[g][0], gs));
                    PCS_CUDA(cudaStreamWaitEvent(st, g_multi.gather_ev[g][0], 0));
                }
            } else {
                for (size_t c = 0; c < plan.chunks; c++) {
                    rc = extend_chunk(c);
                    if (rc) return rc;
                }
            }
            // ---- blinding: the caller's salt columns are in natural LDE order (oracle.rs:119-123); this shard takes the
            //      leaf-order slice of its own leaf range ----
            if (salt_w) {
                DevBuf col, slice;
                PCS_CUDA(col.alloc(n * 8, st));
                PCS_CUDA(slice.alloc(salt_w * n_loc * 8, st));
                std::vector<const uint64_t*> rows(salt_w);
                for (size_t k = 0; k < salt_w; k++) {
                    if (!salts[k]) return fail(PCS_ERR_ARG, "NULL salt pointer");
                    PCS_CUDA(cudaMemcpyAsync(col.p, salts[k], n * 8, cudaMemcpyDefault, st));
                    PCS_CUDA(launch_bitrev_gather(col.u64(), lg_d + rate_bits, (size_t)g * n_loc, n_loc, slice.u64() + k * n_loc, st));
                    rows[k] = slice.u64() + k * n_loc;
                }
                rc = pcs_shard_set_rows(sh, w, salt_w, rows.data(), 1);
                if (rc) return rc;
            }
            return pcs_shard_finish(sh, mb->local_caps.data() + (size_t)g * n_local_cap * 4);   // synchronises this device
        };
        rcs[g] = body();
        if (rcs[g]) {
            errs[g] = pcs_last_error();
            abort_flag.store(1);
            // peers may be waiting for this device's chunk events: publish them all so nobody spins forever
            for (size_t c = 0; c < MULTI_MAX_CHUNKS; c++) recorded[g * MULTI_MAX_CHUNKS + c].store(1, std::memory_order_release);
        }
        cudaStreamSynchronize((cudaStream_t)pcs_stream());
        cudaStreamSynchronize(g_multi.copy_stream[g]);
        cudaStreamSynchronize(g_multi.gather_stream[g]);
    };
    if (G == 1) {
        worker(0);
    } else {
        std::vector<std::thread> th;
        for (int g = 0; g < G; g++) th.emplace_back(worker, g);
        for (auto& t : th) t.join();
    }
    pcs_init(prev >= 0 ? prev : g_multi.devices[0], nullptr);   // pcs_two_to_one below runs on the caller's device
    for (int g = 0; g < G; g++)
        if (rcs[g]) return fail(rcs[g], "device " + std::to_string(g_multi.devices[g]) + ": " + errs[g]);
    if (staged && !keep) mb->poly_ptr.clear();   // the blocks go back to the pool: PolynomialBatch.polynomials was not asked for

    // ---- cap: local caps in device order; above them log2(G) - cap_height levels of two_to_one (merkle_tree.rs:69-96) ----
    mb->cap = mb->local_caps;
    if (int rc = combine_top_levels(mb->cap, plan.top_levels, 0, nullptr)) return rc;
    if (cap_out) memcpy(cap_out, mb->cap.data(), mb->cap.size() * 8);
    guard.armed = false;
    *out = mb;
    return PCS_OK;
}

int pcs_multi_commit_from_coeffs(const uint64_t* const* polys, size_t w, unsigned lg_d, unsigned rate_bits, unsigned cap_height,
                                 const uint64_t* const* salts, size_t salt_w, unsigned flags, uint64_t* cap_out,
                                 pcs_multi_batch** out) {
    return multi_commit(polys, false, w, lg_d, rate_bits, cap_height, salts, salt_w, flags, nullptr, cap_out, out);
}

int pcs_multi_commit_from_values(const uint64_t* const* values, size_t w, unsigned lg_d, unsigned rate_bits, unsigned cap_height,
                                 const uint64_t* const* salts, size_t salt_w, unsigned flags, uint64_t* const* coeffs_out,
                                 uint64_t* cap_out, pcs_multi_batch** out) {
    return multi_commit(values, true, w, lg_d, rate_bits, cap_height, salts, salt_w, flags, coeffs_out, cap_out, out);
}

int pcs_multi_batch_shape(const pcs_multi_batch* mb, size_t* n_leaves, size_t* leaf_len, int* n_shards, unsigned* cap_height) {
    if (!mb) return fail(PCS_ERR_ARG, "batch is NULL");
    if (n_leaves) *n_leaves = ((size_t)1 << mb->lg_d) << mb->rate_bits;
    if (leaf_len) *leaf_len = mb->w + mb->salt_w;
    if (n_shards) *n_shards = mb->n_dev;
    if (cap_height) *cap_height = mb->cap_height;
    return PCS_OK;
}

int pcs_multi_batch_cap(const pcs_multi_batch* mb, uint64_t* cap) {
    if (!mb || !cap) return fail(PCS_ERR_ARG, "NULL pointer");
    memcpy(cap, mb->cap.data(), mb->cap.size() * 8);
    return PCS_OK;
}

pcs_batch* pcs_multi_batch_shard(const pcs_multi_batch* mb, int i) {
    return (mb && i >= 0 && i < mb->n_dev) ? mb->shard[i] : nullptr;
}

int pcs_multi_batch_poly_ptrs(const pcs_multi_batch* mb, const uint64_t** ptrs) {
    if (!mb || !ptrs) return fail(PCS_ERR_ARG, "NULL pointer");
    if (mb->poly_ptr.empty()) return fail(PCS_ERR_ARG, "coefficients were not kept (PCS_KEEP_COEFFS)");
    for (size_t j = 0; j < mb->w; j++) ptrs[j] = mb->poly_ptr[j];
    return PCS_OK;
}

int pcs_multi_batch_get_rows(const pcs_multi_batch* mb, const uint64_t* leaf_indices, size_t n, uint64_t* rows) {
    if (!mb || (n && (!leaf_indices || !rows))) return fail(PCS_ERR_ARG, "NULL pointer");
    const size_t n_leaves = ((size_t)1 << mb->lg_d) << mb->rate_bits, n_loc = n_leaves >> mb->lg_dev, wt = mb->w + mb->salt_w;
    for (size_t k = 0; k < n; k++)
        if (leaf_indices[k] >= n_leaves) return fail(PCS_ERR_ARG, "leaf index out of bounds");
    std::vector<uint64_t> idx, tmp;
    std::vector<size_t> pos;
    for (int g = 0; g < mb->n_dev; g++) {
        idx.clear();
        pos.clear();
        for (size_t k = 0; k < n; k++)
            if (leaf_indices[k] / n_loc == (size_t)g) {
                idx.push_back(leaf_indices[k] % n_loc);
                pos.push_back(k);
            }
        if (idx.empty()) continue;
        tmp.resize(idx.size() * wt);
        int rc = pcs_batch_get_rows(mb->shard[g], idx.data(), idx.size(), tmp.data());
        if (rc) return rc;
        for (size_t i = 0; i < idx.size(); i++) memcpy(rows + pos[i] * wt, tmp.data() + i * wt, wt * 8);
    }
    return PCS_OK;
}

int pcs_multi_batch_prove(const pcs_multi_batch* mb, size_t leaf_index, uint64_t* siblings) {
    if (!mb) return fail(PCS_ERR_ARG, "NULL pointer");
    const size_t n_leaves = ((size_t)1 << mb->lg_d) << mb->rate_bits, n_loc = n_leaves >> mb->lg_dev;
    if (leaf_index >= n_leaves) return fail(PCS_ERR_ARG, "leaf index out of bounds");
    const unsigned n_local = mb->lg_local - mb->local_cap_height;
    if (n_local + mb->top_levels == 0) return PCS_OK;
    if (!siblings) return fail(PCS_ERR_ARG, "NULL pointer");
    const int g = (int)(leaf_index / n_loc);
    int rc = pcs_batch_prove(mb->shard[g], leaf_index % n_loc, siblings);
    if (rc) return rc;
    // above the device's root (n_dev > 2^cap_height): siblings from the other devices' roots, combined level by level
    std::vector<uint64_t> level = mb->local_caps;   // local_cap_height == 0 here: one root per device
    return combine_top_levels(level, mb->top_levels, (size_t)g, siblings + (size_t)n_local * 4);
}

int pcs_multi_batch_timings(const pcs_multi_batch* mb, float ms[5]) {
    if (!mb || !ms) return fail(PCS_ERR_ARG, "NULL pointer");
    for (int i = 0; i < 5; i++) ms[i] = 0;
    for (int g = 0; g < mb->n_dev; g++) {
        float t[5];
        int rc = pcs_batch_timings(mb->shard[g], t);
        if (rc) return rc;
        for (int i = 0; i < 5; i++) ms[i] = t[i] > ms[i] ? t[i] : ms[i];
    }
    return PCS_OK;
}

}  // extern "C"
