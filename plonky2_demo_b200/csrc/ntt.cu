// Batched Goldilocks NTT / coset low-degree extension for sm_100a.
//
// What the reference computes (per polynomial, on the CPU):
//   PolynomialCoeffs::lde          field/src/polynomial/mod.rs:201-203   zero-pad d -> N = d*2^r
//   coset_fft_with_options         field/src/polynomial/mod.rs:282-295   c_i *= 7^i, then
//   fft_classic (radix-2 DIT)      field/src/fft.rs:169-206              bit-reverse + lg N stages
//   transpose + reverse_index_bits plonky2/src/fri/oracle.rs:83-84       -> leaf order
//   ifft_with_options              field/src/fft.rs:72-95
//
// What this file computes instead (same values, different algorithm -- SURVEY 8a identity):
//   the length-N transform with N - d trailing zero coefficients, run as a natural-order-in /
//   bit-reversed-order-out Cooley-Tukey NTT whose twiddles depend only on the butterfly BLOCK:
//       stage sigma, block B:  (u, v) <- (u + w v, u - w v),
//       w = shift^(N / 2^(sigma+1)) * omega_N^((N / 2^(sigma+1)) * brev_sigma(B))
//   The first r stages see v = 0 and are plain copies, so coset c in [0, 2^r) is an independent
//   length-d transform of the SAME coefficients whose output IS the contiguous leaf range
//   [c*d, (c+1)*d): no zero padding, no 7^i pass, no transpose, no bit-reversal pass.
//   The coset shift is absorbed into the twiddles (zero extra multiplies per element).
//
// Decomposition: lg d stages are split into passes of <= 10 stages.  A pass handles, per CTA, tiles of R = 2^nb "rows"
// (the nb index bits it transforms) x C "columns" (index bits below the pass, and/or different polynomials).  Inside a
// tile every twiddle factors as
//       w(i, q) = gamma_i(G) * psi[q],   gamma_{i-1} = gamma_i^2,
// with G = (coset, high index bits) fixed per CTA: one table lookup (Gamma[G]), nb-1 squarings and the products with
// psi give all twiddles once per CTA, shared by all columns and by every tile the CTA walks.
// The stages themselves run on REGISTERS (32 values per thread, two rounds of <= 5 stages, one shared-memory exchange
// in between): see the pass kernel below.
//
// Roofline: HBM traffic is 8 B/elem per pass per direction, but a butterfly costs 37 integer instructions (4 IMAD.WIDE +
// carry-chain reduction + canonicalisation + add + sub), so the kernel is bound by the integer ALU pipe, not by HBM:
// 10 butterflies per output element = 370 instructions per 9 algorithmic bytes (DESIGN.md 4.2).
#include <map>
#include <tuple>
#include <vector>

#include <list>
#include <mutex>

#include "common.cuh"
#include "gl64.cuh"

namespace pcs {

constexpr int NTT_MAX_NB = 10;          // stages per pass
constexpr int NTT_TILE_LOG = 13;        // 8192 elements (64 KiB) per tile
constexpr int NTT_THREADS = 256;          // x 32 registers = one tile

struct NttPass {
    unsigned s0, nb;   // stages [s0, s0+nb)
    unsigned L;        // index bits below the pass
    uint64_t* gamma;   // [2^(r+s0)]  Gamma[G] = (shift * root_N^brev(G))^(2^L)
    uint64_t* psi;     // [2^(nb-1)]  psi[q] = omega_{2^nb}^{brev_{nb-1}(q)}
};

struct NttPlan {
    unsigned lg_d, r;
    bool inverse;
    uint64_t shift;
    uint64_t scale;  // 1/d for the inverse transform (applied by the bit-reversal permutation that follows), else 1
    std::vector<NttPass> passes;
    cudaEvent_t ready = nullptr;      // the table fill has finished (recorded on the stream that built the plan)
    cudaStream_t built_on = nullptr;
    int device = -1;
    ~NttPlan() {
        for (auto& ps : passes) {
            if (ps.gamma) cudaFree(ps.gamma);
            if (ps.psi) cudaFree(ps.psi);
        }
        if (ready) cudaEventDestroy(ready);
    }
};

// -------------------------------------------------------------------------------------------------
// plan construction (device-side table fill)
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t brev32(uint32_t x, unsigned bits) { return bits ? __brev(x) >> (32 - bits) : 0; }

__global__ void k_fill_gamma(uint64_t* gamma, unsigned gbits, uint64_t root_n, uint64_t shift, unsigned L) {
    uint32_t G = blockIdx.x * blockDim.x + threadIdx.x;
    if (G >= (1u << gbits)) return;
    uint64_t beta = gl::mul(shift, gl::pow(root_n, brev32(G, gbits)));
    for (unsigned i = 0; i < L; i++) beta = gl::sqr(beta);
    gamma[G] = beta;
}

__global__ void k_fill_psi(uint64_t* psi, unsigned nb, uint64_t root_2nb) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (1u << (nb - 1))) return;
    psi[q] = gl::pow(root_2nb, brev32(q, nb - 1));
}

// Plan cache: one per CUDA device (twiddle tables live in that device's memory).  The commit path uses a handful of plans
// (shift 7 and the inverse transform per degree); FRI layer shifts and caller-chosen shifts (pcs_coset_lde, pcs_coset_intt)
// are arbitrary, so the cache is LRU-bounded.
struct PlanCache {
    typedef std::tuple<unsigned, unsigned, bool, uint64_t> Key;
    std::list<std::pair<Key, NttPlan*>> lru;   // front = most recently used
    std::map<Key, std::list<std::pair<Key, NttPlan*>>::iterator> index;
};
constexpr size_t NTT_MAX_PLANS = 48;
constexpr int NTT_MAX_DEVICES = 64;
static PlanCache g_plan_cache[NTT_MAX_DEVICES];
static std::mutex g_plan_mutex;

static std::vector<unsigned> split_stages(unsigned lg_d) {
    // equal-ish passes of at most NTT_MAX_NB stages; the FIRST pass gets the remainder so the
    // contiguous last pass is the biggest.
    std::vector<unsigned> v;
    if (lg_d == 0) return v;
    unsigned n = (lg_d + NTT_MAX_NB - 1) / NTT_MAX_NB;
    unsigned base = lg_d / n, extra = lg_d % n;
    for (unsigned i = 0; i < n; i++) v.push_back(base + (i >= n - extra ? 1 : 0));
    return v;
}

NttPlan* ntt_plan_get(unsigned lg_d, unsigned r, bool inverse, uint64_t shift, cudaStream_t st) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= NTT_MAX_DEVICES) return nullptr;
    shift %= gl::P;
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    PlanCache& pc = g_plan_cache[dev];
    const auto key = std::make_tuple(lg_d, r, inverse, shift);
    auto it = pc.index.find(key);
    if (it != pc.index.end()) {
        pc.lru.splice(pc.lru.begin(), pc.lru, it->second);
        NttPlan* p = it->second->second;
        // a plan filled on another stream (pcs_init re-bound the engine's stream): order this stream behind the fill
        if (p->built_on != st && p->ready) cudaStreamWaitEvent(st, p->ready, 0);
        return p;
    }
    unsigned lg_n = lg_d + r;
    uint64_t root = glh::primitive_root_of_unity(lg_n);
    if (inverse) root = glh::inverse(root);
    NttPlan* p = new NttPlan();
    p->lg_d = lg_d;
    p->r = r;
    p->inverse = inverse;
    p->shift = shift;
    p->scale = inverse ? gl::P - ((gl::P - 1) >> lg_d) : 1;  // inverse_2exp, types.rs:227-262
    p->device = dev;
    p->built_on = st;
    unsigned s0 = 0;
    for (unsigned nb : split_stages(lg_d)) {
        NttPass ps;
        ps.s0 = s0;
        ps.nb = nb;
        ps.L = lg_d - s0 - nb;
        ps.gamma = ps.psi = nullptr;
        unsigned gbits = r + s0;
        // plain cudaMalloc (tables outlive any stream); a failure part-way frees what this plan already holds
        bool ok = cudaMalloc(&ps.gamma, sizeof(uint64_t) << gbits) == cudaSuccess;
        ok = ok && cudaMalloc(&ps.psi, sizeof(uint64_t) << (nb - 1)) == cudaSuccess;
        p->passes.push_back(ps);
        if (!ok) {
            cudaGetLastError();
            delete p;
            return nullptr;
        }
        size_t ng = (size_t)1 << gbits;
        k_fill_gamma<<<(unsigned)((ng + 255) / 256), 256, 0, st>>>(ps.gamma, gbits, root, p->shift, ps.L);
        uint64_t root_2nb = glh::powmod(root, 1ULL << (lg_n - nb));
        size_t nq = (size_t)1 << (nb - 1);
        k_fill_psi<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(ps.psi, nb, root_2nb);
        s0 += nb;
    }
    if (cudaEventCreateWithFlags(&p->ready, cudaEventDisableTiming) == cudaSuccess) cudaEventRecord(p->ready, st);
    pc.lru.emplace_front(key, p);
    pc.index[key] = pc.lru.begin();
    while (pc.lru.size() > NTT_MAX_PLANS) {
        // evict the least recently used plan; kernels already enqueued may still read its tables, and cudaFree only
        // returns once the device is idle, so the tables outlive them
        auto& victim = pc.lru.back();
        pc.index.erase(victim.first);
        delete victim.second;
        pc.lru.pop_back();
    }
    return p;
}

// frees the CURRENT device's plans (pcs_shutdown walks the contexts)
void ntt_plans_free() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= NTT_MAX_DEVICES) return;
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    PlanCache& pc = g_plan_cache[dev];
    for (auto& kv : pc.lru) delete kv.second;
    pc.lru.clear();
    pc.index.clear();
}

// -------------------------------------------------------------------------------------------------
// the pass kernel (register-blocked)
//
// A tile is 2^13 elements = R x C, R = 2^nb rows (the nb index bits this pass transforms), C columns
// (2^lcl contiguous low index bits x 2^(lc-lcl) polynomials).  Tile coordinate, in memory order:
//       E = [ pcol | rho (nb bits) | lcol (lcl bits) ]                      (13 bits)
// 256 threads x 32 registers.  The nb stages run as (at most) two register ROUNDS of K1 and K2 stages:
// in a round a thread owns all 2^K values of a K-bit field of rho (and 2^(5-K) polynomials) and does
// the K stages on registers; between the two rounds the tile goes once through shared memory.
// Stages inside a round use a constant-geometry butterfly (pairs (j, j+16), results to (2j, 2j+1)),
// so the stage loop is rolled: ~12 KB of SASS instead of 50 KB, and register indices stay static.
// Twiddles of one (coset, high bits) prefix G are built once per CTA in shared memory, replicated
// per butterfly slot so that every twiddle load is [thread base + immediate]; a CTA then walks
// several column groups (tiles) with the same G.
// -------------------------------------------------------------------------------------------------
struct PassArgs {
    const uint64_t* in;
    const uint64_t* const* in_ptrs;   // first pass only, or null: per-polynomial base pointers (may be PEER memory:
                                      // a shard reads the coefficient blocks of the other GPUs over NVLink in place)
    uint64_t* out;
    size_t in_poly_stride, out_poly_stride;
    size_t in_coset_stride, out_coset_stride;  // in: 0 for the first pass (all cosets read the coefficients)
    const uint64_t* gamma;
    const uint64_t* psi;
    uint32_t n_polys;
    uint32_t r, s0, L, lg_d;   // r = log2(cosets computed by this launch)
    uint32_t c0;               // first coset (leaf order) of this launch: shard commits compute a sub-range
    uint32_t lcl;              // log2(columns per tile taken from the low index bits)
    uint32_t lgroups;          // 2^(L - lcl) column groups per block of polynomials
    uint32_t n_cg;             // column groups in total (lgroups * poly groups)
    uint32_t tiles_per_cta;
    int last;                  // last pass: outputs leave the engine => canonical
};

// Shared-memory swizzle of a tile coordinate.  XOR-linear: sw(a ^ b) = sw(a) ^ sw(b), so an access at
// (thread base | compile-time field value) costs one LOP3 with an immediate: sw(base) ^ sw(const).
__host__ __device__ constexpr uint32_t sw(uint32_t E) { return E ^ ((E >> 5) & 31u); }
__device__ __forceinline__ uint64_t& tile_at(uint64_t* tile, uint32_t base_bytes, uint32_t c) {
    return *reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(tile) + (base_bytes ^ (sw(c) << 3)));
}

// K stages on 32 registers; stage s pairs (j, j+16) with twiddle twp[s*16*STRIDE + j*STRIDE] and
// rotates the register index left by one bit.  The butterfly adds with gl::add_lc, not gl::add_lc_wide: the wide add puts one
// more instruction on the ALU pipe, which bounds this kernel.
template <int STRIDE>
__device__ __forceinline__ void run_stages(uint64_t (&x)[32], const uint64_t* twp, int k) {
#pragma unroll 1
    for (int s = 0; s < k; s++, twp += 16 * STRIDE) {
        uint64_t y[32];
#pragma unroll
        for (int j = 0; j < 16; j++) {
            uint64_t t = gl::canon(gl::mul(x[j + 16], twp[j * STRIDE]));
            y[2 * j] = gl::add_lc(x[j], t);
            y[2 * j + 1] = gl::sub_lc(x[j], t);
        }
#pragma unroll
        for (int j = 0; j < 32; j++) x[j] = y[j];
    }
}

template <int K1, int K2, int LCL>
__global__ void __launch_bounds__(NTT_THREADS, 2) k_ntt_pass(const PassArgs a) {
    constexpr int NB = K1 + K2;
    constexpr int LC = NTT_TILE_LOG - NB;
    constexpr uint32_t TILE = 1u << NTT_TILE_LOG;
    extern __shared__ uint64_t smem[];
    uint64_t* tile = smem;                 // [TILE], swizzled by sw()
    uint64_t* tw1 = tile + TILE;           // [K1][16]
    uint64_t* tw2 = tw1 + 16 * K1;         // [K2][16][32]
    uint64_t* gam = tw2 + 512 * K2;        // [NB]
    const uint32_t tid = threadIdx.x;
    constexpr uint32_t lcl = LCL;          // log2(columns taken from the low index bits); compile time so that
    constexpr uint32_t PB = LC - lcl;      // every tile / shared-memory address folds to base + immediate

    // ---- which prefix / which column groups ----
    const uint32_t gbits = a.r + a.s0;
    const uint32_t G = blockIdx.x & ((1u << gbits) - 1);   // G fastest: the 2^r cosets of an input tile are neighbours
    const uint32_t c = G >> a.s0, H = G & ((1u << a.s0) - 1);   // c: coset index local to this launch
    const uint32_t cg0 = (blockIdx.x >> gbits) * a.tiles_per_cta;
    const size_t h_off = (size_t)H << (a.lg_d - a.s0);

    // ---- twiddles of this prefix: gam[i] = gamma_i, entry(stage i, q) = gamma_i * psi[q] ----
    if (tid < NB) {
        uint64_t g = a.gamma[G + ((size_t)a.c0 << a.s0)];  // gamma_{NB-1} of the global (coset, high bits) prefix
        for (int i = NB - 1; i > (int)tid; i--) g = gl::sqr(g);
        gam[tid] = g;
    }
    __syncthreads();
    for (uint32_t e = tid; e < 16 * K1; e += NTT_THREADS) {
        uint32_t s = e >> 4, j = e & 15;
        tw1[e] = gl::canon(gl::mul(gam[s], a.psi[j & ((1u << s) - 1)]));
    }
    if (K2 > 0) {
        for (uint32_t e = tid; e < (uint32_t)(K2 * 16) << K1; e += NTT_THREADS) {
            uint32_t ra = e & ((1u << K1) - 1), j = (e >> K1) & 15, s = e >> (K1 + 4);
            uint32_t q = (ra << s) | (j & ((1u << s) - 1));
            tw2[(s * 16 + j) * 32 + ra] = gl::canon(gl::mul(gam[K1 + s], a.psi[q]));
        }
    }
    __syncthreads();

    // ---- per-thread coordinates (same for every tile) ----
    // round 1: field = rho bits [NB-1 .. K2]; thread bits = [pcol_low | rho_lo (K2) | lcol]
    constexpr uint32_t lmask = (1u << lcl) - 1;
    const uint32_t lcol1 = tid & lmask;
    const uint32_t rlo1 = (tid >> lcl) & ((1u << K2) - 1);
    const uint32_t pl1 = tid >> (lcl + K2);
    constexpr uint32_t xsh1 = PB - (5 - K1);               // extras -> top polynomial bits
    const uint32_t E1 = (pl1 << (NB + lcl)) | (rlo1 << lcl) | lcol1;
    const uint32_t sb1 = sw(E1) << 3;                       // byte offset of the thread's round-1 base
    constexpr uint32_t p1 = lcl + K2;
    // round 2: field = rho bits [K2-1 .. 0]; thread bits = [pcol_low | rho_hi (K1) | lcol]
    const uint32_t rhi2 = (tid >> lcl) & ((1u << K1) - 1);
    const uint32_t pl2 = tid >> (lcl + K1);
    constexpr uint32_t xsh2 = K2 > 0 ? PB - (5 - K2) : 0;
    const uint32_t E2 = (pl2 << (NB + lcl)) | (rhi2 << (K2 + lcl)) | (tid & lmask);
    const uint32_t sb2 = sw(E2) << 3;
    constexpr bool staged_out = K2 > 0 && lcl < 3;

    for (uint32_t ti = 0; ti < a.tiles_per_cta; ti++) {
        const uint32_t cg = cg0 + ti;
        if (cg >= a.n_cg) break;
        const uint32_t lgroup = cg % a.lgroups, pgroup = cg / a.lgroups;
        const uint32_t poly_base = pgroup << PB;
        const size_t l_base = (size_t)lgroup << lcl;
        const size_t in_off = (size_t)c * a.in_coset_stride + h_off + l_base;
        uint64_t* out_t = a.out + (size_t)c * a.out_coset_stride + h_off + l_base;

        uint64_t x[32];
        // ---- acquire round 1 straight from global memory ----
        {
            const size_t row_stride = (size_t)1 << (K2 + a.L);   // elements between consecutive field values
#pragma unroll
            for (int xv = 0; xv < (1 << (5 - K1)); xv++) {
                // polynomials past the end of the batch read the last one's data: their results are never stored
                uint32_t poly = poly_base + pl1 + (xv << xsh1);
                poly = poly < a.n_polys ? poly : a.n_polys - 1;
                const uint64_t* pp = (a.in_ptrs ? a.in_ptrs[poly] : a.in + (size_t)poly * a.in_poly_stride) + in_off +
                                     ((size_t)rlo1 << a.L) + lcol1;
#pragma unroll
                for (int av = 0; av < (1 << K1); av++, pp += row_stride) x[(av << (5 - K1)) | xv] = *pp;
            }
        }
        run_stages<1>(x, tw1, K1);
        if (K2 > 0) {
            // after K1 rotations register m holds field value m & (2^K1-1), extra m >> K1
#pragma unroll
            for (int m = 0; m < 32; m++) {
                const uint32_t av = m & ((1 << K1) - 1), xv = m >> K1;
                tile_at(tile, sb1, (av << p1) | (xv << (8 + K1))) = x[m];
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const uint32_t av = j >> (5 - K2), xv = j & ((1 << (5 - K2)) - 1);
                x[j] = tile_at(tile, sb2, (av << lcl) | (xv << (8 + K2)));
            }
            run_stages<32>(x, tw2 + rhi2, K2);
        }
        // ---- release ----
        constexpr int KL = K2 > 0 ? K2 : K1;   // field width of the last round
        if (a.last) {
#pragma unroll
            for (int m = 0; m < 32; m++) x[m] = gl::canon(x[m]);
        }
        if (staged_out) {
            // the last round's field is the lowest index bits: regroup through shared memory so that
            // a warp stores 256 contiguous bytes
#pragma unroll
            for (int m = 0; m < 32; m++) {
                const uint32_t av = m & ((1 << KL) - 1), xv = m >> KL;
                tile_at(tile, sb2, (av << lcl) | (xv << (8 + KL))) = x[m];
            }
            __syncthreads();
#pragma unroll 8
            for (uint32_t e = tid; e < TILE; e += NTT_THREADS) {
                const uint32_t poly = poly_base + (e >> (NB + lcl));
                // staged mode is used by last passes (L == lcl == 0: rho is contiguous in memory)
                const uint32_t within = e & ((1u << (NB + lcl)) - 1);
                if (poly < a.n_polys)
                    out_t[(size_t)poly * a.out_poly_stride + ((size_t)(within >> lcl) << a.L) + (within & lmask)] = tile[sw(e)];
            }
        } else {
            const uint32_t rbase = K2 > 0 ? (rhi2 << K2) : rlo1;   // K2 == 0: round-1 coordinates (rlo1 == 0)
            const uint32_t plx = K2 > 0 ? pl2 : pl1, xshx = K2 > 0 ? xsh2 : xsh1, lc_ = K2 > 0 ? (tid & lmask) : lcol1;
            const size_t row_stride = (size_t)1 << a.L;
#pragma unroll
            for (int xv = 0; xv < (1 << (5 - KL)); xv++) {
                const uint32_t poly = poly_base + plx + (xv << xshx);
                uint64_t* pp = out_t + (size_t)poly * a.out_poly_stride + ((size_t)rbase << a.L) + lc_;
                if (poly < a.n_polys) {
#pragma unroll
                    for (int av = 0; av < (1 << KL); av++, pp += row_stride) *pp = x[(xv << KL) | av];
                }
            }
        }
        __syncthreads();   // the tile buffer is rewritten by the next iteration
    }
}

// d == 1: every output of the coset LDE equals the single coefficient.
__global__ void k_broadcast_const(const uint64_t* in, size_t in_stride, uint64_t* out, size_t out_stride, size_t w,
                                  size_t n, uint64_t scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w * n) return;
    size_t j = i / n, k = i % n;
    out[j * out_stride + k] = gl::canon(gl::mul(gl::canon(in[j * in_stride]), scale));
}

// columns from the low index bits when a pass has stages below it: as many as fit the tile (13 - nb bits) while a
// thread's round-2 twiddle row still depends on its thread index only (lcl + K1 <= 8)
constexpr int lcl_max(int k1, int k2) { return (13 - k1 - k2) < (8 - k1) ? (13 - k1 - k2) : (8 - k1); }

template <int K1, int K2, int LCL>
static cudaError_t launch_pass(const PassArgs& a, unsigned grid, cudaStream_t st) {
    constexpr size_t smem = ((size_t)(1u << NTT_TILE_LOG) + 16 * K1 + 512 * K2 + 16) * sizeof(uint64_t);
    static bool attr_set[NTT_MAX_DEVICES] = {false};   // the opt-in to > 48 KB of dynamic shared memory is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= NTT_MAX_DEVICES) return cudaErrorInvalidDevice;
    if (!attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(k_ntt_pass<K1, K2, LCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    k_ntt_pass<K1, K2, LCL><<<grid, NTT_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

template <int K1, int K2>
static cudaError_t launch_pass_lcl(const PassArgs& a, unsigned grid, cudaStream_t st) {
    return a.lcl ? launch_pass<K1, K2, lcl_max(K1, K2)>(a, grid, st) : launch_pass<K1, K2, 0>(a, grid, st);
}

static cudaError_t run_passes(const NttPlan* plan, const uint64_t* in, size_t in_stride, uint64_t* out,
                              size_t out_stride, size_t w, unsigned coset_first, unsigned lg_cosets, cudaStream_t st,
                              const uint64_t* const* in_ptrs = nullptr) {
    const unsigned lg_d = plan->lg_d, r = lg_cosets;
    const size_t d = (size_t)1 << lg_d;
    if (w == 0) return cudaSuccess;
    if (lg_cosets > plan->r || ((size_t)coset_first + ((size_t)1 << lg_cosets)) > ((size_t)1 << plan->r))
        return cudaErrorInvalidValue;
    if (lg_d == 0) {
        if (in_ptrs) return cudaErrorInvalidValue;   // callers stage single-coefficient polynomials
        size_t n = (size_t)1 << r;
        k_broadcast_const<<<(unsigned)((w * n + 255) / 256), 256, 0, st>>>(in, in_stride, out, out_stride, w, n,
                                                                          plan->scale);
        return cudaGetLastError();
    }
    for (size_t pi = 0; pi < plan->passes.size(); pi++) {
        const NttPass& ps = plan->passes[pi];
        PassArgs a;
        bool first = pi == 0, last = pi + 1 == plan->passes.size();
        const unsigned nb = ps.nb, k1 = nb <= 5 ? nb : (nb + 1) / 2, lc = NTT_TILE_LOG - nb;
        a.in = first ? in : out;
        a.in_ptrs = first ? in_ptrs : nullptr;
        a.out = out;
        a.in_poly_stride = first ? in_stride : out_stride;
        a.out_poly_stride = out_stride;
        a.in_coset_stride = first ? 0 : d;
        a.out_coset_stride = d;
        a.gamma = ps.gamma;
        a.psi = ps.psi;
        a.n_polys = (uint32_t)w;
        a.r = r; a.s0 = ps.s0; a.L = ps.L; a.lg_d = lg_d;
        a.c0 = coset_first;
        // columns from the low index bits: at most L, at most lc, and few enough that a thread's
        // round-2 twiddle row depends on its thread index only (lcl + k1 <= 8)
        // L is 0 (last pass) or the stage count of the later passes (>= 5 for every plan split_stages makes); the
        // kernels are instantiated for lcl = 0 and lcl = lcl_max only
        unsigned lclm = lc < 8 - k1 ? lc : 8 - k1;
        unsigned lcl = ps.L >= lclm ? lclm : 0;
        a.lcl = lcl;
        a.lgroups = 1u << (ps.L - lcl);
        uint32_t polys_per_tile = 1u << (lc - lcl);
        uint32_t pgroups = (uint32_t)((w + polys_per_tile - 1) / polys_per_tile);
        size_t n_cg = (size_t)a.lgroups * pgroups;
        if (n_cg > 0xffffffffULL) return cudaErrorInvalidConfiguration;
        a.n_cg = (uint32_t)n_cg;
        // enough CTAs for ~8 waves of 2 CTAs/SM, but amortise the twiddle build over up to 16 tiles
        size_t total_tiles = n_cg << (r + ps.s0);
        size_t tpc = total_tiles / (148 * 2 * 8);
        if (tpc < 1) tpc = 1;
        if (tpc > 32) tpc = 32;
        if (tpc > n_cg) tpc = n_cg;
        tpc = (n_cg + ((n_cg + tpc - 1) / tpc) - 1) / ((n_cg + tpc - 1) / tpc);   // even chunks
        a.tiles_per_cta = (uint32_t)tpc;
        a.last = last ? 1 : 0;
        size_t n_blocks = ((n_cg + tpc - 1) / tpc) << (r + ps.s0);
        if (n_blocks > 0x7fffffffULL) return cudaErrorInvalidConfiguration;
        unsigned grid = (unsigned)n_blocks;
        cudaError_t e;
        switch (nb) {
            case 1: e = launch_pass_lcl<1, 0>(a, grid, st); break;
            case 2: e = launch_pass_lcl<2, 0>(a, grid, st); break;
            case 3: e = launch_pass_lcl<3, 0>(a, grid, st); break;
            case 4: e = launch_pass_lcl<4, 0>(a, grid, st); break;
            case 5: e = launch_pass_lcl<5, 0>(a, grid, st); break;
            case 6: e = launch_pass_lcl<3, 3>(a, grid, st); break;
            case 7: e = launch_pass_lcl<4, 3>(a, grid, st); break;
            case 8: e = launch_pass_lcl<4, 4>(a, grid, st); break;
            case 9: e = launch_pass_lcl<5, 4>(a, grid, st); break;
            case 10: e = launch_pass_lcl<5, 5>(a, grid, st); break;
            default: e = cudaErrorInvalidConfiguration;
        }
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t ntt_lde(const NttPlan* plan, const uint64_t* coeffs, size_t in_stride, uint64_t* out, size_t out_stride,
                    size_t w, cudaStream_t st) {
    return run_passes(plan, coeffs, in_stride, out, out_stride, w, 0, plan->r, st);
}

cudaError_t ntt_lde_cosets(const NttPlan* plan, const uint64_t* coeffs, size_t in_stride, uint64_t* out,
                           size_t out_stride, size_t w, unsigned coset_first, unsigned lg_cosets, cudaStream_t st,
                           const uint64_t* const* coeff_ptrs_dev) {
    return run_passes(plan, coeffs, in_stride, out, out_stride, w, coset_first, lg_cosets, st, coeff_ptrs_dev);
}

cudaError_t ntt_inverse_bitrev(const NttPlan* plan, const uint64_t* values, size_t in_stride, uint64_t* out,
                               size_t out_stride, size_t w, cudaStream_t st) {
    return run_passes(plan, values, in_stride, out, out_stride, w, 0, plan->r, st);
}

// -------------------------------------------------------------------------------------------------
// data-movement helpers
// -------------------------------------------------------------------------------------------------
// out[j][brev(i)] = in[j][i] * scale   (scale = 1/d after an inverse transform, ifft_with_options fft.rs:88-93)
__global__ void k_bitrev_permute(const uint64_t* __restrict__ in, size_t in_stride, uint64_t* __restrict__ out,
                                 size_t out_stride, unsigned lg_n, uint64_t scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t j = blockIdx.y;
    if (i >= ((size_t)1 << lg_n)) return;
    size_t bi = brev_bits(i, lg_n);
    uint64_t v = in[j * in_stride + i];
    if (scale != 1) v = gl::canon(gl::mul(v, scale));
    out[j * out_stride + bi] = v;
}

// out[i] = canon(in[brev_{lg_n}(first + i)]) for i < count: the leaf-order slice [first, first + count) of a column given
// in natural LDE order (salt columns of a shard, oracle.rs:119-123 + :84)
__global__ void k_bitrev_gather(const uint64_t* __restrict__ in, unsigned lg_n, size_t first, size_t count,
                                uint64_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    // the sum inside the branch: brev_bits(first + i, lg_n) compiles to a select instead of this branch
    size_t src = lg_n ? (size_t)(__brevll((unsigned long long)(first + i)) >> (64 - lg_n)) : 0;
    out[i] = gl::canon(in[src]);
}

cudaError_t launch_bitrev_gather(const uint64_t* in, unsigned lg_n, size_t first, size_t count, uint64_t* out,
                                 cudaStream_t st) {
    if (count == 0) return cudaSuccess;
    k_bitrev_gather<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(in, lg_n, first, count, out);
    return cudaGetLastError();
}

uint64_t ntt_plan_scale(const NttPlan* plan) { return plan->scale; }

// The same permutation with both sides coalesced (lg_n >= 10): the index is [hi (5 bits) | mid | lo (5 bits)] and
// brev(i) = [brev(lo) | brev(mid) | brev(hi)], so for a fixed mid the 32 x 32 values (hi, lo) are read as 32 contiguous
// runs over lo and written as 32 contiguous runs over brev(hi): one shared-memory transpose per tile.
__global__ void __launch_bounds__(256) k_bitrev_permute_tiled(const uint64_t* __restrict__ in, size_t in_stride,
                                                             uint64_t* __restrict__ out, size_t out_stride, unsigned lg_n,
                                                             uint64_t scale) {
    __shared__ uint64_t t[32][33];
    const unsigned m = lg_n - 10;
    const size_t mid = blockIdx.x, j = blockIdx.y;
    const uint64_t* src = in + j * in_stride;
    uint64_t* dst = out + j * out_stride;
    const unsigned x = threadIdx.x;
    for (unsigned hi = threadIdx.y; hi < 32; hi += 8) {
        uint64_t v = src[((size_t)hi << (m + 5)) | (mid << 5) | x];
        if (scale != 1) v = gl::canon(gl::mul(v, scale));
        t[hi][x] = v;
    }
    __syncthreads();
    const size_t rmid = brev_bits(mid, m);
    const unsigned hi_src = __brev(x) >> 27;
    for (unsigned lo = threadIdx.y; lo < 32; lo += 8)
        dst[((size_t)(__brev(lo) >> 27) << (m + 5)) | (rmid << 5) | x] = t[hi_src][lo];
}

cudaError_t launch_bitrev_permute(const uint64_t* in, size_t in_stride, uint64_t* out, size_t out_stride, size_t w,
                                  unsigned lg_n, cudaStream_t st, uint64_t scale) {
    if (w == 0) return cudaSuccess;
    size_t n = (size_t)1 << lg_n;
    for (size_t j0 = 0; j0 < w; j0 += 65535) {
        size_t wj = w - j0 < 65535 ? w - j0 : 65535;
        if (lg_n >= 10 && lg_n <= 40) {
            dim3 grid((unsigned)(n >> 10), (unsigned)wj);
            k_bitrev_permute_tiled<<<grid, dim3(32, 8), 0, st>>>(in + j0 * in_stride, in_stride, out + j0 * out_stride, out_stride, lg_n, scale);
        } else {
            dim3 grid((unsigned)((n + 255) / 256), (unsigned)wj);
            k_bitrev_permute<<<grid, 256, 0, st>>>(in + j0 * in_stride, in_stride, out + j0 * out_stride, out_stride, lg_n, scale);
        }
    }
    return cudaGetLastError();
}

// out[c][r] = in[r][c]; 32x32 tiles through shared memory, both sides coalesced.
__global__ void k_transpose(const uint64_t* __restrict__ in, size_t in_pitch, uint64_t* __restrict__ out,
                            size_t out_pitch, size_t rows, size_t cols) {
    __shared__ uint64_t t[32][33];
    size_t c0 = (size_t)blockIdx.x * 32, r0 = (size_t)blockIdx.y * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        size_t r = r0 + k, c = c0 + threadIdx.x;
        if (r < rows && c < cols) t[k][threadIdx.x] = in[r * in_pitch + c];
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        size_t c = c0 + k, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out[c * out_pitch + r] = t[threadIdx.x][k];
    }
}

cudaError_t launch_transpose(const uint64_t* in, size_t in_pitch, uint64_t* out, size_t out_pitch, size_t rows,
                             size_t cols, cudaStream_t st) {
    if (rows == 0 || cols == 0) return cudaSuccess;
    // grid.y limit 65535: put the long dimension on x
    size_t bx = (cols + 31) / 32, by = (rows + 31) / 32;
    if (by > 65535) {
        // process in row slabs
        size_t slab_rows = (size_t)65535 * 32;
        for (size_t rr = 0; rr < rows; rr += slab_rows) {
            size_t nr = rows - rr < slab_rows ? rows - rr : slab_rows;
            dim3 grid((unsigned)bx, (unsigned)((nr + 31) / 32));
            k_transpose<<<grid, dim3(32, 8), 0, st>>>(in + rr * in_pitch, in_pitch, out + rr, out_pitch, nr, cols);
        }
    } else {
        dim3 grid((unsigned)bx, (unsigned)by);
        k_transpose<<<grid, dim3(32, 8), 0, st>>>(in, in_pitch, out, out_pitch, rows, cols);
    }
    return cudaGetLastError();
}

__global__ void k_gather_rows(const uint64_t* __restrict__ cols, size_t col_stride, uint32_t width,
                              const uint64_t* __restrict__ idx, size_t n_idx, uint64_t* __restrict__ out) {
    size_t k = blockIdx.x;
    if (k >= n_idx) return;
    size_t leaf = idx[k];
    for (uint32_t j = threadIdx.x; j < width; j += blockDim.x) out[k * width + j] = cols[(size_t)j * col_stride + leaf];
}

cudaError_t launch_gather_rows(const uint64_t* cols, size_t col_stride, uint32_t width, const uint64_t* idx,
                               size_t n_idx, uint64_t* out, cudaStream_t st) {
    if (n_idx == 0 || width == 0) return cudaSuccess;
    k_gather_rows<<<(unsigned)n_idx, 128, 0, st>>>(cols, col_stride, width, idx, n_idx, out);
    return cudaGetLastError();
}

// data[j][i] *= base^i   (coset_ifft: coefficients of P(shift x) -> coefficients of P, base = shift^-1; polynomial/mod.rs:68-72)
// base^i = hi[i >> 10] * lo[i & 1023] from two small tables (n / 1024 + 1024 exponentiations in all) instead of one
// exponentiation per element: two multiplications per element, HBM bound.
__global__ void k_power_tables(uint64_t base, size_t n, uint64_t* lo, uint64_t* hi) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 1024) lo[i] = gl::pow(base, i);
    size_t n_hi = (n + 1023) >> 10;
    if (i < n_hi) hi[i] = gl::pow(base, i << 10);
}

__global__ void k_mul_powers(uint64_t* data, size_t stride, size_t n, const uint64_t* __restrict__ lo,
                             const uint64_t* __restrict__ hi) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t* p = data + blockIdx.y * stride + i;
    *p = gl::canon(gl::mul(gl::mul(*p, lo[i & 1023]), hi[i >> 10]));
}

cudaError_t launch_mul_powers(uint64_t* data, size_t stride, size_t w, size_t n, uint64_t base, cudaStream_t st) {
    if (w == 0 || n == 0) return cudaSuccess;
    const size_t n_hi = (n + 1023) >> 10;
    uint64_t* tab = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&tab, (1024 + n_hi) * 8, st);
    if (e != cudaSuccess) return e;
    const size_t nt = n_hi > 1024 ? n_hi : 1024;
    k_power_tables<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(base % gl::P, n, tab, tab + 1024);
    for (size_t j0 = 0; j0 < w; j0 += 65535) {
        size_t wj = w - j0 < 65535 ? w - j0 : 65535;
        k_mul_powers<<<dim3((unsigned)((n + 255) / 256), (unsigned)wj), 256, 0, st>>>(data + j0 * stride, stride, n, tab, tab + 1024);
    }
    e = cudaGetLastError();
    cudaFreeAsync(tab, st);
    return e;
}

// rows in NATURAL LDE order with a stride: out[k][j] = cols[j][brev_{lg_n}((index_start + k) * step)], k < count, j < width --
// what get_lde_values(index_start + k, step) returns (oracle.rs:128-133), for a whole range of points at once.  Writes are
// coalesced (a warp writes one 256-byte piece of a row); reads are one sector per element (bit-reversed order has no locality).
__global__ void __launch_bounds__(256) k_lde_natural(const uint64_t* __restrict__ cols, size_t col_stride, uint32_t width,
                                                    unsigned lg_n, size_t index_start, size_t step, size_t count,
                                                    uint64_t* __restrict__ out) {
    const size_t k = (size_t)blockIdx.x * 8 + threadIdx.y;
    if (k >= count) return;
    const size_t idx = (index_start + k) * step;
    const size_t leaf = brev_bits(idx, lg_n);
    for (uint32_t j = threadIdx.x; j < width; j += 32) out[k * width + j] = __ldg(cols + (size_t)j * col_stride + leaf);
}

cudaError_t launch_lde_natural(const uint64_t* cols, size_t col_stride, uint32_t width, unsigned lg_n, size_t index_start,
                               size_t step, size_t count, uint64_t* out, cudaStream_t st) {
    if (count == 0 || width == 0) return cudaSuccess;
    k_lde_natural<<<(unsigned)((count + 7) / 8), dim3(32, 8), 0, st>>>(cols, col_stride, width, lg_n, index_start, step, count, out);
    return cudaGetLastError();
}

__global__ void k_canon(uint64_t* data, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) data[i] = gl::canon(data[i]);
}

cudaError_t launch_canonicalize(uint64_t* data, size_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_canon<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(data, n);
    return cudaGetLastError();
}

}  // namespace pcs
