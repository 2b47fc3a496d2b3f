// Element-wise Goldilocks field operations on the device (pcs_field_op): the device counterpart of the reference's
// field-arithmetic grid test (field/src/prime_field_testing.rs:7-17,78-125, instantiated goldilocks_field.rs:405-411).
// Every arithmetic routine of gl64.cuh that the kernels build on is reachable here, including the 128-bit reduction that
// the Poseidon S-boxes and the NTT butterflies are built with, so the tests can compare each of them with
// big-int arithmetic on the boundary inputs {0..9, 2^31+-10, 2^32+-10, 2^63+-10, p-10..p-1, non-canonical values}.
#include "common.cuh"
#include "gl64.cuh"

namespace pcs {

__global__ void k_field_op(int op, const uint64_t* __restrict__ a, const uint64_t* __restrict__ b, size_t n,
                           uint64_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t x = a[i], y = b ? b[i] : 0;
    uint64_t r;
    switch (op) {
        case PCS_OP_ADD: r = gl::add_lc(x, gl::canon(y)); break;             // loose + canonical, goldilocks_field.rs:199-221
        case PCS_OP_SUB: r = gl::sub_lc(x, gl::canon(y)); break;             // :223-243
        case PCS_OP_MUL: r = gl::mul(x, y); break;                            // :267-274 + reduce128 :356-369
        case PCS_OP_SQUARE: r = gl::sqr(x); break;
        case PCS_OP_CANON: r = x; break;                                      // to_canonical_u64 :171-178
        case PCS_OP_NEG: r = gl::sub_lc(0, gl::canon(x)); break;              // :245-255
        case PCS_OP_REDUCE96: r = gl::reduce96(x, (uint32_t)y); break;        // x + (y mod 2^32) * 2^64, :347-354
        case PCS_OP_MUL_2EXP: r = gl::mul(x, gl::pow(2, y % 192)); break;     // x * 2^y: 2 has order 192 (types.rs:227-262 relies on it)
        default: r = 0;
    }
    out[i] = gl::canon(r);
}

cudaError_t launch_field_op(int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_field_op<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(op, a, b, n, out);
    return cudaGetLastError();
}

}  // namespace pcs
