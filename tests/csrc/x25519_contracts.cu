// x25519_contracts.cu -- test-only harness: the field functions of x25519_device.cuh one by one, so that
// tests/test_x25519_contracts_gpu.py can hold each to its documented limb bounds against Python integers.  Not part of the
// product: built as build/libx25519_contracts.so by `make contracts`.
//
// ABI (ctypes): every pointer is device memory; launches go to `stream` and return a cudaError_t.  Field elements are n x 10
// uint32 limbs; op kFreeze writes n x 8 uint32 words (the canonical value), every other op n x 10 limbs.
#include "../../crystals-kyber_b200/csrc/x25519_device.cuh"

#include <cuda_runtime.h>

namespace {
using namespace x25519;

enum Op { kAdd = 0, kSub, kMul, kSq, kMul121665, kFreeze, kCarry };

__global__ void __launch_bounds__(256) k_field(int op, long long n, const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                               uint32_t *__restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        fe x, y, r;
#pragma unroll
        for (int k = 0; k < 10; k++) x.v[k] = a[10 * i + k], y.v[k] = b[10 * i + k];
        if (op == kFreeze) {
            uint32_t w[8];
            fe_freeze(x, w);
#pragma unroll
            for (int k = 0; k < 8; k++) out[8 * i + k] = w[k];
            continue;
        }
        switch (op) {
        case kAdd: r = fe_add(x, y); break;
        case kSub: r = fe_sub(x, y); break;
        case kMul: r = fe_mul(x, y); break;
        case kSq: r = fe_sq(x); break;
        case kMul121665: r = fe_mul121665(x); break;
        default: r = fe_carry(x); break;
        }
#pragma unroll
        for (int k = 0; k < 10; k++) out[10 * i + k] = r.v[k];
    }
}

}  // namespace

extern "C" __attribute__((visibility("default"))) int x25519_contracts_field(int op, long long n, const void *a, const void *b, void *out,
                                                                            void *stream) {
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (blocks < 1) blocks = 1;
    k_field<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(op, n, (const uint32_t *)a, (const uint32_t *)b, (uint32_t *)out);
    return (int)cudaGetLastError();
}
