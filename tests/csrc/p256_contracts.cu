// p256_contracts.cu -- test-only harness: the field, point and scalar functions of p256_device.cuh one by one, so that
// tests/test_p256_contracts_gpu.py can hold each to its documented bounds against Python integers.  Not part of the product:
// built as build/libp256_contracts.so by `make contracts`.
//
// ABI (ctypes): every pointer is device memory; launches go to `stream` and return a cudaError_t.  Rows are uint32 words:
// a field element is 8 little-endian words, a point 24 (X, Y, Z), a byte string its bytes in memory order.  p256_op(op, n, a,
// a_words, b, b_words, out, out_words) runs `op` on row i of a and b (row lengths in words) and writes row i of out.
#include "../../crystals-kyber_b200/csrc/p256_device.cuh"

namespace {
using namespace p256;

enum Op {
    kAdd = 0,   // a, b: fe -> fe
    kSub,       // a, b: fe -> fe
    kMul,       // a, b: fe -> fe (Montgomery product)
    kSqr,       // a: fe -> fe
    kCanon,     // a: 256-bit -> fe
    kInv,       // a: fe -> fe
    kToMont,    // a: 256-bit -> fe
    kFromMont,  // a: fe -> fe
    kPtAdd,     // a, b: pt -> pt
    kPtDbl,     // a: pt -> pt
    kSeed,      // a: 40 bytes -> 8 words
    kScalarOk,  // a: 8 words -> 1 word (the mask)
    kDecode,    // a: 65 bytes -> 1 word (the mask) + pt
    kMulPoint,  // a: 8-word scalar, b: pt -> pt
};

P256_HD fe fe_at(const uint32_t *p) {
    fe r;
    for (int i = 0; i < 8; i++) r.v[i] = p[i];
    return r;
}
P256_HD void fe_put(uint32_t *p, const fe &a) {
    for (int i = 0; i < 8; i++) p[i] = a.v[i];
}
P256_HD pt pt_at(const uint32_t *p) { return {fe_at(p), fe_at(p + 8), fe_at(p + 16)}; }
P256_HD void pt_put(uint32_t *p, const pt &P) {
    fe_put(p, P.X), fe_put(p + 8, P.Y), fe_put(p + 16, P.Z);
}

P256_HD void run_op(int op, const uint32_t *a, const uint32_t *b, uint32_t *out) {
    switch (op) {
    case kAdd: fe_put(out, fe_add(fe_at(a), fe_at(b))); break;
    case kSub: fe_put(out, fe_sub(fe_at(a), fe_at(b))); break;
    case kMul: fe_put(out, fe_mul(fe_at(a), fe_at(b))); break;
    case kSqr: fe_put(out, fe_sqr(fe_at(a))); break;
    case kCanon: fe_put(out, fe_canon(fe_at(a))); break;
    case kInv: fe_put(out, fe_inv(fe_at(a))); break;
    case kToMont: fe_put(out, fe_to_mont(fe_at(a))); break;
    case kFromMont: fe_put(out, fe_from_mont(fe_at(a))); break;
    case kPtAdd: pt_put(out, pt_add(pt_at(a), pt_at(b))); break;
    case kPtDbl: pt_put(out, pt_dbl(pt_at(a))); break;
    case kSeed: seed_scalar(reinterpret_cast<const uint8_t *>(a), reinterpret_cast<const uint8_t *>(a) + 32, out); break;
    case kScalarOk: out[0] = scalar_ok_mask(a); break;
    case kDecode: {
        pt P;
        out[0] = point_decode(reinterpret_cast<const uint8_t *>(a), P);
        pt_put(out + 1, P);
        break;
    }
    default: pt_put(out, scalarmult(a, pt_at(b))); break;
    }
}

}  // namespace

#ifdef __CUDACC__
#include <cuda_runtime.h>

namespace {
__global__ void __launch_bounds__(128) k_op(int op, long long n, const uint32_t *__restrict__ a, int aw, const uint32_t *__restrict__ b, int bw,
                                            uint32_t *__restrict__ out, int ow) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        run_op(op, a + aw * i, b + bw * i, out + ow * i);
}
}  // namespace

extern "C" __attribute__((visibility("default"))) int p256_op(int op, long long n, const void *a, int aw, const void *b, int bw, void *out,
                                                              int ow, void *stream) {
    long long blocks = (n + 127) / 128;
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (blocks < 1) blocks = 1;
    k_op<<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(op, n, (const uint32_t *)a, aw, (const uint32_t *)b, bw,
                                                                         (uint32_t *)out, ow);
    return (int)cudaGetLastError();
}
#else
// host build of the same functions (a CPU check of p256_device.cuh): g++ -x c++ -shared -fPIC
extern "C" __attribute__((visibility("default"))) int p256_op(int op, long long n, const void *a, int aw, const void *b, int bw, void *out,
                                                              int ow, void *) {
    for (long long i = 0; i < n; i++)
        run_op(op, (const uint32_t *)a + aw * i, (const uint32_t *)b + bw * i, (uint32_t *)out + ow * i);
    return 0;
}
#endif
