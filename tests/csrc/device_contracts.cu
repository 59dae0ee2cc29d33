// device_contracts.cu -- test-only harness: the device functions of mlkem_device.cuh called one by one, on the tables the
// library builds (mlkem_tables.inl), so that tests/test_device_contracts_gpu.py can hold each of them to its documented
// input domain against an exact reference.  Not part of the product: built as build/libmlkem_b200_contracts.so by
// `make contracts`.
//
// ABI (ctypes): every pointer is device memory; every launch goes to `stream` and returns a cudaError_t.  Polynomials are
// n x 256 uint16 in natural order; the kernels load and store them in the layouts the product's kernels use (the forward
// transforms take layout A and leave layout C, the inverse ones take layout C and leave layout A).
#include "../../crystals-kyber_b200/csrc/mlkem_device.cuh"

#include <stddef.h>
#include <string.h>

namespace {
using namespace mlkem;
#include "../../crystals-kyber_b200/csrc/mlkem_tables.inl"

// ------------------------------------------------------------------------------------------------ transforms
// One instantiation per kernel, as the product's callers use them (mlkem_kernels.cuh):
enum Transform {
    kNttFma = 0,       // ntt_warp<kFmaPipe>             k_noise
    kNttBalanced,      // ntt_warp<kBalanced>            k_decrypt, k_ntt_batch (all inputs < q)
    kNttExact,         // ntt_warp_exact                 k_ntt_batch (some input >= q)
    kInttFmaLazy,      // intt_warp<kFmaPipe, false>     matvec_row_tail, k_matvec_table, k_encrypt_v
    kInttBalanced,     // intt_warp<kBalanced, true>     k_decrypt, k_intt_batch
    kRoundTripFma,     // ntt_warp<kFmaPipe> then intt_warp<kFmaPipe, false>
};
constexpr int kTPB = 256;

template <int T>
__global__ void __launch_bounds__(kTPB) k_transform(int n, const uint16_t *__restrict__ in, uint16_t *__restrict__ out) {
    __shared__ __align__(16) uint16_t s_scratch[(kTPB / 32) * kScratchU16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = s_scratch + warp * kScratchU16;
    constexpr bool kForward = T == kNttFma || T == kNttBalanced || T == kNttExact || T == kRoundTripFma;
    constexpr bool kFma = T == kNttFma || T == kInttFmaLazy || T == kRoundTripFma;
    LaneTwiddles tw, twi;
    load_lane_twiddles<kFma>(tw, lane);
    load_lane_twiddles_inv<kFma>(twi, lane);
    for (long long p = (long long)blockIdx.x * (kTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kTPB / 32)) {
        const uint16_t *src = in + 256 * p;
        uint16_t *dst = out + 256 * p;
        uint32_t x[8];
#pragma unroll
        for (int r = 0; r < 8; r++) x[r] = src[kForward ? idxA(lane, r) : idxC(lane, r)];
        if (T == kNttFma || T == kRoundTripFma) ntt_warp<kFmaPipe>(x, scratch, lane, tw);
        if (T == kNttBalanced) ntt_warp<kBalanced>(x, scratch, lane, tw);
        if (T == kNttExact) ntt_warp_exact(x, scratch, lane);
        if (T == kInttFmaLazy || T == kRoundTripFma) intt_warp<kFmaPipe, false>(x, scratch, lane, twi);
        if (T == kInttBalanced) intt_warp<kBalanced, true>(x, scratch, lane, twi);
        constexpr bool kOutC = T == kNttFma || T == kNttBalanced || T == kNttExact;
#pragma unroll
        for (int r = 0; r < 8; r++) dst[kOutC ? idxC(lane, r) : idxA(lane, r)] = (uint16_t)x[r];
        __syncwarp();  // the next polynomial's first transpose reuses the scratch
    }
}

// ------------------------------------------------------------------------------------------------ base-case products
// sum over j < k of basemul_acc(a[j], b[j]) in layout C (lane owns coefficient pairs 4 lane .. 4 lane + 3, as k_encrypt_v and
// k_decrypt hold them), then the reductions its consumers apply: raw accumulators, barrett32 (matvec_row_tail, k_encrypt_v,
// k_decrypt with the FMA pipe), canon32 (k_decrypt with the balanced pipe).  out: n x 3 x 256 uint32.
__global__ void __launch_bounds__(kTPB) k_basemul(int n, int k, const uint16_t *__restrict__ a, const uint16_t *__restrict__ b,
                                                  uint32_t *__restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint2 gam[4];
#pragma unroll
    for (int i = 0; i < 4; i++) gam[i] = lane_gamma(4 * lane + i);
    for (long long p = (long long)blockIdx.x * (kTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kTPB / 32)) {
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
        for (int j = 0; j < k; j++) {
            const uint16_t *aj = a + 256 * (p * k + j) + 8 * lane, *bj = b + 256 * (p * k + j) + 8 * lane;
#pragma unroll
            for (int i = 0; i < 4; i++) basemul_acc(acc[2 * i], acc[2 * i + 1], aj[2 * i], aj[2 * i + 1], bj[2 * i], bj[2 * i + 1], gam[i]);
        }
        uint32_t *o = out + 3 * 256 * p + 8 * lane;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            o[r] = acc[r];
            o[256 + r] = barrett32(acc[r]);
            o[512 + r] = canon32(acc[r]);
        }
    }
}

// ------------------------------------------------------------------------------------------------ scalars
// out[j nx + i] = op(x_i, y0 + j), x_i = xs[i] (or i when xs is null).  The second operand is the d of Compress / Decompress,
// the table word of mul_shoup (0..127 zeta, 128..129 zeta_inv_last), the noise code, or the nibble position.
enum Scalar {
    kBarrett16 = 0,
    kCanon16,
    kCanonFma,
    kCompress,       // compress<y>, y = 1..11
    kCompressCanon,  // compress_canon<y>, y in {1, 4, 5, 10, 11}
    kCompressResid,  // compress_resid<y>, y in {1, 4, 5}
    kDecompress,     // decompress<y>, y = 1..11
    kMulShoup,       // mul_shoup(x, balanced word y)
    kNoiseCode,      // noise_code_to_coeff(x)
    kAddNoiseCode,   // add_noise_code(x, code y)
    kNibble,         // nibble_fma(x, nibble_weight(y))
};
#define MLKEM_D1_11(F) \
    F(1) F(2) F(3) F(4) F(5) F(6) F(7) F(8) F(9) F(10) F(11)
__device__ uint32_t scalar_op(int op, uint32_t x, uint32_t y) {
    switch (op) {
    case kBarrett16: return barrett16(x);
    case kCanon16: return canon16(x);
    case kCanonFma: return canon_fma(x);
    case kCompress:
        switch (y) {
#define MLKEM_CASE(d) case d: return compress<d>(x);
            MLKEM_D1_11(MLKEM_CASE)
#undef MLKEM_CASE
        }
        break;
    case kCompressCanon:
        switch (y) {
        case 1: return compress_canon<1>(x);
        case 4: return compress_canon<4>(x);
        case 5: return compress_canon<5>(x);
        case 10: return compress_canon<10>(x);
        case 11: return compress_canon<11>(x);
        }
        break;
    case kCompressResid:
        switch (y) {
        case 1: return compress_resid<1>(x);
        case 4: return compress_resid<4>(x);
        case 5: return compress_resid<5>(x);
        }
        break;
    case kDecompress:
        switch (y) {
#define MLKEM_CASE(d) case d: return decompress<d>(x);
            MLKEM_D1_11(MLKEM_CASE)
#undef MLKEM_CASE
        }
        break;
    case kMulShoup: return mul_shoup(x, y < 128 ? c_tw.zeta[y] : c_tw.zeta_inv_last[y - 128]);
    case kNoiseCode: return noise_code_to_coeff(x);
    case kAddNoiseCode: return add_noise_code(x, y);
    case kNibble: return nibble_fma(x, nibble_weight((int)y));
    }
    return 0xFFFFFFFFu;  // an (op, y) the harness does not know: fails any comparison
}
#undef MLKEM_D1_11
__global__ void __launch_bounds__(kTPB) k_scalar(int op, long long nx, const uint32_t *__restrict__ xs, uint32_t y0, int ny,
                                                 uint32_t *__restrict__ out) {
    for (long long t = (long long)blockIdx.x * kTPB + threadIdx.x; t < nx * ny; t += (long long)gridDim.x * kTPB) {
        const long long i = t % nx;
        const uint32_t j = (uint32_t)(t / nx);
        out[t] = scalar_op(op, xs ? xs[i] : (uint32_t)i, y0 + j);
    }
}

// Checks too large to copy back are counted on the device against 64-bit arithmetic.  result[0] = number of failures,
// result[1] = smallest failing index (the caller initialises it to ~0).
enum Sweep {
    kBarrett32All = 0,  // index = x, every x < 2^32: barrett32(x) < 2q and congruent, canon32(x) == x mod q
    kMulShoupFma,       // index = j n + i: mul_shoup_fma(a_i, word j) < 2q and congruent, j over the 258 FMA-table words
};
__device__ __forceinline__ uint2 fma_word(int j) {  // 0..127 zeta32, 128..255 gamma32, 256..257 zeta_inv_last32
    return j < 128 ? c_tw.zeta32[j] : j < 256 ? c_tw.gamma32[j - 128] : c_tw.zeta_inv_last32[j - 256];
}
constexpr int kFmaWords = 258;
__global__ void __launch_bounds__(kTPB) k_sweep(int op, long long n, const uint32_t *__restrict__ as,
                                                unsigned long long *__restrict__ result) {
    const long long total = op == kBarrett32All ? (1ll << 32) : n * kFmaWords;
    unsigned long long bad = 0, first = ~0ull;
    for (long long t = (long long)blockIdx.x * kTPB + threadIdx.x; t < total; t += (long long)gridDim.x * kTPB) {
        bool ok;
        if (op == kBarrett32All) {
            const uint32_t x = (uint32_t)t, want = (uint32_t)((unsigned long long)x % kQ), b = barrett32(x);
            ok = b < 2 * kQ && b % kQ == want && canon32(x) == want;
        } else {
            const uint32_t a = as[t % n];
            const uint2 w = fma_word((int)(t / n));
            const uint32_t r = mul_shoup_fma(a, w.x, w.y);
            ok = r < 2 * kQ && r % kQ == (uint32_t)((unsigned long long)a * w.x % kQ);
        }
        if (!ok) {
            bad++;
            first = min(first, (unsigned long long)t);
        }
    }
    if (bad) {
        atomicAdd(result, bad);
        atomicMin(result + 1, first);
    }
}

unsigned grid_for(long long work) {
    const long long blocks = (work + kTPB - 1) / kTPB;
    return (unsigned)(blocks < 148 * 16 ? (blocks > 0 ? blocks : 1) : 148 * 16);
}

}  // namespace

#define CONTRACTS_API extern "C" __attribute__((visibility("default")))

// The TwiddleTables and Keccak round constants that build_tables() produces (host only, no device needed).  Returns
// sizeof(TwiddleTables), or -1 when tw_cap is smaller.
CONTRACTS_API long long contracts_tables(void *tw, size_t tw_cap, void *rc24) {
    if (tw_cap < sizeof(TwiddleTables)) return -1;
    TwiddleTables t;
    uint2 rc[24];
    build_tables(t, rc);
    memcpy(tw, &t, sizeof t);
    memcpy(rc24, rc, sizeof rc);
    return (long long)sizeof t;
}

// Upload the tables to the harness's copies of c_tw, g_tw, c_keccak_rc and c_pow2 on the current device (what the library's
// acquire() does for its own).
CONTRACTS_API int contracts_init(void) {
    TwiddleTables t;
    uint2 rc[24];
    build_tables(t, rc);
    uint32_t pow2[32];
    for (int k = 0; k < 32; k++) pow2[k] = 1u << k;
    cudaError_t e;
    if ((e = cudaMemcpyToSymbol(c_tw, &t, sizeof t)) != cudaSuccess) return e;
    if ((e = cudaMemcpyToSymbol(g_tw, &t, sizeof t)) != cudaSuccess) return e;
    if ((e = cudaMemcpyToSymbol(c_keccak_rc, rc, sizeof rc)) != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_pow2, pow2, sizeof pow2);
}

// which: a Transform.  in, out: n x 256 uint16.
CONTRACTS_API int contracts_transform(int which, int n, const uint16_t *in, uint16_t *out, cudaStream_t stream) {
    const unsigned grid = grid_for((long long)n * 32);
    switch (which) {
    case kNttFma: k_transform<kNttFma><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    case kNttBalanced: k_transform<kNttBalanced><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    case kNttExact: k_transform<kNttExact><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    case kInttFmaLazy: k_transform<kInttFmaLazy><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    case kInttBalanced: k_transform<kInttBalanced><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    case kRoundTripFma: k_transform<kRoundTripFma><<<grid, kTPB, 0, stream>>>(n, in, out); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// a, b: n x k x 256 uint16 (any 12-bit values); out: n x 3 x 256 uint32 (raw, barrett32, canon32).
CONTRACTS_API int contracts_basemul(int n, int k, const uint16_t *a, const uint16_t *b, uint32_t *out, cudaStream_t stream) {
    k_basemul<<<grid_for((long long)n * 32), kTPB, 0, stream>>>(n, k, a, b, out);
    return cudaGetLastError();
}

// op: a Scalar.  xs: nx uint32 or null (x = index).  out: ny x nx uint32.
CONTRACTS_API int contracts_scalar(int op, long long nx, const uint32_t *xs, uint32_t y0, int ny, uint32_t *out, cudaStream_t stream) {
    k_scalar<<<grid_for(nx * ny), kTPB, 0, stream>>>(op, nx, xs, y0, ny, out);
    return cudaGetLastError();
}

// op: a Sweep.  as: n uint32 (kMulShoupFma only).  result: 2 x uint64, initialised by the caller to {0, ~0}.
CONTRACTS_API int contracts_sweep(int op, long long n, const uint32_t *as, unsigned long long *result, cudaStream_t stream) {
    k_sweep<<<148 * 16, kTPB, 0, stream>>>(op, n, as, result);
    return cudaGetLastError();
}
