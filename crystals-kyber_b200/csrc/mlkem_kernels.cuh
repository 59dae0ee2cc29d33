// mlkem_kernels.cuh -- the CUDA kernels of the batched ML-KEM engine (sm_100a).
//
// Work decomposition (DESIGN.md has the full picture):
//   * every Keccak sponge is run by ONE THREAD (state in registers); a warp therefore runs 32 sponges of
//     the same kind in lock step.  Kernels are split by sponge kind so warps never mix roles.  (Small batches are the
//     exception: the k_*_warp hash kernels run one sponge per WARP, the latency form -- keccak_f1600_warp.)
//   * every polynomial operation (NTT, inverse NTT, multiply-accumulate, compress, pack) is run by ONE
//     WARP per polynomial, 8 coefficients per lane.
//   * the matrix expansion is fused with its consumer: k_sample_matvec samples the k entries of one matrix
//     row with k threads straight into shared memory (exactly three XOF blocks per sponge, straight-line code) and
//     the warps of the block then multiply them with the vector, accumulate, (inverse-)transform, add the noise,
//     compress and pack -- the matrix never exists in HBM.  The 2.7 % of rows that own a sponge needing a fourth
//     block go to a list that k_sample_matvec_list works off with the general sampler.
//   * keys that are resident on the device (mlkem_b200_keys) are addressed through a per-item index (KeySel); with an
//     expanded key table the matrix is sampled once per KEY and k_matvec_table reads it back instead.
//
// All byte buffers are dense and item-major (item i of an array with per-item size S starts at i*S);
// every per-item size on this path is a multiple of 16 bytes, so with 16-byte aligned bases every item,
// row and hash input is 8-byte aligned.
#pragma once
#include "mlkem_device.cuh"

namespace mlkem {

template <int K_, int ETA1_, int ETA2_, int DU_, int DV_>
struct ParamSet {  // ml_kem.c:1363 init()
    static constexpr int K = K_, ETA1 = ETA1_, ETA2 = ETA2_, DU = DU_, DV = DV_;
    static constexpr int EK = 384 * K + 32;            // encapsulation key bytes (ml_kem.c:730)
    static constexpr int DKPKE = 384 * K;              // K-PKE decryption key bytes (ml_kem.c:731)
    static constexpr int DK = 768 * K + 96;            // decapsulation key bytes (ml_kem.c:1050)
    static constexpr int C1ROW = 32 * DU;              // bytes of one compressed u row
    static constexpr int C2 = 32 * DV;                 // bytes of compressed v
    static constexpr int C = C1ROW * K + C2;           // ciphertext bytes (ml_kem.c:1105)
};
using P512 = ParamSet<2, 3, 2, 10, 4>;
using P768 = ParamSet<3, 2, 2, 10, 4>;
using P1024 = ParamSet<4, 2, 2, 11, 5>;

// Which key an item uses.  Unkeyed calls: item i reads row i of the key array it was given.  Keyed calls (the resident
// key tables of mlkem_b200_keys_*): row index[i], or row (base + i) % nkeys when the caller passed no index array
// (keys reused cyclically, base = global index of the chunk's first item).
struct KeySel {
    const uint32_t *index;
    uint32_t base, nkeys;
};
__device__ __forceinline__ size_t key_row(const KeySel &k, int item) {
    if (k.index) return min(__ldg(k.index + item), k.nkeys - 1u);  // clamped: memory safety for device-memory callers
    if (k.nkeys) return (k.base + (uint32_t)item) % k.nkeys;
    return (size_t)item;
}

constexpr int kHashTPB = 128;   // threads per block of the thread-per-item hash kernels
constexpr int kNoiseTPB = 128;  // threads (= sponges) per block of k_noise
constexpr int kSlotWords = 129; // shared-memory words per sampled polynomial slot (odd: conflict-free per-thread writes)
constexpr int kMatTableTPB = 128; // threads per block of k_matvec_table (4 rows in flight per block)

// =================================================================================================
// Reference cell layout <-> dense bytes
// =================================================================================================
// The reference keeps one byte per 4-byte `union byte` cell (ml_kem.h:35-38; value in the low 8 bits, upper bits ignored on
// input -- D5).  Thread = four cells = one dense 32-bit word: a 128-bit access on the cell side, a 32-bit one on the
// dense side, both coalesced.  HBM-bound (20 bytes moved per 4 payload bytes).
__global__ void __launch_bounds__(256) k_cells_to_bytes(size_t nwords, const uint4 *__restrict__ cells, uint32_t *__restrict__ dense) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nwords) return;
    const uint4 c = __ldg(cells + i);
    dense[i] = (c.x & 0xFFu) | ((c.y & 0xFFu) << 8) | ((c.z & 0xFFu) << 16) | (c.w << 24);
}
__global__ void __launch_bounds__(256) k_bytes_to_cells(size_t nwords, const uint32_t *__restrict__ dense, uint4 *__restrict__ cells) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nwords) return;
    const uint32_t w = __ldg(dense + i);
    cells[i] = make_uint4(w & 0xFFu, (w >> 8) & 0xFFu, (w >> 16) & 0xFFu, w >> 24);
}

// =================================================================================================
// Hash kernels: one item per thread
// =================================================================================================

// (rho, sigma) = G(d || k)   (ml_kem.c:674-681).  33-byte message, SHA3-512: one permutation.
// Also places rho at the tail of ek (ml_kem.c:745-747) and, for the full decapsulation key, inside dk (:1058-1062):
// rho_out + i*rho_stride, rho_out2 + i*rho_stride2 (nullable).
__global__ void __launch_bounds__(kHashTPB) k_keygen_G(int n, const uint8_t *__restrict__ d, uint32_t kbyte,
                                                       uint8_t *__restrict__ rs, uint8_t *__restrict__ rho_out, size_t rho_stride,
                                                       uint8_t *__restrict__ rho_out2, size_t rho_stride2) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane a[25];
    keccak_zero(a);
#pragma unroll
    for (int w = 0; w < 4; w++) a[w] = load_lane(d + 32 * (size_t)i + 8 * w);
    a[4].lo = kbyte | (kSfxHash << 8);
    a[kRateSha3_512 - 1].hi ^= 0x80000000u;
    keccak_f1600(a);
#pragma unroll
    for (int w = 0; w < 8; w++) store_lane(rs + 64 * (size_t)i + 8 * w, a[w]);
#pragma unroll
    for (int w = 0; w < 4; w++) {
        store_lane(rho_out + rho_stride * i + 8 * w, a[w]);
        if (rho_out2) store_lane(rho_out2 + rho_stride2 * i + 8 * w, a[w]);
    }
}

// SHA3-256 over `P::EK` bytes at `ek`; result in h[0..3].
template <class P>
__device__ __forceinline__ void hash_H_ek(const uint8_t *ek, Lane h[4]) {
    Lane a[25];
    sponge_absorb_words<kRateSha3_256>(a, P::EK / 8, kSfxHash, [&](int w) { return load_lane(ek + 8 * w); });
#pragma unroll
    for (int w = 0; w < 4; w++) h[w] = a[w];
}

// SHA3-512 over the 64-byte message x || y; output lanes 0..7 left in a[].
__device__ __forceinline__ void hash_G_64(Lane a[25], const Lane x[4], const Lane y[4]) {
    keccak_zero(a);
#pragma unroll
    for (int w = 0; w < 4; w++) {
        a[w] = x[w];
        a[4 + w] = y[w];
    }
    a[8].lo = kSfxHash;
    a[8].hi = 0x80000000u;
    keccak_f1600(a);
}

// KeyGen tail (ml_kem.c:1064-1077): dk[768k+32 .. +32) = H(ek), dk[768k+64 .. +32) = z.
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_keygen_H(int n, const uint8_t *__restrict__ ek, const uint8_t *__restrict__ z,
                                                       uint8_t *__restrict__ dk) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane h[4];
    hash_H_ek<P>(ek + (size_t)P::EK * i, h);
    uint8_t *tail = dk + (size_t)P::DK * i + 768 * P::K + 32;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        store_lane(tail + 8 * w, h[w]);
        store_lane(tail + 32 + 8 * w, load_lane(z + 32 * (size_t)i + 8 * w));
    }
}

// Encaps front (ml_kem.c:1108-1124): h = H(ek); (K, r) = G(m || h).
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_encaps_HG(int n, const uint8_t *__restrict__ ek, const uint8_t *__restrict__ m,
                                                        uint8_t *__restrict__ Kout, uint8_t *__restrict__ r) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane h[4], mm[4], a[25];
    hash_H_ek<P>(ek + (size_t)P::EK * i, h);
#pragma unroll
    for (int w = 0; w < 4; w++) mm[w] = load_lane(m + 32 * (size_t)i + 8 * w);
    hash_G_64(a, mm, h);
#pragma unroll
    for (int w = 0; w < 4; w++) {
        store_lane(Kout + 32 * (size_t)i + 8 * w, a[w]);
        store_lane(r + 32 * (size_t)i + 8 * w, a[4 + w]);
    }
}

// Keyed Encaps front: h = H(ek) was computed once when the key table was loaded (k_hash_ek_table), so only
// (K, r) = G(m || h) is left (ml_kem.c:1116-1124).
__global__ void __launch_bounds__(kHashTPB) k_encaps_G_keyed(int n, const uint8_t *__restrict__ hek, KeySel keys, const uint8_t *__restrict__ m,
                                                             uint8_t *__restrict__ Kout, uint8_t *__restrict__ r) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane h[4], mm[4], a[25];
    const uint8_t *hp = hek + 32 * key_row(keys, i);
#pragma unroll
    for (int w = 0; w < 4; w++) {
        mm[w] = load_lane(m + 32 * (size_t)i + 8 * w);
        h[w] = load_lane(hp + 8 * w);
    }
    hash_G_64(a, mm, h);
#pragma unroll
    for (int w = 0; w < 4; w++) {
        store_lane(Kout + 32 * (size_t)i + 8 * w, a[w]);
        store_lane(r + 32 * (size_t)i + 8 * w, a[4 + w]);
    }
}
// h[i] = H(ek_i) for the rows of a key table (ek_i at ek + i*ek_stride): run once per table.
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_hash_ek_table(int n, const uint8_t *__restrict__ ek, size_t ek_stride, uint8_t *__restrict__ hek) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane h[4];
    hash_H_ek<P>(ek + ek_stride * i, h);
#pragma unroll
    for (int w = 0; w < 4; w++) store_lane(hek + 32 * (size_t)i + 8 * w, h[w]);
}

// Plain H over ek (used by the public-wrapper hash check, ml_kem.c:1336-1350): status[i] = -5 on mismatch.
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_check_dk_hash(int n, const uint8_t *__restrict__ dk, int *__restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *base = dk + (size_t)P::DK * i;
    Lane h[4];
    hash_H_ek<P>(base + 384 * P::K, h);
    uint32_t diff = 0;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        Lane s = load_lane(base + 768 * P::K + 32 + 8 * w);
        diff |= (s.lo ^ h[w].lo) | (s.hi ^ h[w].hi);
    }
    status[i] = diff ? -5 : 0;
}

// The modulus check of ML-KEM.Encaps (FIPS 203 section 7.2; ml_kem.c:1273-1291 where it cannot fail, D4):
// status[i] = -4 when any 12-bit coefficient of ek is >= q.  FIPS mode only.
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_check_ek_modulus(int n, const uint8_t *__restrict__ ek, int *__restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(ek + (size_t)P::EK * i);
    uint32_t bad = 0;
    for (int t = 0; t < 96 * P::K; t += 3) {  // 3 words = 8 coefficients
        uint32_t w0 = __ldg(w + t), w1 = __ldg(w + t + 1), w2 = __ldg(w + t + 2);
        uint32_t c[8] = {w0 & 0xFFF, (w0 >> 12) & 0xFFF, (w0 >> 24) | ((w1 & 0xF) << 8), (w1 >> 4) & 0xFFF,
                         (w1 >> 16) & 0xFFF, (w1 >> 28) | ((w2 & 0xFF) << 4), (w2 >> 8) & 0xFFF, w2 >> 20};
#pragma unroll
        for (int k = 0; k < 8; k++) bad |= (c[k] >= kQ);
    }
    status[i] = bad ? -4 : 0;
}

// KEM_Decaps returns NULL for an item that fails its input checks (ml_kem.c:1344-1350): the batched form
// zeroes that item's key instead (status[i] != 0 tells the caller).
__global__ void __launch_bounds__(kHashTPB) k_mask_keys(int n, const int *__restrict__ status, uint8_t *__restrict__ K) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (status[i] != 0) {
        uint4 zero = make_uint4(0, 0, 0, 0);
        reinterpret_cast<uint4 *>(K + 32 * (size_t)i)[0] = zero;
        reinterpret_cast<uint4 *>(K + 32 * (size_t)i)[1] = zero;
    }
}

// Decaps (ml_kem.c:1181-1193): (K', r') = G(m' || h), h = dk[768k+32 .. +32).
template <class P>
__global__ void __launch_bounds__(kHashTPB) k_decaps_G(int n, const uint8_t *__restrict__ mprime, const uint8_t *__restrict__ dk, KeySel keys,
                                                       uint8_t *__restrict__ Kr) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Lane h[4], mm[4], a[25];
    const uint8_t *hp = dk + (size_t)P::DK * key_row(keys, i) + 768 * P::K + 32;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        mm[w] = load_lane(mprime + 32 * (size_t)i + 8 * w);
        h[w] = load_lane(hp + 8 * w);
    }
    hash_G_64(a, mm, h);
#pragma unroll
    for (int w = 0; w < 8; w++) store_lane(Kr + 64 * (size_t)i + 8 * w, a[w]);
}

// Decaps tail (ml_kem.c:1196-1215): Kbar = J(z || c) -- SHAKE128 in the reference (D2) -- then a
// branch-free select between K' and Kbar on the re-encryption mismatch flag.  The reference's compare is
// an early-exit loop; the selected key is the same.
template <class P, int RATE = kRateShake128>
__global__ void __launch_bounds__(kHashTPB) k_decaps_J_select(int n, const uint8_t *__restrict__ dk, KeySel keys, const uint8_t *__restrict__ c,
                                                              const uint8_t *__restrict__ Kr, const uint32_t *__restrict__ flags,
                                                              uint8_t *__restrict__ Kout) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *z = dk + (size_t)P::DK * key_row(keys, i) + 768 * P::K + 64;
    const uint8_t *ci = c + (size_t)P::C * i;
    Lane a[25];
    // RATE 21 = SHAKE128 (the reference's J, D2); RATE 17 = SHAKE256 (FIPS 203)
    sponge_absorb_words<RATE>(a, 4 + P::C / 8, kSfxXof,
                              [&](int w) { return w < 4 ? load_lane(z + 8 * w) : load_lane(ci + 8 * (w - 4)); });
    uint32_t mask = flags[i] ? 0xFFFFFFFFu : 0u;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        Lane kp = load_lane(Kr + 64 * (size_t)i + 8 * w);
        Lane o{(a[w].lo & mask) | (kp.lo & ~mask), (a[w].hi & mask) | (kp.hi & ~mask)};
        store_lane(Kout + 32 * (size_t)i + 8 * w, o);
    }
}

// -------------------------------------------------------------------------------------------------
// The same hash kernels with one item per WARP (keccak_f1600_warp): small batches, where the chains of dependent
// permutations -- 9 for H(ek), 7 for J(z || c) at ML-KEM-768 -- are latency, not throughput.  The host picks these when the
// batch has at most kWarpHashMaxItems items (MLKEM_B200_WARP_HASH_MAX); results are identical.
// -------------------------------------------------------------------------------------------------
constexpr int kWarpHashTPB = 128;        // 4 items per block
constexpr int kWarpHashMaxItems = 1024;  // one warp per item costs ~8 x the issue slots of one thread per item: past ~2 000 items the
                                         // thread form is faster again (DESIGN.md section 5)

// SHA3-256 over P::EK bytes at `ek`: lanes 0..3 of the result hold the digest words.
template <class P>
__device__ __forceinline__ Lane warp_hash_H_ek(const uint8_t *ek, int lane, const WarpSponge &w) {
    return warp_sponge_absorb_words<kRateSha3_256>(lane, w, P::EK / 8, kSfxHash, [&](int i) { return load_lane(ek + 8 * i); });
}
// SHA3-512 over x || y, x = 32 bytes in memory, y = the words held by lanes 0..3 of `y03`: lanes 0..7 hold the digest words.
__device__ __forceinline__ Lane warp_hash_G_64(const uint8_t *x, Lane y03, int lane, const WarpSponge &w) {
    const Lane y = shfl_lane(y03, (lane - 4) & 31);  // lanes 4..7 take y[0..3]
    Lane a{0u, 0u};
    if (lane < 4) a = load_lane(x + 8 * lane);
    else if (lane < 8) a = y;
    else if (lane == 8) a = Lane{kSfxHash, 0x80000000u};  // 64-byte message: suffix and pad share lane 8 = RATE - 1
    keccak_f1600_warp(a, w);
    return a;
}

template <class P>
__global__ void __launch_bounds__(kWarpHashTPB) k_keygen_H_warp(int n, const uint8_t *__restrict__ ek, const uint8_t *__restrict__ z,
                                                                uint8_t *__restrict__ dk) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * (kWarpHashTPB / 32) + (threadIdx.x >> 5);
    if (i >= n) return;  // warp-uniform
    const WarpSponge w = warp_sponge_init(lane);
    const Lane h = warp_hash_H_ek<P>(ek + (size_t)P::EK * i, lane, w);
    uint8_t *tail = dk + (size_t)P::DK * i + 768 * P::K + 32;  // dk tail = H(ek) || z, ml_kem.c:1064-1077
    if (lane < 4) store_lane(tail + 8 * lane, h);
    else if (lane < 8) store_lane(tail + 8 * lane, load_lane(z + 32 * (size_t)i + 8 * (lane - 4)));
}

template <class P>
__global__ void __launch_bounds__(kWarpHashTPB) k_encaps_HG_warp(int n, const uint8_t *__restrict__ ek, const uint8_t *__restrict__ m,
                                                                 uint8_t *__restrict__ Kout, uint8_t *__restrict__ r) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * (kWarpHashTPB / 32) + (threadIdx.x >> 5);
    if (i >= n) return;
    const WarpSponge w = warp_sponge_init(lane);
    const Lane h = warp_hash_H_ek<P>(ek + (size_t)P::EK * i, lane, w);   // ml_kem.c:1108
    const Lane a = warp_hash_G_64(m + 32 * (size_t)i, h, lane, w);       // (K, r) = G(m || h), ml_kem.c:1116-1124
    if (lane < 4) store_lane(Kout + 32 * (size_t)i + 8 * lane, a);
    else if (lane < 8) store_lane(r + 32 * (size_t)i + 8 * (lane - 4), a);
}

template <class P>
__global__ void __launch_bounds__(kWarpHashTPB) k_check_dk_hash_warp(int n, const uint8_t *__restrict__ dk, int *__restrict__ status) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * (kWarpHashTPB / 32) + (threadIdx.x >> 5);
    if (i >= n) return;
    const WarpSponge w = warp_sponge_init(lane);
    const uint8_t *base = dk + (size_t)P::DK * i;
    const Lane h = warp_hash_H_ek<P>(base + 384 * P::K, lane, w);
    bool diff = false;
    if (lane < 4) {
        const Lane s = load_lane(base + 768 * P::K + 32 + 8 * lane);
        diff = ((s.lo ^ h.lo) | (s.hi ^ h.hi)) != 0;
    }
    const bool any = __any_sync(kFullMask, diff);
    if (lane == 0) status[i] = any ? -5 : 0;
}

template <class P, int RATE = kRateShake128>
__global__ void __launch_bounds__(kWarpHashTPB) k_decaps_J_select_warp(int n, const uint8_t *__restrict__ dk, KeySel keys, const uint8_t *__restrict__ c,
                                                                       const uint8_t *__restrict__ Kr, const uint32_t *__restrict__ flags,
                                                                       uint8_t *__restrict__ Kout) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * (kWarpHashTPB / 32) + (threadIdx.x >> 5);
    if (i >= n) return;
    const WarpSponge w = warp_sponge_init(lane);
    const uint8_t *z = dk + (size_t)P::DK * key_row(keys, i) + 768 * P::K + 64;
    const uint8_t *ci = c + (size_t)P::C * i;
    const Lane a = warp_sponge_absorb_words<RATE>(lane, w, 4 + P::C / 8, kSfxXof,
                                                  [&](int t) { return t < 4 ? load_lane(z + 8 * t) : load_lane(ci + 8 * (t - 4)); });
    const uint32_t mask = flags[i] ? 0xFFFFFFFFu : 0u;  // branch-free select, as in k_decaps_J_select
    if (lane < 4) {
        const Lane kp = load_lane(Kr + 64 * (size_t)i + 8 * lane);
        store_lane(Kout + 32 * (size_t)i + 8 * lane, Lane{(a.lo & mask) | (kp.lo & ~mask), (a.hi & mask) | (kp.hi & ~mask)});
    }
}

// Generic batched hash over equal-length messages, length a multiple of 8 bytes.  RATE (lanes) and the suffix select the
// function, OUTW the output lanes: H = <17, 4> + 0x06, G = <9, 8> + 0x06, J = <21, 4> + 0x1F (the host maps `which` to these).
template <int RATE, int OUTW>
__global__ void __launch_bounds__(kHashTPB) k_hash_words(int n, const uint8_t *__restrict__ in, int nwords, uint32_t sfx,
                                                         uint8_t *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *p = in + (size_t)nwords * 8 * i;
    Lane a[25];
    sponge_absorb_words<RATE>(a, nwords, sfx, [&](int w) { return load_lane(p + 8 * w); });
#pragma unroll
    for (int w = 0; w < OUTW; w++) store_lane(out + (size_t)OUTW * 8 * i + 8 * w, a[w]);
}

// General sponge over pre-padded messages (the SHA-3 front-end sha3_b / sha3_h / sha3_s, sha3.c:408-494).
// The host lays out N || suffix || pad (sha3.c:226,257-277, a pure bit-layout step) as `nblocks` blocks of
// `rl` 64-bit lanes per message; the device absorbs them and squeezes `out_bytes` bytes following
// sha3.c:298-311 (a permutation only when more output is still needed).  One message per thread.
__global__ void __launch_bounds__(kHashTPB) k_sponge_padded(int n, const uint8_t *__restrict__ padded, int nblocks, int rl,
                                                            uint8_t *__restrict__ out, int out_bytes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *p = padded + (size_t)i * nblocks * rl * 8;
    Lane a[25];
    keccak_zero(a);
    for (int b = 0; b < nblocks; b++) {
#pragma unroll
        for (int l = 0; l < 25; l++)
            if (l < rl) {
                Lane w = load_lane(p + ((size_t)b * rl + l) * 8);
                a[l].lo ^= w.lo;
                a[l].hi ^= w.hi;
            }
        keccak_f1600(a);
    }
    const int out_stride = (out_bytes + 7) & ~7;
    uint8_t *o = out + (size_t)i * out_stride;
    int done = 0;
    while (done < out_bytes) {
        int take = min(rl * 8, out_bytes - done);
#pragma unroll
        for (int l = 0; l < 25; l++)
            if (l * 8 < take) store_lane(o + done + l * 8, a[l]);
        done += take;
        if (done < out_bytes) keccak_f1600(a);
    }
}

// =================================================================================================
// Noise: PRF_eta(seed, nonce) = SHAKE128(seed || nonce) (D1) -> SamplePolyCBD_eta -> [NTT]
// =================================================================================================

// ml_kem.c:253 SamplePolyCBD on one 32-bit word of PRF output for eta = 2: 8 coefficients, returned as
// 4-bit codes (coefficient + 3).
__device__ __forceinline__ uint32_t cbd2_word(uint32_t w) {
    uint32_t t = w - ((w >> 1) & 0x55555555u);  // per bit pair: b0 + b1 (= 2 b1 + b0 - b1), one instruction less than masking both
    uint32_t x = t & 0x33333333u, y = (t >> 2) & 0x33333333u;
    return x + (0x33333333u - y);
}
// eta = 3: 96 bits (w0,w1,w2) -> 16 coefficients -> two words of 4-bit codes.
__device__ __forceinline__ uint32_t cbd3_chunk(uint32_t c24) {  // 4 coefficients -> 4 codes in the low 16 bits
    uint32_t t = (c24 & 0x249249u) + ((c24 >> 1) & 0x249249u) + ((c24 >> 2) & 0x249249u);
    uint32_t out = 0;
#pragma unroll
    for (int m = 0; m < 4; m++) {
        uint32_t x = (t >> (6 * m)) & 7u, y = (t >> (6 * m + 3)) & 7u;
        out |= (x + 3u - y) << (4 * m);
    }
    return out;
}
__device__ __forceinline__ void cbd3_words(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t &o0, uint32_t &o1) {
    uint32_t c0 = w0 & 0xFFFFFFu, c1 = (w0 >> 24) | ((w1 & 0xFFFFu) << 8), c2 = (w1 >> 16) | ((w2 & 0xFFu) << 16), c3 = w2 >> 8;
    o0 = cbd3_chunk(c0) | (cbd3_chunk(c1) << 16);
    o1 = cbd3_chunk(c2) | (cbd3_chunk(c3) << 16);
}

// PRF + CBD for one (seed, nonce): 32 words of 4-bit codes written through `put(word_index, value)`.
// RATE = 21 lanes: SHAKE128, what the reference's PRF is (D1, ml_kem.c:508).  RATE = 17 lanes: SHAKE256, the PRF of
// FIPS 203 (library flag MLKEM_B200_FLAG_FIPS203).
template <int ETA, int RATE, typename PUT>
__device__ __forceinline__ void prf_cbd_codes(const Lane seed[4], uint32_t nonce, PUT put) {
    Lane a[25];
    keccak_zero(a);
#pragma unroll
    for (int w = 0; w < 4; w++) a[w] = seed[w];
    a[4].lo = nonce | (kSfxXof << 8);  // 33-byte message, then suffix 1111 + first pad bit
    a[RATE - 1].hi ^= 0x80000000u;
    keccak_f1600(a);
    if (ETA == 2) {  // 128 bytes = lanes 0..15 (fits one block at either rate)
#pragma unroll
        for (int l = 0; l < 16; l++) {
            put(2 * l, cbd2_word(a[l].lo));
            put(2 * l + 1, cbd2_word(a[l].hi));
        }
    } else {  // 192 bytes = 48 words = 16 groups of 96 bits; the second block is squeezed as in sha3.c:298-311
        constexpr int W1 = 2 * RATE;      // words in the first block: 42 or 34
        constexpr int G1 = W1 / 3;        // whole groups in the first block: 14 or 11
        uint32_t o0, o1;
#pragma unroll
        for (int g = 0; g < G1; g++) {
            const int w = 3 * g;
            uint32_t w0 = (w & 1) ? a[w >> 1].hi : a[w >> 1].lo, w1 = ((w + 1) & 1) ? a[(w + 1) >> 1].hi : a[(w + 1) >> 1].lo,
                     w2 = ((w + 2) & 1) ? a[(w + 2) >> 1].hi : a[(w + 2) >> 1].lo;
            cbd3_words(w0, w1, w2, o0, o1);
            put(2 * g, o0);
            put(2 * g + 1, o1);
        }
        constexpr int LEFT = W1 - 3 * G1;  // words of a group that straddles the blocks: 0 (rate 168) or 1 (rate 136)
        uint32_t carry = 0;
        if (LEFT) carry = ((W1 - 1) & 1) ? a[(W1 - 1) >> 1].hi : a[(W1 - 1) >> 1].lo;
        keccak_f1600(a);
        int next = 0;  // next unread word of the second block
        if (LEFT) {
            cbd3_words(carry, a[0].lo, a[0].hi, o0, o1);
            put(2 * G1, o0);
            put(2 * G1 + 1, o1);
            next = 2;
        }
#pragma unroll
        for (int g = G1 + (LEFT ? 1 : 0); g < 16; g++) {
            const int w = next + 3 * (g - G1 - (LEFT ? 1 : 0));
            uint32_t w0 = (w & 1) ? a[w >> 1].hi : a[w >> 1].lo, w1 = ((w + 1) & 1) ? a[(w + 1) >> 1].hi : a[(w + 1) >> 1].lo,
                     w2 = ((w + 2) & 1) ? a[(w + 2) >> 1].hi : a[(w + 2) >> 1].lo;
            cbd3_words(w0, w1, w2, o0, o1);
            put(2 * g, o0);
            put(2 * g + 1, o1);
        }
    }
}

// A polynomial in layout C is one 16-byte vector per lane: natural-order global stores / loads are single
// fully coalesced 128-bit accesses (512 contiguous bytes per warp).
__device__ __forceinline__ void store_layoutC_global(const uint32_t x[8], int lane, uint16_t *dst) {
    reinterpret_cast<uint4 *>(dst)[lane] = pack_pairs(x);
}
__device__ __forceinline__ void load_layoutC_global(uint32_t x[8], int lane, const uint16_t *src) {
    unpack_pairs(__ldg(reinterpret_cast<const uint4 *>(src) + lane), x);
}

// Grid: (ceil(n / kNoiseTPB), npoly).  Thread = one (item, nonce) sponge; blockIdx.y selects the nonce,
// so a block is uniform in eta and in whether its polynomials get transformed.
//   seeds       : 32-byte PRF key of item i at seeds + i*seed_stride
//   NTT_OUT     : out16 + i*out16_stride + p*256   <- NTT(CBD(...)) as uint16, natural order  (s^, e^, y^)
//                 enc12 + i*enc12_stride + p*384   <- ByteEncode12 of the same polynomial for p < enc12_polys
//                                                     (KeyGen: dk_pke rows = ByteEncode12(s^[p]), ml_kem.c:750-756)
//   otherwise   : outc  + i*outc_stride  + p*32    <- 4-bit codes of CBD(...)                 (e1, e2)
template <int ETA, bool NTT_OUT, int RATE = kRateShake128>
__global__ void __launch_bounds__(kNoiseTPB) k_noise(int n, const uint8_t *__restrict__ seeds, size_t seed_stride, int nonce0,
                                                     uint16_t *__restrict__ out16, size_t out16_stride,
                                                     uint32_t *__restrict__ outc, size_t outc_stride,
                                                     uint8_t *__restrict__ enc12, size_t enc12_stride, int enc12_polys) {
    __shared__ uint32_t s_codes[NTT_OUT ? kNoiseTPB * 33 : 1];
    __shared__ __align__(16) uint16_t s_scratch[NTT_OUT ? (kNoiseTPB / 32) * kScratchU16 : 2];
    const int p = blockIdx.y;
    const int item = blockIdx.x * kNoiseTPB + threadIdx.x;
    Lane seed[4];
#pragma unroll
    for (int w = 0; w < 4; w++) seed[w] = item < n ? load_lane(seeds + seed_stride * item + 8 * w) : Lane{0u, 0u};
    if (NTT_OUT) {
        uint32_t *mine = s_codes + 33 * threadIdx.x;
        prf_cbd_codes<ETA, RATE>(seed, (uint32_t)(nonce0 + p), [&](int w, uint32_t v) { mine[w] = v; });
        __syncwarp();  // a warp only ever reads the 32 slots its own lanes wrote
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        uint16_t *scratch = s_scratch + warp * kScratchU16;
        LaneTwiddles tw;
        load_lane_twiddles<kFmaPipe>(tw, lane);  // this kernel's alu pipe belongs to Keccak
        const uint32_t pw = nibble_weight(lane & 7);
        for (int t = 0; t < 32; t++) {
            int it = blockIdx.x * kNoiseTPB + warp * 32 + t;
            if (it >= n) break;
            const uint32_t *codes = s_codes + 33 * (warp * 32 + t) + (lane >> 3);
            uint32_t x[8];
#pragma unroll
            for (int r = 0; r < 8; r++) x[r] = nibble_fma(codes[4 * r], pw) + (kQ - 3);  // coefficient lane + 32 r as a residue <= q + 3
            ntt_warp<kFmaPipe>(x, scratch, lane, tw);
            store_layoutC_global(x, lane, out16 + out16_stride * it + 256 * p);
            if (p < enc12_polys) {  // block-uniform: blockIdx.y selects the polynomial
                // 8 consecutive 12-bit coefficients = 12 bytes = three words per lane, 384 contiguous bytes per warp
                uint32_t *row = reinterpret_cast<uint32_t *>(enc12 + enc12_stride * it + 384 * p) + 3 * lane;
                row[0] = x[0] | (x[1] << 12) | (x[2] << 24);
                row[1] = (x[2] >> 8) | (x[3] << 4) | (x[4] << 16) | (x[5] << 28);
                row[2] = (x[5] >> 4) | (x[6] << 8) | (x[7] << 20);
            }
        }
    } else {
        if (item >= n) return;
        uint32_t buf[32];
        prf_cbd_codes<ETA, RATE>(seed, (uint32_t)(nonce0 + p), [&](int w, uint32_t v) { buf[w] = v; });
        uint4 *dst = reinterpret_cast<uint4 *>(outc + outc_stride * item + 32 * p);
#pragma unroll
        for (int v = 0; v < 8; v++) dst[v] = make_uint4(buf[4 * v], buf[4 * v + 1], buf[4 * v + 2], buf[4 * v + 3]);
    }
}

// =================================================================================================
// SampleNTT (ml_kem.c:189), one sponge per thread, output into a shared-memory slot
// =================================================================================================
// The reference squeezes 840 bytes (5 blocks) up front, consumes three-byte groups until it has 256
// coefficients, gives up after the 279th group (even when that group completed the polynomial) and then
// restarts with B[32] and B[33] incremented.  Here blocks are squeezed on demand (3 suffice 99.1 % of the
// time); the accepted coefficients, the give-up rule and the restart are identical.  `group_limit` is 278
// (= groups that may be consumed by a successful run); tests lower it to exercise the restart path.
//
// Returns with 256 canonical coefficients in slot[0..255]; b32/b33 are updated like the caller's buffer.
//
// Parsing cost matters (112 candidates per block against 4320 instructions per permutation), so the
// inner loop is arranged for the alu pipe: the 12-bit field is moved to the top of a register (a multiply
// by a power of two on the fma pipe, or one funnel shift when it straddles two words), compared there
// against q << 20 without masking, and stored through a running shared-memory address.  Bounds are only
// checked in blocks that can complete the polynomial (CHECKED); the give-up rule is applied by
// overwriting the groups beyond the limit with 0xFFF fields, which are always rejected.
template <bool CHECKED>
__device__ __forceinline__ void parse_block(const Lane a[25], uint32_t &addr, uint32_t end_addr) {
#pragma unroll
    for (int ch = 0; ch < 7; ch++) {  // 3 lanes = 6 words = 16 candidates
        const uint32_t w[7] = {a[3 * ch].lo, a[3 * ch].hi, a[3 * ch + 1].lo, a[3 * ch + 1].hi, a[3 * ch + 2].lo, a[3 * ch + 2].hi, 0u};
#pragma unroll
        for (int m = 0; m < 16; m++) {  // candidate m = bits [12 m, 12 m + 12): d1 / d2 of group m / 2 (ml_kem.c:208-209)
            const int bit = 12 * m, wi = bit >> 5, sh = bit & 31;
            uint32_t t;  // the field in bits [20, 32), don't-care bits below
            if (sh == 20) t = w[wi];
            else if (sh < 20) t = w[wi] * (1u << (20 - sh));
            else t = __funnelshift_r(w[wi], w[wi + 1], sh - 20);
            bool ok = t < (kQ << 20);                         // d < q  (:211, :216)
            if (CHECKED) ok = ok && (addr < end_addr);         // j < N  (:203, :216)
            uint32_t d;
            asm("mul.hi.u32 %0, %1, 4096;" : "=r"(d) : "r"(t));  // t >> 20 on the fma pipe
            if (ok) {
                asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)d) : "memory");
                addr += 2;
            }
        }
    }
}

// Replace every three-byte group of the block at index >= usable by 0xFFFFFF (both candidates rejected).
__device__ __forceinline__ void mask_groups(Lane a[25], int usable) {
    const int cut = 24 * max(usable, 0);
#pragma unroll
    for (int k = 0; k < 42; k++) {
        const int lo = 32 * k;
        uint32_t m = cut <= lo ? 0xFFFFFFFFu : (cut >= lo + 32 ? 0u : (0xFFFFFFFFu << (cut - lo)));
        if (k & 1) a[k >> 1].hi |= m;
        else a[k >> 1].lo |= m;
    }
}

__device__ __forceinline__ void sample_ntt_thread(const Lane rho[4], uint32_t &b32, uint32_t &b33, uint16_t *slot, bool active,
                                                  int group_limit) {
    Lane a[25];
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(slot), end_addr = base + 2 * kN;
    uint32_t addr = active ? base : end_addr;  // inactive lanes (beyond the batch) just follow along
    int groups_left = 0;
    bool need_init = true;
    // Loop until every lane of the warp holds a full polynomial.
    while (__any_sync(kFullMask, addr < end_addr)) {
        if (need_init) {  // XOF.Init + Absorb(rho || b32 || b33), ml_kem.c:200-201
            keccak_zero(a);
#pragma unroll
            for (int w = 0; w < 4; w++) a[w] = rho[w];
            a[4].lo = (b32 & 0xFFu) | ((b33 & 0xFFu) << 8) | (kSfxXof << 16);
            a[kRateShake128 - 1].hi ^= 0x80000000u;
            groups_left = group_limit;
            need_init = false;
        }
        keccak_f1600(a);  // one 168-byte block = 56 three-byte groups
        const bool running = addr < end_addr;
        // give-up rule (:221-227): only `groups_left` more groups may be consumed.  Rare (block 5 with the
        // reference's limit), so it is handled by masking; safe in place because such a lane either completes
        // within this block or restarts from a fresh state.
        if (__any_sync(kFullMask, running && groups_left < 56)) {
            if (running && groups_left < 56) mask_groups(a, groups_left);
        }
        if (__all_sync(kFullMask, addr + 2 * 112 <= end_addr)) parse_block<false>(a, addr, end_addr);
        else parse_block<true>(a, addr, end_addr);
        groups_left -= 56;
        // (:237-242) out of groups without a full polynomial -> bump the seed in the caller's buffer, restart
        if (groups_left <= 0 && addr < end_addr) {
            b32 = (b32 + 1) & 0xFFu;
            b33 = (b33 + 1) & 0xFFu;
            addr = base;
            need_init = true;
        }
    }
}

// =================================================================================================
// SampleNTT, fast path: exactly three squeezed blocks per sponge
// =================================================================================================
// 99.1 % of all sponges are complete after three blocks (336 candidates, 256 needed, acceptance 0.813).  A warp
// that waits for its slowest lane pays a fourth permutation in one case out of four, and its block mates wait at
// the barrier meanwhile.  The fused kernel therefore runs EXACTLY three blocks per sponge, marks the rows that own
// an incomplete sponge and leaves them to a dense clean-up pass (k_sample_matvec_list) that re-runs them through
// the general sampler.  Straight-line code, no votes in the first two blocks, every warp does identical work.
//
// Candidate loop: the 12-bit field is brought to the top of a register (multiply by a constant-bank power of two --
// ptxas would turn a literal one into a shift -- or a funnel shift when the field straddles two words), compared there
// against q << 20 without masking, shifted down and stored UNCONDITIONALLY at the running position, which advances
// under the predicate; a rejected value is overwritten by the next candidate.  Blocks 1 and 2 cannot overflow the slot
// (2 * 112 < 256); block 3 also tests the position, the slot's spare 129th word absorbing the stores of lanes that are
// already complete.  (Running the chunks of block 3 unchecked while every lane still has room for 16 coefficients saves
// instructions but doubles the code of that block: 9.27 vs 9.19 ms -- this kernel feels its instruction footprint,
// unrolling Keccak four-fold costs 7 %.  One checked parser for all three blocks is smaller still but slower, 9.37 ms.)
// (Measured alternatives, 2^20 Encaps, fused kernel: rejection bit and position by multiply-high / multiply-add, value
// by multiply-high, i.e. nothing on the alu pipe: 9.50 ms; value by shift: 9.40 ms; this form: 9.31 ms.  IMAD.HI is
// the costliest neighbour a LOP3 stream can have: profiles/coissue_r01.jsonl.)
#ifdef MLKEM_B200_EXPERIMENT
#define MLKEM_CHECK_SLOT_STORE(st, lim) \
    if ((st) + 512 < end_addr || (st) > (lim)) __trap();  // own bounds check: compute-sanitizer is not available on the pool
#else
#define MLKEM_CHECK_SLOT_STORE(st, lim)
#endif
template <bool CHECKED>
__device__ __forceinline__ void parse_chunk3(const uint32_t w[7], uint32_t &addr, uint32_t end_addr) {
#ifndef MLKEM_B200_PARSE_ALU_ADDR
    const uint32_t one = c_pow2[0], two = c_pow2[1];  // values the compiler cannot see through
#endif
#pragma unroll
    for (int m = 0; m < 16; m++) {  // candidate m = bits [12 m, 12 m + 12): d1 / d2 of group m / 2 (ml_kem.c:208-209)
        const int bit = 12 * m, wi = bit >> 5, sh = bit & 31;
        uint32_t t;  // the field in bits [20, 32), don't-care bits below
        if (sh == 20) t = w[wi];
        else if (sh < 20) t = shl_fma(w[wi], 20 - sh);
        else t = __funnelshift_r(w[wi], w[wi + 1], sh - 20);
        const bool ok = t < (kQ << 20);  // d < q  (:211, :216)
        MLKEM_CHECK_SLOT_STORE(addr, CHECKED ? end_addr : end_addr - 2)
        // (t >> 20 as the high word of an IMAD.WIDE by 4096 -- the fma pipe again -- needs an aligned register pair and a move per
        // candidate: 9.38 vs 8.97 ms, rejected.)
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)(t >> 20)) : "memory");
#ifndef MLKEM_B200_PARSE_ALU_ADDR
        // The position advances by a PREDICATED multiply-add (1 * 2 + addr, both factors opaque to the compiler: IMAD, fma pipe, one
        // issue cycle) instead of a predicated add (VIADD, alu pipe, two); in the checked block the two conditions meet in one
        // predicate (setp.and), where the compiler's own code spent a SEL on them.  Inline PTX because nvcc turns the C form into
        // SEL + IMAD.IADD.  1 704 -> 1 594 instructions in the sampling loop, fused kernel 9.015 -> 8.964 ms per 2^20 Encaps
        // (-DMLKEM_B200_PARSE_ALU_ADDR restores the old form).
        if (CHECKED)
            asm volatile("{.reg .pred p; setp.lt.u32 p, %1, %2; setp.lt.and.u32 p, %0, %3, p; @p mad.lo.u32 %0, %4, %5, %0;}"
                         : "+r"(addr) : "r"(t), "r"(kQ << 20), "r"(end_addr), "r"(one), "r"(two));
        else
            asm volatile("{.reg .pred p; setp.lt.u32 p, %1, %2; @p mad.lo.u32 %0, %3, %4, %0;}" : "+r"(addr) : "r"(t), "r"(kQ << 20), "r"(one), "r"(two));
        (void)ok;
#else
        if (CHECKED) {
            if (ok && addr < end_addr) addr += 2;  // j < N  (:203, :216)
        } else {
            if (ok) addr += 2;
        }
#endif
    }
}
template <bool CHECKED>  // false: blocks 1 and 2 (cannot fill the slot), true: block 3
__device__ __forceinline__ void parse_block3(const Lane a[25], uint32_t &addr, uint32_t end_addr) {
#pragma unroll
    for (int ch = 0; ch < 7; ch++) {  // 3 lanes = 6 words = 16 candidates
        const uint32_t w[7] = {a[3 * ch].lo, a[3 * ch].hi, a[3 * ch + 1].lo, a[3 * ch + 1].hi, a[3 * ch + 2].lo, a[3 * ch + 2].hi, 0u};
        parse_chunk3<CHECKED>(w, addr, end_addr);
    }
}
// Returns true when the slot holds the complete polynomial.  No group limit applies: three blocks are 168 of the 278
// groups a run may consume (ml_kem.c:221-227), so the fast path is only used with group_limit >= 168.
__device__ __forceinline__ bool sample_ntt_three_blocks(const Lane rho[4], uint32_t b32, uint32_t b33, uint16_t *slot, int experiment = 0) {
    Lane a[25];
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(slot), end_addr = base + 2 * kN;
    uint32_t addr = base;
    keccak_zero(a);
#pragma unroll
    for (int w = 0; w < 4; w++) a[w] = rho[w];
    a[4].lo = (b32 & 0xFFu) | ((b33 & 0xFFu) << 8) | (kSfxXof << 16);  // XOF.Init + Absorb(rho || b32 || b33), ml_kem.c:200-201
    a[kRateShake128 - 1].hi ^= 0x80000000u;
#pragma unroll 1
    for (int blk = 0; blk < 3; blk++) {
        keccak_f1600(a);  // one 168-byte block = 56 three-byte groups = 112 candidates
#ifdef MLKEM_B200_EXPERIMENT
        if (experiment & 2) {
            addr += a[0].lo & 2;
            continue;
        }
#endif
        if (blk < 2) parse_block3<false>(a, addr, end_addr);
        else parse_block3<true>(a, addr, end_addr);
    }
    return addr >= end_addr;
}

// =================================================================================================
// Fused matrix expansion + matrix-vector product (the heavy kernel of KeyGen and Encrypt)
// =================================================================================================
enum MatvecMode { kModeKeyGen = 0, kModeEncrypt = 1, kModeEncryptCompare = 2 };

struct MatvecArgs {
    int n;
    int group_limit;
    const uint8_t *rho;      // 32-byte matrix seed of item i at rho + key_row(keys, i)*rho_stride
    size_t rho_stride;
    KeySel keys;
    const uint16_t *vec;     // s^ (KeyGen) or y^ (Encrypt): item i, polynomial j at vec + i*vec_stride + 256 j
    size_t vec_stride;
    const uint16_t *add16;   // KeyGen: e^ as uint16, same addressing as vec (polynomial index = row)
    size_t add16_stride;
    const uint32_t *addc;    // Encrypt: e1 as 4-bit codes, row r of item i at addc + i*addc_stride + 32 r
    size_t addc_stride;
    uint8_t *out;            // KeyGen: ek (row r at +384 r); Encrypt: c (row r at +32 du r)
    size_t out_stride;
    uint8_t *out2;           // KeyGen: second copy of the row inside dk (dk + 384k), or nullptr
    size_t out2_stride;
    const uint8_t *cmp;      // EncryptCompare: the received ciphertext, addressed like out
    uint32_t *flags;         // EncryptCompare: flags[i] |= 1 when a re-encrypted row differs
    int *defer_list;         // rows (item * K + row) left to the clean-up pass; nullptr for the list kernel = all rows
    int *defer_count;        // number of entries in defer_list (zeroed by the host before the fused kernel)
#ifdef MLKEM_B200_EXPERIMENT
    int experiment;          // build/libmlkem_b200_exp.so only (make exp): 1 = skip phase 2, 2 = skip parsing, 4 = phase 2 twice, 8 = skip phase 1
#endif
};

// Dynamic shared memory of the matvec kernels: 32 K sampling slots, then per warp a 512-byte transform scratch and a
// 384-byte staging row for the packed output, then the row index of each of the 32 groups (-1 = nothing to do) and
// one "incomplete" byte per sponge.
constexpr int kMatvecWarpBytes = 512 + 384;
template <class P>
__host__ __device__ constexpr size_t matvec_slots_bytes() {
    return ((size_t)32 * P::K * kSlotWords * 4 + 15) & ~(size_t)15;
}
template <class P>
constexpr size_t matvec_smem_bytes() {
    return matvec_slots_bytes<P>() + (size_t)P::K * kMatvecWarpBytes + 32 * 4 + 32 * P::K;
}

// Phase 2 of the matvec kernels: the warps of the block take the 32 groups round-robin and finish the rows whose
// K sampled entries sit in the slots grp*K .. grp*K+K-1.  s_gg[grp] = item * K + row, or -1 to skip the group.
// (Tried twice and measured slower both times, 31.7 vs 32.4 M pairs/s early on and 9.09 vs 9.03 ms per 2^20 Encaps with
// the final phase 2: giving every warp the groups sampled by its own lanes, with named barriers for the two groups that
// straddle a warp boundary at K = 3, so that no block-wide barrier separates the phases.  The barrier wait it removes
// -- 9 % of the warp samples -- is not on the critical path.)
// Lane constants of phase 2.  Loaded BEFORE the block barrier that ends phase 1, so that the barrier wait hides their
// latency (they used to be the first long-scoreboard stall of every block).
struct MatvecLaneConsts {
    uint2 gam[4];
    LaneTwiddles tw;
    uint32_t pw;
};
template <int MODE>
__device__ __forceinline__ void matvec_load_consts(MatvecLaneConsts &c, int lane) {
#pragma unroll
    for (int r = 0; r < 4; r++) c.gam[r] = lane_gamma(lane + 32 * r);
    if (MODE != kModeKeyGen) load_lane_twiddles_inv<kFmaPipe>(c.tw, lane);
    c.pw = nibble_weight(lane & 7);
}
// The global operands of one group (row): the vector, the noise codes (Encrypt) or e^ (KeyGen), the received ciphertext
// row (compare mode).  Fetched one group ahead (see matvec_finish_rows); the first group's before the block barrier.
template <class P>
struct MatvecOperands {
    static constexpr int kCmpWords = (8 * P::DU + 31) / 32;
    uint32_t v[8 * P::K], cw[8], cmp[kCmpWords], ev[4];
};
template <class P, int MODE>
__device__ __forceinline__ void matvec_prefetch(MatvecOperands<P> &o, const MatvecArgs &g, int gg, int lane) {
    constexpr int K = P::K;
    if (gg < 0) return;
    const int item = gg / K, row = gg - item * K;
    const uint16_t *vec = g.vec + g.vec_stride * item;
    // (16-bit loads instead of 32-bit loads + mask/shift: the load/store pipe has slack, the alu pipe does not.)
#pragma unroll
    for (int j = 0; j < K; j++)
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int t = lane + 32 * r;
            o.v[8 * j + 2 * r] = __ldg(vec + 256 * j + 2 * t);
            o.v[8 * j + 2 * r + 1] = __ldg(vec + 256 * j + 2 * t + 1);
        }
    if (MODE == kModeEncryptCompare) {
        const uint32_t *cw = reinterpret_cast<const uint32_t *>(g.cmp + g.out_stride * item + (size_t)P::C1ROW * row);
#pragma unroll
        for (int i = 0; i < MatvecOperands<P>::kCmpWords; i++) o.cmp[i] = (lane + 32 * i < 8 * P::DU) ? __ldg(cw + lane + 32 * i) : 0u;
    }
    if (MODE != kModeKeyGen) {
        const uint32_t *codes = g.addc + g.addc_stride * item + 32 * row + (lane >> 3);
#pragma unroll
        for (int r = 0; r < 8; r++) o.cw[r] = __ldg(codes + 4 * r);
    } else {
        const uint32_t *ev = reinterpret_cast<const uint32_t *>(g.add16 + g.add16_stride * item + 256 * row);
#pragma unroll
        for (int r = 0; r < 4; r++) o.ev[r] = __ldg(ev + lane + 32 * r);
    }
}

// The rest of a row once its K base-case products are accumulated: (KeyGen) + e^ and ByteEncode12, or (Encrypt) inverse
// transform, + e1, Compress_du, ByteEncode_du; then store the row or compare it with the received ciphertext.
template <class P, int MODE>
__device__ __forceinline__ void matvec_row_tail(const MatvecArgs &g, int item, int row, uint32_t acc[8], const uint32_t cw8[8],
                                                const uint32_t *cmpw, const uint32_t ev4[4], uint16_t *scratch, uint8_t *stage, int lane,
                                                const LaneTwiddles &tw, uint32_t pw) {
    constexpr int kCmpWords = MatvecOperands<P>::kCmpWords;
    int nwords;
    if (MODE == kModeKeyGen) {
        // t^[row] = A[row] . s^ + e^[row]   (ml_kem.c:723-727), then ByteEncode12 (:736-742)
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int t = lane + 32 * r;
            uint32_t e = ev4[r];
            uint32_t c0 = csubq(canon32(acc[2 * r]) + (e & 0xFFFFu)), c1 = csubq(canon32(acc[2 * r + 1]) + (e >> 16));
            uint32_t v = c0 | (c1 << 12);
            stage[3 * t] = (uint8_t)v;
            stage[3 * t + 1] = (uint8_t)(v >> 8);
            stage[3 * t + 2] = (uint8_t)(v >> 16);
        }
        nwords = 96;
    } else {
        // u[row] = InverseNTT(At[row] . y^) + e1[row]  (ml_kem.c:854-864); Compress_du + ByteEncode_du (:886-896)
        uint32_t *sw = reinterpret_cast<uint32_t *>(scratch);
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int t = lane + 32 * r;
            sw[sidx(2 * t) >> 1] = barrett32(acc[2 * r]) + barrett32(acc[2 * r + 1]) * 65536u;  // < 2q each
        }
        __syncwarp();
        uint32_t x[8];
        load_scratch_C(x, scratch, lane);
        __syncwarp();
        intt_warp<kFmaPipe, false>(x, scratch, lane, tw);  // [0, 2q)
#pragma unroll
        for (int r = 0; r < 8; r++) {  // (x + e1) mod q, exact, then Compress_du: everything but the final mask on the fma pipe
            uint32_t y = x[r] + nibble_fma(cw8[r], pw) + (kQ - 3);  // < 3q + 4
            x[r] = compress_canon<P::DU>(canon_fma(y));
        }
        store_scratch_A(x, scratch, lane);
        __syncwarp();
        load_scratch_C(x, scratch, lane);
        pack8<P::DU>(x, stage + P::DU * lane);
        nwords = 8 * P::DU;
    }
    __syncwarp();
    const uint32_t *stw = reinterpret_cast<const uint32_t *>(stage);
    const size_t row_off = (MODE == kModeKeyGen ? 384 : P::C1ROW) * (size_t)row;
    if (MODE == kModeEncryptCompare) {
        uint32_t d = 0;
#pragma unroll
        for (int i = 0; i < kCmpWords; i++)
            if (lane + 32 * i < nwords) d |= stw[lane + 32 * i] ^ cmpw[i];
        d = __any_sync(kFullMask, d != 0) ? 1u : 0u;
        if (lane == 0) atomicOr(g.flags + item, d);  // unconditional: no data-dependent control flow
    } else {
        uint32_t *ow = reinterpret_cast<uint32_t *>(g.out + g.out_stride * item + row_off);
        for (int w = lane; w < nwords; w += 32) ow[w] = stw[w];
        if (MODE == kModeKeyGen && g.out2) {
            uint32_t *ow2 = reinterpret_cast<uint32_t *>(g.out2 + g.out2_stride * item + row_off);
            for (int w = lane; w < nwords; w += 32) ow2[w] = stw[w];
        }
    }
    __syncwarp();
}

template <class P, int MODE>
__device__ __forceinline__ void matvec_finish_rows(const MatvecArgs &g, uint32_t *s_slots, const int *s_gg, int lane, int warp,
                                                   const MatvecLaneConsts &lc, MatvecOperands<P> &nx) {
    constexpr int K = P::K;
    uint8_t *warp_area = reinterpret_cast<uint8_t *>(s_slots) + matvec_slots_bytes<P>() + warp * kMatvecWarpBytes;
    uint16_t *scratch = reinterpret_cast<uint16_t *>(warp_area);
    uint8_t *stage = warp_area + 512;
    const uint2 *gam = lc.gam;
    const LaneTwiddles &tw = lc.tw;
    const uint32_t pw = lc.pw;

    // Every global operand of a group is fetched one group ahead into a second register set (nx; the caller has already
    // issued the loads of this warp's first group) and copied over at the top of the iteration: one wait per iteration,
    // for loads that were issued a whole iteration earlier.  (Loading the codes and the ciphertext row at the top of the
    // iteration that uses them left 32 % of the phase-2 warp time in long-scoreboard stalls: consumers of early loads
    // also wait for later loads that share their scoreboard.)
    constexpr int kCmpWords = MatvecOperands<P>::kCmpWords;
    // (Measured and rejected, round 2: two operand sets that swap roles every row -- the loop unrolled by two -- instead of
    // one set copied over per row: 15 instructions less per row, 147 registers, twice the code: 9.63 vs 9.02 ms per 2^20 Encaps.)
#pragma unroll 1
    for (int grp = warp; grp < 32; grp += K) {
        const int gg = s_gg[grp];
        uint32_t v[8 * K], cw8[8], cmpw[kCmpWords], ev4[4];
#pragma unroll
        for (int i = 0; i < 8 * K; i++) v[i] = nx.v[i];
#pragma unroll
        for (int i = 0; i < 8; i++) cw8[i] = nx.cw[i];
#pragma unroll
        for (int i = 0; i < kCmpWords; i++) cmpw[i] = nx.cmp[i];
#pragma unroll
        for (int i = 0; i < 4; i++) ev4[i] = nx.ev[i];
        matvec_prefetch<P, MODE>(nx, g, grp + K < 32 ? s_gg[grp + K] : -1, lane);
        if (gg < 0) continue;  // beyond the batch, or left to the clean-up pass
        const int item = gg / K, row = gg - item * K;
        const uint32_t slot0 = (uint32_t)__cvta_generic_to_shared(s_slots + kSlotWords * (grp * K));
        // ---- row . vector in the NTT domain (ml_kem.c:618 VectorMultiply), lazily accumulated.
        // Lane handles coefficient pairs t = lane + 32 r (conflict-free slot reads, coalesced vector reads).
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
#pragma unroll
        for (int j = 0; j < K; j++) {
#pragma unroll
            for (int r = 0; r < 4; r++) {
                // two 16-bit shared loads (inline PTX: the compiler would merge them into one 32-bit load plus a mask
                // and a shift on the alu pipe)
                uint16_t a0, a1;
                const uint32_t ad = slot0 + 4 * (kSlotWords * j + lane + 32 * r);
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(a0) : "r"(ad));
                asm volatile("ld.shared.u16 %0, [%1+2];" : "=h"(a1) : "r"(ad));
                basemul_acc(acc[2 * r], acc[2 * r + 1], a0, a1, v[8 * j + 2 * r], v[8 * j + 2 * r + 1], gam[r]);
            }
        }
        matvec_row_tail<P, MODE>(g, item, row, acc, cw8, cmpw, ev4, scratch, stage, lane, tw, pw);
    }
}

template <class P>
__device__ __forceinline__ int *matvec_gg(uint32_t *s_slots) {
    return reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(s_slots) + matvec_slots_bytes<P>() + P::K * kMatvecWarpBytes);
}

// The fused kernel.  Block = 32 K threads = 32 (item,row) groups x K matrix columns.  Phase 1: each thread samples one
// matrix entry into its slot with the three-block sampler.  Phase 2: the warps finish the complete rows; rows with an
// incomplete entry (2.7 % at K = 3) are appended to g.defer_list for k_sample_matvec_list.
template <class P, int MODE>
__global__ void __launch_bounds__(32 * P::K) k_sample_matvec(MatvecArgs g) {
    constexpr int K = P::K;
    extern __shared__ __align__(16) uint32_t s_slots[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *s_gg = matvec_gg<P>(s_slots);
    uint8_t *s_inc = reinterpret_cast<uint8_t *>(s_gg + 32);
    {
        const int grp = tid / K, col = tid - grp * K;
        const int gg = blockIdx.x * 32 + grp;
        const int item = gg / K, row = gg - item * K;
        const bool active = item < g.n;
        Lane rho[4];
#pragma unroll
        for (int w = 0; w < 4; w++) rho[w] = active ? load_lane(g.rho + g.rho_stride * key_row(g.keys, item) + 8 * w) : Lane{0u, 0u};
        // KeyGen: A[row][col] = SampleNTT(rho || col || row)      (ml_kem.c:686-693)
        // Encrypt: At[row][col] = SampleNTT(rho || row || col)    (ml_kem.c:817-823, stored transposed)
        const uint32_t b32 = MODE == kModeKeyGen ? col : row, b33 = MODE == kModeKeyGen ? row : col;
        // threads beyond the batch sample a dummy sponge into their own slot (the straight-line sampler has no idle mode)
#ifdef MLKEM_B200_EXPERIMENT
        // bit 8: phase 2 alone, on whatever the slots hold (what does the polynomial arithmetic cost when no Keccak runs next to it?)
        const bool complete = (g.experiment & 8) ? true
                                                 : sample_ntt_three_blocks(rho, b32, b33, reinterpret_cast<uint16_t *>(s_slots + kSlotWords * tid), g.experiment);
#else
        const bool complete = sample_ntt_three_blocks(rho, b32, b33, reinterpret_cast<uint16_t *>(s_slots + kSlotWords * tid));
#endif
        s_inc[tid] = active && !complete;
    }
    MatvecLaneConsts lc;
    matvec_load_consts<MODE>(lc, lane);
    // the operands of this warp's first group: their addresses do not depend on what the other warps sampled, so the loads
    // go out before the barrier (if the row turns out to be deferred they were for nothing)
    MatvecOperands<P> nx;
    {
        const int gg = blockIdx.x * 32 + warp;
        matvec_prefetch<P, MODE>(nx, g, gg / K < g.n ? gg : -1, lane);
    }
    __syncthreads();
    {  // every warp resolves the groups it is going to finish itself (warp, warp + K, ...): no second block barrier
        const int grp = warp + K * lane;
        if (grp < 32) {
            const int gg = blockIdx.x * 32 + grp;
            bool deferred = false;
#pragma unroll
            for (int j = 0; j < K; j++) deferred |= s_inc[grp * K + j] != 0;
            const bool active = gg / K < g.n;
            s_gg[grp] = (active && !deferred) ? gg : -1;
            if (active && deferred) g.defer_list[atomicAdd(g.defer_count, 1)] = gg;
        }
        __syncwarp();
    }
#ifdef MLKEM_B200_EXPERIMENT
    if (g.experiment & 1) return;
    if (g.experiment & 4) {
        matvec_finish_rows<P, MODE>(g, s_slots, s_gg, lane, warp, lc, nx);
        matvec_prefetch<P, MODE>(nx, g, s_gg[warp], lane);
    }
#endif
    matvec_finish_rows<P, MODE>(g, s_slots, s_gg, lane, warp, lc, nx);
}

// The general kernel: rows taken from g.defer_list (or all rows of the batch when it is nullptr), sampled with the
// general sampler (any number of blocks, give-up rule and restart of ml_kem.c:221-242).  Persistent blocks.
template <class P, int MODE>
__global__ void __launch_bounds__(32 * P::K) k_sample_matvec_list(MatvecArgs g) {
    constexpr int K = P::K;
    extern __shared__ __align__(16) uint32_t s_slots[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *s_gg = matvec_gg<P>(s_slots);
    MatvecLaneConsts lc;
    matvec_load_consts<MODE>(lc, lane);
    const int count = g.defer_list ? *g.defer_count : g.n * K;
    for (int base = blockIdx.x * 32; base < count; base += gridDim.x * 32) {
        {
            const int grp = tid / K, col = tid - grp * K;
            const int e = base + grp;
            const int gg = e < count ? (g.defer_list ? g.defer_list[e] : e) : -1;
            const bool active = gg >= 0;
            const int item = active ? gg / K : 0, row = gg - item * K;
            if (col == 0) s_gg[grp] = gg;
            Lane rho[4];
#pragma unroll
            for (int w = 0; w < 4; w++) rho[w] = active ? load_lane(g.rho + g.rho_stride * key_row(g.keys, item) + 8 * w) : Lane{0u, 0u};
            uint32_t b32 = MODE == kModeKeyGen ? col : row, b33 = MODE == kModeKeyGen ? row : col;
            sample_ntt_thread(rho, b32, b33, reinterpret_cast<uint16_t *>(s_slots + kSlotWords * tid), active, g.group_limit);
        }
        __syncthreads();
        MatvecOperands<P> nx;
        matvec_prefetch<P, MODE>(nx, g, s_gg[warp], lane);
        matvec_finish_rows<P, MODE>(g, s_slots, s_gg, lane, warp, lc, nx);
        __syncthreads();  // the slots are reused by the next batch of rows
    }
}

// =================================================================================================
// Expanded key tables: the matrix of a resident key is sampled once, not once per ciphertext
// =================================================================================================
// A^ depends only on rho, i.e. on the key.  A resident key table (mlkem_b200_keys_*, MLKEM_B200_FLAG_EXPAND_KEYS) keeps
// At[row][col] = SampleNTT(rho || row || col) (ml_kem.c:817-823, the order K-PKE.Encrypt consumes it in) as uint16
// polynomials, K*K*512 bytes per key, so that keyed Encaps / Decaps run 8 / 15 Keccak permutations per item instead of
// 44 / 42 at ML-KEM-768: what is left of the matrix-vector product is HBM-fed polynomial arithmetic.

// Seeds of the matrix entries of n keys: seeds[(key*K + row)*K + col] = rho_key || row || col (34 bytes each).
template <class P>
__global__ void __launch_bounds__(256) k_matrix_seeds(int n, const uint8_t *__restrict__ ek, size_t ek_stride, uint8_t *__restrict__ seeds) {
    constexpr int K = P::K;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * K * K) return;
    const int key = e / (K * K), rc = e - key * K * K, row = rc / K, col = rc - row * K;
    const uint8_t *rho = ek + ek_stride * key + 384 * K;
    uint8_t *out = seeds + 34 * (size_t)e;
    for (int b = 0; b < 32; b++) out[b] = rho[b];
    out[32] = (uint8_t)row;
    out[33] = (uint8_t)col;
}

// Key rotation (mlkem_b200_keys_replace*): row i of src (src + i*src_stride) is copied to row key_row(slots, i) of dst,
// 16 bytes per thread.  The new dk / ek rows, their H(ek) and their matrices are computed in scratch beforehand, so this is
// the only kernel that writes into a live table, and it writes nothing outside the listed rows.  Strides and row sizes are
// multiples of 16 (DK, EK, 384 K, 32, K*K*512).
__global__ void __launch_bounds__(256) k_scatter_rows(int n, int row_words, const uint8_t *__restrict__ src, size_t src_stride, KeySel slots,
                                                      uint8_t *__restrict__ dst, size_t dst_stride) {
    const size_t total = (size_t)n * row_words;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int i = (int)(t / row_words), w = (int)(t - (size_t)i * row_words);
        const uint4 v = reinterpret_cast<const uint4 *>(src + src_stride * i)[w];
        reinterpret_cast<uint4 *>(dst + dst_stride * key_row(slots, i))[w] = v;
    }
}

// Randomness of the seeded calls (mlkem_b200_kem_*_seeded_batch, _kem_encaps_keyed_batch, _keys_generate, _keys_replace_generate):
// R_j = SHAKE256(seed[32] || LE64(first + j) || LE64(tag)), 48 bytes = 6 lanes, one block at rate 136, one permutation.  R_j[0:32]
// goes to out0 + 32 j (d of KeyGen, m of Encaps) and, when out1 is not null, R_j[32:64] to out1 + 32 j (z of KeyGen): the two
// arrays enqueue_keygen takes.  `first` is the index within the whole call of this launch's first item, so the result does not
// depend on the chunking.  The 32-byte call seed is read from device memory, never passed as a kernel argument.
__global__ void __launch_bounds__(kHashTPB) k_expand_seed(int n, const uint8_t *__restrict__ seed, unsigned long long first, uint32_t tag,
                                                          uint8_t *__restrict__ out0, uint8_t *__restrict__ out1) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const unsigned long long idx = first + (unsigned long long)j;
    Lane a[25];
    sponge_absorb_words<kRateSha3_256>(a, 6, kSfxXof, [&](int w) {
        if (w < 4) return load_lane(seed + 8 * w);
        return w == 4 ? Lane{(uint32_t)idx, (uint32_t)(idx >> 32)} : Lane{tag, 0u};
    });
#pragma unroll
    for (int w = 0; w < 4; w++) store_lane(out0 + 32 * (size_t)j + 8 * w, a[w]);
    if (out1) {
#pragma unroll
        for (int w = 0; w < 4; w++) store_lane(out1 + 32 * (size_t)j + 8 * w, a[4 + w]);
    }
}

// u rows of K-PKE.Encrypt from the table (ml_kem.c:854-896): persistent warps, warp = one (item, row); the K matrix
// polynomials of the row come from HBM / L2 with coalesced 32-bit loads (a coefficient pair per lane and load), the
// vector, noise codes and ciphertext row are fetched one row ahead like in the fused kernel.
#ifndef MLKEM_B200_MATTABLE_PREFETCH
#define MLKEM_B200_MATTABLE_PREFETCH 1  // 1: operands of the next row in a second register set (118 registers, 16 warps per SM)
#endif                                  // 0: loaded at the top of the row, latency left to occupancy (MLKEM_B200_MATTABLE_BLOCKS per SM)
#ifndef MLKEM_B200_MATTABLE_BLOCKS
#define MLKEM_B200_MATTABLE_BLOCKS 1
#endif
template <class P, int MODE>
__global__ void __launch_bounds__(kMatTableTPB, MLKEM_B200_MATTABLE_BLOCKS) k_matvec_table(MatvecArgs g, const uint16_t *__restrict__ table) {
    static_assert(MODE != kModeKeyGen, "the table is kept in Encrypt order");
    constexpr int K = P::K, NW = kMatTableTPB / 32;
    __shared__ __align__(16) uint8_t s_warp[NW * kMatvecWarpBytes];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = reinterpret_cast<uint16_t *>(s_warp + warp * kMatvecWarpBytes);
    uint8_t *stage = s_warp + warp * kMatvecWarpBytes + 512;
    MatvecLaneConsts lc;
    matvec_load_consts<MODE>(lc, lane);
    const int rows = g.n * K, stride = gridDim.x * NW;
    int gg = blockIdx.x * NW + warp;
    MatvecOperands<P> nx;
    if (MLKEM_B200_MATTABLE_PREFETCH) matvec_prefetch<P, MODE>(nx, g, gg < rows ? gg : -1, lane);
    constexpr int kCmpWords = MatvecOperands<P>::kCmpWords;
#pragma unroll 1
    for (; gg < rows; gg += stride) {
        if (!MLKEM_B200_MATTABLE_PREFETCH) matvec_prefetch<P, MODE>(nx, g, gg, lane);
        const int item = gg / K, row = gg - item * K;
        const uint32_t *arow = reinterpret_cast<const uint32_t *>(table + ((size_t)key_row(g.keys, item) * K + row) * K * 256);
        uint32_t aw[4 * K];
#pragma unroll
        for (int j = 0; j < K; j++)
#pragma unroll
            for (int r = 0; r < 4; r++) aw[4 * j + r] = __ldg(arow + 128 * j + lane + 32 * r);
        uint32_t v[8 * K], cw8[8], cmpw[kCmpWords], ev4[4];
#pragma unroll
        for (int i = 0; i < 8 * K; i++) v[i] = nx.v[i];
#pragma unroll
        for (int i = 0; i < 8; i++) cw8[i] = nx.cw[i];
#pragma unroll
        for (int i = 0; i < kCmpWords; i++) cmpw[i] = nx.cmp[i];
#pragma unroll
        for (int i = 0; i < 4; i++) ev4[i] = 0;
        if (MLKEM_B200_MATTABLE_PREFETCH) matvec_prefetch<P, MODE>(nx, g, gg + stride < rows ? gg + stride : -1, lane);
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
#pragma unroll
        for (int j = 0; j < K; j++)
#pragma unroll
            for (int r = 0; r < 4; r++)
                basemul_acc(acc[2 * r], acc[2 * r + 1], aw[4 * j + r] & 0xFFFFu, aw[4 * j + r] >> 16, v[8 * j + 2 * r], v[8 * j + 2 * r + 1], lc.gam[r]);
        matvec_row_tail<P, MODE>(g, item, row, acc, cw8, cmpw, ev4, scratch, stage, lane, lc.tw, lc.pw);
    }
}

// =================================================================================================
// Remaining K-PKE pieces, one item per warp
// =================================================================================================
constexpr int kWarpTPB = 128;  // 4 items per block
// Transform variant of k_decrypt and of the stand-alone NTT / InverseNTT kernels.  No Keccak runs next to them, so the
// balanced form (quotient by multiply + shift) wins: measured 3.28 vs 2.97 G NTT/s and 1.81 vs 1.95 ms per 2^20
// decryptions against the multiply-high form (IMAD.HI issues at half the IMAD rate; tools/time_prims.py).
#ifndef MLKEM_B200_PRIM_PIPE
#define MLKEM_B200_PRIM_PIPE false
#endif
constexpr bool kPrimPipe = MLKEM_B200_PRIM_PIPE;

struct EncVArgs {
    int n;
    const uint8_t *ek;      // item i at ek + key_row(keys, i)*ek_stride: ByteEncode12(t^) (384 K bytes) || rho
    size_t ek_stride;
    KeySel keys;
    const uint16_t *yhat;   // y^ polynomials, item stride in uint16
    size_t yhat_stride;
    const uint32_t *addc;   // noise codes, e2 is row K
    size_t addc_stride;
    const uint8_t *m;       // 32-byte message of item i at m + 32 i
    uint8_t *c;             // ciphertext base (c2 is written at + 32 du K)
    size_t c_stride;
    const uint8_t *cmp;
    uint32_t *flags;
};

// Bulk asynchronous global -> shared copies (cp.async.bulk, the 1-D form of the TMA engine, completion signalled on an
// mbarrier): the persistent warps of k_encrypt_v / k_decrypt fetch the inputs of their NEXT item while they work on the
// current one (two buffers and two mbarriers per warp).  ONE lane issues one instruction per contiguous row -- 1 to 2 KB
// each -- where round 1 had every lane issue 16-byte cp.async copies (140 per item in k_decrypt), and the copy engine,
// not the LSU pipe, moves the data.  Sources and destinations are 16-byte aligned and sizes are multiples of 16 (every
// per-item size on this path is).
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// v = InverseNTT(t^ . y^) + e2 + Decompress_1(m)  (ml_kem.c:867-880); c2 = ByteEncode_dv(Compress_dv(v)) (:899-904).
// One item per warp; every lane owns 8 consecutive coefficients (= 12 bytes of each ByteEncode12 row).
// COMPARE: OR the mismatch against the received ciphertext into flags instead of storing.
// (Blocks per SM: 8 would cap the kernel at 64 registers, which it no longer fits without spilling 8 of them; 7 = 72 registers.)
#ifndef MLKEM_B200_ENCV_BLOCKS
#define MLKEM_B200_ENCV_BLOCKS 7
#endif
template <class P, bool COMPARE>
__global__ void __launch_bounds__(kWarpTPB, MLKEM_B200_ENCV_BLOCKS) k_encrypt_v(EncVArgs g) {
    constexpr int K = P::K, NW = kWarpTPB / 32;
    constexpr int kRowsBytes = 384 * K, kVecBytes = 512 * K, kBufBytes = kRowsBytes + kVecBytes + 16;  // t^ rows | y^ | slack
    __shared__ __align__(16) uint16_t s_scratch[NW * kScratchU16];
    __shared__ __align__(16) uint8_t s_in[NW * 2 * kBufBytes];
    __shared__ __align__(16) uint8_t s_stage[NW * 32 * P::DV];
    __shared__ __align__(8) uint64_t s_bar[NW * 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = s_scratch + warp * kScratchU16;
    uint8_t *inbuf = s_in + warp * 2 * kBufBytes;
    uint8_t *stage = s_stage + warp * 32 * P::DV;
    uint64_t *bar = s_bar + 2 * warp;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        mbar_fence_init();
    }
    __syncwarp();
    uint2 gam[4];
#pragma unroll
    for (int i = 0; i < 4; i++) gam[i] = lane_gamma(4 * lane + i);
    LaneTwiddles tw;
    load_lane_twiddles_inv<kFmaPipe>(tw, lane);
    const uint32_t pw = nibble_weight(lane & 7);
    auto fetch = [&](int item, int b) {  // lane 0 only: the t^ rows of the key and the y^ polynomials of the item
        uint8_t *buf = inbuf + b * kBufBytes;
        mbar_expect_tx(bar + b, kRowsBytes + kVecBytes);
        bulk_g2s(buf, g.ek + g.ek_stride * key_row(g.keys, item), kRowsBytes, bar + b);
        bulk_g2s(buf + kRowsBytes, g.yhat + g.yhat_stride * item, kVecBytes, bar + b);
    };
    const int stride = gridDim.x * NW;
    int item = blockIdx.x * NW + warp, cur = 0;
    uint32_t phase = 0;  // bit b = parity the next wait on buffer b expects
    if (item < g.n && lane == 0) fetch(item, 0);
    for (; item < g.n; item += stride, cur ^= 1) {  // persistent warps
        // the other buffer was last read in the previous iteration, which ended with __syncwarp()
        if (item + stride < g.n && lane == 0) fetch(item + stride, cur ^ 1);
        mbar_wait(bar + cur, (phase >> cur) & 1u);  // this item's rows have landed
        phase ^= 1u << cur;
        const uint8_t *rows = inbuf + cur * kBufBytes;
        const uint16_t *yv = reinterpret_cast<const uint16_t *>(rows + kRowsBytes);
        // e2 codes and the message bits are needed after the inverse transform: issue their loads now
        const uint32_t *codes = g.addc + g.addc_stride * item + 32 * K;
        const uint32_t *mw = reinterpret_cast<const uint32_t *>(g.m + 32 * (size_t)item);
        uint32_t cw8[8], mw8[8];
#pragma unroll
        for (int r = 0; r < 8; r++) {
            cw8[r] = __ldg(codes + (lane >> 3) + 4 * r);
            mw8[r] = __ldg(mw + r);
        }
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
#pragma unroll
        for (int j = 0; j < K; j++) {
            uint32_t t[8], y[8];
            unpack8<12>(rows + 384 * j, lane, t);  // ByteDecode12 without reduction (ml_kem.c:806-808, D4)
            unpack_pairs(*reinterpret_cast<const uint4 *>(yv + 256 * j + 8 * lane), y);
#pragma unroll
            for (int i = 0; i < 4; i++) basemul_acc(acc[2 * i], acc[2 * i + 1], t[2 * i], t[2 * i + 1], y[2 * i], y[2 * i + 1], gam[i]);
        }
        uint32_t x[8];
#pragma unroll
        for (int r = 0; r < 8; r++) x[r] = barrett32(acc[r]);  // < 2q
        intt_warp<kFmaPipe, false>(x, scratch, lane, tw);  // layout C in, layout A out, [0, 2q)
#pragma unroll
        for (int r = 0; r < 8; r++) {
            uint32_t mu = ((mw8[r] >> lane) & 1u) * 1665u;  // Decompress_1(bit) = 1665 bit (ml_kem.c:867-870)
            // v = x + e2 + mu as a residue < 4q: Compress_dv is exact on residues for d <= 5 (compress_resid)
            x[r] = compress_resid<P::DV>(x[r] + nibble_fma(cw8[r], pw) + (kQ - 3) + mu);
        }
        store_scratch_A(x, scratch, lane);
        __syncwarp();
        load_scratch_C(x, scratch, lane);
        pack8<P::DV>(x, stage + P::DV * lane);
        __syncwarp();
        const uint32_t *stw = reinterpret_cast<const uint32_t *>(stage);
        const size_t off = (size_t)P::C1ROW * K;
        if (COMPARE) {
            const uint32_t *cw = reinterpret_cast<const uint32_t *>(g.cmp + g.c_stride * item + off);
            uint32_t d = 0;
            for (int w = lane; w < 8 * P::DV; w += 32) d |= stw[w] ^ __ldg(cw + w);
            d = __any_sync(kFullMask, d != 0) ? 1u : 0u;
            if (lane == 0) atomicOr(g.flags + item, d);
        } else {
            uint32_t *ow = reinterpret_cast<uint32_t *>(g.c + g.c_stride * item + off);
            for (int w = lane; w < 8 * P::DV; w += 32) ow[w] = stw[w];
        }
        __syncwarp();
    }
}

// ml_kem.c:942 PKE_Decrypt: m' = ByteEncode_1(Compress_1(v - InverseNTT(s^ . NTT(u)))).  One item per warp; the
// ciphertext and the ByteEncode12 rows of s^ are staged in shared memory with 128-bit loads.
template <class P>
__global__ void __launch_bounds__(kWarpTPB) k_decrypt(int n, const uint8_t *__restrict__ dk, size_t dk_stride, KeySel keys,
                                                      const uint8_t *__restrict__ c, uint8_t *__restrict__ mout) {
    constexpr int K = P::K, NW = kWarpTPB / 32;
    constexpr int kSkBytes = 384 * K, kBufBytes = P::C + kSkBytes + 32;  // ciphertext | s^ rows | slack
    __shared__ __align__(16) uint16_t s_scratch[NW * kScratchU16];
    __shared__ __align__(16) uint8_t s_in[NW * 2 * kBufBytes];
    __shared__ __align__(8) uint64_t s_bar[NW * 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = s_scratch + warp * kScratchU16;
    uint8_t *inbuf = s_in + warp * 2 * kBufBytes;
    uint64_t *bar = s_bar + 2 * warp;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        mbar_fence_init();
    }
    __syncwarp();
    uint2 gam[4];
#pragma unroll
    for (int i = 0; i < 4; i++) gam[i] = lane_gamma(4 * lane + i);
    LaneTwiddles tw, twi;
    load_lane_twiddles<kPrimPipe>(tw, lane);
    load_lane_twiddles_inv<kPrimPipe>(twi, lane);
    auto fetch = [&](int item, int b) {  // lane 0 only: the ciphertext of the item and the s^ rows of its key
        uint8_t *buf = inbuf + b * kBufBytes;
        mbar_expect_tx(bar + b, P::C + kSkBytes);
        bulk_g2s(buf, c + (size_t)P::C * item, P::C, bar + b);
        bulk_g2s(buf + P::C, dk + dk_stride * key_row(keys, item), kSkBytes, bar + b);
    };
    const int stride = gridDim.x * NW;
    int item = blockIdx.x * NW + warp, cur = 0;
    uint32_t phase = 0;  // bit b = parity the next wait on buffer b expects
    if (item < n && lane == 0) fetch(item, 0);
    for (; item < n; item += stride, cur ^= 1) {  // persistent warps
        if (item + stride < n && lane == 0) fetch(item + stride, cur ^ 1);
        mbar_wait(bar + cur, (phase >> cur) & 1u);
        phase ^= 1u << cur;
        const uint8_t *ct = inbuf + cur * kBufBytes, *sk = ct + P::C;
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
        for (int i = 0; i < K; i++) {
            // u^[i] = NTT(Decompress_du(ByteDecode_du(c1[i])))   (ml_kem.c:978-987)
            uint32_t x[8], sh[8];
            unpack8<P::DU>(ct + P::C1ROW * i, lane, x);
#pragma unroll
            for (int r = 0; r < 8; r++) x[r] = decompress<P::DU>(x[r]);
            store_scratch_C(x, scratch, lane);
            __syncwarp();
            load_scratch_A(x, scratch, lane);
            __syncwarp();
            ntt_warp<kPrimPipe>(x, scratch, lane, tw);  // layout C out: 8 consecutive coefficients = 4 base-case pairs
            unpack8<12>(sk + 384 * i, lane, sh);  // s^[i] = ByteDecode12(dk_pke[i]) (ml_kem.c:996-998), no reduction
#pragma unroll
            for (int p = 0; p < 4; p++) basemul_acc(acc[2 * p], acc[2 * p + 1], sh[2 * p], sh[2 * p + 1], x[2 * p], x[2 * p + 1], gam[p]);
        }
        uint32_t x[8];
#pragma unroll
        for (int r = 0; r < 8; r++) x[r] = kPrimPipe ? barrett32(acc[r]) : canon32(acc[r]);
        intt_warp<kPrimPipe>(x, scratch, lane, twi);
        // w = v - x (ml_kem.c:1001-1003), m' bit = Compress_1(w) (:1009-1012); coefficient lane+32r is bit lane of word r
        uint32_t myword = 0;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            uint32_t v = decompress<P::DV>(unpack1<P::DV>(ct + P::C1ROW * K, idxA(lane, r)));
            uint32_t w = csubq(v + kQ - x[r]);
            uint32_t word = __ballot_sync(kFullMask, compress_canon<1>(w) & 1u);
            if (lane == r) myword = word;
        }
        if (lane < 8) reinterpret_cast<uint32_t *>(mout + 32 * (size_t)item)[lane] = myword;
        __syncwarp();
    }
}

// =================================================================================================
// Stand-alone batched primitives (the C-ABI's mlkem_*_batch entry points; BASELINE config 2)
// =================================================================================================
constexpr int kPrimTPB = 256;  // 8 polynomials per block

// ml_kem.c:287 NTT over n polynomials of 256 uint16 (natural order in, natural order out).
// Loads: 8 x 16-bit per lane in layout A (each warp instruction reads 64 contiguous bytes); stores: one
// 128-bit vector per lane (layout C = natural order).
__global__ void __launch_bounds__(kPrimTPB) k_ntt_batch(int n, const uint16_t *__restrict__ in, uint16_t *__restrict__ out) {
    __shared__ __align__(16) uint16_t s_scratch[(kPrimTPB / 32) * kScratchU16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = s_scratch + warp * kScratchU16;
    LaneTwiddles tw;
    load_lane_twiddles<kPrimPipe>(tw, lane);
    const long long stride = (long long)gridDim.x * (kPrimTPB / 32);
    long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp;
    uint32_t nxt[8];  // the next polynomial of this warp is in flight while the current one is transformed
    if (p < n) {
#pragma unroll
        for (int r = 0; r < 8; r++) nxt[r] = __ldg(in + 256 * p + idxA(lane, r));
    }
    for (; p < n; p += stride) {
        uint32_t x[8];
#pragma unroll
        for (int r = 0; r < 8; r++) x[r] = nxt[r] & 0xFFFu;
        if (p + stride < n) {
#pragma unroll
            for (int r = 0; r < 8; r++) nxt[r] = __ldg(in + 256 * (p + stride) + idxA(lane, r));
        }
        bool big = false;
#pragma unroll
        for (int r = 0; r < 8; r++) big |= x[r] >= kQ;
        if (__any_sync(kFullMask, big)) ntt_warp_exact(x, scratch, lane);  // a coefficient in [q, 4096): ml_kem.c:317-318 literally
        else ntt_warp<kPrimPipe>(x, scratch, lane, tw);
        store_layoutC_global(x, lane, out + 256 * p);
    }
}
// ml_kem.c:336 InverseNTT: 128-bit loads (layout C), 16-bit stores in layout A.
__global__ void __launch_bounds__(kPrimTPB) k_intt_batch(int n, const uint16_t *__restrict__ in, uint16_t *__restrict__ out) {
    __shared__ __align__(16) uint16_t s_scratch[(kPrimTPB / 32) * kScratchU16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *scratch = s_scratch + warp * kScratchU16;
    LaneTwiddles tw;
    load_lane_twiddles_inv<kPrimPipe>(tw, lane);
    const long long stride = (long long)gridDim.x * (kPrimTPB / 32);
    long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp;
    uint4 nxt = make_uint4(0, 0, 0, 0);
    if (p < n) nxt = __ldg(reinterpret_cast<const uint4 *>(in + 256 * p) + lane);
    for (; p < n; p += stride) {
        uint32_t x[8];
        unpack_pairs(nxt, x);
        if (p + stride < n) nxt = __ldg(reinterpret_cast<const uint4 *>(in + 256 * (p + stride)) + lane);
#pragma unroll
        for (int r = 0; r < 8; r++) x[r] &= 0xFFFu;
        intt_warp<kPrimPipe>(x, scratch, lane, tw);
        uint16_t *dst = out + 256 * p;
#pragma unroll
        for (int r = 0; r < 8; r++) dst[idxA(lane, r)] = (uint16_t)x[r];
    }
}
// ml_kem.c:415 MultiplyNTTs (operands may be any 12-bit value, D4).
__global__ void __launch_bounds__(kPrimTPB) k_mulntt_batch(int n, const uint16_t *__restrict__ f, const uint16_t *__restrict__ gq,
                                                           uint16_t *__restrict__ h) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint2 gam[4];
#pragma unroll
    for (int r = 0; r < 4; r++) gam[r] = lane_gamma(lane + 32 * r);
    for (long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kPrimTPB / 32)) {
        const uint32_t *fw = reinterpret_cast<const uint32_t *>(f + 256 * p), *gw = reinterpret_cast<const uint32_t *>(gq + 256 * p);
        uint32_t *hw = reinterpret_cast<uint32_t *>(h + 256 * p);
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int t = lane + 32 * r;
            uint32_t a = __ldg(fw + t), b = __ldg(gw + t), c0 = 0, c1 = 0;
            basemul_acc(c0, c1, a & 0xFFFu, (a >> 16) & 0xFFFu, b & 0xFFFu, (b >> 16) & 0xFFFu, gam[r]);
            hw[t] = canon32(c0) | (canon32(c1) << 16);
        }
    }
}

// ml_kem.c:580 PolyAddition / :599 PolySubtraction, element-wise on 12-bit coefficients (8 per thread).  Restated literally:
// the sum is reduced ((u + v) % q), the difference is `u < v ? q - (v - u) : u - v` kept in a 12-bit field -- it stays
// unreduced when u - v >= q, like in the reference.  On the KEM path both are fused into their consumers (matvec_row_tail,
// k_encrypt_v, k_decrypt); these kernels serve the stand-alone entry points.
template <bool SUB>
__global__ void __launch_bounds__(kPrimTPB) k_poly_addsub(long long nvec, const uint4 *__restrict__ u, const uint4 *__restrict__ v,
                                                          uint4 *__restrict__ z) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        const uint4 a4 = __ldg(u + i), b4 = __ldg(v + i);
        const uint32_t a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            uint32_t r[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t x = (a[k] >> (16 * h)) & 0xFFFu, y = (b[k] >> (16 * h)) & 0xFFFu;
                r[h] = SUB ? ((x < y ? kQ - (y - x) : x - y) & 0xFFFu) : canon16(x + y);
            }
            o[k] = r[0] | (r[1] << 16);
        }
        z[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}
// ml_kem.c:618 VectorMultiply: w = sum over i < k of MultiplyNTTs(u[i], v[i]); one item per warp, operands any 12-bit value.
__global__ void __launch_bounds__(kPrimTPB) k_vecmul_batch(int n, int k, const uint16_t *__restrict__ u, const uint16_t *__restrict__ v,
                                                           uint16_t *__restrict__ w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint2 gam[4];
#pragma unroll
    for (int r = 0; r < 4; r++) gam[r] = lane_gamma(lane + 32 * r);
    for (long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kPrimTPB / 32)) {
        uint32_t acc[8];
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = 0;
        for (int j = 0; j < k; j++) {
            const uint32_t *uw = reinterpret_cast<const uint32_t *>(u + 256 * (p * k + j)), *vw = reinterpret_cast<const uint32_t *>(v + 256 * (p * k + j));
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const uint32_t a = __ldg(uw + lane + 32 * r), b = __ldg(vw + lane + 32 * r);
                uint32_t c0 = 0, c1 = 0;  // every product is reduced before it is added (MultiplyNTTs then PolyAddition)
                basemul_acc(c0, c1, a & 0xFFFu, (a >> 16) & 0xFFFu, b & 0xFFFu, (b >> 16) & 0xFFFu, gam[r]);
                acc[2 * r] += canon32(c0);
                acc[2 * r + 1] += canon32(c1);
            }
        }
        uint32_t *ww = reinterpret_cast<uint32_t *>(w + 256 * p);
#pragma unroll
        for (int r = 0; r < 4; r++) ww[lane + 32 * r] = canon16(acc[2 * r]) | (canon16(acc[2 * r + 1]) << 16);
    }
}

// ml_kem.c:189 SampleNTT over n 34-byte seeds; out = n x 256 uint16; seeds_after (optional) receives the
// caller-visible B after the call (only bytes 32, 33 can change).
__global__ void __launch_bounds__(128) k_sample_ntt_batch(int n, const uint8_t *__restrict__ seeds, uint16_t *__restrict__ out,
                                                          uint8_t *__restrict__ seeds_after, int group_limit) {
    extern __shared__ __align__(16) uint32_t s_slots[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int item = blockIdx.x * 128 + tid;
    const bool active = item < n;
    Lane rho[4];
    uint32_t b32 = 0, b33 = 0;
    if (active) {
        const uint8_t *s = seeds + 34 * (size_t)item;  // 34-byte stride: byte loads
#pragma unroll
        for (int w = 0; w < 4; w++) {
            uint32_t lo = 0, hi = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                lo |= (uint32_t)s[8 * w + b] << (8 * b);
                hi |= (uint32_t)s[8 * w + 4 + b] << (8 * b);
            }
            rho[w] = Lane{lo, hi};
        }
        b32 = s[32];
        b33 = s[33];
    } else {
#pragma unroll
        for (int w = 0; w < 4; w++) rho[w] = Lane{0u, 0u};
    }
    sample_ntt_thread(rho, b32, b33, reinterpret_cast<uint16_t *>(s_slots + kSlotWords * tid), active, group_limit);
    if (active && seeds_after) {
        uint8_t *sa = seeds_after + 34 * (size_t)item;
        const uint8_t *s = seeds + 34 * (size_t)item;
        for (int b = 0; b < 32; b++) sa[b] = s[b];
        sa[32] = (uint8_t)b32;
        sa[33] = (uint8_t)b33;
    }
    __syncwarp();
    for (int t = 0; t < 32; t++) {  // coalesced copy-out, one polynomial at a time
        int it = blockIdx.x * 128 + warp * 32 + t;
        if (it >= n) break;
        const uint32_t *src = s_slots + kSlotWords * (warp * 32 + t);
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + 256 * (size_t)it);
#pragma unroll
        for (int r = 0; r < 4; r++) dst[lane + 32 * r] = src[lane + 32 * r];
    }
}

// ml_kem.c:253 SamplePolyCBD over n byte strings of 64 eta bytes (no PRF); one polynomial per warp.
template <int ETA>
__global__ void __launch_bounds__(kPrimTPB) k_cbd_batch(int n, const uint8_t *__restrict__ in, uint16_t *__restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kPrimTPB / 32)) {
        const uint8_t *src = in + (size_t)64 * ETA * p;
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + 256 * p);
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int t = lane + 32 * r;  // coefficients 2t, 2t+1 = 4 eta bits starting at bit 4 eta t
            uint32_t c[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int bit = 2 * ETA * (2 * t + h);
                uint32_t w = (uint32_t)src[bit >> 3] | ((uint32_t)src[min((bit >> 3) + 1, 64 * ETA - 1)] << 8);
                w >>= (bit & 7);
                uint32_t x = __popc(w & ((1u << ETA) - 1u)), y = __popc((w >> ETA) & ((1u << ETA) - 1u));
                c[h] = x >= y ? x - y : kQ - (y - x);
            }
            dst[t] = c[0] | (c[1] << 16);
        }
    }
}

// PRF + CBD (+ optional NTT) exposed as a primitive: n (seed, nonce) pairs -> uint16 polynomials.
template <int ETA, int RATE = kRateShake128>
__global__ void __launch_bounds__(kNoiseTPB) k_prf_cbd_batch(int n, const uint8_t *__restrict__ seeds, const uint8_t *__restrict__ nonces,
                                                             uint16_t *__restrict__ out) {
    __shared__ uint32_t s_codes[kNoiseTPB * 33];
    const int item = blockIdx.x * kNoiseTPB + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Lane seed[4];
#pragma unroll
    for (int w = 0; w < 4; w++) seed[w] = item < n ? load_lane(seeds + 32 * (size_t)item + 8 * w) : Lane{0u, 0u};
    uint32_t nonce = item < n ? nonces[item] : 0u;
    uint32_t *mine = s_codes + 33 * threadIdx.x;
    prf_cbd_codes<ETA, RATE>(seed, nonce, [&](int w, uint32_t v) { mine[w] = v; });
    __syncwarp();
    for (int t = 0; t < 32; t++) {
        int it = blockIdx.x * kNoiseTPB + warp * 32 + t;
        if (it >= n) break;
        const uint32_t *codes = s_codes + 33 * (warp * 32 + t);
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + 256 * (size_t)it);
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int tt = lane + 32 * r;  // coefficients 2tt, 2tt+1
            uint32_t wd = codes[tt >> 2] >> (8 * (tt & 3));
            dst[tt] = noise_code_to_coeff(wd & 15u) | (noise_code_to_coeff((wd >> 4) & 15u) << 16);
        }
    }
}

// ByteEncode_d(Compress_d(.)) and Decompress_d(ByteDecode_d(.)) (ml_kem.c:83-177), HBM-bound:
// one polynomial per warp, 128-bit loads of 8 coefficients per lane, bytes staged in shared memory and
// written back with 128-bit stores.  COMPRESS=false gives the plain codec (for d = 12: no reduction, D4).
template <int D, bool COMPRESS>
__global__ void __launch_bounds__(kPrimTPB) k_encode_batch(int n, const uint16_t *__restrict__ in, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t s_stage[(kPrimTPB / 32) * 32 * D];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *stage = s_stage + warp * 32 * D;
    const long long stride = (long long)gridDim.x * (kPrimTPB / 32);
    long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp;
    uint4 nxt = make_uint4(0, 0, 0, 0);
    if (p < n) nxt = __ldg(reinterpret_cast<const uint4 *>(in + 256 * p) + lane);  // coefficients 8 lane .. 8 lane + 7
    for (; p < n; p += stride) {
        uint4 q4 = nxt;
        if (p + stride < n) nxt = __ldg(reinterpret_cast<const uint4 *>(in + 256 * (p + stride)) + lane);  // next polynomial in flight
        uint32_t w[4] = {q4.x, q4.y, q4.z, q4.w}, v[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint32_t c = (w[i >> 1] >> (16 * (i & 1))) & 0xFFFu;
            v[i] = (COMPRESS ? compress<D>(c) : c) & ((1u << D) - 1u);
        }
        pack8<D>(v, stage + D * lane);
        __syncwarp();
        const uint4 *sv = reinterpret_cast<const uint4 *>(stage);
        uint4 *ov = reinterpret_cast<uint4 *>(out + (size_t)32 * D * p);
        for (int i = lane; i < 2 * D; i += 32) ov[i] = sv[i];
        __syncwarp();
    }
}
template <int D, bool DECOMPRESS>
__global__ void __launch_bounds__(kPrimTPB) k_decode_batch(int n, const uint8_t *__restrict__ in, uint16_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t s_stage[(kPrimTPB / 32) * 32 * D + 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *stage = s_stage + warp * 32 * D;
    for (long long p = (long long)blockIdx.x * (kPrimTPB / 32) + warp; p < n; p += (long long)gridDim.x * (kPrimTPB / 32)) {
        const uint4 *iv = reinterpret_cast<const uint4 *>(in + (size_t)32 * D * p);
        uint4 *sv = reinterpret_cast<uint4 *>(stage);
        for (int i = lane; i < 2 * D; i += 32) sv[i] = __ldg(iv + i);
        __syncwarp();
        uint32_t v[8];
        unpack8<D>(stage, lane, v);
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = DECOMPRESS ? decompress<D>(v[i]) : v[i];
        reinterpret_cast<uint4 *>(out + 256 * p)[lane] =
            make_uint4(v[0] | (v[1] << 16), v[2] | (v[3] << 16), v[4] | (v[5] << 16), v[6] | (v[7] << 16));
        __syncwarp();
    }
}
// Element-wise Compress_d / Decompress_d on uint16 arrays (8 coefficients per thread).
template <int D, bool DECOMPRESS>
__global__ void __launch_bounds__(kPrimTPB) k_compress_batch(long long nvec, const uint4 *__restrict__ in, uint4 *__restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        uint4 q4 = __ldg(in + i);
        uint32_t w[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            uint32_t lo = w[k] & 0xFFFu, hi = (w[k] >> 16) & 0xFFFu;
            if (DECOMPRESS) {
                lo = decompress<D>(lo & ((1u << D) - 1u));
                hi = decompress<D>(hi & ((1u << D) - 1u));
            } else {
                lo = compress<D>(lo);
                hi = compress<D>(hi);
            }
            w[k] = lo | (hi << 16);
        }
        out[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

}  // namespace mlkem
