// mlkem_device.cuh -- device-side building blocks of the B200 batched ML-KEM engine (sm_100a).
//
// Everything here is integer work on the 32-bit ALU/FMA pipes; there is no dense contraction on this
// path, so no tensor cores (see DESIGN.md).  Three families of routines:
//
//   1. field arithmetic mod q = 3329 (Shoup multiplication by constants, Barrett for products),
//   2. Keccak-f[1600] with one sponge per THREAD (25 lanes as 50 x 32-bit registers, funnel-shift
//      rotates), plus absorb/squeeze helpers for SHA3-256 / SHA3-512 / SHAKE128; and (2b) the same permutation with one
//      sponge per WARP (state lanes spread over the lanes, neighbours by shuffle) for the hash chains of small batches,
//   3. polynomial routines with one polynomial per WARP: NTT / inverse NTT (8 coefficients per lane,
//      three register-local passes with two transposes through a swizzled shared-memory scratch, no
//      shuffles), NTT-domain multiply-accumulate, Compress/Decompress and ByteEncode/ByteDecode.
//
// Bit-exactness contract: results equal the reference rsjahnige/CRYSTALS-Kyber `ml_kem.c`
// (see SURVEY.md section 0 for where it differs from FIPS 203).  File:line citations below refer to
// /root/reference/ml_kem.c unless stated otherwise.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mlkem {

constexpr int kN = 256;
constexpr uint32_t kQ = 3329;
constexpr uint32_t kFullMask = 0xFFFFFFFFu;

// ------------------------------------------------------------------------------------------------
// Constant tables (filled once per device by the host: build_tables() / acquire() in mlkem_b200.cu)
// ------------------------------------------------------------------------------------------------
// zeta_i = 17^BitRev7(i) mod q (ml_kem.c:300-307) as {w, floor(w * 2^16 / q)} for Shoup multiplication.
// gamma_i = 17^(2 BitRev7(i) + 1) mod q (ml_kem.c:424-433), same packing.
// The inverse transform walks the same table downwards (ml_kem.c:345-357: i = 127 .. 1); its last layer
// is pre-multiplied by 3303 = 128^-1 (ml_kem.c:378-381).
struct TwiddleTables {
    uint2 zeta[128];
    uint2 zeta_inv_last[2];  // {zeta[1] * 3303 mod q, 3303}
    uint2 gamma[128];        // {w, floor(w 2^16 / q)}
    uint2 gamma32[128];      // {w, floor(w 2^32 / q)} for mul_shoup_fma
    uint2 zeta32[128];       // zeta as {w, floor(w 2^32 / q)}: the transforms that run next to Keccak (kFmaPipe variants)
    uint2 zeta_inv_last32[2];
};
// The library is a single translation unit (mlkem_b200.cu), so the tables are defined right here.
// c_tw (constant bank) serves the warp-uniform lookups; g_tw (global memory, read through L1 with __ldg) serves
// the lane-dependent ones -- a constant-bank load with 8..32 distinct addresses per warp is replayed once per
// address, which showed up as the top stall reason per instruction in the first ncu capture.
__constant__ TwiddleTables c_tw;
__device__ TwiddleTables g_tw;
__constant__ uint2 c_keccak_rc[24];
// c_pow2[k] = 2^k.  A left shift written as x * c_pow2[k] is an IMAD with a constant-bank operand: ptxas cannot see the
// value, so it cannot turn the multiply back into a shift on the alu pipe (which it does for literal powers of two).
__constant__ uint32_t c_pow2[32];
__device__ __forceinline__ uint32_t shl_fma(uint32_t x, int k) { return x * c_pow2[k]; }
__device__ __forceinline__ uint2 lane_zeta(int i) { return __ldg(&g_tw.zeta[i]); }
__device__ __forceinline__ uint2 lane_zeta32(int i) { return __ldg(&g_tw.zeta32[i]); }
__device__ __forceinline__ uint2 lane_gamma(int i) { return __ldg(&g_tw.gamma32[i]); }

// ------------------------------------------------------------------------------------------------
// 1. Field arithmetic
// ------------------------------------------------------------------------------------------------

// High half of a 32 x 32-bit product: IMAD.HI.  (The co-issue microbenchmark prices an IMAD.HI next to a LOP3 stream at
// 1.71 lost LOP3 issues and an IMAD.WIDE at 0.29, profiles/coissue_r01.jsonl, but in the kernels the IMAD.WIDE form --
// -DMLKEM_B200_MULHI_WIDE, inline PTX so that ptxas keeps it -- is slower: fused kernel 9.42 vs 9.29 ms, k_noise 1.58 vs
// 1.55 ms per 2^20 items.  It needs an aligned register pair per product.)
__device__ __forceinline__ uint32_t mulhi(uint32_t a, uint32_t b) {
#ifndef MLKEM_B200_MULHI_WIDE
    return __umulhi(a, b);
#else
    [[maybe_unused]] uint32_t lo;
    uint32_t hi;
    asm volatile("{.reg .b64 t; mul.wide.u32 t, %2, %3; mov.b64 {%0, %1}, t;}" : "=r"(lo), "=r"(hi) : "r"(a), "r"(b));
    return hi;
#endif
}

// a * w mod q for a < 2^16 and a constant w given as {w, floor(w 2^16 / q)}; result in [0, 2q).
__device__ __forceinline__ uint32_t mul_shoup(uint32_t a, uint2 w) {
    uint32_t qh = (a * w.y) >> 16;
    return a * w.x - qh * kQ;
}
// Same product with the quotient estimate taken by a high multiply (a < 2^32, w32 = floor(w 2^32 / q)): three
// fma-pipe instructions and none on the alu pipe.  Used where the alu pipe is the bottleneck (next to Keccak).
__device__ __forceinline__ uint32_t mul_shoup_fma(uint32_t a, uint32_t w, uint32_t w32) {
    uint32_t qh = mulhi(a, w32);
    return a * w - qh * kQ;
}
// Pipe policy of the transforms.  The hashing kernels saturate the alu pipe (LOP3 / SHF) and leave the fma pipe idle,
// so every transform that shares an SM with Keccak (k_sample_matvec, k_noise) is instantiated with FMA = true: quotient
// estimates by multiply-high (IMAD.HI, fma pipe, half rate) instead of multiply + shift (IMAD + SHF), exact
// canonicalisation by multiply-high instead of Barrett + min.  The stand-alone transforms keep the balanced form.
constexpr bool kFmaPipe = true, kBalanced = false;
template <bool FMA>
__device__ __forceinline__ uint32_t mulz(uint32_t a, uint2 z) {  // z from the zeta32 (FMA) or zeta (balanced) table; result < 2q
    return FMA ? mul_shoup_fma(a, z.x, z.y) : mul_shoup(a, z);
}
// x mod q, exact, for x < 2^21 (1290168 = ceil(2^32 / q); checked exhaustively in
// tests/test_abi_cpu.py::test_arithmetic_lemmas): two fma-pipe instructions, none on the alu pipe.
__device__ __forceinline__ uint32_t canon_fma(uint32_t x) { return x - mulhi(x, 1290168u) * kQ; }
// x mod q for x < 2^16, result in [0, q + 1]: q + 1 only for x = 56594, 59923, 63252, so the result is <= q for x < 16q
// (checked exhaustively in tests/test_abi_cpu.py::test_arithmetic_lemmas).
__device__ __forceinline__ uint32_t barrett16(uint32_t x) {
    uint32_t qh = (x * 40317u) >> 27;  // floor(2^27 / q) = 40317
    return x - qh * kQ;
}
// x mod q for any x < 2^32, result in [0, 2q).
__device__ __forceinline__ uint32_t barrett32(uint32_t x) {
    uint32_t qh = mulhi(x, 1290167u);  // floor(2^32 / q)
    return x - qh * kQ;
}
// r in [0, 2q) -> [0, q)
__device__ __forceinline__ uint32_t csubq(uint32_t r) { return min(r, r - kQ); }
// canonical value of any x < 2^16
__device__ __forceinline__ uint32_t canon16(uint32_t x) { return csubq(barrett16(x)); }
// canonical value of any x < 2^32
__device__ __forceinline__ uint32_t canon32(uint32_t x) { return csubq(barrett32(x)); }

// ml_kem.c:83 Compress_d for canonical x: floor((2^d x + 1664) / q) mod 2^d  (SURVEY 8(a) a5: closed form
// verified exhaustively against the reference's quotient/remainder formulation).
template <int D>
__device__ __forceinline__ uint32_t compress(uint32_t x) {
    if (D >= 12) return x;
    uint32_t t = (x << D) + 1664u;  // < 2^23
    uint32_t qh = mulhi(t, 1290167u);
    uint32_t r = t - qh * kQ;  // [0, 2q)
    qh += (r >= kQ);
    return qh & ((1u << D) - 1u);
}
// The same for CANONICAL x (< q) and the d of the parameter sets: a single multiply-high.  The constants were found
// by exhaustive search over all x < q (tools/find_compress_constants.py): floor(((x << d) + c) M / 2^32) mod 2^d equals
// Compress_d(x) with (c, M) = (1665, 1290167) for d in {1, 4, 5} and (1664, 1290168) for d in {10, 11}.
template <int D>
__device__ __forceinline__ uint32_t compress_canon(uint32_t x) {
    static_assert(D == 1 || D == 4 || D == 5 || D == 10 || D == 11, "no verified constants for this d");
    constexpr uint32_t c = (D >= 10) ? 1664u : 1665u, M = (D >= 10) ? 1290168u : 1290167u;
    return mulhi(x * (1u << D) + c, M) & ((1u << D) - 1u);
}

// Compress_d of a RESIDUE x < 4q (any representative of the coefficient) for d <= 5: for these d the single
// multiply-high stays exact far beyond q (exhaustive check in tests/test_abi_cpu.py::test_arithmetic_lemmas), and a
// multiple of q added to x only adds a multiple of 2^d to the quotient.  Not valid for d = 10, 11.
template <int D>
__device__ __forceinline__ uint32_t compress_resid(uint32_t x) {
    static_assert(D == 1 || D == 4 || D == 5, "single multiply-high is not exact on residues for this d");
    return mulhi(x * (1u << D) + 1664u, 1290168u) & ((1u << D) - 1u);
}

// ml_kem.c:104 Decompress_d: (q y + 2^(d-1)) >> d.
template <int D>
__device__ __forceinline__ uint32_t decompress(uint32_t y) {
    if (D >= 12) return y;
    return (kQ * y + (1u << (D - 1))) >> D;
}

// ------------------------------------------------------------------------------------------------
// 2. Keccak-f[1600], one sponge per thread
// ------------------------------------------------------------------------------------------------
// A lane is kept as two 32-bit halves so that rotates are single funnel shifts (SHF.L.W) and the
// theta / chi steps are single three-input LOP3s: 122 LOP3 + 58 SHF = 180 instructions per round,
// all on the alu pipe (profiles/: 99 % of the measured LOP3/SHF issue rate).
struct Lane {
    uint32_t lo, hi;
};

template <int R>
__device__ __forceinline__ Lane rotl64(Lane x) {
    Lane r = x;
    if constexpr (R == 32) {
        r.lo = x.hi;
        r.hi = x.lo;
    } else if constexpr (R > 0 && R < 32) {
        r.hi = __funnelshift_l(x.lo, x.hi, R);
        r.lo = __funnelshift_l(x.hi, x.lo, R);
    } else if constexpr (R > 32) {
        r.hi = __funnelshift_l(x.hi, x.lo, R - 32);
        r.lo = __funnelshift_l(x.lo, x.hi, R - 32);
    }
    return r;
}
__device__ __forceinline__ Lane xor3(Lane a, Lane b, Lane c) { return Lane{a.lo ^ b.lo ^ c.lo, a.hi ^ b.hi ^ c.hi}; }
__device__ __forceinline__ Lane xor5(Lane a, Lane b, Lane c, Lane d, Lane e) {
    return Lane{a.lo ^ b.lo ^ c.lo ^ d.lo ^ e.lo, a.hi ^ b.hi ^ c.hi ^ d.hi ^ e.hi};
}
__device__ __forceinline__ Lane chi3(Lane a, Lane b, Lane c) { return Lane{a.lo ^ (~b.lo & c.lo), a.hi ^ (~b.hi & c.hi)}; }

// sha3.c:207 Keccak_f = 24 x Iota(Chi(Pi(Rho(Theta(S))))) (sha3.c:15,53,88,116,182).
// Kept as a loop of two rounds per iteration: 360 instructions fit the instruction cache even with several inlined
// call sites, ptxas renames registers across the back edge without moves, and the loop overhead is halved
// (measured: +0.9 % over one round per iteration; three / four rounds per iteration cost the fused matrix kernel 0.8 % / 7 %;
// 24 rounds unrolled overflow the instruction cache: -19 %).
__device__ __forceinline__ void keccak_f1600(Lane a[25]) {
#pragma unroll 2
    for (int rnd = 0; rnd < 24; rnd++) {
        Lane c0 = xor5(a[0], a[5], a[10], a[15], a[20]), c1 = xor5(a[1], a[6], a[11], a[16], a[21]),
             c2 = xor5(a[2], a[7], a[12], a[17], a[22]), c3 = xor5(a[3], a[8], a[13], a[18], a[23]),
             c4 = xor5(a[4], a[9], a[14], a[19], a[24]);
        Lane r0 = rotl64<1>(c0), r1 = rotl64<1>(c1), r2 = rotl64<1>(c2), r3 = rotl64<1>(c3), r4 = rotl64<1>(c4);
#define MLKEM_TH(x, cm, rp)             \
    a[x] = xor3(a[x], cm, rp);          \
    a[x + 5] = xor3(a[x + 5], cm, rp);  \
    a[x + 10] = xor3(a[x + 10], cm, rp); \
    a[x + 15] = xor3(a[x + 15], cm, rp); \
    a[x + 20] = xor3(a[x + 20], cm, rp);
        MLKEM_TH(0, c4, r1) MLKEM_TH(1, c0, r2) MLKEM_TH(2, c1, r3) MLKEM_TH(3, c2, r4) MLKEM_TH(4, c3, r0)
#undef MLKEM_TH
        Lane b[25];
        b[0] = a[0];             b[10] = rotl64<1>(a[1]);   b[20] = rotl64<62>(a[2]);  b[5] = rotl64<28>(a[3]);   b[15] = rotl64<27>(a[4]);
        b[16] = rotl64<36>(a[5]); b[1] = rotl64<44>(a[6]);   b[11] = rotl64<6>(a[7]);   b[21] = rotl64<55>(a[8]);  b[6] = rotl64<20>(a[9]);
        b[7] = rotl64<3>(a[10]);  b[17] = rotl64<10>(a[11]); b[2] = rotl64<43>(a[12]);  b[12] = rotl64<25>(a[13]); b[22] = rotl64<39>(a[14]);
        b[23] = rotl64<41>(a[15]); b[8] = rotl64<45>(a[16]); b[18] = rotl64<15>(a[17]); b[3] = rotl64<21>(a[18]);  b[13] = rotl64<8>(a[19]);
        b[14] = rotl64<18>(a[20]); b[24] = rotl64<2>(a[21]); b[9] = rotl64<61>(a[22]);  b[19] = rotl64<56>(a[23]); b[4] = rotl64<14>(a[24]);
#pragma unroll
        for (int y = 0; y < 25; y += 5) {
#pragma unroll
            for (int x = 0; x < 5; x++) a[y + x] = chi3(b[y + x], b[y + (x + 1) % 5], b[y + (x + 2) % 5]);
        }
        uint2 rc = c_keccak_rc[rnd];
        a[0].lo ^= rc.x;
        a[0].hi ^= rc.y;
    }
}

__device__ __forceinline__ void keccak_zero(Lane a[25]) {
#pragma unroll
    for (int i = 0; i < 25; i++) a[i] = Lane{0u, 0u};
}

// Domain-suffix bytes (suffix bits followed by the first pad bit, sha3.c:408-431 + sha3.c:226):
constexpr uint32_t kSfxHash = 0x06;  // sfx {0,1}      SHA3-256 / SHA3-512
constexpr uint32_t kSfxXof = 0x1F;   // sfx {1,1,1,1}  SHAKE
constexpr int kRateShake128 = 21;    // lanes: c = 256  (PRF, J and the matrix XOF -- D1, D2)
constexpr int kRateSha3_256 = 17;    // lanes: c = 512  (H)
constexpr int kRateSha3_512 = 9;     // lanes: c = 1024 (G)

// Absorb a message given as 64-bit little-endian words (all ML-KEM hash inputs except G(d||k) are
// multiples of 8 bytes) and apply pad10*1 (sha3.c:226,257-291).  `word(i)` returns message word i as a
// Lane; `nwords` is uniform across the warp.  Leaves the state after the last absorbing permutation,
// i.e. ready to read the first output block.
template <int RATE, typename F>
__device__ __forceinline__ void sponge_absorb_words(Lane a[25], int nwords, uint32_t sfx, F word) {
    keccak_zero(a);
    int base = 0;
    for (; base + RATE <= nwords; base += RATE) {
#pragma unroll
        for (int i = 0; i < RATE; i++) {
            Lane w = word(base + i);
            a[i].lo ^= w.lo;
            a[i].hi ^= w.hi;
        }
        keccak_f1600(a);
    }
    int rem = nwords - base;  // 0 .. RATE-1 words in the final block
#pragma unroll
    for (int i = 0; i < RATE; i++) {
        if (i < rem) {
            Lane w = word(base + i);
            a[i].lo ^= w.lo;
            a[i].hi ^= w.hi;
        } else if (i == rem) {
            a[i].lo ^= sfx;
        }
    }
    a[RATE - 1].hi ^= 0x80000000u;
    keccak_f1600(a);
}

__device__ __forceinline__ Lane load_lane(const uint8_t *p) {  // p must be 8-byte aligned
    uint2 v = *reinterpret_cast<const uint2 *>(p);
    return Lane{v.x, v.y};
}
__device__ __forceinline__ void store_lane(uint8_t *p, Lane v) { *reinterpret_cast<uint2 *>(p) = make_uint2(v.lo, v.hi); }

// ------------------------------------------------------------------------------------------------
// 2b. Keccak-f[1600], one sponge per WARP: the latency form, for small batches
// ------------------------------------------------------------------------------------------------
// One sponge per thread is the throughput form: 4 320 dependent-issue instructions per permutation, 4.4 us on a warp that has a
// scheduler to itself.  A batch of one (what a caller of the reference's KEM_Encaps / KEM_Decaps gets) spends most of its time
// in such chains -- H(ek) alone is 9 permutations one after the other -- with 31 lanes of the warp idle.  Here lane l < 25
// holds state lane A[x][y], l = x + 5 y, as two registers, and the round's neighbours come by shuffle: theta's column
// parities from the four other lanes of the column (then C[x-1] and C[x+1] from row 0), rho as a funnel shift by the lane's
// own offset, pi as one permuting shuffle, chi from the two next lanes of the row; 18 SHFL + ~16 alu instructions per round
// instead of 180, a dependent chain of four shuffle latencies.  Lanes 25..31 carry zeros and shuffle from themselves.
// (tests/test_abi_cpu.py::test_warp_keccak_model pins this index arithmetic against hashlib with a numpy model of the 32 lanes.)
struct WarpSponge {
    int s5, s10, s15, s20;  // the other four lanes of this lane's column
    int xm, xp;             // row-0 lanes holding C[x-1] and C[x+1]
    int pi;                 // source of this lane after rho: B[y][2x+3y] = A[x][y] read backwards
    int c1, c2;             // the next two lanes of this lane's row
    uint32_t shift;         // rho offset mod 32
    bool swap, first;       // rho offset >= 32; lane 0 (iota)
};
__device__ __forceinline__ WarpSponge warp_sponge_init(int lane) {
    // rho offsets by lane index x + 5 y (sha3.c:53-87 computes them from the (t+1)(t+2)/2 walk): the same constants as the
    // rotl64<> amounts of keccak_f1600 above, packed four per word
    constexpr uint32_t kRho[7] = {0u | 1u << 8 | 62u << 16 | 28u << 24,  27u | 36u << 8 | 44u << 16 | 6u << 24,  55u | 20u << 8 | 3u << 16 | 10u << 24,
                                  43u | 25u << 8 | 39u << 16 | 41u << 24, 45u | 15u << 8 | 21u << 16 | 8u << 24, 18u | 2u << 8 | 61u << 16 | 56u << 24,
                                  14u};
    WarpSponge w;
    const bool act = lane < 25;
    const int x = lane % 5, y = lane / 5;
    w.s5 = act ? (lane + 5) % 25 : lane;
    w.s10 = act ? (lane + 10) % 25 : lane;
    w.s15 = act ? (lane + 15) % 25 : lane;
    w.s20 = act ? (lane + 20) % 25 : lane;
    w.xm = act ? (x + 4) % 5 : lane;
    w.xp = act ? (x + 1) % 5 : lane;
    w.pi = act ? (x + 3 * y) % 5 + 5 * x : lane;
    w.c1 = act ? 5 * y + (x + 1) % 5 : lane;
    w.c2 = act ? 5 * y + (x + 2) % 5 : lane;
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < 7; k++) word = (lane >> 2) == k ? kRho[k] : word;
    const uint32_t rot = act ? (word >> (8 * (lane & 3))) & 63u : 0u;
    w.shift = rot & 31u;
    w.swap = (rot & 32u) != 0;
    w.first = lane == 0;
    return w;
}
__device__ __forceinline__ Lane shfl_lane(Lane v, int src) {
    return Lane{__shfl_sync(kFullMask, v.lo, src), __shfl_sync(kFullMask, v.hi, src)};
}
// sha3.c:207 Keccak_f on the state spread over the warp; every lane of the warp must call it.
__device__ __forceinline__ void keccak_f1600_warp(Lane &a, const WarpSponge &w) {
#pragma unroll 2
    for (int rnd = 0; rnd < 24; rnd++) {
        const Lane c = xor5(a, shfl_lane(a, w.s5), shfl_lane(a, w.s10), shfl_lane(a, w.s15), shfl_lane(a, w.s20));  // theta, sha3.c:15
        a = xor3(a, shfl_lane(c, w.xm), rotl64<1>(shfl_lane(c, w.xp)));
        const uint32_t lo = w.swap ? a.hi : a.lo, hi = w.swap ? a.lo : a.hi;                                       // rho, sha3.c:53
        a.hi = __funnelshift_l(lo, hi, w.shift);
        a.lo = __funnelshift_l(hi, lo, w.shift);
        const Lane b = shfl_lane(a, w.pi);                                                                          // pi, sha3.c:88
        a = chi3(b, shfl_lane(b, w.c1), shfl_lane(b, w.c2));                                                        // chi, sha3.c:116
        const uint2 rc = c_keccak_rc[rnd];                                                                          // iota, sha3.c:182
        a.lo ^= w.first ? rc.x : 0u;
        a.hi ^= w.first ? rc.y : 0u;
    }
}
// The warp form of sponge_absorb_words: `word(i)` is evaluated by lane (i mod RATE) only.  Returns this lane's state lane
// after the last absorbing permutation: lanes 0 .. RATE-1 hold the first output block.
template <int RATE, typename F>
__device__ __forceinline__ Lane warp_sponge_absorb_words(int lane, const WarpSponge &w, int nwords, uint32_t sfx, F word) {
    Lane a{0u, 0u};
    int base = 0;
    for (; base + RATE <= nwords; base += RATE) {
        if (lane < RATE) {
            const Lane v = word(base + lane);
            a.lo ^= v.lo;
            a.hi ^= v.hi;
        }
        keccak_f1600_warp(a, w);
    }
    const int rem = nwords - base;  // 0 .. RATE-1 words in the final block, then the suffix and the pad (sha3.c:226)
    if (lane < rem) {
        const Lane v = word(base + lane);
        a.lo ^= v.lo;
        a.hi ^= v.hi;
    } else if (lane == rem) {
        a.lo ^= sfx;
    }
    if (lane == RATE - 1) a.hi ^= 0x80000000u;
    keccak_f1600_warp(a, w);
    return a;
}

// ------------------------------------------------------------------------------------------------
// 3. Polynomials, one per warp
// ------------------------------------------------------------------------------------------------
// Register layouts for the 256 coefficients of one polynomial held by a warp, 8 per lane
// (coefficient index bits b7..b0):
//   layout A: x[r] = f[lane + 32 r]                        r = b7 b6 b5        lane = b4 b3 b2 b1 b0
//   layout B: x[r] = f[32 (lane >> 2) + 4 r + (lane & 3)]  r = b4 b3 b2        lane = b7 b6 b5 b1 b0
//   layout C: x[r] = f[8 lane + r]                         r = b2 b1 b0        lane = b7 b6 b5 b4 b3
// The forward transform (layers len = 128 .. 2 act on index bits b7 .. b1) runs three register-local
// passes, A: len 128/64/32, B: len 16/8/4, C: len 2, with two transposes through the warp's shared-memory
// scratch in between; it consumes layout A and leaves layout C, i.e. every lane ends up owning 8
// consecutive coefficients = one 16-byte vector of the natural-order output.  The inverse transform runs
// the same passes backwards: C in, A out.  No shuffles, no redundant multiplications: 28 butterflies per lane.
//
// Scratch polynomials are 256 uint16 (512 B, 16-byte aligned) with an XOR swizzle that makes all three
// access patterns bank-conflict free: coefficient c lives at uint16 index  c ^ (((c >> 6) & 3) << 3)
// (index bits b4 b3 are XORed with b7 b6; 8-coefficient groups stay contiguous and 16-byte aligned).
constexpr int kScratchU16 = 256;
__device__ __forceinline__ int sidx(int c) { return c ^ (((c >> 6) & 3) << 3); }
__device__ __forceinline__ int idxA(int lane, int r) { return lane + 32 * r; }
__device__ __forceinline__ int idxB(int lane, int r) { return ((lane >> 2) << 5) | (r << 2) | (lane & 3); }
__device__ __forceinline__ int idxC(int lane, int r) { return 8 * lane + r; }

// Per-lane twiddles for the passes whose zeta depends on the lane.
struct LaneTwiddles {
    uint2 z16;    // len 16: block = lane >> 2                 (layout B)
    uint2 z8[2];  // len 8 : block = 2 (lane >> 2) + (r >> 2)
    uint2 z4[4];  // len 4 : block = 4 (lane >> 2) + (r >> 1)
    uint2 z2[2];  // len 2 : block = 2 lane + (r >> 2)         (layout C)
};
// Forward: block `blk` of the layer with n blocks uses zeta[n + blk] (ml_kem.c:296-308, i counts up from 1).
template <bool FMA = false>
__device__ __forceinline__ uint2 lane_z(int i) { return FMA ? lane_zeta32(i) : lane_zeta(i); }
template <bool FMA = false>
__device__ __forceinline__ uint2 uniform_z(int i) { return FMA ? c_tw.zeta32[i] : c_tw.zeta[i]; }
template <bool FMA = false>
__device__ __forceinline__ void load_lane_twiddles(LaneTwiddles &t, int lane) {
    int g = lane >> 2;
    t.z16 = lane_z<FMA>(8 + g);
#pragma unroll
    for (int i = 0; i < 2; i++) t.z8[i] = lane_z<FMA>(16 + 2 * g + i);
#pragma unroll
    for (int i = 0; i < 4; i++) t.z4[i] = lane_z<FMA>(32 + 4 * g + i);
#pragma unroll
    for (int i = 0; i < 2; i++) t.z2[i] = lane_z<FMA>(64 + 2 * lane + i);
}
// Inverse: block `blk` of the layer with n blocks uses zeta[2n - 1 - blk] (ml_kem.c:345-357, i counts down from 127).
template <bool FMA = false>
__device__ __forceinline__ void load_lane_twiddles_inv(LaneTwiddles &t, int lane) {
    int g = lane >> 2;
    t.z16 = lane_z<FMA>(15 - g);
#pragma unroll
    for (int i = 0; i < 2; i++) t.z8[i] = lane_z<FMA>(31 - (2 * g + i));
#pragma unroll
    for (int i = 0; i < 4; i++) t.z4[i] = lane_z<FMA>(63 - (4 * g + i));
#pragma unroll
    for (int i = 0; i < 2; i++) t.z2[i] = lane_z<FMA>(127 - (2 * lane + i));
}

// Transposes between layouts through the swizzled scratch.  Values must be < 2^16.
__device__ __forceinline__ void store_scratch_A(const uint32_t x[8], uint16_t *s, int lane) {
#pragma unroll
    for (int r = 0; r < 8; r++) s[sidx(idxA(lane, r))] = (uint16_t)x[r];
}
__device__ __forceinline__ void load_scratch_A(uint32_t x[8], const uint16_t *s, int lane) {
#pragma unroll
    for (int r = 0; r < 8; r++) x[r] = s[sidx(idxA(lane, r))];
}
__device__ __forceinline__ void store_scratch_B(const uint32_t x[8], uint16_t *s, int lane) {
#pragma unroll
    for (int r = 0; r < 8; r++) s[sidx(idxB(lane, r))] = (uint16_t)x[r];
}
__device__ __forceinline__ void load_scratch_B(uint32_t x[8], const uint16_t *s, int lane) {
#pragma unroll
    for (int r = 0; r < 8; r++) x[r] = s[sidx(idxB(lane, r))];
}
// Layout C is one 16-byte vector per lane (8 consecutive coefficients).
__device__ __forceinline__ uint4 pack_pairs(const uint32_t x[8]) {
    return make_uint4(x[0] + x[1] * 65536u, x[2] + x[3] * 65536u, x[4] + x[5] * 65536u, x[6] + x[7] * 65536u);  // IMAD, fma pipe
}
__device__ __forceinline__ void unpack_pairs(uint4 v, uint32_t x[8]) {
    x[0] = v.x & 0xFFFFu; x[1] = v.x >> 16; x[2] = v.y & 0xFFFFu; x[3] = v.y >> 16;
    x[4] = v.z & 0xFFFFu; x[5] = v.z >> 16; x[6] = v.w & 0xFFFFu; x[7] = v.w >> 16;
}
__device__ __forceinline__ void store_scratch_C(const uint32_t x[8], uint16_t *s, int lane) {
    *reinterpret_cast<uint4 *>(s + sidx(8 * lane)) = pack_pairs(x);
}
__device__ __forceinline__ void load_scratch_C(uint32_t x[8], const uint16_t *s, int lane) {
    unpack_pairs(*reinterpret_cast<const uint4 *>(s + sidx(8 * lane)), x);
}

// Cooley-Tukey butterfly, lazy: inputs < 2^16 - 2q, outputs grow by at most 2q.
template <bool FMA = false>
__device__ __forceinline__ void ct_bfly(uint32_t &a, uint32_t &b, uint2 z) {
    uint32_t t = mulz<FMA>(b, z);
    b = a - t + 2 * kQ;
    a = a + t;
}

// ml_kem.c:287 NTT.  x in layout A with values < 4096 (values >= q are treated as residues here; callers that can see
// such values -- the stand-alone k_ntt_batch -- switch to ntt_warp_exact, which reproduces the reference).  Returns the
// transform in layout C, canonical.  `scratch` = this warp's 512-byte scratch; tw from load_lane_twiddles<FMA>.
template <bool FMA = false>
__device__ __forceinline__ void ntt_warp(uint32_t x[8], uint16_t *scratch, int lane, const LaneTwiddles &tw) {
    // pass A -- len = 128, 64, 32: register index bits 2, 1, 0
#pragma unroll
    for (int r = 0; r < 4; r++) ct_bfly<FMA>(x[r], x[r + 4], uniform_z<FMA>(1));
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], uniform_z<FMA>(2 + h));
#pragma unroll
    for (int h = 0; h < 4; h++) ct_bfly<FMA>(x[2 * h], x[2 * h + 1], uniform_z<FMA>(4 + h));
    store_scratch_A(x, scratch, lane);  // values < 4096 + 6q < 2^16
    __syncwarp();
    load_scratch_B(x, scratch, lane);
    __syncwarp();
    // pass B -- len = 16, 8, 4
#pragma unroll
    for (int r = 0; r < 4; r++) ct_bfly<FMA>(x[r], x[r + 4], tw.z16);
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], tw.z8[h]);
#pragma unroll
    for (int h = 0; h < 4; h++) ct_bfly<FMA>(x[2 * h], x[2 * h + 1], tw.z4[h]);
    store_scratch_B(x, scratch, lane);  // values < 4096 + 12q < 2^16
    __syncwarp();
    load_scratch_C(x, scratch, lane);
    __syncwarp();
    // pass C -- len = 2: coefficient pairs (i, i + 2) inside each group of four
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], tw.z2[h]);
#pragma unroll
    for (int r = 0; r < 8; r++) x[r] = FMA ? canon_fma(x[r]) : canon16(x[r]);  // < 4096 + 14q < 2^16
}

// ml_kem.c:309-320 restated literally, for polynomials that contain coefficients in [q, 4096).  The reference's update
//     t = zeta f[j+len] % q;   f[j+len] = f[j] >= t ? f[j] - t : q - (t - f[j]);   f[j] = (f[j] + t) % q
// reduces the sum but not the difference: a 12-bit value >= q in the f[j] role survives as f[j] - t, so some outputs
// are the canonical residue plus q.  Which ones depends on the whole chain of comparisons, hence this separate path,
// taken (warp-uniformly) only when such an input is present -- never on the KEM path, whose NTT inputs are CBD samples
// and Decompress outputs, all < q.
__device__ __forceinline__ void ct_bfly_exact(uint32_t &a, uint32_t &b, uint2 z) {
    const uint32_t t = csubq(mul_shoup(b, z)), lo = a;  // b < 4096
    b = lo >= t ? lo - t : kQ - (t - lo);
    a = canon16(lo + t);                                // lo + t < 4096 + q
}
__device__ __forceinline__ void ntt_warp_exact(uint32_t x[8], uint16_t *scratch, int lane) {
    LaneTwiddles tw;
    load_lane_twiddles<false>(tw, lane);
#pragma unroll
    for (int r = 0; r < 4; r++) ct_bfly_exact(x[r], x[r + 4], uniform_z<false>(1));
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly_exact(x[4 * h + r], x[4 * h + r + 2], uniform_z<false>(2 + h));
#pragma unroll
    for (int h = 0; h < 4; h++) ct_bfly_exact(x[2 * h], x[2 * h + 1], uniform_z<false>(4 + h));
    store_scratch_A(x, scratch, lane);
    __syncwarp();
    load_scratch_B(x, scratch, lane);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 4; r++) ct_bfly_exact(x[r], x[r + 4], tw.z16);
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly_exact(x[4 * h + r], x[4 * h + r + 2], tw.z8[h]);
#pragma unroll
    for (int h = 0; h < 4; h++) ct_bfly_exact(x[2 * h], x[2 * h + 1], tw.z4[h]);
    store_scratch_B(x, scratch, lane);
    __syncwarp();
    load_scratch_C(x, scratch, lane);
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) ct_bfly_exact(x[4 * h + r], x[4 * h + r + 2], tw.z2[h]);
}

// Gentleman-Sande butterfly for the inverse transform (ml_kem.c:359-373): a' = a + b, b' = zeta (b - a).
// `bias` is a multiple of q not smaller than the bound of a.
template <bool FMA = false>
__device__ __forceinline__ void gs_bfly(uint32_t &a, uint32_t &b, uint2 z, uint32_t bias) {
    uint32_t t = a;
    a = t + b;
    b = mulz<FMA>(b - t + bias, z);
}

// ml_kem.c:336 InverseNTT including the final multiplication by 3303 (:378-381).
// x in layout C; returns layout A.  tw from load_lane_twiddles_inv<FMA>.
//   balanced form: inputs < 4096, output canonical.
//   FMA form:      inputs < 8192 (so the lazily reduced sums of the base-case products, < 2q, can be fed directly);
//                  output canonical when CANON, else in [0, 2q) for a consumer that reduces anyway.
template <bool FMA = false, bool CANON = true>
__device__ __forceinline__ void intt_warp(uint32_t x[8], uint16_t *scratch, int lane, const LaneTwiddles &tw) {
    // pass C -- len = 2.  inputs < 4096 <= 2q (FMA: < 8192 <= 3q): sums < 8192 (16384), products < 2q
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) gs_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], tw.z2[h], (FMA ? 3 : 2) * kQ);
    store_scratch_C(x, scratch, lane);
    __syncwarp();
    load_scratch_B(x, scratch, lane);
    __syncwarp();
    // pass B -- len = 4: inputs < 8192 (16384), sums < 16384 (16384 + 2q < 2^16); the bias must be a multiple of q
    // >= 8191 (16383): 3q (5q)
#pragma unroll
    for (int h = 0; h < 4; h++) {
        gs_bfly<FMA>(x[2 * h], x[2 * h + 1], tw.z4[h], (FMA ? 5 : 3) * kQ);
        x[2 * h] = FMA ? barrett32(x[2 * h]) : barrett16(x[2 * h]);  // <= q (FMA: < 2q), keeps the later sums below 2^16
    }
    // len = 8: inputs < 2q: sums < 4q, bias 2q
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) gs_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], tw.z8[h], 2 * kQ);
    // len = 16: inputs < 4q: sums < 8q, bias 4q
#pragma unroll
    for (int r = 0; r < 4; r++) gs_bfly<FMA>(x[r], x[r + 4], tw.z16, 4 * kQ);
    store_scratch_B(x, scratch, lane);  // < 8q = 26632
    __syncwarp();
    load_scratch_A(x, scratch, lane);
    __syncwarp();
    // pass A -- len = 32: inputs < 8q: sums < 16q = 53264 < 2^16, bias 8q; reduce the sums
#pragma unroll
    for (int h = 0; h < 4; h++) {
        gs_bfly<FMA>(x[2 * h], x[2 * h + 1], uniform_z<FMA>(7 - h), 8 * kQ);
        x[2 * h] = FMA ? barrett32(x[2 * h]) : barrett16(x[2 * h]);
    }
    // len = 64: inputs < 2q: sums < 4q, bias 2q
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
        for (int r = 0; r < 2; r++) gs_bfly<FMA>(x[4 * h + r], x[4 * h + r + 2], uniform_z<FMA>(3 - h), 2 * kQ);
    // len = 128 with the 128^-1 scaling folded in: a' = 3303 (a + b), b' = 3303 zeta (b - a); inputs < 4q
    const uint2 zs = FMA ? c_tw.zeta_inv_last32[1] : c_tw.zeta_inv_last[1], zl = FMA ? c_tw.zeta_inv_last32[0] : c_tw.zeta_inv_last[0];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        uint32_t t = x[r];
        x[r] = mulz<FMA>(t + x[r + 4], zs);
        x[r + 4] = mulz<FMA>(x[r + 4] - t + 4 * kQ, zl);
        if (CANON) {
            x[r] = csubq(x[r]);
            x[r + 4] = csubq(x[r + 4]);
        }
    }
}

// ml_kem.c:395 BaseCaseMultiply + :415 MultiplyNTTs + :618 VectorMultiply, accumulated lazily.
// (a0 + a1 X)(b0 + b1 X) mod (X^2 - gamma) added into (acc0, acc1); operands may be any 12-bit value
// (D4: ByteDecode12 does not reduce), each term is < 3 * 4096^2 so four terms fit 32 bits.
__device__ __forceinline__ void basemul_acc(uint32_t &acc0, uint32_t &acc1, uint32_t a0, uint32_t a1, uint32_t b0,
                                            uint32_t b1, uint2 gamma) {
    uint32_t a1g = mul_shoup_fma(a1, gamma.x, gamma.y);  // gamma = {w, floor(w 2^32 / q)} from the gamma32 table; < 2q
    acc0 += a0 * b0 + a1g * b1;
    acc1 += a0 * b1 + a1 * b0;
}

// ------------------------------------------------------------------------------------------------
// Bit packing.  ByteEncode_d / ByteDecode_d (ml_kem.c:125,153) are little-endian bit strings:
// coefficient i occupies bits [d i, d i + d).  A lane that owns 8 consecutive coefficients therefore
// owns exactly d consecutive bytes.
// ------------------------------------------------------------------------------------------------
// Pack 8 d-bit values into d bytes at `dst` (shared memory; dst = row + d * lane, so it is 2-byte aligned for even d
// and 4-byte aligned for d = 4, 12).  The packed words are built with multiply-adds (the fields are disjoint, so
// + is |) to keep the work on the fma pipe.
template <int D>
__device__ __forceinline__ void pack8(const uint32_t v[8], uint8_t *dst) {
    constexpr int NW = (8 * D + 31) / 32;
    uint32_t w[NW];
#pragma unroll
    for (int k = 0; k < NW; k++) {
        uint32_t acc = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int off = D * i - 32 * k;  // bit offset of field i relative to word k
            if (off >= 0 && off < 32) acc += v[i] * (1u << off);
            else if (off < 0 && off + D > 0) acc += v[i] >> (-off);
        }
        w[k] = acc;
    }
    if (D % 4 == 0) {  // d = 4, 12: whole words
#pragma unroll
        for (int k = 0; k < NW; k++) reinterpret_cast<uint32_t *>(dst)[k] = w[k];
    } else if (D % 2 == 0) {  // d = 10: five half-words
#pragma unroll
        for (int h = 0; h < D / 2; h++) reinterpret_cast<uint16_t *>(dst)[h] = (uint16_t)(w[h >> 1] >> (16 * (h & 1)));
    } else {
#pragma unroll
        for (int b8 = 0; b8 < D; b8++) dst[b8] = (uint8_t)(w[b8 >> 2] >> (8 * (b8 & 3)));
    }
}
// Unpack the 8 d-bit values owned by `lane` (bits [8 d lane, 8 d lane + 8 d) of the row) from a packed row
// in shared memory.  `row` must be 4-byte aligned and readable up to 4 bytes past its end.
template <int D>
__device__ __forceinline__ void unpack8(const uint8_t *row, int lane, uint32_t v[8]) {
    const uint32_t *w = reinterpret_cast<const uint32_t *>(row);
    const int bit = 8 * D * lane, wi = bit >> 5, s = bit & 31;
    constexpr int NA = (8 * D + 31) / 32;  // aligned words holding the lane's 8 d bits
    uint32_t raw[NA + 1], a[NA + 1];
#pragma unroll
    for (int k = 0; k <= NA; k++) raw[k] = ((8 * D) % 32 == 0 && k == NA) ? 0u : w[wi + k];  // s == 0 when 8d is a word multiple
#pragma unroll
    for (int k = 0; k < NA; k++) a[k] = ((8 * D) % 32 == 0) ? raw[k] : __funnelshift_r(raw[k], raw[k + 1], s);
    a[NA] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int o = D * i, k = o >> 5, sh = o & 31;
        uint32_t f = (sh + D <= 32) ? (a[k] >> sh) : __funnelshift_r(a[k], a[k + 1], sh);
        v[i] = f & ((1u << D) - 1u);
    }
}

// Extract the d-bit value of coefficient c from a little-endian packed byte string (shared or global).
template <int D>
__device__ __forceinline__ uint32_t unpack1(const uint8_t *src, int c) {
    if (D == 1) return (src[c >> 3] >> (c & 7)) & 1u;
    if (D == 4) return (src[c >> 1] >> ((c & 1) * 4)) & 15u;
    const int bit = D * c, byte = bit >> 3, sh = bit & 7;
    uint32_t w = (uint32_t)src[byte];
    if (sh + D > 8) w |= (uint32_t)src[byte + 1] << 8;  // never reads past the last byte of the string
    if (D > 9 && sh + D > 16) w |= (uint32_t)src[byte + 2] << 16;
    return (w >> sh) & ((1u << D) - 1u);
}

// x >> S as a multiply-high (IMAD.HI, fma pipe) -- inline PTX so that the compiler does not turn it back into a shift.
template <int S>
__device__ __forceinline__ uint32_t shr_fma(uint32_t x) {
    return mulhi(x, 1u << (32 - S));
}
// Nibble j of w, given sel = nibble_weight(j).
#ifndef MLKEM_B200_NIBBLE_ALU  // multiply + multiply-high with sel = 1 << (28 - 4 j): nothing on the alu pipe (measured: k_noise
                               // 1.551 vs 1.574 ms, k_encrypt_v 0.951 vs 0.977 ms per 2^20 items against the shift + mask form)
__device__ __forceinline__ uint32_t nibble_fma(uint32_t w, uint32_t sel) { return shr_fma<28>(w * sel); }
__device__ __forceinline__ uint32_t nibble_weight(int j) { return 1u << (28 - 4 * j); }
#else  // shift + mask with sel = 4 j
__device__ __forceinline__ uint32_t nibble_fma(uint32_t w, uint32_t sel) { return (w >> sel) & 15u; }
__device__ __forceinline__ uint32_t nibble_weight(int j) { return 4 * j; }
#endif

// Noise polynomials travel between kernels as 4-bit codes (coefficient + 3), 8 per 32-bit word.
__device__ __forceinline__ uint32_t noise_code_to_coeff(uint32_t code) {  // code in 0..6 -> canonical
    return csubq(code + (kQ - 3));
}
// (x + e) mod q for canonical x and the noise coefficient e given by its code: one 3-input add, two min-subtracts.
__device__ __forceinline__ uint32_t add_noise_code(uint32_t x, uint32_t code) {
    return csubq(csubq(x + code + (kQ - 3)));  // x + code + q - 3 < 2q + 3
}

}  // namespace mlkem
