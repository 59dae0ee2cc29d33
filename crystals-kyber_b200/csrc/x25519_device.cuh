// x25519_device.cuh -- X25519 (RFC 7748) for one item per thread: field arithmetic mod p = 2^255 - 19 and the Montgomery ladder.
//
// Representation: 10 unsigned limbs of 26, 25, 26, 25, ... bits (radix 2^25.5), limb i at bit offset ceil(25.5 i), products
// accumulated in 64 bits (IMAD.WIDE.U32).  Every function is plain C++ on 32 / 64-bit integers, so the same code also builds
// for the host (X25519_HD), where tests/csrc/x25519_contracts.cu and a CPU build can check it.
//
// Limb bounds (T_i = 2^26 for even i, 2^25 for odd i; "tight" and "loose" are the two states a value is in):
//   tight  limb_i < T_i for i != 1, limb_1 < 2^25 + 2^18          -- what fe_mul / fe_sq / fe_mul121665 / fe_carry return
//   loose  limb_i < 3 T_i + 2^18                                   -- what fe_add / fe_sub of two tight values return
// fe_mul / fe_sq / fe_mul121665 accept loose inputs: 19 * (3 * 2^26 + 2^18) < 2^32 keeps the pre-multiplied limbs in 32 bits, and
// a product column is at most 10 terms of 2^27.6 * 2^31.9 < 2^62.8 -- no 64-bit accumulator overflows.
//
// Constant flow: nothing below branches on, loops a data-dependent number of times over, or indexes memory with a value
// derived from the scalar or the point.  The ladder runs exactly 255 steps, the swap is a mask (fe_cswap), the inversion is a
// fixed addition chain and the all-zero test is arithmetic.  Everything is forced inline: no call frames, no local memory.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define X25519_HD __host__ __device__ __forceinline__
#else
#define X25519_HD inline
#endif

namespace x25519 {

struct fe {
    uint32_t v[10];
};

constexpr uint32_t kMask26 = (1u << 26) - 1, kMask25 = (1u << 25) - 1;
X25519_HD constexpr int limb_bits(int i) { return (i & 1) ? 25 : 26; }

// 64-bit columns -> tight limbs.  Input: c[i] < 2^63 (each column of fe_mul / fe_sq / fe_mul121665).  The carry out of limb 9 has
// weight 2^255 = 19 mod p; after it, limb 0 is carried once more, which leaves limb 1 up to 2^18 above 2^25.
X25519_HD fe fe_carry_wide(uint64_t c[10]) {
#pragma unroll
    for (int i = 0; i < 9; i++) {
        c[i + 1] += c[i] >> limb_bits(i);
        c[i] &= (i & 1) ? kMask25 : kMask26;
    }
    c[0] += 19 * (c[9] >> 25);  // c[9] < 2^63.7: the carry is < 2^38.7, times 19 < 2^43
    c[9] &= kMask25;
    c[1] += c[0] >> 26;  // < 2^17
    c[0] &= kMask26;
    fe r;
#pragma unroll
    for (int i = 0; i < 10; i++) r.v[i] = (uint32_t)c[i];
    return r;
}

// loose (or tight) -> tight.
X25519_HD fe fe_carry(const fe &a) {
    uint64_t c[10];
#pragma unroll
    for (int i = 0; i < 10; i++) c[i] = a.v[i];
    return fe_carry_wide(c);
}

// a + b, no carry.  Inputs tight, output loose.
X25519_HD fe fe_add(const fe &a, const fe &b) {
    fe r;
#pragma unroll
    for (int i = 0; i < 10; i++) r.v[i] = a.v[i] + b.v[i];
    return r;
}

// a - b + 2p, no carry.  Inputs tight (b_i <= 2p_i limb by limb: 2p_1 = 2^26 - 2 > 2^25 + 2^18), output loose.
X25519_HD fe fe_sub(const fe &a, const fe &b) {
    fe r;
#pragma unroll
    for (int i = 0; i < 10; i++) {
        const uint32_t two_p = i == 0 ? 2 * (kMask26 - 18) : (i & 1) ? 2 * kMask25 : 2 * kMask26;
        r.v[i] = a.v[i] + two_p - b.v[i];
    }
    return r;
}

// a * b mod p.  Inputs loose, output tight.  Limb i times limb j lands in column i + j; a product of two odd limbs carries a
// factor 2 (ceil(25.5 i) + ceil(25.5 j) = ceil(25.5 (i + j)) + 1), and column i + j >= 10 wraps to i + j - 10 times 19.
X25519_HD fe fe_mul(const fe &a, const fe &b) {
    uint32_t b19[10], a2[10];
#pragma unroll
    for (int i = 0; i < 10; i++) {
        b19[i] = 19 * b.v[i];                        // < 2^31.9
        a2[i] = (i & 1) ? 2 * a.v[i] : a.v[i];       // < 2^27
    }
    uint64_t c[10];
#pragma unroll
    for (int k = 0; k < 10; k++) c[k] = 0;
#pragma unroll
    for (int i = 0; i < 10; i++) {
#pragma unroll
        for (int j = 0; j < 10; j++) {
            const uint32_t x = ((i & 1) && (j & 1)) ? a2[i] : a.v[i];
            const uint32_t y = (i + j >= 10) ? b19[j] : b.v[j];
            c[(i + j) % 10] += (uint64_t)x * y;
        }
    }
    return fe_carry_wide(c);
}

// a^2 mod p.  Input loose, output tight.  The 55 products i <= j of fe_mul's table; a cross term (i < j) counts twice.
// The doubled operand is a_i << s, s <= 2: < 2^28.6; a column has at most 6 terms of < 2^28.6 * 2^31.9, below 2^63.
X25519_HD fe fe_sq(const fe &a) {
    uint32_t a19[10];
#pragma unroll
    for (int i = 0; i < 10; i++) a19[i] = 19 * a.v[i];
    uint64_t c[10];
#pragma unroll
    for (int k = 0; k < 10; k++) c[k] = 0;
#pragma unroll
    for (int i = 0; i < 10; i++) {
#pragma unroll
        for (int j = i; j < 10; j++) {
            const int s = (i < j ? 1 : 0) + (((i & j) & 1) ? 1 : 0);
            const uint32_t x = a.v[i] << s;
            const uint32_t y = (i + j >= 10) ? a19[j] : a.v[j];
            c[(i + j) % 10] += (uint64_t)x * y;
        }
    }
    return fe_carry_wide(c);
}

// a * 121665 mod p (a24 = (486662 - 2) / 4, RFC 7748 section 5).  Input loose (< 2^27.6: the product is < 2^44.5), output tight.
X25519_HD fe fe_mul121665(const fe &a) {
    uint64_t c[10];
#pragma unroll
    for (int i = 0; i < 10; i++) c[i] = (uint64_t)a.v[i] * 121665u;
    return fe_carry_wide(c);
}

// Conditional swap of a and b when swap == 1 (swap in {0, 1}): by mask, never by branch.
X25519_HD void fe_cswap(fe &a, fe &b, uint32_t swap) {
    const uint32_t m = 0u - swap;
#pragma unroll
    for (int i = 0; i < 10; i++) {
        const uint32_t t = m & (a.v[i] ^ b.v[i]);
        a.v[i] ^= t;
        b.v[i] ^= t;
    }
}

// Decoding of a u-coordinate (RFC 7748 section 5): 32 little-endian bytes as 8 words, bit 255 cleared; values in [p, 2^255) are
// accepted as they are (the arithmetic is mod p).  Output: limb_i < T_i (tight).
X25519_HD fe fe_from_words(const uint32_t w[8]) {
    const uint32_t w7 = w[7] & 0x7FFFFFFFu;
    fe r;
    r.v[0] = w[0] & kMask26;
    r.v[1] = ((w[0] >> 26) | (w[1] << 6)) & kMask25;
    r.v[2] = ((w[1] >> 19) | (w[2] << 13)) & kMask26;
    r.v[3] = ((w[2] >> 13) | (w[3] << 19)) & kMask25;
    r.v[4] = (w[3] >> 6) & kMask26;
    r.v[5] = w[4] & kMask25;
    r.v[6] = ((w[4] >> 25) | (w[5] << 7)) & kMask26;
    r.v[7] = ((w[5] >> 19) | (w[6] << 13)) & kMask25;
    r.v[8] = ((w[6] >> 12) | (w7 << 20)) & kMask26;
    r.v[9] = (w7 >> 6) & kMask25;
    return r;
}

// The canonical value in [0, p) as 8 little-endian words.  Input loose.  Two carry passes leave every limb below T_i (the
// second pass can only add 1 to limb 1 when the first left it >= 2^25, i.e. when its low 25 bits are < 2^18), so the value is
// v < 2^255; q = floor((v + 19) / 2^255) is 1 exactly when v >= p, and v + 19 q with bit 255 dropped is v - q p.
X25519_HD void fe_freeze(const fe &a, uint32_t out[8]) {
    fe h = fe_carry(fe_carry(a));
    uint32_t q = (h.v[0] + 19) >> 26;
#pragma unroll
    for (int i = 1; i < 10; i++) q = (h.v[i] + q) >> limb_bits(i);
    h.v[0] += 19 * q;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        h.v[i + 1] += h.v[i] >> limb_bits(i);
        h.v[i] &= (i & 1) ? kMask25 : kMask26;
    }
    h.v[9] &= kMask25;
    out[0] = h.v[0] | (h.v[1] << 26);
    out[1] = (h.v[1] >> 6) | (h.v[2] << 19);
    out[2] = (h.v[2] >> 13) | (h.v[3] << 13);
    out[3] = (h.v[3] >> 19) | (h.v[4] << 6);
    out[4] = h.v[5] | (h.v[6] << 25);
    out[5] = (h.v[6] >> 7) | (h.v[7] << 19);
    out[6] = (h.v[7] >> 13) | (h.v[8] << 12);
    out[7] = (h.v[8] >> 20) | (h.v[9] << 6);
}

// z^(p - 2) = z^(2^255 - 21) by the fixed addition chain of the curve's reference implementations: 254 squarings, 11 products.
// Input loose, output tight.
X25519_HD fe fe_invert(const fe &z) {
    auto sq_n = [](fe t, int n) {
#pragma unroll 1
        for (int i = 0; i < n; i++) t = fe_sq(t);  // n is a constant of the chain, not data
        return t;
    };
    const fe z2 = fe_sq(z);                          // 2
    const fe z9 = fe_mul(sq_n(z2, 2), z);            // 9
    const fe z11 = fe_mul(z9, z2);                   // 11
    const fe z5_0 = fe_mul(fe_sq(z11), z9);          // 2^5 - 1
    const fe z10_0 = fe_mul(sq_n(z5_0, 5), z5_0);    // 2^10 - 1
    const fe z20_0 = fe_mul(sq_n(z10_0, 10), z10_0); // 2^20 - 1
    const fe z40_0 = fe_mul(sq_n(z20_0, 20), z20_0); // 2^40 - 1
    const fe z50_0 = fe_mul(sq_n(z40_0, 10), z10_0); // 2^50 - 1
    const fe z100_0 = fe_mul(sq_n(z50_0, 50), z50_0);   // 2^100 - 1
    const fe z200_0 = fe_mul(sq_n(z100_0, 100), z100_0); // 2^200 - 1
    const fe z250_0 = fe_mul(sq_n(z200_0, 50), z50_0);   // 2^250 - 1
    return fe_mul(sq_n(z250_0, 5), z11);                 // 2^255 - 32 + 11 = p - 2
}

// X25519(k, u) of RFC 7748 section 5: k and u as 8 little-endian words each (k unclamped: clamped here), result in out.
// Returns 1 when the result is all zero (u of small order), else 0 -- computed without a branch.
X25519_HD uint32_t scalarmult(uint32_t out[8], const uint32_t k_in[8], const uint32_t u_in[8]) {
    uint32_t k[8];
#pragma unroll
    for (int i = 0; i < 8; i++) k[i] = k_in[i];
    k[0] &= ~7u;                               // clamping: clear bits 0, 1, 2,
    k[7] = (k[7] & 0x7FFFFFFFu) | 0x40000000u; // clear bit 255, set bit 254
    // bit 254 to the top of k[7]: every step reads the top bit and shifts the 256-bit scalar left by one (a funnel shift per
    // word), so the scalar is never indexed by a loop counter
#pragma unroll
    for (int i = 7; i > 0; i--) k[i] = (k[i] << 1) | (k[i - 1] >> 31);
    k[0] <<= 1;
    const fe x1 = fe_from_words(u_in);
    fe x2 = {{1, 0, 0, 0, 0, 0, 0, 0, 0, 0}}, z2 = {{0}}, x3 = x1, z3 = {{1, 0, 0, 0, 0, 0, 0, 0, 0, 0}};
    uint32_t swap = 0;
#pragma unroll 1
    for (int t = 254; t >= 0; t--) {  // exactly 255 steps
        const uint32_t kt = k[7] >> 31;
#pragma unroll
        for (int i = 7; i > 0; i--) k[i] = (k[i] << 1) | (k[i - 1] >> 31);
        k[0] <<= 1;
        swap ^= kt;
        fe_cswap(x2, x3, swap);
        fe_cswap(z2, z3, swap);
        swap = kt;
        const fe A = fe_add(x2, z2), B = fe_sub(x2, z2), C = fe_add(x3, z3), D = fe_sub(x3, z3);
        const fe AA = fe_sq(A), BB = fe_sq(B), DA = fe_mul(D, A), CB = fe_mul(C, B);
        const fe E = fe_sub(AA, BB);
        x3 = fe_sq(fe_add(DA, CB));
        z3 = fe_mul(x1, fe_sq(fe_sub(DA, CB)));
        x2 = fe_mul(AA, BB);
        z2 = fe_mul(E, fe_add(AA, fe_mul121665(E)));
    }
    fe_cswap(x2, x3, swap);
    fe_cswap(z2, z3, swap);
    fe_freeze(fe_mul(x2, fe_invert(z2)), out);
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc |= out[i];
    return ((acc | (0u - acc)) >> 31) ^ 1u;  // 1 iff acc == 0
}

}  // namespace x25519
