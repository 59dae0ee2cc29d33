// p256_device.cuh -- NIST P-256 (FIPS 186-5, SP 800-186) for one item per thread: field arithmetic mod
// p = 2^256 - 2^224 + 2^192 + 2^96 - 1, the complete projective formulas of Renes, Costello and Batina (2016) for a = -3, a
// Montgomery ladder over them, point decoding with SP 800-56A partial public-key validation, and the scalar range check and
// FIPS 186-5 A.2.1 reduction of the seeded calls.
//
// Representation: a field element is 8 little-endian 32-bit words in the Montgomery domain (x R mod p, R = 2^256), multiplied
// by CIOS with 64-bit products (IMAD.WIDE.U32).  p = -1 mod 2^32, so -p^-1 mod 2^32 = 1 and the reduction factor of each
// round is the low word itself.  Every function is plain C++ on 32 / 64-bit integers, so the same code also builds for the host
// (P256_HD), where tests/csrc/p256_contracts.cu and a CPU build can check it.
//
// Bounds: every field element a function takes or returns is canonical, in [0, p), with three exceptions that take any
// 256-bit value: fe_canon (returns a mod p), fe_mul when the other operand is canonical (a b < p 2^256 is all CIOS needs for a
// result below 2p, which one subtraction brings into [0, p)), and fe_to_mont (fe_mul by R^2 mod p).  Since 2^256 < 2p, one
// masked subtraction of p canonicalises any 256-bit value.
//
// Constant flow: nothing below branches on, loops a data-dependent number of times over, or indexes memory with a value
// derived from a scalar or a point.  The ladder runs exactly 256 steps, the swap is a mask (pt_cswap), the scalar is shifted
// through registers, the inversion is a fixed addition chain, the complete formulas have no exceptional case (the identity and
// P = Q need no branch), and every comparison is a borrow turned into a mask.  Everything is forced inline: no call frames,
// no local memory.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define P256_HD __host__ __device__ __forceinline__
#else
#define P256_HD inline
#endif

namespace p256 {

struct fe {
    uint32_t v[8];  // little-endian words
};

struct pt {
    fe X, Y, Z;  // projective (X : Y : Z), Montgomery-domain coordinates; the identity is (0 : 1 : 0)
};

// p and the group order n, word by word (constant folded wherever a loop is unrolled).
P256_HD constexpr uint32_t p_word(int i) { return i < 3 ? 0xFFFFFFFFu : i < 6 ? 0u : i == 6 ? 1u : 0xFFFFFFFFu; }
P256_HD constexpr uint32_t n_word(int i) {
    return i == 0 ? 0xFC632551u : i == 1 ? 0xF3B9CAC2u : i == 2 ? 0xA7179E84u : i == 3 ? 0xBCE6FAADu : i == 6 ? 0u : 0xFFFFFFFFu;
}

P256_HD fe fe_zero() { return {{0, 0, 0, 0, 0, 0, 0, 0}}; }
P256_HD fe fe_one() { return {{0x00000001u, 0, 0, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFEu, 0}}; }  // R mod p
P256_HD fe fe_r2() { return {{0x00000003u, 0, 0xFFFFFFFFu, 0xFFFFFFFBu, 0xFFFFFFFEu, 0xFFFFFFFFu, 0xFFFFFFFDu, 0x00000004u}}; }  // R^2 mod p
P256_HD fe fe_b() {  // b R mod p
    return {{0x29C4BDDFu, 0xD89CDF62u, 0x78843090u, 0xACF005CDu, 0xF7212ED6u, 0xE5A220ABu, 0x04874834u, 0xDC30061Du}};
}
P256_HD pt base_point() {  // G, Montgomery domain, Z = 1
    return {{{0x18A9143Cu, 0x79E730D4u, 0x5FEDB601u, 0x75BA95FCu, 0x77622510u, 0x79FB732Bu, 0xA53755C6u, 0x18905F76u}},
            {{0xCE95560Au, 0xDDF25357u, 0xBA19E45Cu, 0x8B4AB8E4u, 0xDD21F325u, 0xD2E88688u, 0x25885D85u, 0x8571FF18u}},
            fe_one()};
}

// r = a - m (mod 2^256) where m = mask & p; returns the borrow out of the top word (1 when a < (mask & p)).
P256_HD uint32_t sub_p_masked(fe &r, const fe &a, uint32_t mask) {
    uint64_t br = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint64_t d = (uint64_t)a.v[i] - (p_word(i) & mask) - br;
        r.v[i] = (uint32_t)d;
        br = (d >> 32) & 1;
    }
    return (uint32_t)br;
}

// mask ? b : a, word by word.
P256_HD fe fe_select(const fe &a, const fe &b, uint32_t mask) {
    fe r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = a.v[i] ^ (mask & (a.v[i] ^ b.v[i]));
    return r;
}

// a mod p for any 256-bit a (2^256 < 2p: at most one subtraction).
P256_HD fe fe_canon(const fe &a) {
    fe d;
    const uint32_t br = sub_p_masked(d, a, 0xFFFFFFFFu);
    return fe_select(d, a, 0u - br);  // a < p: keep a
}

// a + b mod p.  Inputs and output in [0, p).
P256_HD fe fe_add(const fe &a, const fe &b) {
    fe s;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)a.v[i] + b.v[i];
        s.v[i] = (uint32_t)c;
        c >>= 32;
    }
    fe d;
    const uint32_t br = sub_p_masked(d, s, 0xFFFFFFFFu);
    // s + 2^256 c >= p  <=>  c == 1 or no borrow; then d (taken mod 2^256) is the sum minus p
    return fe_select(s, d, 0u - ((uint32_t)c | (br ^ 1u)));
}

// a - b mod p.  Inputs and output in [0, p).
P256_HD fe fe_sub(const fe &a, const fe &b) {
    fe d;
    uint64_t br = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint64_t t = (uint64_t)a.v[i] - b.v[i] - br;
        d.v[i] = (uint32_t)t;
        br = (t >> 32) & 1;
    }
    const uint32_t m = 0u - (uint32_t)br;  // borrow: add p back (mod 2^256)
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)d.v[i] + (p_word(i) & m);
        d.v[i] = (uint32_t)c;
        c >>= 32;
    }
    return d;
}

// a b R^-1 mod p (Montgomery product, CIOS).  Requires a b < p 2^256 -- one operand in [0, p), the other any 256-bit value;
// output in [0, p).  Invariant of the rounds: t < a + p < 2^257, so t fits 8 words and a carry bit (t[8]) between rounds and
// the 64-bit column sums t_j + a_j b_i + carry never exceed 2^64 - 1.
P256_HD fe fe_mul(const fe &a, const fe &b) {
    uint32_t t[9];
#pragma unroll
    for (int j = 0; j < 9; j++) t[j] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            c = (uint64_t)a.v[j] * b.v[i] + t[j] + (c >> 32);
            t[j] = (uint32_t)c;
        }
        c = (uint64_t)t[8] + (c >> 32);
        t[8] = (uint32_t)c;
        const uint32_t t9 = (uint32_t)(c >> 32);
        const uint32_t m = t[0];  // t[0] * (-p^-1 mod 2^32), and -p^-1 = 1 mod 2^32
        c = (uint64_t)m * p_word(0) + t[0];
#pragma unroll
        for (int j = 1; j < 8; j++) {
            c = (uint64_t)m * p_word(j) + t[j] + (c >> 32);
            t[j - 1] = (uint32_t)c;
        }
        c = (uint64_t)t[8] + (c >> 32);
        t[7] = (uint32_t)c;
        t[8] = t9 + (uint32_t)(c >> 32);
    }
    fe lo, d;
#pragma unroll
    for (int j = 0; j < 8; j++) lo.v[j] = t[j];
    const uint32_t br = sub_p_masked(d, lo, 0xFFFFFFFFu);
    return fe_select(lo, d, 0u - (t[8] | (br ^ 1u)));
}

// a^2 R^-1 mod p.  Input and output in [0, p).
P256_HD fe fe_sqr(const fe &a) { return fe_mul(a, a); }

// x R mod p for any 256-bit x; x R^-1 mod p (out of the Montgomery domain) for x in [0, p).  Outputs in [0, p).
P256_HD fe fe_to_mont(const fe &x) { return fe_mul(x, fe_r2()); }
P256_HD fe fe_from_mont(const fe &x) { return fe_mul(x, {{1, 0, 0, 0, 0, 0, 0, 0}}); }

// 0xFFFFFFFF when a == b (word by word), else 0.
P256_HD uint32_t fe_eq_mask(const fe &a, const fe &b) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc |= a.v[i] ^ b.v[i];
    return ((acc | (0u - acc)) >> 31) - 1u;
}

// z^(p - 2) = z^-1 (0 for z = 0), Montgomery domain in and out.  p - 2 = 1^32 0^31 1 0^96 1^94 0 1 (most significant bit
// first); x_k below is z^(2^k - 1).  255 squarings and 13 products, whatever z is.  Input and output in [0, p).
P256_HD fe fe_inv(const fe &z) {
    auto sq_n = [](fe t, int n) {
#pragma unroll 1
        for (int i = 0; i < n; i++) t = fe_sqr(t);  // n is a constant of the chain, not data
        return t;
    };
    const fe x2 = fe_mul(fe_sqr(z), z);
    const fe x4 = fe_mul(sq_n(x2, 2), x2);
    const fe x8 = fe_mul(sq_n(x4, 4), x4);
    const fe x16 = fe_mul(sq_n(x8, 8), x8);
    const fe x24 = fe_mul(sq_n(x16, 8), x8);
    const fe x28 = fe_mul(sq_n(x24, 4), x4);
    const fe x30 = fe_mul(sq_n(x28, 2), x2);
    const fe x32 = fe_mul(sq_n(x30, 2), x2);
    fe t = fe_mul(sq_n(x32, 32), z);  // 1^32 0^31 1
    t = sq_n(t, 96);                  // 0^96
    t = fe_mul(sq_n(t, 32), x32);     // 1^32
    t = fe_mul(sq_n(t, 32), x32);     // 1^64
    t = fe_mul(sq_n(t, 30), x30);     // 1^94
    return fe_mul(sq_n(t, 2), z);     // 0 1
}

// P + Q, Renes-Costello-Batina 2016 Algorithm 4 (complete, a = -3): 12 products, 2 products by b, no exceptional case.
P256_HD pt pt_add(const pt &P, const pt &Q) {
    const fe b = fe_b();
    fe t0 = fe_mul(P.X, Q.X), t1 = fe_mul(P.Y, Q.Y), t2 = fe_mul(P.Z, Q.Z);
    fe t3 = fe_mul(fe_add(P.X, P.Y), fe_add(Q.X, Q.Y));
    fe t4 = fe_add(t0, t1);
    t3 = fe_sub(t3, t4);
    t4 = fe_mul(fe_add(P.Y, P.Z), fe_add(Q.Y, Q.Z));
    fe X3 = fe_add(t1, t2);
    t4 = fe_sub(t4, X3);
    X3 = fe_mul(fe_add(P.X, P.Z), fe_add(Q.X, Q.Z));
    fe Y3 = fe_add(t0, t2);
    Y3 = fe_sub(X3, Y3);
    fe Z3 = fe_mul(b, t2);
    X3 = fe_sub(Y3, Z3);
    Z3 = fe_add(X3, X3);
    X3 = fe_add(X3, Z3);
    Z3 = fe_sub(t1, X3);
    X3 = fe_add(t1, X3);
    Y3 = fe_mul(b, Y3);
    t1 = fe_add(t2, t2);
    t2 = fe_add(t1, t2);
    Y3 = fe_sub(Y3, t2);
    Y3 = fe_sub(Y3, t0);
    t1 = fe_add(Y3, Y3);
    Y3 = fe_add(t1, Y3);
    t1 = fe_add(t0, t0);
    t0 = fe_add(t1, t0);
    t0 = fe_sub(t0, t2);
    t1 = fe_mul(t4, Y3);
    t2 = fe_mul(t0, Y3);
    Y3 = fe_mul(X3, Z3);
    Y3 = fe_add(Y3, t2);
    X3 = fe_mul(t3, X3);
    X3 = fe_sub(X3, t1);
    Z3 = fe_mul(t4, Z3);
    t1 = fe_mul(t3, t0);
    Z3 = fe_add(Z3, t1);
    return {X3, Y3, Z3};
}

// 2P, Renes-Costello-Batina 2016 Algorithm 6 (complete, a = -3): 8 products, 3 squarings, 2 products by b.
P256_HD pt pt_dbl(const pt &P) {
    const fe b = fe_b();
    fe t0 = fe_sqr(P.X), t1 = fe_sqr(P.Y), t2 = fe_sqr(P.Z);
    fe t3 = fe_mul(P.X, P.Y);
    t3 = fe_add(t3, t3);
    fe Z3 = fe_mul(P.X, P.Z);
    Z3 = fe_add(Z3, Z3);
    fe Y3 = fe_mul(b, t2);
    Y3 = fe_sub(Y3, Z3);
    fe X3 = fe_add(Y3, Y3);
    Y3 = fe_add(X3, Y3);
    X3 = fe_sub(t1, Y3);
    Y3 = fe_add(t1, Y3);
    Y3 = fe_mul(X3, Y3);
    X3 = fe_mul(X3, t3);
    t3 = fe_add(t2, t2);
    t2 = fe_add(t2, t3);
    Z3 = fe_mul(b, Z3);
    Z3 = fe_sub(Z3, t2);
    Z3 = fe_sub(Z3, t0);
    t3 = fe_add(Z3, Z3);
    Z3 = fe_add(Z3, t3);
    t3 = fe_add(t0, t0);
    t0 = fe_add(t3, t0);
    t0 = fe_sub(t0, t2);
    t0 = fe_mul(t0, Z3);
    Y3 = fe_add(Y3, t0);
    t0 = fe_mul(P.Y, P.Z);
    t0 = fe_add(t0, t0);
    Z3 = fe_mul(t0, Z3);
    X3 = fe_sub(X3, Z3);
    Z3 = fe_mul(t0, t1);
    Z3 = fe_add(Z3, Z3);
    Z3 = fe_add(Z3, Z3);
    return {X3, Y3, Z3};
}

// Conditional swap of P and Q when swap == 1 (swap in {0, 1}): by mask, never by branch.
P256_HD void pt_cswap(pt &P, pt &Q, uint32_t swap) {
    const uint32_t m = 0u - swap;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint32_t t = m & (P.X.v[i] ^ Q.X.v[i]);
        P.X.v[i] ^= t, Q.X.v[i] ^= t;
        t = m & (P.Y.v[i] ^ Q.Y.v[i]);
        P.Y.v[i] ^= t, Q.Y.v[i] ^= t;
        t = m & (P.Z.v[i] ^ Q.Z.v[i]);
        P.Z.v[i] ^= t, Q.Z.v[i] ^= t;
    }
}

// k P for a 256-bit k (8 little-endian words, any value: k = 0 or a multiple of the order gives the identity), by the
// Montgomery ladder over the complete formulas: exactly 256 steps of one addition and one doubling, R1 - R0 = P throughout.
P256_HD pt scalarmult(const uint32_t k_in[8], const pt &P) {
    uint32_t k[8];
#pragma unroll
    for (int i = 0; i < 8; i++) k[i] = k_in[i];
    pt R0 = {fe_zero(), fe_one(), fe_zero()}, R1 = P;
    uint32_t swap = 0;
#pragma unroll 1
    for (int t = 0; t < 256; t++) {  // exactly 256 steps
        // the top bit of k, then k <<= 1 (a funnel shift per word): the scalar is never indexed by the loop counter
        const uint32_t kt = k[7] >> 31;
#pragma unroll
        for (int i = 7; i > 0; i--) k[i] = (k[i] << 1) | (k[i - 1] >> 31);
        k[0] <<= 1;
        swap ^= kt;
        pt_cswap(R0, R1, swap);
        swap = kt;
        R1 = pt_add(R0, R1);
        R0 = pt_dbl(R0);
    }
    pt_cswap(R0, R1, swap);
    return R0;
}

// ---- encodings: big-endian bytes <-> little-endian words ----------------------------------------------------------------
P256_HD uint32_t load_be32(const uint8_t *p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}
P256_HD void store_be32(uint8_t *p, uint32_t w) {
    p[0] = (uint8_t)(w >> 24), p[1] = (uint8_t)(w >> 16), p[2] = (uint8_t)(w >> 8), p[3] = (uint8_t)w;
}
// 32 big-endian bytes -> 8 little-endian words (no reduction).
P256_HD void words_from_be(const uint8_t *in, uint32_t w[8]) {
#pragma unroll
    for (int i = 0; i < 8; i++) w[7 - i] = load_be32(in + 4 * i);
}
P256_HD void words_to_be(const uint32_t w[8], uint8_t *out, uint32_t mask) {
#pragma unroll
    for (int i = 0; i < 8; i++) store_be32(out + 4 * i, w[7 - i] & mask);
}

// 0xFFFFFFFF when the 256-bit a is below the 256-bit bound `word(i)` (a borrow out of a - bound), else 0.
template <class Word>
P256_HD uint32_t lt_mask(const uint32_t a[8], Word word) {
    uint64_t br = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) br = (((uint64_t)a[i] - word(i) - br) >> 32) & 1;
    return 0u - (uint32_t)br;
}

// Scalar range check: 0xFFFFFFFF when 1 <= k <= n - 1, else 0 (k as 8 little-endian words).
P256_HD uint32_t scalar_ok_mask(const uint32_t k[8]) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc |= k[i];
    const uint32_t nz = 0u - ((acc | (0u - acc)) >> 31);
    return nz & lt_mask(k, [](int i) { return n_word(i); });
}

// TLS 1.3 UncompressedPointRepresentation (65 bytes: 0x04 || X || Y, big-endian) -> affine point in the Montgomery domain
// (Z = 1), with SP 800-56A partial public-key validation: returns 0xFFFFFFFF when the prefix is 0x04, X < p, Y < p and
// Y^2 = X^3 - 3X + b mod p, else 0.  The point is decoded the same way whatever the verdict.  (The identity has no 65-byte
// encoding, and with cofactor 1 every other curve point has order n.)
P256_HD uint32_t point_decode(const uint8_t *in, pt &P) {
    uint32_t x[8], y[8];
    words_from_be(in + 1, x);
    words_from_be(in + 33, y);
    const auto pw = [](int i) { return p_word(i); };
    uint32_t ok = lt_mask(x, pw) & lt_mask(y, pw);
    const uint32_t pre = (uint32_t)in[0] ^ 4u;
    ok &= ((pre | (0u - pre)) >> 31) - 1u;
    fe xf, yf;
#pragma unroll
    for (int i = 0; i < 8; i++) xf.v[i] = x[i], yf.v[i] = y[i];
    P.X = fe_to_mont(xf);
    P.Y = fe_to_mont(yf);
    P.Z = fe_one();
    const fe rhs = fe_add(fe_sub(fe_mul(fe_sqr(P.X), P.X), fe_add(P.X, fe_add(P.X, P.X))), fe_b());
    return ok & fe_eq_mask(fe_sqr(P.Y), rhs);
}

// The affine coordinates of P (canonical, out of the Montgomery domain) as little-endian words.  The identity gives (0, 0).
P256_HD void to_affine(const pt &P, uint32_t x[8], uint32_t y[8]) {
    const fe zi = fe_inv(P.Z);
    const fe ax = fe_from_mont(fe_mul(P.X, zi)), ay = fe_from_mont(fe_mul(P.Y, zi));
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = ax.v[i], y[i] = ay.v[i];
}

// 65-byte encoding 0x04 || X || Y of affine (x, y), every byte ANDed with `mask` (0 or 0xFFFFFFFF).
P256_HD void point_encode(const uint32_t x[8], const uint32_t y[8], uint8_t *out, uint32_t mask) {
    out[0] = (uint8_t)(4u & mask);
    words_to_be(x, out + 1, mask);
    words_to_be(y, out + 33, mask);
}

// FIPS 186-5 A.2.1 ("extra random bits"): d = (c mod (n - 1)) + 1 for the 320-bit big-endian c = hi[0..32) || lo[0..8), as 8
// little-endian words.  c = T 2^64 + L: T mod (n - 1) by one masked subtraction (T < 2^256 < 2 (n - 1)), then the 64 bits of L shifted in,
// x = 2 x + bit, each followed by one masked subtraction of n - 1 (x < n - 1 before the step, so 2 x + bit < 2 (n - 1); the
// bit shifted out of the top word takes part in the comparison).  Always 1 <= d <= n - 1.
P256_HD void seed_scalar(const uint8_t *hi, const uint8_t *lo, uint32_t d[8]) {
    const auto nm1 = [](int i) { return i == 0 ? n_word(0) - 1u : n_word(i); };  // n is odd: no borrow out of word 0
    uint32_t x[8];
    words_from_be(hi, x);
    uint64_t L = ((uint64_t)load_be32(lo) << 32) | load_be32(lo + 4);
    auto sub_nm1_masked = [&](uint32_t force) {  // x -= n - 1 when x >= n - 1 or force
        uint32_t r[8];
        uint64_t br = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint64_t t = (uint64_t)x[i] - nm1(i) - br;
            r[i] = (uint32_t)t;
            br = (t >> 32) & 1;
        }
        const uint32_t m = 0u - (force | ((uint32_t)br ^ 1u));
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] ^= m & (x[i] ^ r[i]);
    };
    sub_nm1_masked(0);
#pragma unroll 1
    for (int s = 0; s < 64; s++) {
        const uint32_t top = x[7] >> 31, bit = (uint32_t)(L >> 63);
        L <<= 1;
#pragma unroll
        for (int i = 7; i > 0; i--) x[i] = (x[i] << 1) | (x[i - 1] >> 31);
        x[0] = (x[0] << 1) | bit;
        sub_nm1_masked(top);
    }
    uint64_t c = 1;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += x[i];
        d[i] = (uint32_t)c;
        c >>= 32;
    }
}

}  // namespace p256
