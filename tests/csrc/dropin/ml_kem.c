/*
 * tests/csrc/dropin/ml_kem.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Stands in for the reference's ml_kem.c when oracle/ref_shim.c is built against libmlkem_b200.so (Makefile target
 * `dropin` -> build/libref_dropin.so).  ref_shim.c `#include`s "ml_kem.c" and so finds this file through
 * -Itests/csrc/dropin; everything it calls then resolves to the drop-in API of include/ml_kem.h and include/sha3.h,
 * except seven functions that are internal to the reference (static in its ml_kem.c) and that the drop-in does not
 * export: PolyAddition, PolySubtraction, VectorMultiply, H, G, J and PRF.
 *
 * Those seven are defined below, static, so that none of them is exported from or shadows anything in the library.
 * They are NOT part of the drop-in.  Each converts the reference's 4-byte cells to dense values, calls the batched
 * entry point of include/mlkem_b200.h that reproduces the reference function, and returns malloc'ed cells (upper
 * bits zero) as the reference does.  The hashes follow the reference's parameters: H = SHA3-256, G = SHA3-512,
 * J = SHAKE128 with 256 output bits (SURVEY D2), PRF_eta(s, b) = SHAKE128(s || b) with 512 eta output bits (D1).
 */
#include "ml_kem.h"
#include "mlkem_b200.h"

#include <stdint.h>

static uint16_t *dropin_coeffs(const union integer *f, size_t n) {
    uint16_t *o = malloc(sizeof(uint16_t) * n);
    for (size_t i = 0; i < n; i++) o[i] = (uint16_t)f[i].t;
    return o;
}
static union integer *dropin_cells_of_coeffs(const uint16_t *f, size_t n) {
    union integer *o = calloc(n, sizeof(union integer));
    for (size_t i = 0; i < n; i++) o[i].t = f[i];
    return o;
}
static union byte *dropin_cells_of_bytes(const uint8_t *b, size_t n) {
    union byte *o = calloc(n, sizeof(union byte));
    for (size_t i = 0; i < n; i++) o[i].e = b[i];
    return o;
}

/* ml_kem.c:580 / :599: one polynomial through mlkem_b200_poly_add_batch / mlkem_b200_poly_sub_batch. */
static union integer *dropin_poly_op(const union integer *u, const union integer *v, int sub) {
    uint16_t *a = dropin_coeffs(u, N), *b = dropin_coeffs(v, N), z[N];
    int rc = sub ? mlkem_b200_poly_sub_batch(1, a, b, z, NULL) : mlkem_b200_poly_add_batch(1, a, b, z, NULL);
    free(a);
    free(b);
    return rc ? NULL : dropin_cells_of_coeffs(z, N);
}
static union integer *PolyAddition(const union integer *u, const union integer *v) { return dropin_poly_op(u, v, 0); }
static union integer *PolySubtraction(const union integer *u, const union integer *v) { return dropin_poly_op(u, v, 1); }

/* ml_kem.c:618: k polynomials each, given as k pointers, through mlkem_b200_vector_multiply_batch. */
static union integer *VectorMultiply(union integer **u, union integer **v, unsigned int k) {
    uint16_t *a = malloc(sizeof(uint16_t) * N * (k ? k : 1)), *b = malloc(sizeof(uint16_t) * N * (k ? k : 1)), w[N];
    for (unsigned i = 0; i < k; i++)
        for (unsigned j = 0; j < N; j++) {
            a[N * i + j] = (uint16_t)u[i][j].t;
            b[N * i + j] = (uint16_t)v[i][j].t;
        }
    int rc = mlkem_b200_vector_multiply_batch((int)k, 1, a, b, w, NULL);
    free(a);
    free(b);
    return rc ? NULL : dropin_cells_of_coeffs(w, N);
}

/* One sponge of the reference's sha3_b (sha3.c:408) on len whole bytes, through mlkem_b200_sha3_bits_batch. */
static union byte *dropin_sponge(const uint8_t *msg, size_t len, int xof, unsigned c, size_t d_bits) {
    static const uint8_t hash_sfx[4] = {0, 1, 0, 0}, xof_sfx[4] = {1, 1, 1, 1};
    uint8_t *out = malloc(d_bits / 8);
    int rc = mlkem_b200_sha3_bits_batch(1, msg, 8 * len, xof ? xof_sfx : hash_sfx, c, d_bits, out, NULL);
    union byte *o = rc ? NULL : dropin_cells_of_bytes(out, d_bits / 8);
    free(out);
    return o;
}
static union byte *dropin_hash(const union byte *in, unsigned int len, int xof, unsigned c, size_t d_bits) {
    uint8_t *msg = malloc(len + 1u);
    for (unsigned i = 0; i < len; i++) msg[i] = (uint8_t)in[i].e;
    union byte *o = dropin_sponge(msg, len, xof, c, d_bits);
    free(msg);
    return o;
}
static union byte *H(const union byte *in, unsigned int len) { return dropin_hash(in, len, 0, 512, 256); }   /* ml_kem.c:521 */
static union byte *G(const union byte *in, unsigned int len) { return dropin_hash(in, len, 0, 1024, 512); }  /* ml_kem.c:559 */
static union byte *J(const union byte *in, unsigned int len) { return dropin_hash(in, len, 1, 256, 256); }    /* ml_kem.c:540 */
/* ml_kem.c:496 */
static union byte *PRF(const union byte *s, union byte b, unsigned int eta) {
    uint8_t msg[33];
    for (unsigned i = 0; i < 32; i++) msg[i] = (uint8_t)s[i].e;
    msg[32] = (uint8_t)b.e;
    return dropin_sponge(msg, 33, 1, 256, 512 * (size_t)eta);
}
