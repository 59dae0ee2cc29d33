/*
 * mlkem_b200.h -- C ABI of the B200-native batched ML-KEM engine (libmlkem_b200.so).
 *
 * This is the drop-in boundary for the hot path of rsjahnige/CRYSTALS-Kyber.  The reference has no
 * plugin / FFI layer: its boundary is the C header ml_kem.h plus the symbols of ml_kem.o.  Two headers
 * therefore describe this library:
 *
 *   include/ml_kem.h      the reference's own API (same unions, structs, enum and prototypes), each call a
 *                         batch of one -- what an existing caller links against unchanged;
 *   include/mlkem_b200.h  (this file) the batched entry points the reference-signature functions are
 *                         built on, dense bytes / uint16 instead of the reference's 4-byte unions.
 *
 * Every function below names the reference function (file:line in /root/reference) whose results it
 * reproduces bit for bit.  All arithmetic runs in CUDA kernels for sm_100a; there is no CPU fallback:
 * without a usable CUDA device every call returns MLKEM_B200_ERR_CUDA.
 *
 * Layout conventions
 *   - byte strings are dense uint8_t, item-major: item i of an array with per-item size S is at base + i*S;
 *   - polynomials are 256 x uint16_t, natural coefficient order, item-major;
 *   - keys and ciphertexts use the byte layouts of ml_kem.c: ek = ByteEncode12(t^)[384k] || rho[32]
 *     (ml_kem.c:736-747), dk = dk_pke[384k] || ek || H(ek)[32] || z[32] (ml_kem.c:1050-1077),
 *     c = c1[32 du k] || c2[32 dv] (ml_kem.c:907-918).
 *
 * Memory spaces (mlkem_b200_opts.mem)
 *   MLKEM_B200_MEM_HOST    pointers are host memory (pinned memory from mlkem_b200_host_alloc gives the
 *                          full PCIe rate).  The call stages chunks through device memory with copies and
 *                          kernels overlapped on several streams and returns when the results are in place.
 *   MLKEM_B200_MEM_DEVICE  pointers are device memory on opts.device, 16-byte aligned.  The call enqueues
 *                          its kernels on opts.stream (NULL = the CUDA default stream) and returns
 *                          without synchronising; the caller orders its own work through that stream.
 *
 * Threads, streams and devices.  Calls may come from several host threads and name different streams or devices: the
 * per-device workspaces are shared, each use is fenced by an event, so calls on different streams never touch each
 * other's intermediates (they serialise on the workspace instead).  A call switches the calling thread's current
 * CUDA device to opts.device only for its own duration.
 */
#ifndef MLKEM_B200_H
#define MLKEM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library itself is built with -fvisibility=hidden */
#endif

#define MLKEM_B200_MEM_HOST 0
#define MLKEM_B200_MEM_DEVICE 1

/* Return codes.  -1, -3 and -5 keep the meaning of the reference's ml_errno (ml_kem.c:1243-1391). */
#define MLKEM_B200_OK 0
#define MLKEM_B200_ERR_PARAM (-1)     /* unknown parameter set (ml_errno -1, ml_kem.c:1391) */
#define MLKEM_B200_ERR_LENGTH (-3)    /* length / type check failed (ml_errno -3, ml_kem.c:1269,1323,1331) */
#define MLKEM_B200_ERR_HASH (-5)      /* dk hash check failed (ml_errno -5, ml_kem.c:1347) */
#define MLKEM_B200_ERR_CUDA (-10)     /* CUDA runtime error or no device; see mlkem_b200_last_error() */
#define MLKEM_B200_ERR_ARG (-11)      /* NULL / misaligned pointer, unsupported d or eta */

typedef struct mlkem_b200_opts {
    int device;             /* CUDA device ordinal, -1 = the calling thread's current device */
    int mem;                /* MLKEM_B200_MEM_HOST or MLKEM_B200_MEM_DEVICE */
    void *stream;           /* cudaStream_t for MEM_DEVICE calls; NULL = the CUDA default stream */
    int chunk_items;        /* items per internal chunk, 0 = default */
    int sample_group_limit; /* test hook for the SampleNTT give-up rule (ml_kem.c:221-227); 0 = 278 (the reference) */
    int flags;              /* 0 = bit-exact to the reference; MLKEM_B200_FLAG_FIPS203 see below */
} mlkem_b200_opts;
/* A NULL opts pointer means {device -1, MEM_HOST, NULL, 0, 0, 0}.
 *
 * Tuning knobs read from the environment (defaults in brackets; measured on B200 in profiles/experiments_r01.txt):
 *   MLKEM_B200_CHUNK       items per chunk of a device-memory call [262144]; workspace is about 4.3 KB per item and stream
 *   MLKEM_B200_STREAMS     internal streams the chunks of a device-memory call take turns on [4]; read once at load time,
 *                          mlkem_b200_set_streams() overrides it
 *   MLKEM_B200_HOST_CHUNK  items per staged chunk of a host-memory call [65536]
 *   MLKEM_B200_HOST_SLOTS  staging slots (H2D / kernels / D2H overlap) of a host-memory call [3]; consecutive host-memory
 *                          calls alternate between two such groups of slots
 *   MLKEM_B200_WARP_HASH_MAX  chunks of at most this many items run their long hash chains (H(ek), G(m || h), J(z || c), the dk
 *                          hash check) with one sponge per warp instead of one per thread [1024]: the latency form, 13-21 % off a
 *                          batch of one (profiles/latency_r02_warp_hash_ab.jsonl); 0 = one sponge per thread everywhere */

/* FIPS 203 mode (SURVEY.md 8(f) N1).  The reference deviates from FIPS 203: its PRF and J are SHAKE128 (SURVEY D1, D2)
 * and its ByteDecode12 never reduces, so the modulus check of KEM_Encaps cannot fail (D4).  With this flag PRF and J are
 * SHAKE256 and mlkem_b200_kem_encaps_batch performs a real modulus check (-4): the outputs are those of a conformant
 * ML-KEM (pinned in tests against an independent FIPS 203 implementation), NOT those of the reference. */
#define MLKEM_B200_FLAG_FIPS203 1
#define MLKEM_B200_ERR_MODULUS (-4)   /* FIPS mode only: an encapsulation key has a coefficient >= q (ml_errno -4) */
/* Host-memory calls only: return as soon as the copies and kernels are enqueued on the library's streams instead of
 * waiting for the results.  The buffers must be pinned (mlkem_b200_host_alloc) and stay untouched until
 * mlkem_b200_synchronize(device, NULL) returns.  Consecutive asynchronous calls pipeline through the staging slots:
 * the device-to-host tail of one overlaps the host-to-device head of the next.  Ignored by the calls that use their results
 * on the host before they return: the public-wrapper batches (mlkem_b200_kem_*_batch), mlkem_b200_sha3_bits_batch and the
 * set-up calls mlkem_b200_keys_*. */
#define MLKEM_B200_FLAG_ASYNC 2
/* mlkem_b200_keys_load / _load_ek / _from_seeds only: also keep the expanded matrix A^ of every key in the table
 * (At[row][col] = SampleNTT(rho || row || col), ml_kem.c:817-823; k*k*512 bytes per key, 4.6 KB at ML-KEM-768).  The matrix
 * depends on the key alone, so keyed Encaps / Decaps then skip the 27 of their 44 / 42 Keccak permutations that
 * re-sample it for every item.  Results are unchanged.  (sample_group_limit, the test hook, is fixed at load time.) */
#define MLKEM_B200_FLAG_EXPAND_KEYS 4

const char *mlkem_b200_version(void);
const char *mlkem_b200_last_error(void);          /* text of the last CUDA error seen by this thread */
unsigned long long mlkem_b200_launch_count(void); /* kernels launched by this library so far (all threads) */
int mlkem_b200_device_count(void);
int mlkem_b200_synchronize(int device, void *stream);
void *mlkem_b200_host_alloc(size_t bytes);        /* pinned host memory (cudaHostAlloc) */
void *mlkem_b200_host_alloc_wc(size_t bytes);     /* the same, write-combined: for INPUT buffers the CPU only ever fills sequentially */
void mlkem_b200_host_free(void *p);
void mlkem_b200_release(int device);              /* wait for the device, wipe and drop its cached workspaces (key tables stay) */

/* Sizes of a parameter set (512 / 768 / 1024), 0 for an unknown set.  ml_kem.c:730-731,1050,1105 */
unsigned mlkem_b200_ek_bytes(int param_set);
unsigned mlkem_b200_dk_bytes(int param_set);
unsigned mlkem_b200_dkpke_bytes(int param_set);
unsigned mlkem_b200_ct_bytes(int param_set);

/* ---- ML-KEM internal algorithms (FIPS 203 Alg. 16-18 as implemented by the reference) -------------- */

/* KeyGen_internal, ml_kem.c:1034.  d, z: n x 32.  ek: n x (384k+32).  dk: n x (768k+96). */
int mlkem_b200_keygen_batch(int param_set, size_t n, const uint8_t *d, const uint8_t *z, uint8_t *ek, uint8_t *dk,
                            const mlkem_b200_opts *opts);
/* Encaps_internal, ml_kem.c:1093.  ek: n x (384k+32), m: n x 32.  c: n x 32(du k + dv), K: n x 32. */
int mlkem_b200_encaps_batch(int param_set, size_t n, const uint8_t *ek, const uint8_t *m, uint8_t *c, uint8_t *K,
                            const mlkem_b200_opts *opts);
/* Decaps_internal, ml_kem.c:1136, including FO re-encryption and implicit rejection on the device.
 * dk: n x (768k+96), c: n x 32(du k + dv).  K: n x 32. */
int mlkem_b200_decaps_batch(int param_set, size_t n, const uint8_t *dk, const uint8_t *c, uint8_t *K,
                            const mlkem_b200_opts *opts);
/* The dk hash check of KEM_Decaps, ml_kem.c:1336-1350: status[i] = 0 or -5.  status: n x int32. */
int mlkem_b200_check_dk_batch(int param_set, size_t n, const uint8_t *dk, int32_t *status, const mlkem_b200_opts *opts);

/* ---- resident key tables: keyed Encaps / Decaps (SURVEY 8(f) N4, fewer bytes per operation) ---------------- */

/* A decapsulation key is 768k+96 bytes and a server uses the same few keys for every ciphertext it receives, so on
 * the host path mlkem_b200_decaps_batch spends 69 % of its PCIe bytes re-sending keys.  A key table is loaded into the
 * memory of opts->device once; the keyed calls then take only the ciphertexts (or messages) and a 4-byte key index
 * per item.  Results are bit-identical to the unkeyed calls with dk[i] = table[key_index[i]] (Decaps_internal,
 * ml_kem.c:1136; Encaps_internal, ml_kem.c:1093).  Loading is a set-up call: it returns when the table is complete. */
typedef struct mlkem_b200_keys mlkem_b200_keys;

/* n_keys decapsulation keys (n_keys x (768k+96) bytes, host or device memory per opts->mem).  status (HOST memory, may
 * be NULL): the dk hash check of KEM_Decaps (ml_kem.c:1336-1350) once per key, status[i] = 0 or -5; failing keys are
 * loaded all the same (Decaps_internal does not validate either).  On an error return *out is NULL: no table is left behind. */
int mlkem_b200_keys_load(int param_set, size_t n_keys, const uint8_t *dk, int32_t *status, const mlkem_b200_opts *opts,
                         mlkem_b200_keys **out);
/* n_keys encapsulation keys only (n_keys x (384k+32) bytes): a table for mlkem_b200_encaps_keyed_batch. */
int mlkem_b200_keys_load_ek(int param_set, size_t n_keys, const uint8_t *ek, const mlkem_b200_opts *opts,
                            mlkem_b200_keys **out);
/* The same table as mlkem_b200_keys_load(KeyGen_internal(d, z)) built on the device from the 64-byte seeds
 * (ml_kem.c:1034): 64 instead of 2400 bytes per key cross PCIe.  d, z: n_keys x 32. */
int mlkem_b200_keys_from_seeds(int param_set, size_t n_keys, const uint8_t *d, const uint8_t *z,
                               const mlkem_b200_opts *opts, mlkem_b200_keys **out);
size_t mlkem_b200_keys_count(const mlkem_b200_keys *keys);
void mlkem_b200_keys_free(mlkem_b200_keys *keys); /* wipes the decapsulation keys, then frees the table */

/* Key rotation: overwrite the keys in slots slot[0..n) of an existing table, in place.  The table keeps its parameter set,
 * device, size and memory: pointers that keyed calls already enqueued hold stay valid.
 *   Results    afterwards keyed Encaps / Decaps on slot[i] give byte for byte what the unkeyed calls give with the new key i;
 *              every other slot is unchanged.  In a table loaded with MLKEM_B200_FLAG_EXPAND_KEYS the matrices of the replaced
 *              slots are re-expanded with the sample_group_limit the table was loaded with, not this call's.
 *   Buffers    slot is always HOST memory (n x uint32).  The key material lives in opts->mem; device-memory sources are read
 *              in order on opts->stream.  opts->device must be -1 or the table's.
 *   Ordering   a set-up call: it returns once the table is updated.  It is ordered after every library call already enqueued
 *              on the table's device (MLKEM_B200_FLAG_ASYNC host-memory calls and device-memory calls on any stream
 *              included), and every call enqueued after it returns sees the new keys.
 *   Errors     MLKEM_B200_ERR_ARG, with nothing written, for a slot >= n_keys, a slot listed twice, a NULL pointer, or the
 *              wrong kind of table (see each function).  n == 0 does nothing and returns MLKEM_B200_OK.
 *   Secrets    the old dk rows are overwritten in place; device scratch that held new dk bytes or seeds is zeroed before it
 *              is freed. */
/* New decapsulation keys: dk is n x (768k+96).  Not for a table of encapsulation keys only.  status (HOST memory, may be NULL)
 * as in mlkem_b200_keys_load: status[i] = 0 or -5 from the dk hash check of key i (ml_kem.c:1336-1350); a failing key is
 * written all the same. */
int mlkem_b200_keys_replace(mlkem_b200_keys *keys, size_t n, const uint32_t *slot, const uint8_t *dk, int32_t *status,
                            const mlkem_b200_opts *opts);
/* New encapsulation keys: ek is n x (384k+32).  Only for a table of encapsulation keys (mlkem_b200_keys_load_ek): in a table
 * with decapsulation keys the dk rows would contradict their ek. */
int mlkem_b200_keys_replace_ek(mlkem_b200_keys *keys, size_t n, const uint32_t *slot, const uint8_t *ek,
                               const mlkem_b200_opts *opts);
/* The same as mlkem_b200_keys_replace with the dk of KeyGen_internal(d, z) (ml_kem.c:1034), run on the device: d, z are
 * n x 32.  KeyGen honours opts->flags & MLKEM_B200_FLAG_FIPS203 and opts->sample_group_limit, as mlkem_b200_keys_from_seeds
 * does.  Not for a table of encapsulation keys only. */
int mlkem_b200_keys_replace_from_seeds(mlkem_b200_keys *keys, size_t n, const uint32_t *slot, const uint8_t *d,
                                       const uint8_t *z, const mlkem_b200_opts *opts);
/* Read back the encapsulation keys of rows [first, first + n) of a table (either kind) into ek (n x (384k+32), host or device
 * memory per opts->mem): the public keys of a table built with mlkem_b200_keys_from_seeds, without a second KeyGen.  Ordered
 * like a replace; a host-memory export returns when ek is filled, a device-memory one is enqueued on opts->stream.
 * MLKEM_B200_ERR_ARG for a range outside the table or a NULL ek (n == 0: nothing to do, MLKEM_B200_OK). */
int mlkem_b200_keys_export_ek(const mlkem_b200_keys *keys, size_t first, size_t n, uint8_t *ek, const mlkem_b200_opts *opts);

/* Encaps_internal / Decaps_internal for n items, item i under key key_index[i] of the table.  key_index: n x uint32 in
 * the same memory space as the other buffers, or NULL = key (i mod n_keys).  Host-memory calls reject an index >=
 * n_keys (MLKEM_B200_ERR_ARG); device-memory calls clamp it to n_keys-1.  opts->device must be -1 or the table's. */
int mlkem_b200_encaps_keyed_batch(const mlkem_b200_keys *keys, size_t n, const uint32_t *key_index, const uint8_t *m,
                                  uint8_t *c, uint8_t *K, const mlkem_b200_opts *opts);
int mlkem_b200_decaps_keyed_batch(const mlkem_b200_keys *keys, size_t n, const uint32_t *key_index, const uint8_t *c,
                                  uint8_t *K, const mlkem_b200_opts *opts);

/* ---- the reference's cell layout, batched (SURVEY 8(f) N4) ------------------------------------------------------ */

/* KeyGen_internal / Encaps_internal / Decaps_internal on arrays in the layout the reference itself uses: one byte per
 * 4-byte `union byte` cell (ml_kem.h:35-38; uint32_t here, layout-compatible), item-major, value in the low 8 bits,
 * upper bits ignored on input and zero on output.  Same sizes in CELLS as the dense calls have in bytes.  The
 * conversion to and from dense bytes runs on the device inside the chunk pipeline (host-memory calls ship the cells as
 * they are: four PCIe bytes per payload byte -- the price of not touching every byte on the host). */
int mlkem_b200_keygen_cells_batch(int param_set, size_t n, const uint32_t *d, const uint32_t *z, uint32_t *ek, uint32_t *dk,
                                  const mlkem_b200_opts *opts);
int mlkem_b200_encaps_cells_batch(int param_set, size_t n, const uint32_t *ek, const uint32_t *m, uint32_t *c, uint32_t *K,
                                  const mlkem_b200_opts *opts);
int mlkem_b200_decaps_cells_batch(int param_set, size_t n, const uint32_t *dk, const uint32_t *c, uint32_t *K,
                                  const mlkem_b200_opts *opts);
/* The conversion alone, n_bytes (a multiple of 4) payload bytes: for callers that keep dense copies around. */
int mlkem_b200_cells_from_bytes(size_t n_bytes, const uint8_t *bytes, uint32_t *cells, const mlkem_b200_opts *opts);
int mlkem_b200_cells_to_bytes(size_t n_bytes, const uint32_t *cells, uint8_t *bytes, const mlkem_b200_opts *opts);

/* ---- batched forms of the public wrappers: entropy + input checks around the internal algorithms --------- */

/* KEM_KeyGen, ml_kem.c:1233: (d, z) come from the host entropy source (/dev/urandom, as getRandomBytes ml_kem.c:458).
 * Returns -2 when the entropy source fails (ml_errno -2). */
int mlkem_b200_kem_keygen_batch(int param_set, size_t n, uint8_t *ek, uint8_t *dk, const mlkem_b200_opts *opts);
/* KEM_Encaps, ml_kem.c:1257: type check on ek_len (-3), the reference's modulus check is an identity (SURVEY D4),
 * m from the entropy source. */
int mlkem_b200_kem_encaps_batch(int param_set, size_t n, const uint8_t *ek, size_t ek_len, uint8_t *c, uint8_t *K,
                                const mlkem_b200_opts *opts);
/* KEM_Decaps, ml_kem.c:1310: type checks on dk_len and c_len (-3, whole call), then per item the hash check
 * (status[i] = -5, K[i] zeroed -- the reference returns NULL for such an item) and Decaps_internal. */
int mlkem_b200_kem_decaps_batch(int param_set, size_t n, const uint8_t *dk, size_t dk_len, const uint8_t *c, size_t c_len,
                                uint8_t *K, int32_t *status, const mlkem_b200_opts *opts);

/* ---- randomness expanded on the device: KEM_KeyGen / KEM_Encaps, keyed KEM_Encaps, generated key tables -------------- */

/* The calls above read every random byte from /dev/urandom on one host thread (64 bytes per KeyGen, 32 per Encaps), far
 * below what the device computes.  The calls below take ONE 32-byte call seed and expand it on the device.  Item j of a call
 * (its position in the call, 0 <= j < n, whatever the chunking) gets
 *
 *     R_j = SHAKE256(seed[0..32) || LE64(j) || LE64(tag), 64 bytes)    -- 48 input bytes: one block, one Keccak-f[1600]
 *
 *   tag 1 (KeyGen):  d_j = R_j[0..32), z_j = R_j[32..64)
 *   tag 2 (Encaps):  m_j = R_j[0..32)
 *
 * and the call returns exactly what the named existing call returns with that randomness.
 *
 *   seed     always HOST memory, 32 bytes, or NULL.  NULL: 32 fresh bytes from the host entropy source (/dev/urandom) for this
 *            call; -2 when that source fails, as in mlkem_b200_kem_keygen_batch.  A non-NULL seed makes the call deterministic:
 *            that form is for tests and known-answer checks, like the *_internal calls.  A repeated seed repeats EVERY secret
 *            of the call (every d, z, m and so every dk and shared key): never pass one twice outside a test.
 *   Not a DRBG  this is a SHAKE256 expansion of 32 OS bytes per call, not an SP 800-90A DRBG.  Callers that need every random
 *            byte from the OS keep mlkem_b200_kem_keygen_batch / _kem_encaps_batch.
 *   Flags    the derivation does not depend on MLKEM_B200_FLAG_FIPS203; the KEM computations honour it as usual.
 *   Secrets  the seed is copied into the device's pooled scratch; the library's host copy is zeroed with explicit_bzero and the
 *            device copy once the call's work has drained, before the call returns: it never sits in a kernel-parameter
 *            buffer.  The expanded d, z, m live only in the chunk workspaces or in scratch that is zeroed, like every other
 *            per-item secret, and host-memory calls never send them over PCIe (a seeded KeyGen copies nothing to the device
 *            but the seed).
 *   Synchrony  so every call here is SYNCHRONOUS in both memory spaces: a device-memory call returns once opts->stream has
 *            drained, and MLKEM_B200_FLAG_ASYNC is ignored.
 * The other buffers follow opts->mem. */

/* mlkem_b200_keygen_batch(d_j, z_j).  ek: n x (384k+32), dk: n x (768k+96). */
int mlkem_b200_kem_keygen_seeded_batch(int param_set, size_t n, const uint8_t *seed, uint8_t *ek, uint8_t *dk,
                                       const mlkem_b200_opts *opts);
/* The checks of mlkem_b200_kem_encaps_batch (-1 unknown set, -3 ek_len, in FIPS mode -4 when any coefficient of any ek is
 * >= q), then mlkem_b200_encaps_batch(ek, m_j). */
int mlkem_b200_kem_encaps_seeded_batch(int param_set, size_t n, const uint8_t *ek, size_t ek_len, const uint8_t *seed,
                                       uint8_t *c, uint8_t *K, const mlkem_b200_opts *opts);
/* mlkem_b200_encaps_keyed_batch(keys, key_index, m_j), with its index rules (host memory rejects an index >= n_keys, device
 * memory clamps it, NULL = i mod n_keys), on a table of either kind. */
int mlkem_b200_kem_encaps_keyed_batch(const mlkem_b200_keys *keys, size_t n, const uint32_t *key_index, const uint8_t *seed,
                                      uint8_t *c, uint8_t *K, const mlkem_b200_opts *opts);
/* mlkem_b200_keys_from_seeds(d_j, z_j) for j < n_keys: a key table whose secrets never exist on the host.  Honours
 * MLKEM_B200_FLAG_EXPAND_KEYS, MLKEM_B200_FLAG_FIPS203 and sample_group_limit.  Publish its keys with mlkem_b200_keys_export_ek. */
int mlkem_b200_keys_generate(int param_set, size_t n_keys, const uint8_t *seed, const mlkem_b200_opts *opts,
                             mlkem_b200_keys **out);
/* mlkem_b200_keys_replace_from_seeds(slot, d_j, z_j), j the position in slot[]: the checks, ordering and errors of the other
 * replaces. */
int mlkem_b200_keys_replace_generate(mlkem_b200_keys *keys, size_t n, const uint32_t *slot, const uint8_t *seed,
                                     const mlkem_b200_opts *opts);

/* ---- K-PKE (FIPS 203 Alg. 13-15) -------------------------------------------------------------------- */

/* PKE_KeyGen, ml_kem.c:651.  d: n x 32.  ek: n x (384k+32).  dk_pke: n x 384k. */
int mlkem_b200_pke_keygen_batch(int param_set, size_t n, const uint8_t *d, uint8_t *ek, uint8_t *dk_pke,
                                const mlkem_b200_opts *opts);
/* PKE_Encrypt, ml_kem.c:776.  m, r: n x 32. */
int mlkem_b200_pke_encrypt_batch(int param_set, size_t n, const uint8_t *ek, const uint8_t *m, const uint8_t *r,
                                 uint8_t *c, const mlkem_b200_opts *opts);
/* PKE_Decrypt, ml_kem.c:942.  dk_pke: item i at dk_pke + i*dk_stride (384k for bare keys, 768k+96 to read them
 * out of decapsulation keys).  m: n x 32. */
int mlkem_b200_pke_decrypt_batch(int param_set, size_t n, const uint8_t *dk_pke, size_t dk_stride, const uint8_t *c,
                                 uint8_t *m, const mlkem_b200_opts *opts);

/* ---- ring arithmetic ------------------------------------------------------------------------------- */

/* NTT, ml_kem.c:287, for any 12-bit coefficients.  For inputs in [q, 4096) the reference's butterfly leaves the
 * difference f[j] - t unreduced (ml_kem.c:317-318), so some outputs are the residue plus q: reproduced bit for bit
 * (a polynomial that contains such a coefficient takes a literal restatement of the reference's update). */
int mlkem_b200_ntt_batch(size_t n, const uint16_t *f, uint16_t *f_hat, const mlkem_b200_opts *opts);
/* InverseNTT, ml_kem.c:336 (includes the multiplication by 3303).  Coefficients are taken as residues mod q and the
 * output is canonical, which is the reference's result whenever its arithmetic is defined: for a pair with
 * f[j] - f[j+len] > q (needs f[j] >= q) the reference's `Q - (t - f[j+len])` wraps in a 24-bit field and the
 * following product overflows a signed int (ml_kem.c:366-368) -- undefined behaviour, not reproduced. */
int mlkem_b200_intt_batch(size_t n, const uint16_t *f_hat, uint16_t *f, const mlkem_b200_opts *opts);
/* MultiplyNTTs, ml_kem.c:415 (128 BaseCaseMultiply, ml_kem.c:395).  Operands may be any 12-bit value. */
int mlkem_b200_multiply_ntts_batch(size_t n, const uint16_t *f_hat, const uint16_t *g_hat, uint16_t *h_hat,
                                   const mlkem_b200_opts *opts);

/* PolyAddition, ml_kem.c:580: (u + v) mod q coefficient-wise; PolySubtraction, ml_kem.c:599: u < v ? q - (v - u) : u - v,
 * kept in 12 bits (unreduced when u - v >= q, like the reference).  n polynomials each. */
int mlkem_b200_poly_add_batch(size_t n, const uint16_t *u, const uint16_t *v, uint16_t *z, const mlkem_b200_opts *opts);
int mlkem_b200_poly_sub_batch(size_t n, const uint16_t *u, const uint16_t *v, uint16_t *z, const mlkem_b200_opts *opts);
/* VectorMultiply, ml_kem.c:618: w = sum_{i<k} MultiplyNTTs(u[i], v[i]).  u, v: n x k x 256, w: n x 256; 1 <= k <= 16. */
int mlkem_b200_vector_multiply_batch(int k, size_t n, const uint16_t *u, const uint16_t *v, uint16_t *w,
                                     const mlkem_b200_opts *opts);

/* ---- samplers -------------------------------------------------------------------------------------- */

/* SampleNTT, ml_kem.c:189.  seeds: n x 34.  a_hat: n x 256.  seeds_after (may be NULL): n x 34, the caller's
 * buffer B after the call (the reference bumps B[32], B[33] when it gives up and restarts, :237-242). */
int mlkem_b200_sample_ntt_batch(size_t n, const uint8_t *seeds, uint16_t *a_hat, uint8_t *seeds_after,
                                const mlkem_b200_opts *opts);
/* SamplePolyCBD_eta, ml_kem.c:253.  bytes: n x 64 eta, eta in {2, 3}. */
int mlkem_b200_cbd_batch(int eta, size_t n, const uint8_t *bytes, uint16_t *f, const mlkem_b200_opts *opts);
/* SamplePolyCBD_eta(PRF_eta(s, b)), ml_kem.c:496 + :253 (PRF is SHAKE128 in the reference).
 * seeds: n x 32, nonces: n x 1. */
int mlkem_b200_prf_cbd_batch(int eta, size_t n, const uint8_t *seeds, const uint8_t *nonces, uint16_t *f,
                             const mlkem_b200_opts *opts);

/* ---- codec ----------------------------------------------------------------------------------------- */

/* ByteEncode_d, ml_kem.c:125.  F: n x 256 (low d bits used).  B: n x 32 d.  d in {1,4,5,10,11,12}. */
int mlkem_b200_byte_encode_batch(int d, size_t n, const uint16_t *F, uint8_t *B, const mlkem_b200_opts *opts);
/* ByteDecode_d, ml_kem.c:153 (d = 12: no reduction mod q, like the reference). */
int mlkem_b200_byte_decode_batch(int d, size_t n, const uint8_t *B, uint16_t *F, const mlkem_b200_opts *opts);
/* Compress_d / Decompress_d, ml_kem.c:83 / :104, element-wise over n_coeffs values (multiple of 8). */
int mlkem_b200_compress_batch(int d, size_t n_coeffs, const uint16_t *x, uint16_t *y, const mlkem_b200_opts *opts);
int mlkem_b200_decompress_batch(int d, size_t n_coeffs, const uint16_t *y, uint16_t *x, const mlkem_b200_opts *opts);
/* Fused ByteEncode_d(Compress_d(F)) and Decompress_d(ByteDecode_d(B)) as used at ml_kem.c:886-904, :978-993. */
int mlkem_b200_compress_encode_batch(int d, size_t n, const uint16_t *F, uint8_t *B, const mlkem_b200_opts *opts);
int mlkem_b200_decode_decompress_batch(int d, size_t n, const uint8_t *B, uint16_t *F, const mlkem_b200_opts *opts);

/* ---- hashes ---------------------------------------------------------------------------------------- */

/* which = 0: H = SHA3-256 (ml_kem.c:521), 32 B out.  1: G = SHA3-512 (:559), 64 B out.
 * 2: J = SHAKE128 with 32 B out (:540 -- the reference uses capacity 256).  3: SHAKE256 with 32 B out (J of FIPS 203).
 * in: n messages of `len` bytes each, len a multiple of 8 (true of every H/G/J input of ML-KEM except
 * G(d||k), which only occurs inside KeyGen). */
int mlkem_b200_hash_batch(int which, size_t n, size_t len, const uint8_t *in, uint8_t *out, const mlkem_b200_opts *opts);

/* sha3_b, sha3.c:408: the reference's general SHA-3 front-end for messages of any BIT length (SURVEY 8(f) N3).
 * msgs: n messages of nbits bits, packed LSB-first into ceil(nbits/8) bytes each; sfx = the reference's 4 suffix
 * bits (sfx[2] == 1 selects the 4-bit XOF suffix, else the first 2 bits); c = capacity in bits (1600 - c must be a
 * multiple of 64: every SHA-3 / SHAKE instance); d = output bits; out: n x ceil(d/8) bytes, unused top bits zero.
 * Host memory only.  Reproduces the reference's padding deviation for (nbits + |sfx| + 2) % r == 0. */
int mlkem_b200_sha3_bits_batch(size_t n, const uint8_t *msgs, size_t nbits, const uint8_t sfx[4], unsigned c, size_t d,
                               uint8_t *out, const mlkem_b200_opts *opts);

/* ---- measurement hooks (bench.py) -------------------------------------------------------------------- */

/* Per-kernel timing: while enabled, every kernel launch of the library is bracketed by CUDA events on its
 * stream.  mlkem_b200_profile_report() synchronises, writes up to `cap` bytes of JSON
 * ({"kernel name": {"launches": L, "ms": total}, ...}) into buf, clears the records and returns the number of
 * bytes written (0 when nothing was recorded). */
void mlkem_b200_profile(int enable);
/* Device-memory calls interleave their chunks on 4 internal streams by default (kernels of different chunks
 * overlap).  n = 1 serialises them on the caller's stream, which is what per-kernel timing needs; n < 1 restores
 * the default. */
void mlkem_b200_set_streams(int n);
int mlkem_b200_profile_report(char *buf, int cap);

/* Copy-only ceiling of a host-memory call: moves the same bytes through the same chunking, staging slots and streams as
 * a real call with n items and these buffers (n_in inputs copied to the device, n_out outputs copied back), with no
 * kernels in between.  bench.py times it next to the real calls (e2e.copy_ceiling). */
int mlkem_b200_copy_probe(size_t n, int n_in, const void *const *in, const size_t *in_item_bytes, int n_out,
                          void *const *out, const size_t *out_item_bytes, const mlkem_b200_opts *opts);

/* INT32 roofline denominators of the current device, measured now: sustained thread-operations per second
 * of out[0] LOP3, out[1] SHF (alu pipe), out[2] IMAD (fma pipe), out[3] LOP3+IMAD interleaved (both pipes),
 * out[4] IADD3, out[5] IMAD.HI.  MEASURED_PEAKS.json has no integer figure, and the ML-KEM kernels are bound by
 * these pipes, not by HBM or the tensor cores. */
int mlkem_b200_int32_peak(double out[6]);

/* Read-only copies of the device twiddle tables: zeta_i = 17^BitRev7(i), gamma_i = 17^(2 BitRev7(i)+1). */
int mlkem_b200_tables(uint16_t zeta[128], uint16_t gamma[128]);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MLKEM_B200_H */
