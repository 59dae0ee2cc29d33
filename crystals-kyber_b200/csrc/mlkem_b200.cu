// mlkem_b200.cu -- host side of libmlkem_b200.so: the batched C ABI of include/mlkem_b200.h.
//
// Single translation unit: device code (mlkem_device.cuh, mlkem_kernels.cuh) + per-device context
// (streams, workspace, staging buffers) + the pipelines that chain the kernels into KeyGen / Encaps /
// Decaps / K-PKE, + the reference-signature API of include/ml_kem.h (ml_kem_compat.inl).
//
// There is no CPU implementation of any hot-path function in this library: if CUDA is unusable every entry
// point fails with MLKEM_B200_ERR_CUDA.
#include "mlkem_kernels.cuh"

#include "../../include/mlkem_b200.h"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

namespace {

using namespace mlkem;

thread_local char tl_error[512] = "";
std::atomic<unsigned long long> g_launches{0};
int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}
constexpr int kSlots = 6;      // streams / workspaces per device: two groups of kHostSlots for host-memory calls, the first kDevSlots for device-memory calls
constexpr int kDevSlots = 4;
constexpr int kHostSlots = 3;  // measured: 3 slots keep the H2D copy engine at ~50.7 GB/s (2 slots: 48 GB/s)
constexpr int kMaxDevices = 64;
// Streams that device-memory calls interleave their chunks on (1 = serial; measured 31.3 / 32.4 / 32.5 / 32.5 M pairs/s with
// 1 / 2 / 3 / 4).  MLKEM_B200_STREAMS sets the start value ONCE; mlkem_b200_set_streams() overrides it afterwards.
int initial_streams() {
    int v = env_int("MLKEM_B200_STREAMS", 0);
    return v < 1 ? kDevSlots : (v > kDevSlots ? kDevSlots : v);
}
std::atomic<int> g_streams{initial_streams()};
// Batches of at most this many items run their long hash chains (H(ek), J(z || c)) with one sponge per WARP instead of one per
// thread: latency instead of throughput.  MLKEM_B200_WARP_HASH_MAX = 0 switches the warp form off.
int warp_hash_max() {
    static const int v = env_int("MLKEM_B200_WARP_HASH_MAX", kWarpHashMaxItems);
    return v;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) {                                                                              \
            snprintf(tl_error, sizeof tl_error, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return MLKEM_B200_ERR_CUDA;                                                                       \
        }                                                                                                     \
    } while (0)

// Optional per-kernel timing (mlkem_b200_profile): CUDA events recorded on the launching stream around
// every kernel, resolved when the report is read.  Off by default; costs two event records per launch.
struct ProfEntry {
    const char *name;
    cudaEvent_t e0, e1;
};
std::atomic<int> g_profile{0};
std::mutex g_prof_mutex;
std::vector<ProfEntry> g_prof_entries;

inline void prof_begin(const char *name, cudaStream_t st, ProfEntry &pe, bool &on) {
    on = g_profile.load(std::memory_order_relaxed) != 0;
    if (!on) return;
    pe.name = name;
    cudaEventCreate(&pe.e0);
    cudaEventCreate(&pe.e1);
    cudaEventRecord(pe.e0, st);
}
inline void prof_end(cudaStream_t st, ProfEntry &pe, bool on) {
    if (!on) return;
    cudaEventRecord(pe.e1, st);
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    g_prof_entries.push_back(pe);
}

// kernel<<<...>>>(...) with launch accounting, optional timing and error capture
#define LAUNCH(kernel, grid, block, smem, stream, ...)           \
    do {                                                         \
        auto kern_ = kernel;                                     \
        ProfEntry pe_;                                           \
        bool prof_on_;                                           \
        prof_begin(#kernel, (stream), pe_, prof_on_);            \
        kern_<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__); \
        prof_end((stream), pe_, prof_on_);                       \
        g_launches.fetch_add(1, std::memory_order_relaxed);      \
        CU(cudaGetLastError());                                  \
    } while (0)

inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }
inline unsigned warp_hash_grid(int n) { return cdiv((size_t)n, kWarpHashTPB / 32); }
// grid of the persistent warp-per-item kernels: enough blocks to fill the machine several times over, then grid-stride
inline unsigned warp_grid(size_t items, int warps_per_block) {
    size_t blocks = (items + warps_per_block - 1) / warps_per_block;
    const size_t cap = 148 * 16;
    return (unsigned)(blocks < cap ? blocks : cap);
}

// ------------------------------------------------------------------------------------------------
// Tables
// ------------------------------------------------------------------------------------------------
#include "mlkem_tables.inl"

// ------------------------------------------------------------------------------------------------
// Per-device context
// ------------------------------------------------------------------------------------------------
// Slot k of a device = workspace ws[k] + staging buffer io[k] + library stream stream[k].  A slot may be used from the
// library stream (chunks of large device-memory calls, every host-memory call) or from the CALLER's stream (a
// device-memory call that stays on one stream), so stream order alone does not protect it: ev_slot[k] is recorded after
// the last kernel of every use, and every user makes its stream wait for it first.  call_mutex serialises the enqueueing.
struct DeviceCtx {
    bool ready = false;
    cudaStream_t stream[kSlots] = {};
    void *ws[kSlots] = {};  // kernel workspace (intermediates between kernels)
    size_t ws_bytes[kSlots] = {};
    void *io[kSlots] = {};  // device staging of host-resident inputs / outputs
    size_t io_bytes[kSlots] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[kSlots] = {}, ev_slot[kSlots] = {};
    void *misc = nullptr;  // small pooled device buffer: entropy seeds / status words of the public-wrapper batches
    size_t misc_bytes = 0;
    int host_group = 0;     // consecutive host-memory calls alternate between slots 0..2 and 3..5: with MLKEM_B200_FLAG_ASYNC the
                            // chunks of two calls in flight run side by side (one call's D2H under the other's H2D)
    std::mutex call_mutex;  // one call at a time enqueues on this device's streams / workspaces
    std::mutex misc_mutex;  // one user of `misc` at a time (held until its stream has drained)
};
DeviceCtx g_ctx[kMaxDevices];
std::mutex g_mutex;

// The calling thread's current device is switched for the duration of a call only (torch, for one, follows
// cudaGetDevice): every entry point holds one of these.
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    int enter(int d) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev == d) return 0;
        CU(cudaSetDevice(d));
        changed = true;
        return 0;
    }
    ~DeviceGuard() {
        if (changed && prev >= 0) cudaSetDevice(prev);
    }
};

// Grow-only device buffer.  `last_use` (may be null) is the event after which nothing reads the old buffer any more.
int ensure_buffer(void **p, size_t *have, size_t need, cudaEvent_t last_use = nullptr) {
    if (*have >= need) return 0;
    if (*p) {
        if (last_use) CU(cudaEventSynchronize(last_use));
        CU(cudaMemset(*p, 0, *have));  // intermediates are secret-dependent (sigma, s^, m', K' || r')
        CU(cudaFree(*p));
    }
    *p = nullptr;
    *have = 0;
    size_t want = need + need / 8;
    CU(cudaMalloc(p, want));
    *have = want;
    return 0;
}

template <class KernelT>
int allow_smem(KernelT kernel, size_t bytes) {
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return 0;
}
template <class P>
int allow_smem_matvec() {
    const size_t b = matvec_smem_bytes<P>();
    if (int rc = allow_smem(k_sample_matvec<P, kModeKeyGen>, b)) return rc;
    if (int rc = allow_smem(k_sample_matvec<P, kModeEncrypt>, b)) return rc;
    if (int rc = allow_smem(k_sample_matvec<P, kModeEncryptCompare>, b)) return rc;
    if (int rc = allow_smem(k_sample_matvec_list<P, kModeKeyGen>, b)) return rc;
    if (int rc = allow_smem(k_sample_matvec_list<P, kModeEncrypt>, b)) return rc;
    if (int rc = allow_smem(k_sample_matvec_list<P, kModeEncryptCompare>, b)) return rc;
    return 0;
}

// Select the device (for the lifetime of `guard`) and make sure its context exists.  Returns the ordinal through *dev.
int acquire(const mlkem_b200_opts *o, int *dev, DeviceCtx **ctx, DeviceGuard &guard) {
    int d = o ? o->device : -1;
    if (d < 0) CU(cudaGetDevice(&d));
    if (d >= kMaxDevices) {
        snprintf(tl_error, sizeof tl_error, "device ordinal %d out of range", d);
        return MLKEM_B200_ERR_ARG;
    }
    if (int rc = guard.enter(d)) return rc;
    std::lock_guard<std::mutex> lock(g_mutex);
    DeviceCtx &c = g_ctx[d];
    if (!c.ready) {
        // all or nothing: streams and events are created into locals and only published when everything succeeded
        cudaStream_t st[kSlots] = {};
        cudaEvent_t ev[2 * kSlots + 1] = {};
        auto create = [&]() -> int {
            TwiddleTables t;
            uint2 rc[24];
            build_tables(t, rc);
            CU(cudaMemcpyToSymbol(c_tw, &t, sizeof t));
            CU(cudaMemcpyToSymbol(g_tw, &t, sizeof t));
            CU(cudaMemcpyToSymbol(c_keccak_rc, rc, sizeof rc));
            uint32_t pow2[32];
            for (int k = 0; k < 32; k++) pow2[k] = 1u << k;
            CU(cudaMemcpyToSymbol(c_pow2, pow2, sizeof pow2));
            for (int s = 0; s < kSlots; s++) CU(cudaStreamCreateWithFlags(&st[s], cudaStreamNonBlocking));
            for (int e = 0; e < 2 * kSlots + 1; e++) CU(cudaEventCreateWithFlags(&ev[e], cudaEventDisableTiming));
            if (int r = allow_smem_matvec<P512>()) return r;
            if (int r = allow_smem_matvec<P768>()) return r;
            if (int r = allow_smem_matvec<P1024>()) return r;
            if (int r = allow_smem(k_sample_ntt_batch, 128 * kSlotWords * 4)) return r;
            return 0;
        };
        if (int r = create()) {
            for (auto s_ : st)
                if (s_) cudaStreamDestroy(s_);
            for (auto e_ : ev)
                if (e_) cudaEventDestroy(e_);
            return r;
        }
        for (int s = 0; s < kSlots; s++) {
            c.stream[s] = st[s];
            c.ev_join[s] = ev[s];
            c.ev_slot[s] = ev[kSlots + s];
        }
        c.ev_fork = ev[2 * kSlots];
        c.ready = true;
    }
    *dev = d;
    *ctx = &c;
    return 0;
}

// Bump allocator over a workspace buffer.
struct Arena {
    uint8_t *base;
    size_t off = 0;
    explicit Arena(void *p) : base(static_cast<uint8_t *>(p)) {}
    template <class T>
    T *take(size_t count) {
        off = (off + 255) & ~size_t(255);
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

template <class P>
constexpr size_t ws_bytes_per_item() {
    // keygen: rs 64 + 2K polys ; encrypt: K polys + (K+1) code rows ; decaps adds m' 32 + K'r' 64 + flag 4
    size_t kg = 64 + 2 * P::K * 512 + 4 * P::K;
    size_t enc = P::K * 512 + (P::K + 1) * 128 + 32 + 4 * P::K;
    size_t dec = enc + 32 + 64 + 4;
    size_t m = kg > dec ? kg : dec;
    return m + 64;
}
constexpr size_t kWsSlack = 16 * 256;

// ------------------------------------------------------------------------------------------------
// Pipelines on device pointers.  Every function only enqueues work on `st`.
// ------------------------------------------------------------------------------------------------

// The fused matrix kernel and its clean-up pass.  With the reference's group limit (278 >= 168 = three blocks) the
// straight-line kernel runs first and appends the rows it could not complete to a list that the general kernel
// then works off; a lowered limit (test hook) sends every row through the general kernel.
template <class P, int MODE>
int launch_matvec(cudaStream_t st, Arena &ws, MatvecArgs a) {
    constexpr int K = P::K;
    const size_t rows = (size_t)a.n * K, smem = matvec_smem_bytes<P>();
    const unsigned blocks = cdiv(rows, 32), list_grid = std::min<unsigned>(blocks, 148 * 4);
#ifdef MLKEM_B200_EXPERIMENT
    static const int env_exp = env_int("MLKEM_B200_EXPERIMENT", 0);
    a.experiment = env_exp;
#endif
    // A batch that fits one block (a batch of one, most of all) goes through the general kernel alone: the same results from
    // one launch instead of a memset and two launches, and nothing to defer when there is no second wave of blocks to keep busy.
    if (a.group_limit >= 168 && rows > 32) {
        a.defer_list = ws.take<int>(rows);
        a.defer_count = ws.take<int>(1);
        CU(cudaMemsetAsync(a.defer_count, 0, sizeof(int), st));
        LAUNCH((k_sample_matvec<P, MODE>), blocks, 32 * K, smem, st, a);
#ifdef MLKEM_B200_EXPERIMENT
        if (env_exp & 16) return 0;  // what would a free clean-up pass buy?
#endif
        LAUNCH((k_sample_matvec_list<P, MODE>), list_grid, 32 * K, smem, st, a);
    } else {
        a.defer_list = nullptr;
        a.defer_count = nullptr;
        LAUNCH((k_sample_matvec_list<P, MODE>), list_grid, 32 * K, smem, st, a);
    }
    return 0;
}

// K-PKE.Encrypt (ml_kem.c:776) for n items; `seed` = 32-byte PRF key r per item.
// Stores c, or (cmp != nullptr) ORs the mismatch of the re-encryption against cmp into flags.
template <class P>
int enqueue_encrypt(cudaStream_t st, Arena &ws, int n, const uint8_t *ek, size_t ek_stride, KeySel keys, const uint8_t *m,
                    const uint8_t *seed, size_t seed_stride, uint8_t *c, const uint8_t *cmp, uint32_t *flags, int group_limit, bool fips,
                    const uint16_t *matrix = nullptr) {
    constexpr int K = P::K;
    uint16_t *yhat = ws.take<uint16_t>((size_t)n * K * 256);
    uint32_t *codes = ws.take<uint32_t>((size_t)n * (K + 1) * 32);
    // y^ = NTT(CBD_eta1(PRF(r, 0..K-1)))            ml_kem.c:826-836
    // (PRF = SHAKE128 as in the reference, or SHAKE256 in FIPS mode)
    if (!fips) {
        LAUNCH((k_noise<P::ETA1, true>), dim3(cdiv(n, kNoiseTPB), K), kNoiseTPB, 0, st, n, seed, seed_stride, 0, yhat, (size_t)K * 256,
               (uint32_t *)nullptr, (size_t)0, (uint8_t *)nullptr, (size_t)0, 0);
        // e1, e2 = CBD_eta2(PRF(r, K..2K))               ml_kem.c:839-851
        LAUNCH((k_noise<P::ETA2, false>), dim3(cdiv(n, kNoiseTPB), K + 1), kNoiseTPB, 0, st, n, seed, seed_stride, K, (uint16_t *)nullptr,
               (size_t)0, codes, (size_t)(K + 1) * 32, (uint8_t *)nullptr, (size_t)0, 0);
    } else {
        LAUNCH((k_noise<P::ETA1, true, kRateSha3_256>), dim3(cdiv(n, kNoiseTPB), K), kNoiseTPB, 0, st, n, seed, seed_stride, 0, yhat,
               (size_t)K * 256, (uint32_t *)nullptr, (size_t)0, (uint8_t *)nullptr, (size_t)0, 0);
        LAUNCH((k_noise<P::ETA2, false, kRateSha3_256>), dim3(cdiv(n, kNoiseTPB), K + 1), kNoiseTPB, 0, st, n, seed, seed_stride, K,
               (uint16_t *)nullptr, (size_t)0, codes, (size_t)(K + 1) * 32, (uint8_t *)nullptr, (size_t)0, 0);
    }
    MatvecArgs a{};
    a.n = n;
    a.group_limit = group_limit;
    a.rho = ek + 384 * K;
    a.rho_stride = ek_stride;
    a.keys = keys;
    a.vec = yhat;
    a.vec_stride = (size_t)K * 256;
    a.addc = codes;
    a.addc_stride = (size_t)(K + 1) * 32;
    a.out = c;
    a.out_stride = P::C;
    a.cmp = cmp;
    a.flags = flags;
    EncVArgs v{};
    v.n = n;
    v.ek = ek;
    v.ek_stride = ek_stride;
    v.keys = keys;
    v.yhat = yhat;
    v.yhat_stride = (size_t)K * 256;
    v.addc = codes;
    v.addc_stride = (size_t)(K + 1) * 32;
    v.m = m;
    v.c = c;
    v.c_stride = P::C;
    v.cmp = cmp;
    v.flags = flags;
    // the u rows: from the expanded key table when there is one, else matrix expansion fused with the product
    const unsigned tgrid = warp_grid((size_t)n * K, kMatTableTPB / 32);
    if (cmp) {
        if (matrix) LAUNCH((k_matvec_table<P, kModeEncryptCompare>), tgrid, kMatTableTPB, 0, st, a, matrix);
        else if (int rc = launch_matvec<P, kModeEncryptCompare>(st, ws, a)) return rc;
        LAUNCH((k_encrypt_v<P, true>), warp_grid(n, kWarpTPB / 32), kWarpTPB, 0, st, v);
    } else {
        if (matrix) LAUNCH((k_matvec_table<P, kModeEncrypt>), tgrid, kMatTableTPB, 0, st, a, matrix);
        else if (int rc = launch_matvec<P, kModeEncrypt>(st, ws, a)) return rc;
        LAUNCH((k_encrypt_v<P, false>), warp_grid(n, kWarpTPB / 32), kWarpTPB, 0, st, v);
    }
    return 0;
}

// KeyGen_internal (ml_kem.c:1034) when z != nullptr, PKE_KeyGen (ml_kem.c:651) otherwise.
template <class P>
int enqueue_keygen(cudaStream_t st, Arena &ws, int n, const uint8_t *d, const uint8_t *z, uint8_t *ek, uint8_t *dk, int group_limit, bool fips) {
    constexpr int K = P::K;
    const bool full = z != nullptr;
    const size_t dk_stride = full ? P::DK : P::DKPKE;
    uint8_t *rs = ws.take<uint8_t>((size_t)n * 64);
    uint16_t *se = ws.take<uint16_t>((size_t)n * 2 * K * 256);
    // G, and rho into the tail of ek and (full key) the ek copy inside dk
    LAUNCH(k_keygen_G, cdiv(n, kHashTPB), kHashTPB, 0, st, n, d, (uint32_t)K, rs, ek + 384 * K, (size_t)P::EK,
           full ? dk + 768 * K : (uint8_t *)nullptr, dk_stride);
    // s^ (nonces 0..K-1) and e^ (nonces K..2K-1), ml_kem.c:696-720; sigma = rs + 32
    if (!fips)
        LAUNCH((k_noise<P::ETA1, true>), dim3(cdiv(n, kNoiseTPB), 2 * K), kNoiseTPB, 0, st, n, rs + 32, (size_t)64, 0, se, (size_t)2 * K * 256,
               (uint32_t *)nullptr, (size_t)0, dk, dk_stride, K);  // dk_pke rows = ByteEncode12(s^) written on the way (:750-756)
    else
        LAUNCH((k_noise<P::ETA1, true, kRateSha3_256>), dim3(cdiv(n, kNoiseTPB), 2 * K), kNoiseTPB, 0, st, n, rs + 32, (size_t)64, 0, se,
               (size_t)2 * K * 256, (uint32_t *)nullptr, (size_t)0, dk, dk_stride, K);
    MatvecArgs a{};
    a.n = n;
    a.group_limit = group_limit;
    a.rho = rs;
    a.rho_stride = 64;
    a.vec = se;
    a.vec_stride = (size_t)2 * K * 256;
    a.add16 = se + K * 256;
    a.add16_stride = (size_t)2 * K * 256;
    a.out = ek;
    a.out_stride = P::EK;
    a.out2 = full ? dk + 384 * K : nullptr;
    a.out2_stride = dk_stride;
    if (int rc = launch_matvec<P, kModeKeyGen>(st, ws, a)) return rc;
    if (full && n <= warp_hash_max()) LAUNCH((k_keygen_H_warp<P>), warp_hash_grid(n), kWarpHashTPB, 0, st, n, ek, z, dk);
    else if (full) LAUNCH((k_keygen_H<P>), cdiv(n, kHashTPB), kHashTPB, 0, st, n, ek, z, dk);
    return 0;
}

template <class P>
int enqueue_encaps(cudaStream_t st, Arena &ws, int n, const uint8_t *ek, const uint8_t *m, uint8_t *c, uint8_t *Kout, int group_limit, bool fips) {
    uint8_t *r = ws.take<uint8_t>((size_t)n * 32);
    if (n <= warp_hash_max()) LAUNCH((k_encaps_HG_warp<P>), warp_hash_grid(n), kWarpHashTPB, 0, st, n, ek, m, Kout, r);
    else LAUNCH((k_encaps_HG<P>), cdiv(n, kHashTPB), kHashTPB, 0, st, n, ek, m, Kout, r);
    return enqueue_encrypt<P>(st, ws, n, ek, P::EK, KeySel{}, m, r, 32, c, nullptr, nullptr, group_limit, fips);
}

// Encaps_internal against a resident key table: ek rows at ek + key*ek_stride, their hashes H(ek) at hek + 32 key.
template <class P>
int enqueue_encaps_keyed(cudaStream_t st, Arena &ws, int n, const uint8_t *ek, size_t ek_stride, const uint8_t *hek, KeySel keys,
                         const uint8_t *m, uint8_t *c, uint8_t *Kout, int group_limit, bool fips, const uint16_t *matrix) {
    uint8_t *r = ws.take<uint8_t>((size_t)n * 32);
    LAUNCH(k_encaps_G_keyed, cdiv(n, kHashTPB), kHashTPB, 0, st, n, hek, keys, m, Kout, r);
    return enqueue_encrypt<P>(st, ws, n, ek, ek_stride, keys, m, r, 32, c, nullptr, nullptr, group_limit, fips, matrix);
}

template <class P>
int enqueue_decaps(cudaStream_t st, Arena &ws, int n, const uint8_t *dk, KeySel keys, const uint8_t *c, uint8_t *Kout, int group_limit, bool fips,
                   const uint16_t *matrix = nullptr) {
    constexpr int K = P::K;
    uint8_t *mp = ws.take<uint8_t>((size_t)n * 32);
    uint8_t *Kr = ws.take<uint8_t>((size_t)n * 64);
    uint32_t *flags = ws.take<uint32_t>((size_t)n);
    CU(cudaMemsetAsync(flags, 0, (size_t)n * 4, st));
    LAUNCH((k_decrypt<P>), warp_grid(n, kWarpTPB / 32), kWarpTPB, 0, st, n, dk, (size_t)P::DK, keys, c, mp);
    LAUNCH((k_decaps_G<P>), cdiv(n, kHashTPB), kHashTPB, 0, st, n, mp, dk, keys, Kr);
    // c' = K-PKE.Encrypt(ek_pke, m', r') compared on the fly (ml_kem.c:1206-1215)
    if (int rc = enqueue_encrypt<P>(st, ws, n, dk + 384 * K, P::DK, keys, mp, Kr + 32, 64, nullptr, c, flags, group_limit, fips, matrix)) return rc;
    if (n <= warp_hash_max()) {
        if (!fips) LAUNCH((k_decaps_J_select_warp<P>), warp_hash_grid(n), kWarpHashTPB, 0, st, n, dk, keys, c, Kr, flags, Kout);
        else LAUNCH((k_decaps_J_select_warp<P, kRateSha3_256>), warp_hash_grid(n), kWarpHashTPB, 0, st, n, dk, keys, c, Kr, flags, Kout);
        return 0;
    }
    if (!fips) LAUNCH((k_decaps_J_select<P>), cdiv(n, kHashTPB), kHashTPB, 0, st, n, dk, keys, c, Kr, flags, Kout);
    else LAUNCH((k_decaps_J_select<P, kRateSha3_256>), cdiv(n, kHashTPB), kHashTPB, 0, st, n, dk, keys, c, Kr, flags, Kout);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Generic batched driver: handles host / device memory, chunking and the multi-slot pipelines.
// ------------------------------------------------------------------------------------------------
struct Buf {
    const void *in;   // non-null for inputs
    void *out;        // non-null for outputs
    size_t item_bytes;
    bool cells = false;  // the caller's array is in the reference's cell layout: one byte per 4-byte `union byte` (ml_kem.h:35-38)
};

// Cell layout <-> dense bytes, on the device (SURVEY 8(f) N4: the stride-4 conversion off the host's critical path).
int launch_narrow(cudaStream_t st, const void *cells, void *dense, size_t bytes) {
    const size_t nw = bytes / 4;
    if (nw) LAUNCH(k_cells_to_bytes, cdiv(nw, 256), 256, 0, st, nw, (const uint4 *)cells, (uint32_t *)dense);
    return 0;
}
int launch_widen(cudaStream_t st, const void *dense, void *cells, size_t bytes) {
    const size_t nw = bytes / 4;
    if (nw) LAUNCH(k_bytes_to_cells, cdiv(nw, 256), 256, 0, st, nw, (const uint32_t *)dense, (uint4 *)cells);
    return 0;
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// run(stream, arena, n_chunk, ptrs[], first) where ptrs[i] is the device address of buffer i for this chunk and `first`
// the index of the chunk's first item within the call.
template <class Run>
int drive(const mlkem_b200_opts *o, size_t n, size_t ws_per_item, std::vector<Buf> bufs, Run run) {
    if (n == 0) return MLKEM_B200_OK;
    if (n > 0x7FFFFFFFull / 8) {
        snprintf(tl_error, sizeof tl_error, "batch too large");
        return MLKEM_B200_ERR_ARG;
    }
    for (auto &b : bufs)
        if (!b.in && !b.out) {
            snprintf(tl_error, sizeof tl_error, "NULL buffer");
            return MLKEM_B200_ERR_ARG;
        }
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
    // Calls from several host threads are serialised per device while they enqueue.  The slots (workspace + staging
    // buffer) are shared between calls and may be used from different streams: see DeviceCtx::ev_slot.
    std::unique_lock<std::mutex> call_lock(ctx->call_mutex);
    const bool on_device = o && o->mem == MLKEM_B200_MEM_DEVICE;
    static const int env_chunk = env_int("MLKEM_B200_CHUNK", 0);  // tuning knobs
    static const int env_hchunk = env_int("MLKEM_B200_HOST_CHUNK", 0);
    static const int host_slots = std::min(kHostSlots, std::max(1, env_int("MLKEM_B200_HOST_SLOTS", kHostSlots)));
    size_t chunk = (o && o->chunk_items > 0) ? (size_t)o->chunk_items
                   : (on_device ? (env_chunk > 0 ? (size_t)env_chunk : (size_t)1 << 18) : (env_hchunk > 0 ? (size_t)env_hchunk : (size_t)1 << 16));
    if (chunk > ((size_t)1 << 26)) chunk = (size_t)1 << 26;  // the kernels index rows (items x k) and list entries with int
    if (chunk > n) chunk = n;
    const size_t nchunks = (n + chunk - 1) / chunk;
    std::vector<void *> ptrs(bufs.size());
    size_t cell_dense_per_item = 0;  // dense images of cell-layout buffers live in the workspace (device path) / staging buffer (host path)
    for (auto &b : bufs)
        if (b.cells) cell_dense_per_item += (b.item_bytes + 15) & ~size_t(15);

    if (on_device) {
        for (auto &b : bufs)
            if (!aligned16(b.in ? b.in : b.out)) {
                snprintf(tl_error, sizeof tl_error, "device pointers must be 16-byte aligned");
                return MLKEM_B200_ERR_ARG;
            }
        // NULL is the CUDA default stream (what torch hands over for its default stream), not a library stream:
        // the caller orders its own work against ours through the stream it names.
        cudaStream_t st = static_cast<cudaStream_t>(o->stream);
        // Large batches are cut into chunks that take turns on the library's streams (forked from and joined back
        // into the caller's stream): the kernels of a chunk are a dependent chain that alternates between alu-bound
        // hashing and fma-heavy polynomial arithmetic, so several chains in flight fill each other's tails (the
        // clean-up pass of the matrix kernel, for one, fills barely more than one wave of blocks).
        if (!(o && o->chunk_items > 0) && n >= ((size_t)1 << 16) && nchunks < 2 && g_streams.load() > 1) {
            chunk = ((n + 1) / 2 + 1023) & ~(size_t)1023;
        }
        const size_t nch = (n + chunk - 1) / chunk;
        int nstreams = g_streams.load();
        if (nstreams > kDevSlots) nstreams = kDevSlots;
        if ((size_t)nstreams > nch) nstreams = (int)nch;
        if (nstreams < 1) nstreams = 1;
        {
            std::lock_guard<std::mutex> lock(g_mutex);
            for (int k = 0; k < nstreams; k++)
                if (int rc = ensure_buffer(&ctx->ws[k], &ctx->ws_bytes[k], chunk * (ws_per_item + cell_dense_per_item) + kWsSlack + 256 * bufs.size(),
                                           ctx->ev_slot[k]))
                    return rc;
        }
        const bool fork = nstreams > 1;
        if (fork) CU(cudaEventRecord(ctx->ev_fork, st));
        for (int k = 0; k < nstreams; k++) {
            cudaStream_t sk = fork ? ctx->stream[k] : st;
            if (fork) CU(cudaStreamWaitEvent(sk, ctx->ev_fork, 0));
            CU(cudaStreamWaitEvent(sk, ctx->ev_slot[k], 0));  // the previous user of slot k, whatever stream it was on
        }
        int rc = 0;
        for (size_t ci = 0; ci < nch && !rc; ci++) {
            size_t i0 = ci * chunk, cn = (i0 + chunk <= n) ? chunk : n - i0;
            const int k = fork ? (int)(ci % nstreams) : 0;
            cudaStream_t sk = fork ? ctx->stream[k] : st;
            Arena arena(ctx->ws[k]);
            for (size_t b = 0; b < bufs.size() && !rc; b++) {
                const uint8_t *base = static_cast<const uint8_t *>(bufs[b].in ? bufs[b].in : bufs[b].out);
                if (!bufs[b].cells) {
                    ptrs[b] = const_cast<uint8_t *>(base) + i0 * bufs[b].item_bytes;
                } else {  // dense image in the workspace; inputs are narrowed now, outputs widened after the pipeline
                    ptrs[b] = arena.take<uint8_t>(cn * bufs[b].item_bytes);
                    if (bufs[b].in) rc = launch_narrow(sk, base + 4 * i0 * bufs[b].item_bytes, ptrs[b], cn * bufs[b].item_bytes);
                }
            }
            if (!rc) rc = run(sk, arena, (int)cn, ptrs.data(), i0);
            for (size_t b = 0; b < bufs.size() && !rc; b++)
                if (bufs[b].cells && bufs[b].out)
                    rc = launch_widen(sk, ptrs[b], static_cast<uint8_t *>(bufs[b].out) + 4 * i0 * bufs[b].item_bytes, cn * bufs[b].item_bytes);
        }
        // also on the error path: whatever was enqueued is joined back into the caller's stream and the slots are marked
        for (int k = 0; k < nstreams; k++) {
            cudaStream_t sk = fork ? ctx->stream[k] : st;
            cudaError_t e = cudaEventRecord(ctx->ev_slot[k], sk);
            if (fork && e == cudaSuccess) e = cudaEventRecord(ctx->ev_join[k], sk);
            if (fork && e == cudaSuccess) e = cudaStreamWaitEvent(st, ctx->ev_join[k], 0);
            if (e != cudaSuccess && !rc) {
                snprintf(tl_error, sizeof tl_error, "stream join failed: %s", cudaGetErrorString(e));
                rc = MLKEM_B200_ERR_CUDA;
            }
        }
        return rc;
    }

    // host memory: stage each chunk through device buffers, rotating over the staging slots / streams so that the
    // copies of one chunk overlap the kernels of the other
    size_t io_per_item = 0;
    for (auto &b : bufs) io_per_item += ((b.item_bytes + 15) & ~size_t(15)) * (b.cells ? 5 : 1);  // cells: 4x image + dense image
    const int nslots = nchunks > 1 ? (int)std::min<size_t>(host_slots, nchunks) : 1;
    const int s0 = ctx->host_group * kHostSlots;  // this call's slot group
    ctx->host_group ^= 1;
    {
        std::lock_guard<std::mutex> lock(g_mutex);
        for (int s = s0; s < s0 + nslots; s++) {
            if (int rc = ensure_buffer(&ctx->ws[s], &ctx->ws_bytes[s], chunk * ws_per_item + kWsSlack, ctx->ev_slot[s])) return rc;
            if (int rc = ensure_buffer(&ctx->io[s], &ctx->io_bytes[s], chunk * io_per_item + 512 * bufs.size(), ctx->ev_slot[s])) return rc;
        }
    }
    for (int s = s0; s < s0 + nslots; s++) CU(cudaStreamWaitEvent(ctx->stream[s], ctx->ev_slot[s], 0));
    auto chunk_of = [&](size_t ci) -> int {
        const int s = s0 + (int)(ci % nslots);
        cudaStream_t st = ctx->stream[s];
        size_t i0 = ci * chunk, cn = (i0 + chunk <= n) ? chunk : n - i0;
        Arena io(ctx->io[s]);
        std::vector<uint8_t *> wide(bufs.size(), nullptr);  // device image of a cell-layout buffer (4 bytes per byte)
        for (size_t b = 0; b < bufs.size(); b++) {
            const size_t ib = bufs[b].item_bytes, scale = bufs[b].cells ? 4 : 1;
            ptrs[b] = io.take<uint8_t>(chunk * ib);
            uint8_t *land = (uint8_t *)ptrs[b];
            if (bufs[b].cells) land = wide[b] = io.take<uint8_t>(4 * chunk * ib);
            if (bufs[b].in) {
                CU(cudaMemcpyAsync(land, static_cast<const uint8_t *>(bufs[b].in) + scale * i0 * ib, scale * cn * ib, cudaMemcpyHostToDevice, st));
                if (bufs[b].cells)
                    if (int rc = launch_narrow(st, land, ptrs[b], cn * ib)) return rc;
            }
        }
        Arena arena(ctx->ws[s]);
        if (int rc = run(st, arena, (int)cn, ptrs.data(), i0)) return rc;
        for (size_t b = 0; b < bufs.size(); b++)
            if (bufs[b].out) {
                const size_t ib = bufs[b].item_bytes, scale = bufs[b].cells ? 4 : 1;
                const uint8_t *src = (const uint8_t *)ptrs[b];
                if (bufs[b].cells) {
                    if (int rc = launch_widen(st, ptrs[b], wide[b], cn * ib)) return rc;
                    src = wide[b];
                }
                CU(cudaMemcpyAsync(static_cast<uint8_t *>(bufs[b].out) + scale * i0 * ib, src, scale * cn * ib, cudaMemcpyDeviceToHost, st));
            }
        return 0;
    };
    int rc = 0;
    for (size_t ci = 0; ci < nchunks && !rc; ci++) rc = chunk_of(ci);
    for (int s = s0; s < s0 + nslots; s++) cudaEventRecord(ctx->ev_slot[s], ctx->stream[s]);
    // Enqueueing is over: the next call may start filling the slots behind this one (it waits on ev_slot), so that the
    // D2H tail of this call overlaps the H2D head of the next.
    call_lock.unlock();
    // MLKEM_B200_FLAG_ASYNC: return now; the caller keeps its (pinned) buffers untouched until mlkem_b200_synchronize().
    if (!rc && o && (o->flags & MLKEM_B200_FLAG_ASYNC)) return MLKEM_B200_OK;
    // also on the error path: nothing may still be writing into the caller's buffers when the call returns
    for (int s = s0; s < s0 + nslots; s++) {
        cudaError_t e = cudaStreamSynchronize(ctx->stream[s]);
        if (e != cudaSuccess && !rc) {
            snprintf(tl_error, sizeof tl_error, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
            rc = MLKEM_B200_ERR_CUDA;
        }
    }
    return rc;
}

int group_limit_of(const mlkem_b200_opts *o) { return (o && o->sample_group_limit > 0) ? o->sample_group_limit : 278; }
bool fips_of(const mlkem_b200_opts *o) { return o && (o->flags & MLKEM_B200_FLAG_FIPS203); }

#define DISPATCH_SET(param_set, CALL)                   \
    switch (param_set) {                                \
    case 512: { using P = P512; CALL; } break;          \
    case 768: { using P = P768; CALL; } break;          \
    case 1024: { using P = P1024; CALL; } break;        \
    default: return MLKEM_B200_ERR_PARAM;               \
    }

inline unsigned prim_grid(size_t n_polys) {
    size_t blocks = (n_polys + (kPrimTPB / 32) - 1) / (kPrimTPB / 32);
    size_t cap = 148 * 8 * 4;  // a few waves of 8 resident blocks per SM; the kernels grid-stride
    return (unsigned)(blocks < cap ? blocks : cap);
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char *mlkem_b200_version(void) { return "mlkem_b200 0.1 (sm_100a)"; }
const char *mlkem_b200_last_error(void) { return tl_error; }
unsigned long long mlkem_b200_launch_count(void) { return g_launches.load(); }
int mlkem_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
int mlkem_b200_synchronize(int device, void *stream) {
    DeviceGuard guard;
    if (device >= 0)
        if (int rc = guard.enter(device)) return rc;
    if (stream) CU(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    else CU(cudaDeviceSynchronize());
    return 0;
}
void *mlkem_b200_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();  // a failed allocation must not linger as the "last error" of the next kernel launch
        return nullptr;
    }
    return p;
}
void *mlkem_b200_host_alloc_wc(size_t bytes) {
    void *p = nullptr;
    // write-combined mappings are a limited resource (8 processes x 20 GB did not fit on the 8-GPU box): callers fall back
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocWriteCombined) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void mlkem_b200_host_free(void *p) {
    if (p) cudaFreeHost(p);
}
void mlkem_b200_release(int device) {
    if (device < 0 || device >= kMaxDevices) return;
    DeviceCtx &c = g_ctx[device];
    // lock order everywhere: misc_mutex (public-wrapper batches) -> call_mutex (drive) -> g_mutex (buffer growth)
    std::lock_guard<std::mutex> misc_lock(c.misc_mutex);
    std::lock_guard<std::mutex> call_lock(c.call_mutex);
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!c.ready) return;
    DeviceGuard guard;
    if (guard.enter(device)) return;
    cudaDeviceSynchronize();
    // the workspaces hold secret-dependent intermediates (sigma, s^ / e^, m', K' || r') and staged keys: wipe, then free
    auto wipe_free = [](void *&p, size_t &bytes) {
        if (p) {
            cudaMemset(p, 0, bytes);
            cudaFree(p);
        }
        p = nullptr;
        bytes = 0;
    };
    for (int s = 0; s < kSlots; s++) {
        wipe_free(c.ws[s], c.ws_bytes[s]);
        wipe_free(c.io[s], c.io_bytes[s]);
    }
    wipe_free(c.misc, c.misc_bytes);
}

static unsigned k_of(int set) { return set == 512 ? 2 : set == 768 ? 3 : set == 1024 ? 4 : 0; }
unsigned mlkem_b200_ek_bytes(int set) { unsigned k = k_of(set); return k ? 384 * k + 32 : 0; }
unsigned mlkem_b200_dk_bytes(int set) { unsigned k = k_of(set); return k ? 768 * k + 96 : 0; }
unsigned mlkem_b200_dkpke_bytes(int set) { unsigned k = k_of(set); return k ? 384 * k : 0; }
unsigned mlkem_b200_ct_bytes(int set) {
    switch (set) {
    case 512: return P512::C;
    case 768: return P768::C;
    case 1024: return P1024::C;
    default: return 0;
    }
}

int mlkem_b200_keygen_batch(int set, size_t n, const uint8_t *d, const uint8_t *z, uint8_t *ek, uint8_t *dk, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{d, nullptr, 32}, {z, nullptr, 32}, {nullptr, ek, P::EK}, {nullptr, dk, P::DK}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_keygen<P>(st, ws, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint8_t *)p[2], (uint8_t *)p[3], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_pke_keygen_batch(int set, size_t n, const uint8_t *d, uint8_t *ek, uint8_t *dkpke, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{d, nullptr, 32}, {nullptr, ek, P::EK}, {nullptr, dkpke, P::DKPKE}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_keygen<P>(st, ws, cn, (const uint8_t *)p[0], nullptr, (uint8_t *)p[1], (uint8_t *)p[2], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_encaps_batch(int set, size_t n, const uint8_t *ek, const uint8_t *m, uint8_t *c, uint8_t *K, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{ek, nullptr, P::EK}, {m, nullptr, 32}, {nullptr, c, P::C}, {nullptr, K, 32}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_encaps<P>(st, ws, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint8_t *)p[2], (uint8_t *)p[3], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_decaps_batch(int set, size_t n, const uint8_t *dk, const uint8_t *c, uint8_t *K, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{dk, nullptr, P::DK}, {c, nullptr, P::C}, {nullptr, K, 32}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_decaps<P>(st, ws, cn, (const uint8_t *)p[0], KeySel{}, (const uint8_t *)p[1], (uint8_t *)p[2], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_check_dk_batch(int set, size_t n, const uint8_t *dk, int32_t *status, const mlkem_b200_opts *o) {
    DISPATCH_SET(set, return drive(o, n, 0, {{dk, nullptr, P::DK}, {nullptr, status, 4}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
                     if (cn <= warp_hash_max()) LAUNCH((k_check_dk_hash_warp<P>), warp_hash_grid(cn), kWarpHashTPB, 0, st, cn, (const uint8_t *)p[0], (int *)p[1]);
                     else LAUNCH((k_check_dk_hash<P>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], (int *)p[1]);
                     return 0;
                 }));
    return MLKEM_B200_ERR_PARAM;
}

}  // extern "C" (helpers with C++ linkage follow)

// ---- batched forms of the public wrappers (ml_kem.c:1233-1359): entropy, length checks, dk hash check ----------

// ml_kem.c:458 getRandomBytes reads 32 unsigned ints from /dev/urandom and keeps each modulo 256, i.e. 32 uniform
// bytes; here the bytes are read directly.
static int host_entropy(uint8_t *out, size_t bytes) {
    FILE *f = fopen("/dev/urandom", "rb");
    if (!f) return -2;
    size_t got = fread(out, 1, bytes, f);
    fclose(f);
    return got == bytes ? 0 : -2;  // ml_errno -2: random bit generation failed (ml_kem.c:1243,1297)
}

// A lease on the device's pooled scratch buffer (entropy seeds, status words): no cudaMalloc / cudaFree per call.
// Held until the user's stream has drained, then wiped.
struct MiscLease {
    DeviceCtx *ctx = nullptr;
    std::unique_lock<std::mutex> lock;
    uint8_t *ptr = nullptr;
    size_t bytes = 0;
    cudaStream_t st = nullptr;
    int take(DeviceCtx *c, size_t need, cudaStream_t stream) {
        ctx = c;
        st = stream;
        bytes = need;
        lock = std::unique_lock<std::mutex>(c->misc_mutex);
        if (int rc = ensure_buffer(&c->misc, &c->misc_bytes, need)) return rc;
        ptr = static_cast<uint8_t *>(c->misc);
        return 0;
    }
    ~MiscLease() {
        if (!ptr) return;
        cudaMemsetAsync(ptr, 0, bytes, st);  // seeds are secrets
        cudaStreamSynchronize(st);
    }
};

// Runs `call(seed_ptr)` with `bytes` of fresh entropy placed where opts says the buffers live.
template <class F>
static int with_entropy(const mlkem_b200_opts *o, size_t bytes, F call) {
    struct Wiped {  // the host copy of the seeds is zeroed on every exit path
        std::vector<uint8_t> v;
        ~Wiped() { explicit_bzero(v.data(), v.size()); }
    } host{std::vector<uint8_t>(bytes)};
    if (int rc = host_entropy(host.v.data(), bytes)) return rc;
    if (!(o && o->mem == MLKEM_B200_MEM_DEVICE)) return call(host.v.data());
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(o->stream);
    MiscLease lease;
    if (int rc = lease.take(ctx, bytes, st)) return rc;
    // on the caller's stream: ordered before the kernels that read the seeds (pageable source: the call returns once the
    // bytes are staged, and the lease drains the stream before the host copy and the device buffer are wiped)
    CU(cudaMemcpyAsync(lease.ptr, host.v.data(), bytes, cudaMemcpyHostToDevice, st));
    return call(lease.ptr);
}

// The public-wrapper batches read results (status words) or wipe inputs (seeds) on the host right after their inner calls:
// they are synchronous whatever the caller's flags say.
struct SyncOpts {
    mlkem_b200_opts v;
    const mlkem_b200_opts *p;
    explicit SyncOpts(const mlkem_b200_opts *o) : v(o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0}), p(o ? &v : nullptr) {
        v.flags &= ~MLKEM_B200_FLAG_ASYNC;
    }
};

// The modulus check of KEM_Encaps (ml_kem.c:1274-1291) for n keys: an identity in the reference (its ByteDecode12 never
// reduces), see SURVEY D4.  In FIPS mode it is a real check: any coefficient >= q in any key rejects the call with -4.
// Its MiscLease (device-memory calls) is released when it returns.
static int fips_modulus_check(int set, size_t n, const uint8_t *ek, const mlkem_b200_opts *o) {
    if (!fips_of(o)) return 0;
    std::vector<int32_t> st_host(n);
    const bool on_dev = o->mem == MLKEM_B200_MEM_DEVICE;
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    MiscLease lease;
    int32_t *status = st_host.data();
    if (on_dev) {
        if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
        if (int rc = lease.take(ctx, 4 * n, static_cast<cudaStream_t>(o->stream))) return rc;
        status = reinterpret_cast<int32_t *>(lease.ptr);
    }
    int rc = MLKEM_B200_ERR_PARAM;
    switch (set) {
#define MODCHK(PS, PT)                                                                                                              \
    case PS:                                                                                                                        \
        rc = drive(o, n, 0, {{ek, nullptr, PT::EK}, {nullptr, status, 4}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) { \
            LAUNCH((k_check_ek_modulus<PT>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], (int *)p[1]);            \
            return 0;                                                                                                               \
        });                                                                                                                         \
        break;
        MODCHK(512, P512) MODCHK(768, P768) MODCHK(1024, P1024)
#undef MODCHK
    }
    if (!rc && on_dev) {
        cudaStream_t st = static_cast<cudaStream_t>(o->stream);
        if (cudaMemcpyAsync(st_host.data(), status, 4 * n, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            rc = MLKEM_B200_ERR_CUDA;
    }
    if (rc) return rc;
    for (size_t i = 0; i < n; i++)
        if (st_host[i] != 0) return MLKEM_B200_ERR_MODULUS;
    return 0;
}

// ---- seeded randomness (include/mlkem_b200.h, "randomness expanded on the device") -------------------------------------
// The 32-byte call seed of a seeded call: the caller's bytes, or 32 fresh bytes of host_entropy when seed is NULL.  It is
// copied into the device's pooled misc scratch on `st`, ahead of every later use on that stream; the host copy is zeroed with
// explicit_bzero and the device copy by the lease (after `st` has drained) when the object goes out of scope.  A seed decides
// every secret of its call, so it never sits in a kernel-parameter buffer the library cannot wipe.
struct CallSeed {
    struct Host {
        uint8_t b[32] = {};
        ~Host() { explicit_bzero(b, sizeof b); }
    } host;
    MiscLease lease;  // declared after `host`: drained and wiped first
    const uint8_t *dev = nullptr;
    int take(DeviceCtx *ctx, const uint8_t *seed, cudaStream_t st) {
        if (seed) memcpy(host.b, seed, sizeof host.b);
        else if (int rc = host_entropy(host.b, sizeof host.b)) return rc;
        if (int rc = lease.take(ctx, sizeof host.b, st)) return rc;
        CU(cudaMemcpyAsync(lease.ptr, host.b, sizeof host.b, cudaMemcpyHostToDevice, st));
        dev = lease.ptr;
        return 0;
    }
};
constexpr uint32_t kSeedTagKeyGen = 1, kSeedTagEncaps = 2;

// R_j of items first .. first + n - 1 into out0 (and out1): see k_expand_seed.
static int expand_seed(cudaStream_t st, int n, const uint8_t *seed, size_t first, uint32_t tag, uint8_t *out0, uint8_t *out1) {
    LAUNCH(k_expand_seed, cdiv(n, kHashTPB), kHashTPB, 0, st, n, seed, (unsigned long long)first, tag, out0, out1);
    return 0;
}

// Runs `call(seed_on_device)` for a seeded unkeyed / keyed call with synchronous options `o` (SyncOpts): the seed is placed on
// the caller's stream (device memory) or on a library stream that is drained before the call's own streams read it (host memory).
template <class F>
static int with_call_seed(const mlkem_b200_opts *o, const uint8_t *seed, F call) {
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
    const bool on_dev = o && o->mem == MLKEM_B200_MEM_DEVICE;
    cudaStream_t st = on_dev ? static_cast<cudaStream_t>(o->stream) : ctx->stream[0];
    CallSeed cs;
    if (int rc = cs.take(ctx, seed, st)) return rc;
    if (!on_dev) CU(cudaStreamSynchronize(st));
    return call(cs.dev);
}

extern "C" {

int mlkem_b200_kem_keygen_batch(int set, size_t n, uint8_t *ek, uint8_t *dk, const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    if (!mlkem_b200_ek_bytes(set)) return MLKEM_B200_ERR_PARAM;
    if (n == 0) return MLKEM_B200_OK;
    return with_entropy(o, 64 * n, [&](uint8_t *seeds) { return mlkem_b200_keygen_batch(set, n, seeds, seeds + 32 * n, ek, dk, o); });
}

int mlkem_b200_kem_encaps_batch(int set, size_t n, const uint8_t *ek, size_t ek_len, uint8_t *c, uint8_t *K, const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    unsigned want = mlkem_b200_ek_bytes(set);
    if (!want) return MLKEM_B200_ERR_PARAM;
    if (ek_len != want) return MLKEM_B200_ERR_LENGTH;  // type check, ml_kem.c:1267
    // modulus check (ml_kem.c:1274-1291): an identity in the reference (its ByteDecode12 never reduces), see SURVEY D4.
    // In FIPS mode it is a real check: any coefficient >= q in any key rejects the call with -4.
    if (n == 0) return MLKEM_B200_OK;
    if (int rc = fips_modulus_check(set, n, ek, o)) return rc;
    return with_entropy(o, 32 * n, [&](uint8_t *m) { return mlkem_b200_encaps_batch(set, n, ek, m, c, K, o); });
}

int mlkem_b200_kem_decaps_batch(int set, size_t n, const uint8_t *dk, size_t dk_len, const uint8_t *c, size_t c_len, uint8_t *K,
                                int32_t *status, const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    if (!mlkem_b200_ek_bytes(set)) return MLKEM_B200_ERR_PARAM;
    if (c_len != mlkem_b200_ct_bytes(set)) return MLKEM_B200_ERR_LENGTH;   // ml_kem.c:1321
    if (dk_len != mlkem_b200_dk_bytes(set)) return MLKEM_B200_ERR_LENGTH;  // ml_kem.c:1329
    if (!status) return MLKEM_B200_ERR_ARG;
    if (int rc = mlkem_b200_check_dk_batch(set, n, dk, status, o)) return rc;  // hash check, ml_kem.c:1336-1350
    if (int rc = mlkem_b200_decaps_batch(set, n, dk, c, K, o)) return rc;
    if (n == 0) return MLKEM_B200_OK;
    if (o && o->mem == MLKEM_B200_MEM_DEVICE) {
        int dev;
        DeviceCtx *ctx;
        DeviceGuard guard;  // the stream belongs to opts->device, which need not be the calling thread's current device
        if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
        cudaStream_t st = static_cast<cudaStream_t>(o->stream);
        LAUNCH(k_mask_keys, cdiv(n, kHashTPB), kHashTPB, 0, st, (int)n, (const int *)status, K);
    } else {
        for (size_t i = 0; i < n; i++)
            if (status[i] != 0) memset(K + 32 * i, 0, 32);
    }
    return MLKEM_B200_OK;
}

// KEM_KeyGen with (d_j, z_j) expanded on the device from the call seed into the chunk workspace: nothing but the seed crosses
// PCIe host-to-device.
int mlkem_b200_kem_keygen_seeded_batch(int set, size_t n, const uint8_t *seed, uint8_t *ek, uint8_t *dk, const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    if (!mlkem_b200_ek_bytes(set)) return MLKEM_B200_ERR_PARAM;
    if (n == 0) return MLKEM_B200_OK;
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    return with_call_seed(o, seed, [&](const uint8_t *dseed) -> int {
        DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>() + 64, {{nullptr, ek, P::EK}, {nullptr, dk, P::DK}},
                                       [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t first) {
                                           uint8_t *d = ws.take<uint8_t>((size_t)cn * 32), *z = ws.take<uint8_t>((size_t)cn * 32);
                                           if (int rc = expand_seed(st, cn, dseed, first, kSeedTagKeyGen, d, z)) return rc;
                                           return enqueue_keygen<P>(st, ws, cn, d, z, (uint8_t *)p[0], (uint8_t *)p[1], gl, fips);
                                       }));
        return MLKEM_B200_ERR_PARAM;
    });
}

// KEM_Encaps with m_j expanded on the device from the call seed: the checks of mlkem_b200_kem_encaps_batch, then Encaps_internal.
int mlkem_b200_kem_encaps_seeded_batch(int set, size_t n, const uint8_t *ek, size_t ek_len, const uint8_t *seed, uint8_t *c, uint8_t *K,
                                       const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    unsigned want = mlkem_b200_ek_bytes(set);
    if (!want) return MLKEM_B200_ERR_PARAM;
    if (ek_len != want) return MLKEM_B200_ERR_LENGTH;  // type check, ml_kem.c:1267
    if (n == 0) return MLKEM_B200_OK;
    if (int rc = fips_modulus_check(set, n, ek, o)) return rc;  // its lease is released before the seed's is taken
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    return with_call_seed(o, seed, [&](const uint8_t *dseed) -> int {
        DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>() + 32, {{ek, nullptr, P::EK}, {nullptr, c, P::C}, {nullptr, K, 32}},
                                       [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t first) {
                                           uint8_t *m = ws.take<uint8_t>((size_t)cn * 32);
                                           if (int rc = expand_seed(st, cn, dseed, first, kSeedTagEncaps, m, nullptr)) return rc;
                                           return enqueue_encaps<P>(st, ws, cn, (const uint8_t *)p[0], m, (uint8_t *)p[1], (uint8_t *)p[2], gl, fips);
                                       }));
        return MLKEM_B200_ERR_PARAM;
    });
}

int mlkem_b200_pke_encrypt_batch(int set, size_t n, const uint8_t *ek, const uint8_t *m, const uint8_t *r, uint8_t *c, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{ek, nullptr, P::EK}, {m, nullptr, 32}, {r, nullptr, 32}, {nullptr, c, P::C}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_encrypt<P>(st, ws, cn, (const uint8_t *)p[0], P::EK, KeySel{}, (const uint8_t *)p[1], (const uint8_t *)p[2], 32,
                                                                 (uint8_t *)p[3], nullptr, nullptr, gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_pke_decrypt_batch(int set, size_t n, const uint8_t *dk, size_t dk_stride, const uint8_t *c, uint8_t *m, const mlkem_b200_opts *o) {
    if (dk_stride % 16 != 0) {
        snprintf(tl_error, sizeof tl_error, "dk_stride must be a multiple of 16");
        return MLKEM_B200_ERR_ARG;
    }
    DISPATCH_SET(set, {
        if (dk_stride < (size_t)P::DKPKE) return MLKEM_B200_ERR_LENGTH;
        return drive(o, n, 0, {{dk, nullptr, dk_stride}, {c, nullptr, P::C}, {nullptr, m, 32}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
            LAUNCH((k_decrypt<P>), warp_grid(cn, kWarpTPB / 32), kWarpTPB, 0, st, cn, (const uint8_t *)p[0], dk_stride, KeySel{}, (const uint8_t *)p[1], (uint8_t *)p[2]);
            return 0;
        });
    });
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_ntt_batch(size_t n, const uint16_t *f, uint16_t *fh, const mlkem_b200_opts *o) {
    return drive(o, n, 0, {{f, nullptr, 512}, {nullptr, fh, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        LAUNCH(k_ntt_batch, prim_grid(cn), kPrimTPB, 0, st, cn, (const uint16_t *)p[0], (uint16_t *)p[1]);
        return 0;
    });
}
int mlkem_b200_intt_batch(size_t n, const uint16_t *fh, uint16_t *f, const mlkem_b200_opts *o) {
    return drive(o, n, 0, {{fh, nullptr, 512}, {nullptr, f, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        LAUNCH(k_intt_batch, prim_grid(cn), kPrimTPB, 0, st, cn, (const uint16_t *)p[0], (uint16_t *)p[1]);
        return 0;
    });
}
int mlkem_b200_multiply_ntts_batch(size_t n, const uint16_t *f, const uint16_t *g, uint16_t *h, const mlkem_b200_opts *o) {
    return drive(o, n, 0, {{f, nullptr, 512}, {g, nullptr, 512}, {nullptr, h, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        LAUNCH(k_mulntt_batch, prim_grid(cn), kPrimTPB, 0, st, cn, (const uint16_t *)p[0], (const uint16_t *)p[1], (uint16_t *)p[2]);
        return 0;
    });
}

static int addsub_impl(size_t n, const uint16_t *u, const uint16_t *v, uint16_t *z, const mlkem_b200_opts *o, bool sub) {
    return drive(o, n * 32, 0, {{u, nullptr, 16}, {v, nullptr, 16}, {nullptr, z, 16}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        unsigned grid = cdiv(cn, kPrimTPB);
        if (grid > 148 * 32) grid = 148 * 32;
        if (sub) LAUNCH((k_poly_addsub<true>), grid, kPrimTPB, 0, st, (long long)cn, (const uint4 *)p[0], (const uint4 *)p[1], (uint4 *)p[2]);
        else LAUNCH((k_poly_addsub<false>), grid, kPrimTPB, 0, st, (long long)cn, (const uint4 *)p[0], (const uint4 *)p[1], (uint4 *)p[2]);
        return 0;
    });
}
int mlkem_b200_poly_add_batch(size_t n, const uint16_t *u, const uint16_t *v, uint16_t *z, const mlkem_b200_opts *o) { return addsub_impl(n, u, v, z, o, false); }
int mlkem_b200_poly_sub_batch(size_t n, const uint16_t *u, const uint16_t *v, uint16_t *z, const mlkem_b200_opts *o) { return addsub_impl(n, u, v, z, o, true); }
int mlkem_b200_vector_multiply_batch(int k, size_t n, const uint16_t *u, const uint16_t *v, uint16_t *w, const mlkem_b200_opts *o) {
    if (k < 1 || k > 16) return MLKEM_B200_ERR_ARG;
    return drive(o, n, 0, {{u, nullptr, (size_t)512 * k}, {v, nullptr, (size_t)512 * k}, {nullptr, w, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        LAUNCH(k_vecmul_batch, prim_grid(cn), kPrimTPB, 0, st, cn, k, (const uint16_t *)p[0], (const uint16_t *)p[1], (uint16_t *)p[2]);
        return 0;
    });
}

int mlkem_b200_sample_ntt_batch(size_t n, const uint8_t *seeds, uint16_t *a, uint8_t *seeds_after, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    std::vector<Buf> bufs = {{seeds, nullptr, 34}, {nullptr, a, 512}};
    if (seeds_after) bufs.push_back({nullptr, seeds_after, 34});
    const bool has_after = seeds_after != nullptr;
    // 34-byte items are not 16-byte multiples: the chunk size must keep chunk starts aligned
    mlkem_b200_opts oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo.chunk_items <= 0) oo.chunk_items = 1 << 16;
    oo.chunk_items = (oo.chunk_items + 7) & ~7;
    return drive(&oo, n, 0, bufs, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        LAUNCH(k_sample_ntt_batch, cdiv(cn, 128), 128, 128 * kSlotWords * 4, st, cn, (const uint8_t *)p[0], (uint16_t *)p[1],
               has_after ? (uint8_t *)p[2] : (uint8_t *)nullptr, gl);
        return 0;
    });
}

int mlkem_b200_cbd_batch(int eta, size_t n, const uint8_t *bytes, uint16_t *f, const mlkem_b200_opts *o) {
    if (eta != 2 && eta != 3) return MLKEM_B200_ERR_ARG;
    return drive(o, n, 0, {{bytes, nullptr, (size_t)64 * eta}, {nullptr, f, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        if (eta == 2) LAUNCH((k_cbd_batch<2>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint8_t *)p[0], (uint16_t *)p[1]);
        else LAUNCH((k_cbd_batch<3>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint8_t *)p[0], (uint16_t *)p[1]);
        return 0;
    });
}
int mlkem_b200_prf_cbd_batch(int eta, size_t n, const uint8_t *seeds, const uint8_t *nonces, uint16_t *f, const mlkem_b200_opts *o) {
    if (eta != 2 && eta != 3) return MLKEM_B200_ERR_ARG;
    const bool fips = fips_of(o);
    mlkem_b200_opts oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo.chunk_items <= 0) oo.chunk_items = 1 << 16;
    oo.chunk_items = (oo.chunk_items + 15) & ~15;  // 1-byte nonces: keep chunk starts 16-byte aligned
    return drive(&oo, n, 0, {{seeds, nullptr, 32}, {nonces, nullptr, 1}, {nullptr, f, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        if (fips) {
            if (eta == 2) LAUNCH((k_prf_cbd_batch<2, kRateSha3_256>), cdiv(cn, kNoiseTPB), kNoiseTPB, 0, st, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint16_t *)p[2]);
            else LAUNCH((k_prf_cbd_batch<3, kRateSha3_256>), cdiv(cn, kNoiseTPB), kNoiseTPB, 0, st, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint16_t *)p[2]);
            return 0;
        }
        if (eta == 2) LAUNCH((k_prf_cbd_batch<2>), cdiv(cn, kNoiseTPB), kNoiseTPB, 0, st, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint16_t *)p[2]);
        else LAUNCH((k_prf_cbd_batch<3>), cdiv(cn, kNoiseTPB), kNoiseTPB, 0, st, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint16_t *)p[2]);
        return 0;
    });
}

#define DISPATCH_D(d, CALL)                    \
    switch (d) {                               \
    case 1: { constexpr int D = 1; CALL; } break;   \
    case 4: { constexpr int D = 4; CALL; } break;   \
    case 5: { constexpr int D = 5; CALL; } break;   \
    case 10: { constexpr int D = 10; CALL; } break; \
    case 11: { constexpr int D = 11; CALL; } break; \
    case 12: { constexpr int D = 12; CALL; } break; \
    default: return MLKEM_B200_ERR_ARG;        \
    }

static int encode_impl(int d, size_t n, const uint16_t *F, uint8_t *B, const mlkem_b200_opts *o, bool comp) {
    return drive(o, n, 0, {{F, nullptr, 512}, {nullptr, B, (size_t)32 * d}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        DISPATCH_D(d, {
            if (comp) LAUNCH((k_encode_batch<D, true>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint16_t *)p[0], (uint8_t *)p[1]);
            else LAUNCH((k_encode_batch<D, false>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint16_t *)p[0], (uint8_t *)p[1]);
        });
        return 0;
    });
}
static int decode_impl(int d, size_t n, const uint8_t *B, uint16_t *F, const mlkem_b200_opts *o, bool decomp) {
    return drive(o, n, 0, {{B, nullptr, (size_t)32 * d}, {nullptr, F, 512}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        DISPATCH_D(d, {
            if (decomp) LAUNCH((k_decode_batch<D, true>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint8_t *)p[0], (uint16_t *)p[1]);
            else LAUNCH((k_decode_batch<D, false>), prim_grid(cn), kPrimTPB, 0, st, cn, (const uint8_t *)p[0], (uint16_t *)p[1]);
        });
        return 0;
    });
}
int mlkem_b200_byte_encode_batch(int d, size_t n, const uint16_t *F, uint8_t *B, const mlkem_b200_opts *o) { return encode_impl(d, n, F, B, o, false); }
int mlkem_b200_compress_encode_batch(int d, size_t n, const uint16_t *F, uint8_t *B, const mlkem_b200_opts *o) { return encode_impl(d, n, F, B, o, true); }
int mlkem_b200_byte_decode_batch(int d, size_t n, const uint8_t *B, uint16_t *F, const mlkem_b200_opts *o) { return decode_impl(d, n, B, F, o, false); }
int mlkem_b200_decode_decompress_batch(int d, size_t n, const uint8_t *B, uint16_t *F, const mlkem_b200_opts *o) { return decode_impl(d, n, B, F, o, true); }

static int compress_impl(int d, size_t ncoef, const uint16_t *x, uint16_t *y, const mlkem_b200_opts *o, bool decomp) {
    if (ncoef % 8 != 0) return MLKEM_B200_ERR_ARG;
    if (d < 1 || d > 12) return MLKEM_B200_ERR_ARG;
    return drive(o, ncoef / 8, 0, {{x, nullptr, 16}, {nullptr, y, 16}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        unsigned grid = cdiv(cn, kPrimTPB);
        if (grid > 148 * 32) grid = 148 * 32;
#define CASE_D(DD)                                                                                                                        \
    case DD:                                                                                                                              \
        if (decomp) LAUNCH((k_compress_batch<DD, true>), grid, kPrimTPB, 0, st, (long long)cn, (const uint4 *)p[0], (uint4 *)p[1]);        \
        else LAUNCH((k_compress_batch<DD, false>), grid, kPrimTPB, 0, st, (long long)cn, (const uint4 *)p[0], (uint4 *)p[1]);              \
        break;
        switch (d) {
            CASE_D(1) CASE_D(2) CASE_D(3) CASE_D(4) CASE_D(5) CASE_D(6) CASE_D(7) CASE_D(8) CASE_D(9) CASE_D(10) CASE_D(11) CASE_D(12)
        }
#undef CASE_D
        return 0;
    });
}
int mlkem_b200_compress_batch(int d, size_t ncoef, const uint16_t *x, uint16_t *y, const mlkem_b200_opts *o) { return compress_impl(d, ncoef, x, y, o, false); }
int mlkem_b200_decompress_batch(int d, size_t ncoef, const uint16_t *y, uint16_t *x, const mlkem_b200_opts *o) { return compress_impl(d, ncoef, y, x, o, true); }

int mlkem_b200_hash_batch(int which, size_t n, size_t len, const uint8_t *in, uint8_t *out, const mlkem_b200_opts *o) {
    if (len % 8 != 0 || which < 0 || which > 3) return MLKEM_B200_ERR_ARG;
    if (len % 16 != 0 && !(o && o->mem == MLKEM_B200_MEM_DEVICE)) {
        // chunk starts stay 16-byte aligned when the chunk size is even
    }
    mlkem_b200_opts oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo.chunk_items <= 0) oo.chunk_items = 1 << 16;
    oo.chunk_items = (oo.chunk_items + 1) & ~1;
    const int nw = (int)(len / 8);
    return drive(&oo, n, 0, {{in, nullptr, len ? len : 1}, {nullptr, out, which == 1 ? (size_t)64 : (size_t)32}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        if (which == 0) LAUNCH((k_hash_words<kRateSha3_256, 4>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], nw, kSfxHash, (uint8_t *)p[1]);
        else if (which == 1) LAUNCH((k_hash_words<kRateSha3_512, 8>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], nw, kSfxHash, (uint8_t *)p[1]);
        else if (which == 2) LAUNCH((k_hash_words<kRateShake128, 4>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], nw, kSfxXof, (uint8_t *)p[1]);
        else LAUNCH((k_hash_words<kRateSha3_256, 4>), cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], nw, kSfxXof, (uint8_t *)p[1]);
        return 0;
    });
}

// sha3_b of sha3.c:408 for n equal-length messages of `nbits` bits each (bits packed LSB-first into
// ceil(nbits/8) bytes per message, item-major).  Host memory only: this is the reference's general SHA-3
// front-end (SURVEY 8(f) N3), not part of the KEM hot path.
int mlkem_b200_sha3_bits_batch(size_t n, const uint8_t *msgs, size_t nbits, const uint8_t sfx[4], unsigned c, size_t d, uint8_t *out,
                               const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);  // pads into, and reads the digests from, temporary host vectors
    const mlkem_b200_opts *o = so.p;
    if (c == 0 || c >= 1600 || (1600 - c) % 64 != 0 || d == 0 || !sfx || !out || (nbits && !msgs)) return MLKEM_B200_ERR_ARG;
    if (o && o->mem == MLKEM_B200_MEM_DEVICE) return MLKEM_B200_ERR_ARG;
    if (n == 0) return MLKEM_B200_OK;
    const size_t r = 1600 - c, slen = sfx[2] ? 4 : 2, m = nbits + slen;  // sha3.c:414-431
    const size_t x = m % r, padlen = (x == r - 1) ? r + 1 : r - x;       // sha3.c:264-268
    const size_t total = m + padlen, blk_bytes = r / 8, nblocks = total / r, msg_bytes = (nbits + 7) / 8;
    const size_t out_bytes = (d + 7) / 8, out_stride = (out_bytes + 7) & ~size_t(7);
    std::vector<uint8_t> padded(n * nblocks * blk_bytes, 0), res(n * out_stride);
    for (size_t i = 0; i < n; i++) {  // layout only: N || sfx || pad, bit by bit where not byte aligned
        uint8_t *P = padded.data() + i * nblocks * blk_bytes;
        const uint8_t *M = msgs + i * msg_bytes;
        memcpy(P, M, nbits / 8);
        for (size_t b = nbits & ~size_t(7); b < nbits; b++) P[b >> 3] |= (uint8_t)(((M[b >> 3] >> (b & 7)) & 1) << (b & 7));
        for (size_t k = 0; k < slen; k++) P[(nbits + k) >> 3] |= (uint8_t)((sfx[k] & 1) << ((nbits + k) & 7));
        P[m >> 3] |= (uint8_t)(1u << (m & 7));
        // the reference's pad() yields 1 0^r 1 when (m+2) % r == 0 and Sponge copies only its first two bits (sha3.c:228,272-277)
        if ((m + 2) % r != 0) P[(total - 1) >> 3] |= (uint8_t)(1u << ((total - 1) & 7));
    }
    const int rl = (int)(r / 64), nb = (int)nblocks, ob = (int)out_bytes;
    int rc = drive(o, n, 0, {{padded.data(), nullptr, nblocks * blk_bytes}, {nullptr, res.data(), out_stride}},
                   [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
                       LAUNCH(k_sponge_padded, cdiv(cn, kHashTPB), kHashTPB, 0, st, cn, (const uint8_t *)p[0], nb, rl, (uint8_t *)p[1], ob);
                       return 0;
                   });
    if (rc) return rc;
    for (size_t i = 0; i < n; i++) {
        memcpy(out + i * out_bytes, res.data() + i * out_stride, out_bytes);
        if (d % 8) out[i * out_bytes + out_bytes - 1] &= (uint8_t)((1u << (d % 8)) - 1);
    }
    return MLKEM_B200_OK;
}

// ---- the same algorithms on arrays in the reference's cell layout (ml_kem.h:35-38), converted on the device -----------
int mlkem_b200_keygen_cells_batch(int set, size_t n, const uint32_t *d, const uint32_t *z, uint32_t *ek, uint32_t *dk, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{d, nullptr, 32, true}, {z, nullptr, 32, true}, {nullptr, ek, P::EK, true}, {nullptr, dk, P::DK, true}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_keygen<P>(st, ws, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint8_t *)p[2], (uint8_t *)p[3], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}
int mlkem_b200_encaps_cells_batch(int set, size_t n, const uint32_t *ek, const uint32_t *m, uint32_t *c, uint32_t *K, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{ek, nullptr, P::EK, true}, {m, nullptr, 32, true}, {nullptr, c, P::C, true}, {nullptr, K, 32, true}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_encaps<P>(st, ws, cn, (const uint8_t *)p[0], (const uint8_t *)p[1], (uint8_t *)p[2], (uint8_t *)p[3], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}
int mlkem_b200_decaps_cells_batch(int set, size_t n, const uint32_t *dk, const uint32_t *c, uint32_t *K, const mlkem_b200_opts *o) {
    const int gl = group_limit_of(o);
    const bool fips = fips_of(o);
    DISPATCH_SET(set, return drive(o, n, ws_bytes_per_item<P>(), {{dk, nullptr, P::DK, true}, {c, nullptr, P::C, true}, {nullptr, K, 32, true}},
                                   [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t) {
                                       return enqueue_decaps<P>(st, ws, cn, (const uint8_t *)p[0], KeySel{}, (const uint8_t *)p[1], (uint8_t *)p[2], gl, fips);
                                   }));
    return MLKEM_B200_ERR_PARAM;
}
// Layout conversion alone (n_bytes a multiple of 4): dense bytes <-> cells, host or device memory.
int mlkem_b200_cells_from_bytes(size_t n_bytes, const uint8_t *bytes, uint32_t *cells, const mlkem_b200_opts *o) {
    if (n_bytes % 4) return MLKEM_B200_ERR_ARG;
    mlkem_b200_opts oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo.chunk_items <= 0) oo.chunk_items = 1 << 22;  // items are single words here
    return drive(&oo, n_bytes / 4, 0, {{bytes, nullptr, 4}, {nullptr, cells, 4, true}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        CU(cudaMemcpyAsync(p[1], p[0], (size_t)cn * 4, cudaMemcpyDeviceToDevice, st));
        return 0;
    });
}
int mlkem_b200_cells_to_bytes(size_t n_bytes, const uint32_t *cells, uint8_t *bytes, const mlkem_b200_opts *o) {
    if (n_bytes % 4) return MLKEM_B200_ERR_ARG;
    mlkem_b200_opts oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo.chunk_items <= 0) oo.chunk_items = 1 << 22;
    return drive(&oo, n_bytes / 4, 0, {{cells, nullptr, 4, true}, {nullptr, bytes, 4}}, [=](cudaStream_t st, Arena &, int cn, void **p, size_t) {
        CU(cudaMemcpyAsync(p[1], p[0], (size_t)cn * 4, cudaMemcpyDeviceToDevice, st));
        return 0;
    });
}

// ---- resident key tables (SURVEY 8(f) N4: fewer bytes per operation on the host path) ----------------------------
// A server decapsulates many ciphertexts under few keys, and a 2400-byte dk per item is 69 % of the bytes Decaps moves
// over PCIe.  A key table lives in device memory; keyed calls ship only the ciphertext (or message) and a 4-byte index.
}  // extern "C"

struct mlkem_b200_keys {
    int set = 0, device = 0;
    size_t n = 0;
    uint8_t *dk = nullptr;   // n x DK, or nullptr for a table of encapsulation keys only
    uint8_t *ek = nullptr;   // row i at ek + i*ek_stride (inside dk when dk != nullptr)
    size_t ek_stride = 0;
    uint8_t *hek = nullptr;  // n x 32: H(ek_i), computed once at load time
    uint16_t *matrix = nullptr;  // MLKEM_B200_FLAG_EXPAND_KEYS: n x K x K polynomials, At[row][col] = SampleNTT(rho || row || col)
    int group_limit = 278;       // the SampleNTT group limit the matrix was sampled with
};

namespace {

void keys_destroy(mlkem_b200_keys *k) {
    if (!k) return;
    DeviceGuard guard;
    if (guard.enter(k->device) == 0) {
        cudaDeviceSynchronize();
        if (k->dk) {
            cudaMemset(k->dk, 0, k->n * mlkem_b200_dk_bytes(k->set));  // decapsulation keys are secrets
            cudaFree(k->dk);
        } else if (k->ek) {
            cudaFree(k->ek);
        }
        if (k->hek) cudaFree(k->hek);
        if (k->matrix) cudaFree(k->matrix);
    }
    delete k;
}

// Allocates the table and fills it through `fill(ctx, stream, table)`, then hashes the ek rows.
template <class Fill>
int keys_create(int set, size_t n, bool with_dk, const mlkem_b200_opts *o, mlkem_b200_keys **out, Fill fill) {
    if (!out) return MLKEM_B200_ERR_ARG;
    *out = nullptr;
    const unsigned dkb = mlkem_b200_dk_bytes(set), ekb = mlkem_b200_ek_bytes(set), kk = k_of(set);
    if (!dkb) return MLKEM_B200_ERR_PARAM;
    if (n == 0 || n > 0x7FFFFFFFull / 8) {
        snprintf(tl_error, sizeof tl_error, "key table size out of range");
        return MLKEM_B200_ERR_ARG;
    }
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(o, &dev, &ctx, guard)) return rc;
    mlkem_b200_keys *k = new mlkem_b200_keys;
    k->set = set;
    k->device = dev;
    k->n = n;
    auto fail = [&](int rc) {
        keys_destroy(k);
        return rc;
    };
    if (with_dk) {
        if (cudaMalloc(&k->dk, n * dkb) != cudaSuccess) return fail(MLKEM_B200_ERR_CUDA);
        k->ek = k->dk + 384 * kk;
        k->ek_stride = dkb;
    } else {
        if (cudaMalloc(&k->ek, n * ekb) != cudaSuccess) return fail(MLKEM_B200_ERR_CUDA);
        k->ek_stride = ekb;
    }
    if (cudaMalloc(&k->hek, n * 32) != cudaSuccess) return fail(MLKEM_B200_ERR_CUDA);
    cudaStream_t st = (o && o->mem == MLKEM_B200_MEM_DEVICE) ? static_cast<cudaStream_t>(o->stream) : ctx->stream[0];
    if (int rc = fill(ctx, st, k)) return fail(rc);
    auto hash = [&]() -> int {
        switch (set) {
        case 512: LAUNCH((k_hash_ek_table<P512>), cdiv(n, kHashTPB), kHashTPB, 0, st, (int)n, k->ek, k->ek_stride, k->hek); break;
        case 768: LAUNCH((k_hash_ek_table<P768>), cdiv(n, kHashTPB), kHashTPB, 0, st, (int)n, k->ek, k->ek_stride, k->hek); break;
        default: LAUNCH((k_hash_ek_table<P1024>), cdiv(n, kHashTPB), kHashTPB, 0, st, (int)n, k->ek, k->ek_stride, k->hek); break;
        }
        return 0;
    };
    if (int rc = hash()) return fail(rc);
    auto expand = [&]() -> int {  // the matrix of every key, once (mlkem_kernels.cuh: expanded key tables)
        const size_t entries = n * kk * kk;
        uint8_t *seeds = nullptr;
        CU(cudaMalloc(&k->matrix, entries * 512));
        CU(cudaMalloc(&seeds, entries * 34 + 16));
        k->group_limit = group_limit_of(o);
        int rc = 0;
        auto seed_kernel = [&]() -> int {
            switch (set) {
            case 512: LAUNCH((k_matrix_seeds<P512>), cdiv(entries, 256), 256, 0, st, (int)n, k->ek, k->ek_stride, seeds); break;
            case 768: LAUNCH((k_matrix_seeds<P768>), cdiv(entries, 256), 256, 0, st, (int)n, k->ek, k->ek_stride, seeds); break;
            default: LAUNCH((k_matrix_seeds<P1024>), cdiv(entries, 256), 256, 0, st, (int)n, k->ek, k->ek_stride, seeds); break;
            }
            return 0;
        };
        rc = seed_kernel();
        mlkem_b200_opts od{k->device, MLKEM_B200_MEM_DEVICE, st, 0, o ? o->sample_group_limit : 0, 0};
        if (!rc) rc = mlkem_b200_sample_ntt_batch(entries, seeds, k->matrix, nullptr, &od);
        cudaStreamSynchronize(st);
        cudaFree(seeds);
        return rc;
    };
    if (o && (o->flags & MLKEM_B200_FLAG_EXPAND_KEYS))
        if (int rc = expand()) return fail(rc);
    if (cudaStreamSynchronize(st) != cudaSuccess) return fail(MLKEM_B200_ERR_CUDA);  // loading is a set-up call: the table is complete when it returns
    *out = k;
    return MLKEM_B200_OK;
}

// The fill of mlkem_b200_keys_from_seeds / _keys_generate: KeyGen_internal (ml_kem.c:1034) into the table's dk rows from the
// (d, z) that `place(dd, dz)` enqueues on `st` into a temporary, which is zeroed before it is freed.  A scratch ek array in the
// same temporary receives KeyGen's first output (dk embeds the same bytes).
template <class Place>
int keygen_into_table(size_t n_keys, const mlkem_b200_opts *o, cudaStream_t st, mlkem_b200_keys *k, Place place) {
    const unsigned ekb = mlkem_b200_ek_bytes(k->set);
    uint8_t *tmp = nullptr;
    CU(cudaMalloc(&tmp, n_keys * (ekb + 64)));
    uint8_t *dd = tmp + n_keys * ekb, *dz = dd + 32 * n_keys;
    int rc = place(dd, dz);
    mlkem_b200_opts od{k->device, MLKEM_B200_MEM_DEVICE, st, 0, o ? o->sample_group_limit : 0, o ? o->flags : 0};
    if (!rc) rc = mlkem_b200_keygen_batch(k->set, n_keys, dd, dz, tmp, k->dk, &od);
    cudaStreamSynchronize(st);
    cudaMemset(tmp, 0, n_keys * (ekb + 64));
    cudaFree(tmp);
    return rc;
}

// key_index of a keyed host-memory call is checked on the host; device-memory calls clamp in the kernel (key_row).
int check_key_index(const mlkem_b200_keys *k, size_t n, const uint32_t *idx, const mlkem_b200_opts *o) {
    if (!idx || (o && o->mem == MLKEM_B200_MEM_DEVICE)) return 0;
    for (size_t i = 0; i < n; i++)
        if (idx[i] >= k->n) {
            snprintf(tl_error, sizeof tl_error, "key_index[%zu] = %u is outside the table of %zu keys", i, idx[i], k->n);
            return MLKEM_B200_ERR_ARG;
        }
    return 0;
}

// The options of a keyed call: the table decides the device.
int keyed_opts(const mlkem_b200_keys *k, const mlkem_b200_opts *o, mlkem_b200_opts *oo) {
    if (!k) return MLKEM_B200_ERR_ARG;
    *oo = o ? *o : mlkem_b200_opts{-1, MLKEM_B200_MEM_HOST, nullptr, 0, 0, 0};
    if (oo->device >= 0 && oo->device != k->device) {
        snprintf(tl_error, sizeof tl_error, "the key table lives on device %d, the call names device %d", k->device, oo->device);
        return MLKEM_B200_ERR_ARG;
    }
    oo->device = k->device;
    if (oo->chunk_items > 0) oo->chunk_items = (oo->chunk_items + 3) & ~3;  // 4-byte indices: chunk starts stay 16-byte aligned
    return 0;
}

// ---- key rotation: rows of a live table replaced in place, ek rows read back ----------------------------------------
// A replace or an export touches a table that keyed calls may still be reading, on any stream.  It needs no bookkeeping of
// its own: every library call makes its stream wait for the slot events it uses and records them after its last kernel
// (DeviceCtx::ev_slot), so a stream that waits for all kSlots of them, under call_mutex, is ordered after every call already
// enqueued on the device, and recording them all afterwards orders every later call after it.
int wait_all_slots(DeviceCtx *ctx, cudaStream_t st) {
    for (int e = 0; e < kSlots; e++) CU(cudaStreamWaitEvent(st, ctx->ev_slot[e], 0));
    return 0;
}
int record_all_slots(DeviceCtx *ctx, cudaStream_t st) {
    for (int e = 0; e < kSlots; e++) CU(cudaEventRecord(ctx->ev_slot[e], st));
    return 0;
}

// The slots of a replace are HOST memory: each < n_keys and none twice.  Checked before anything is written.
int check_slots(const mlkem_b200_keys *k, size_t n, const uint32_t *slot) {
    std::vector<uint32_t> s(slot, slot + n);
    std::sort(s.begin(), s.end());
    if (s.back() >= k->n) {
        snprintf(tl_error, sizeof tl_error, "slot %u is outside the table of %zu keys", s.back(), k->n);
        return MLKEM_B200_ERR_ARG;
    }
    auto dup = std::adjacent_find(s.begin(), s.end());
    if (dup != s.end()) {
        snprintf(tl_error, sizeof tl_error, "slot %u is listed twice", *dup);
        return MLKEM_B200_ERR_ARG;
    }
    return 0;
}

// Device scratch that holds new key material (dk rows, seeds): wiped once its stream has drained, then freed.  Declared after
// the DeviceGuard of the call, so that it is released on the call's device.
struct WipedScratch {
    void *p = nullptr;
    size_t bytes = 0;
    cudaStream_t st = nullptr;
    ~WipedScratch() {
        if (!p) return;
        cudaStreamSynchronize(st);
        cudaMemsetAsync(p, 0, bytes, st);
        cudaStreamSynchronize(st);
        cudaFree(p);
    }
};

int scatter_rows(cudaStream_t st, size_t n, const uint8_t *src, size_t row_bytes, KeySel slots, uint8_t *dst) {
    const size_t words = n * (row_bytes / 16);
    LAUNCH(k_scatter_rows, std::min<unsigned>(cdiv(words, 256), 148 * 16), 256, 0, st, (int)n, (int)(row_bytes / 16), src, row_bytes, slots, dst,
           row_bytes);
    return 0;
}

enum class NewKeys { kDk, kEk, kSeeds, kGenerate };

// mlkem_b200_keys_replace / _replace_ek / _replace_from_seeds / _replace_generate.  `a` is dk, ek, d (then `z` is z) or the call
// seed (may be NULL: fresh host entropy).  The new rows, their H(ek),
// the hash check and (expanded tables) their matrices are computed in device scratch on `st` first; only then does the stream
// wait for the calls in flight and scatter the results into the listed rows of the table.
int keys_replace(mlkem_b200_keys *k, size_t n, const uint32_t *slot, const uint8_t *a, const uint8_t *z, int32_t *status,
                 const mlkem_b200_opts *o, NewKeys src) {
    mlkem_b200_opts oo;
    if (int rc = keyed_opts(k, o, &oo)) return rc;
    const bool with_dk = src != NewKeys::kEk;
    if (with_dk != (k->dk != nullptr)) {
        snprintf(tl_error, sizeof tl_error, with_dk ? "the key table holds encapsulation keys only"
                                                    : "the key table holds decapsulation keys: replace them, not their ek rows");
        return MLKEM_B200_ERR_ARG;
    }
    if (n == 0) return MLKEM_B200_OK;
    if (!slot || (!a && src != NewKeys::kGenerate) || (src == NewKeys::kSeeds && !z)) {
        snprintf(tl_error, sizeof tl_error, "NULL buffer");
        return MLKEM_B200_ERR_ARG;
    }
    if (int rc = check_slots(k, n, slot)) return rc;
    const int set = k->set;
    const unsigned kk = k_of(set), ekb = mlkem_b200_ek_bytes(set);
    const size_t row = with_dk ? mlkem_b200_dk_bytes(set) : ekb, entries = k->matrix ? n * kk * kk : 0;
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(&oo, &dev, &ctx, guard)) return rc;
    const bool src_dev = oo.mem == MLKEM_B200_MEM_DEVICE;
    // device-memory sources are read in order on the caller's stream
    cudaStream_t st = src_dev ? static_cast<cudaStream_t>(oo.stream) : ctx->stream[0];
    auto up = [](size_t b) { return (b + 255) & ~size_t(255); };
    WipedScratch s;
    s.st = st;
    const bool keygen = src == NewKeys::kSeeds || src == NewKeys::kGenerate;
    s.bytes = up(4 * n) + up(n * row) + up(32 * n) + up(4 * n) + (keygen ? up(64 * n) + up(n * ekb) : 0) +
              (entries ? up(entries * 34 + 16) + up(entries * 512) : 0);
    if (cudaMalloc(&s.p, s.bytes) != cudaSuccess) {
        s.p = nullptr;
        cudaGetLastError();
        snprintf(tl_error, sizeof tl_error, "cudaMalloc of %zu bytes of replace scratch failed", s.bytes);
        return MLKEM_B200_ERR_CUDA;
    }
    Arena ar(s.p);
    uint32_t *d_slot = ar.take<uint32_t>(n);
    uint8_t *rows = ar.take<uint8_t>(n * row), *hek = ar.take<uint8_t>(32 * n);
    int32_t *d_status = ar.take<int32_t>(n);
    const cudaMemcpyKind kind = src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CU(cudaMemcpyAsync(d_slot, slot, 4 * n, cudaMemcpyHostToDevice, st));
    if (keygen) {  // KeyGen_internal (ml_kem.c:1034) into scratch, as mlkem_b200_keys_from_seeds does
        uint8_t *dz = ar.take<uint8_t>(64 * n), *ek_out = ar.take<uint8_t>(n * ekb);
        if (src == NewKeys::kSeeds) {
            CU(cudaMemcpyAsync(dz, a, 32 * n, kind, st));
            CU(cudaMemcpyAsync(dz + 32 * n, z, 32 * n, kind, st));
        } else {  // (d_j, z_j) of the j-th listed slot, expanded from the call seed; its lease ends here, before call_mutex is taken
            CallSeed cs;
            if (int rc = cs.take(ctx, a, st)) return rc;
            if (int rc = expand_seed(st, (int)n, cs.dev, 0, kSeedTagKeyGen, dz, dz + 32 * n)) return rc;
        }
        mlkem_b200_opts od{dev, MLKEM_B200_MEM_DEVICE, st, 0, oo.sample_group_limit, oo.flags & MLKEM_B200_FLAG_FIPS203};
        if (int rc = mlkem_b200_keygen_batch(set, n, dz, dz + 32 * n, ek_out, rows, &od)) return rc;
    } else {
        CU(cudaMemcpyAsync(rows, a, n * row, kind, st));
    }
    const uint8_t *ek_rows = with_dk ? rows + 384 * kk : rows;
    DISPATCH_SET(set, LAUNCH((k_hash_ek_table<P>), cdiv(n, kHashTPB), kHashTPB, 0, st, (int)n, ek_rows, row, hek));
    mlkem_b200_opts od{dev, MLKEM_B200_MEM_DEVICE, st, 0, 0, 0};
    if (status && src == NewKeys::kDk)  // the hash check of KEM_Decaps (ml_kem.c:1336-1350) per new key, as in mlkem_b200_keys_load
        if (int rc = mlkem_b200_check_dk_batch(set, n, rows, d_status, &od)) return rc;
    uint16_t *mat = nullptr;
    if (entries) {  // the matrices of the new keys, sampled with the group limit the table was loaded with
        uint8_t *seeds = ar.take<uint8_t>(entries * 34 + 16);
        mat = ar.take<uint16_t>(entries * 256);
        DISPATCH_SET(set, LAUNCH((k_matrix_seeds<P>), cdiv(entries, 256), 256, 0, st, (int)n, ek_rows, row, seeds));
        od.sample_group_limit = k->group_limit;
        if (int rc = mlkem_b200_sample_ntt_batch(entries, seeds, mat, nullptr, &od)) return rc;
    }
    {
        std::lock_guard<std::mutex> call_lock(ctx->call_mutex);
        if (int rc = wait_all_slots(ctx, st)) return rc;
        const KeySel sel{d_slot, 0, (uint32_t)k->n};
        int rc = scatter_rows(st, n, rows, row, sel, with_dk ? k->dk : k->ek);
        if (!rc) rc = scatter_rows(st, n, hek, 32, sel, k->hek);
        if (!rc && mat) rc = scatter_rows(st, n, (const uint8_t *)mat, (size_t)kk * kk * 512, sel, (uint8_t *)k->matrix);
        const int rc_rec = record_all_slots(ctx, st);  // also after a failed launch: the slots stay ordered
        if (rc || rc_rec) return rc ? rc : rc_rec;
    }
    if (status && src == NewKeys::kDk) CU(cudaMemcpyAsync(status, d_status, 4 * n, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));  // a set-up call: the table is updated when it returns
    return MLKEM_B200_OK;
}

}  // namespace

extern "C" {

int mlkem_b200_keys_load(int set, size_t n_keys, const uint8_t *dk, int32_t *status, const mlkem_b200_opts *o, mlkem_b200_keys **out) {
    if (!dk) return MLKEM_B200_ERR_ARG;
    const unsigned dkb = mlkem_b200_dk_bytes(set);
    const bool src_dev = o && o->mem == MLKEM_B200_MEM_DEVICE;
    int rc = keys_create(set, n_keys, true, o, out, [&](DeviceCtx *, cudaStream_t st, mlkem_b200_keys *k) -> int {
        CU(cudaMemcpyAsync(k->dk, dk, n_keys * dkb, src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        return 0;
    });
    if (rc || !status) return rc;
    // the hash check of KEM_Decaps (ml_kem.c:1336-1350), once per key instead of once per ciphertext; status is HOST memory
    mlkem_b200_opts od{(*out)->device, MLKEM_B200_MEM_DEVICE, nullptr, 0, 0, 0};
    int32_t *d_status = nullptr;
    auto check = [&]() -> int {
        DeviceGuard guard;
        if (int r = guard.enter((*out)->device)) return r;
        CU(cudaMalloc(&d_status, 4 * n_keys));
        int r = mlkem_b200_check_dk_batch(set, n_keys, (*out)->dk, d_status, &od);
        if (!r && cudaMemcpy(status, d_status, 4 * n_keys, cudaMemcpyDeviceToHost) != cudaSuccess) r = MLKEM_B200_ERR_CUDA;
        cudaFree(d_status);
        return r;
    };
    rc = check();
    if (rc) {  // an error leaves no table behind (a FAILED hash check is not an error: status says which keys)
        keys_destroy(*out);
        *out = nullptr;
    }
    return rc;
}

int mlkem_b200_keys_load_ek(int set, size_t n_keys, const uint8_t *ek, const mlkem_b200_opts *o, mlkem_b200_keys **out) {
    if (!ek) return MLKEM_B200_ERR_ARG;
    const unsigned ekb = mlkem_b200_ek_bytes(set);
    const bool src_dev = o && o->mem == MLKEM_B200_MEM_DEVICE;
    return keys_create(set, n_keys, false, o, out, [&](DeviceCtx *, cudaStream_t st, mlkem_b200_keys *k) -> int {
        CU(cudaMemcpyAsync(k->ek, ek, n_keys * ekb, src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        return 0;
    });
}

int mlkem_b200_keys_from_seeds(int set, size_t n_keys, const uint8_t *d, const uint8_t *z, const mlkem_b200_opts *o, mlkem_b200_keys **out) {
    if (!d || !z) return MLKEM_B200_ERR_ARG;
    const bool src_dev = o && o->mem == MLKEM_B200_MEM_DEVICE;
    // KeyGen_internal on the device (ml_kem.c:1034): 64 bytes per key cross PCIe instead of 2400, and KeyGen is faster than
    // the copy it replaces.
    return keys_create(set, n_keys, true, o, out, [&](DeviceCtx *, cudaStream_t st, mlkem_b200_keys *k) -> int {
        return keygen_into_table(n_keys, o, st, k, [&](uint8_t *dd, uint8_t *dz) -> int {
            const cudaMemcpyKind kind = src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
            CU(cudaMemcpyAsync(dd, d, 32 * n_keys, kind, st));
            CU(cudaMemcpyAsync(dz, z, 32 * n_keys, kind, st));
            return 0;
        });
    });
}

// mlkem_b200_keys_from_seeds with (d_j, z_j) expanded on the device from the call seed: the secrets of the table never exist on
// the host.
int mlkem_b200_keys_generate(int set, size_t n_keys, const uint8_t *seed, const mlkem_b200_opts *opts, mlkem_b200_keys **out) {
    const SyncOpts so(opts);
    const mlkem_b200_opts *o = so.p;
    return keys_create(set, n_keys, true, o, out, [&](DeviceCtx *ctx, cudaStream_t st, mlkem_b200_keys *k) -> int {
        return keygen_into_table(n_keys, o, st, k, [&](uint8_t *dd, uint8_t *dz) -> int {
            CallSeed cs;  // one lease at a time: this one ends (device copy wiped) before KeyGen runs
            if (int rc = cs.take(ctx, seed, st)) return rc;
            return expand_seed(st, (int)n_keys, cs.dev, 0, kSeedTagKeyGen, dd, dz);
        });
    });
}

int mlkem_b200_keys_replace_generate(mlkem_b200_keys *k, size_t n, const uint32_t *slot, const uint8_t *seed, const mlkem_b200_opts *o) {
    return keys_replace(k, n, slot, seed, nullptr, nullptr, o, NewKeys::kGenerate);
}

int mlkem_b200_kem_encaps_keyed_batch(const mlkem_b200_keys *k, size_t n, const uint32_t *key_index, const uint8_t *seed, uint8_t *c, uint8_t *K,
                                      const mlkem_b200_opts *opts) {
    const SyncOpts so(opts);
    mlkem_b200_opts oo;
    if (int rc = keyed_opts(k, so.p, &oo)) return rc;
    if (int rc = check_key_index(k, n, key_index, &oo)) return rc;
    if (n == 0) return MLKEM_B200_OK;
    const int gl = group_limit_of(&oo);
    const bool fips = fips_of(&oo), has_idx = key_index != nullptr;
    const uint32_t nk = (uint32_t)k->n;
    std::vector<Buf> bufs = {{nullptr, c, mlkem_b200_ct_bytes(k->set)}, {nullptr, K, 32}};
    if (has_idx) bufs.push_back({key_index, nullptr, 4});
    return with_call_seed(&oo, seed, [&](const uint8_t *dseed) -> int {
        DISPATCH_SET(k->set, return drive(&oo, n, ws_bytes_per_item<P>() + 32, bufs, [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t first) {
                         uint8_t *m = ws.take<uint8_t>((size_t)cn * 32);
                         if (int rc = expand_seed(st, cn, dseed, first, kSeedTagEncaps, m, nullptr)) return rc;
                         KeySel ks{has_idx ? (const uint32_t *)p[2] : nullptr, (uint32_t)(first % nk), nk};
                         return enqueue_encaps_keyed<P>(st, ws, cn, k->ek, k->ek_stride, k->hek, ks, m, (uint8_t *)p[0], (uint8_t *)p[1], gl, fips,
                                                        k->matrix);
                     }));
        return MLKEM_B200_ERR_PARAM;
    });
}

size_t mlkem_b200_keys_count(const mlkem_b200_keys *k) { return k ? k->n : 0; }
void mlkem_b200_keys_free(mlkem_b200_keys *k) { keys_destroy(k); }

int mlkem_b200_keys_replace(mlkem_b200_keys *k, size_t n, const uint32_t *slot, const uint8_t *dk, int32_t *status, const mlkem_b200_opts *o) {
    return keys_replace(k, n, slot, dk, nullptr, status, o, NewKeys::kDk);
}
int mlkem_b200_keys_replace_ek(mlkem_b200_keys *k, size_t n, const uint32_t *slot, const uint8_t *ek, const mlkem_b200_opts *o) {
    return keys_replace(k, n, slot, ek, nullptr, nullptr, o, NewKeys::kEk);
}
int mlkem_b200_keys_replace_from_seeds(mlkem_b200_keys *k, size_t n, const uint32_t *slot, const uint8_t *d, const uint8_t *z,
                                       const mlkem_b200_opts *o) {
    return keys_replace(k, n, slot, d, z, nullptr, o, NewKeys::kSeeds);
}

int mlkem_b200_keys_export_ek(const mlkem_b200_keys *k, size_t first, size_t n, uint8_t *ek, const mlkem_b200_opts *o) {
    mlkem_b200_opts oo;
    if (int rc = keyed_opts(k, o, &oo)) return rc;
    if (first > k->n || n > k->n - first) {
        snprintf(tl_error, sizeof tl_error, "rows [%zu, %zu + %zu) are outside the table of %zu keys", first, first, n, k->n);
        return MLKEM_B200_ERR_ARG;
    }
    if (n == 0) return MLKEM_B200_OK;
    if (!ek) {
        snprintf(tl_error, sizeof tl_error, "NULL buffer");
        return MLKEM_B200_ERR_ARG;
    }
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(&oo, &dev, &ctx, guard)) return rc;
    const bool dst_dev = oo.mem == MLKEM_B200_MEM_DEVICE;
    cudaStream_t st = dst_dev ? static_cast<cudaStream_t>(oo.stream) : ctx->stream[0];
    const size_t ekb = mlkem_b200_ek_bytes(k->set);
    {
        std::lock_guard<std::mutex> call_lock(ctx->call_mutex);  // ordered like a replace (wait_all_slots)
        if (int rc = wait_all_slots(ctx, st)) return rc;
        const cudaError_t e = cudaMemcpy2DAsync(ek, ekb, k->ek + first * k->ek_stride, k->ek_stride, ekb, n,
                                                dst_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st);
        const int rc_rec = record_all_slots(ctx, st);
        if (e != cudaSuccess) {
            snprintf(tl_error, sizeof tl_error, "cudaMemcpy2DAsync failed: %s", cudaGetErrorString(e));
            return MLKEM_B200_ERR_CUDA;
        }
        if (rc_rec) return rc_rec;
    }
    if (!dst_dev) CU(cudaStreamSynchronize(st));
    return MLKEM_B200_OK;
}

int mlkem_b200_encaps_keyed_batch(const mlkem_b200_keys *k, size_t n, const uint32_t *key_index, const uint8_t *m, uint8_t *c, uint8_t *K,
                                  const mlkem_b200_opts *o) {
    mlkem_b200_opts oo;
    if (int rc = keyed_opts(k, o, &oo)) return rc;
    if (int rc = check_key_index(k, n, key_index, &oo)) return rc;
    const int gl = group_limit_of(&oo);
    const bool fips = fips_of(&oo), has_idx = key_index != nullptr;
    const uint32_t nk = (uint32_t)k->n;
    std::vector<Buf> bufs = {{m, nullptr, 32}, {nullptr, c, mlkem_b200_ct_bytes(k->set)}, {nullptr, K, 32}};
    if (has_idx) bufs.push_back({key_index, nullptr, 4});
    DISPATCH_SET(k->set, return drive(&oo, n, ws_bytes_per_item<P>(), bufs, [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t first) {
                     KeySel ks{has_idx ? (const uint32_t *)p[3] : nullptr, (uint32_t)(first % nk), nk};
                     return enqueue_encaps_keyed<P>(st, ws, cn, k->ek, k->ek_stride, k->hek, ks, (const uint8_t *)p[0], (uint8_t *)p[1],
                                                    (uint8_t *)p[2], gl, fips, k->matrix);
                 }));
    return MLKEM_B200_ERR_PARAM;
}

int mlkem_b200_decaps_keyed_batch(const mlkem_b200_keys *k, size_t n, const uint32_t *key_index, const uint8_t *c, uint8_t *K,
                                  const mlkem_b200_opts *o) {
    mlkem_b200_opts oo;
    if (int rc = keyed_opts(k, o, &oo)) return rc;
    if (!k->dk) {
        snprintf(tl_error, sizeof tl_error, "the key table holds encapsulation keys only");
        return MLKEM_B200_ERR_ARG;
    }
    if (int rc = check_key_index(k, n, key_index, &oo)) return rc;
    const int gl = group_limit_of(&oo);
    const bool fips = fips_of(&oo), has_idx = key_index != nullptr;
    const uint32_t nk = (uint32_t)k->n;
    std::vector<Buf> bufs = {{c, nullptr, mlkem_b200_ct_bytes(k->set)}, {nullptr, K, 32}};
    if (has_idx) bufs.push_back({key_index, nullptr, 4});
    DISPATCH_SET(k->set, return drive(&oo, n, ws_bytes_per_item<P>(), bufs, [=](cudaStream_t st, Arena &ws, int cn, void **p, size_t first) {
                     KeySel ks{has_idx ? (const uint32_t *)p[2] : nullptr, (uint32_t)(first % nk), nk};
                     return enqueue_decaps<P>(st, ws, cn, k->dk, ks, (const uint8_t *)p[0], (uint8_t *)p[1], gl, fips, k->matrix);
                 }));
    return MLKEM_B200_ERR_PARAM;
}

// The copy-only ceiling of a host-memory call: the same chunking, staging slots, streams and copy sizes as a real call
// with these buffers, but no kernels in between (bench.py's e2e.copy_ceiling).
int mlkem_b200_copy_probe(size_t n, int n_in, const void *const *in, const size_t *in_item_bytes, int n_out, void *const *out,
                          const size_t *out_item_bytes, const mlkem_b200_opts *o) {
    if (o && o->mem == MLKEM_B200_MEM_DEVICE) return MLKEM_B200_ERR_ARG;
    std::vector<Buf> bufs;
    for (int i = 0; i < n_in; i++) bufs.push_back({in[i], nullptr, in_item_bytes[i]});
    for (int i = 0; i < n_out; i++) bufs.push_back({nullptr, out[i], out_item_bytes[i]});
    if (bufs.empty()) return MLKEM_B200_ERR_ARG;
    return drive(o, n, 0, bufs, [](cudaStream_t, Arena &, int, void **, size_t) { return 0; });
}

int mlkem_b200_tables(uint16_t zeta[128], uint16_t gamma[128]) {
    int dev;
    DeviceCtx *ctx;
    DeviceGuard guard;
    if (int rc = acquire(nullptr, &dev, &ctx, guard)) return rc;
    TwiddleTables t;
    CU(cudaMemcpyFromSymbol(&t, c_tw, sizeof t));
    for (int i = 0; i < 128; i++) {
        zeta[i] = (uint16_t)t.zeta[i].x;
        gamma[i] = (uint16_t)t.gamma[i].x;
    }
    return 0;
}

}  // extern "C"

#include "mlkem_profile.inl"
#include "ml_kem_compat.inl"
#include "sha3_compat.inl"
