"""The launch-geometry constants that tests/test_launch_geometry_gpu.py builds its batch sizes from, checked against the CUDA
sources, and the static check behind its key-index clamp test.

The GPU file picks batch sizes on both sides of every place where a kernel's launch geometry changes: the tail of a
128-thread block, the `rows > 32` switch between the general matrix kernel alone and the fused kernel plus clean-up, the
warp-form / thread-form hashing switch, the 2nd, 3rd and 4th item of a persistent warp, the second grid-stride pass of the
list kernel and of the primitives.  Those sizes are computed from GEOMETRY below.  If a boundary moves in the sources, the
tests here fail, instead of the size table quietly testing one side of it only.
"""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "crystals-kyber_b200", "csrc")

SMS = 148  # the B200's SM count, as the grid caps spell it
GEOMETRY = {
    # mlkem_kernels.cuh: threads per block
    "kHashTPB": 128,  # thread-per-item hash kernels: 128 items per block
    "kNoiseTPB": 128,  # k_noise: 128 sponges per block
    "kWarpTPB": 128,  # k_encrypt_v, k_decrypt: 4 warps (items) per block
    "kMatTableTPB": 128,  # k_matvec_table: 4 rows in flight per block
    "kWarpHashTPB": 128,  # warp-per-item hashes: 4 items per block
    "kWarpHashMaxItems": 1024,  # chunks of at most this many items hash with one sponge per warp
    "kPrimTPB": 256,  # stand-alone primitives: 8 polynomials (or 256 16-byte vectors) per block
    # mlkem_b200.cu: grid caps, in blocks
    "warp_grid_cap": SMS * 16,  # persistent warp-per-item kernels and k_matvec_table
    "list_grid_cap": SMS * 4,  # k_sample_matvec_list, 32 rows per block
    "prim_grid_cap": SMS * 8 * 4,  # prim_grid(): ntt, intt, multiply_ntts, vector_multiply, cbd, codec
    "vector_grid_cap": SMS * 32,  # k_compress_batch and k_poly_addsub
    "fused_min_rows": 32,  # the fused k_sample_matvec runs when rows > 32
    "device_chunk": 1 << 18,  # default chunk of a device-memory call
    "host_chunk": 1 << 16,  # default chunk of a host-memory call, and of the primitives that set their own
    "split_min": 1 << 16,  # device calls of at least this many items in one chunk are split in two
    "max_chunk": 1 << 26,  # chunk_items is clamped to this
}
PERSISTENT_WARPS = GEOMETRY["warp_grid_cap"] * GEOMETRY["kWarpTPB"] // 32  # 9 472 items (or table rows) in flight
LIST_ROWS_PER_PASS = GEOMETRY["list_grid_cap"] * 32  # 18 944 rows
PRIM_POLYS_PER_PASS = GEOMETRY["prim_grid_cap"] * GEOMETRY["kPrimTPB"] // 32  # 37 888 polynomials
VECTORS_PER_PASS = GEOMETRY["vector_grid_cap"] * GEOMETRY["kPrimTPB"]  # 1 212 416 vectors of 8 coefficients


def source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def strip_comments(text):
    """The source without // and /* */ comments; line breaks are kept, so offsets still map to lines."""
    text = re.sub(r"/\*.*?\*/", lambda m: re.sub(r"[^\n]", " ", m.group(0)), text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def function_body(text, signature):
    """(start, end) offsets of the braces of the function whose definition starts with `signature`."""
    at = text.index(signature)
    open_ = text.index("{", at)
    depth = 0
    for i in range(open_, len(text)):
        depth += {"{": 1, "}": -1}.get(text[i], 0)
        if depth == 0:
            return open_, i + 1
    raise ValueError(f"unbalanced braces after {signature!r}")


KEY_ROW = "__device__ __forceinline__ size_t key_row(const KeySel &k, int item)"
CLAMP = "min(__ldg(k.index + item), k.nkeys - 1u)"


def key_index_confined():
    """None when every read of a KeySel's `index` in mlkem_kernels.cuh sits inside key_row and key_row clamps it to
    nkeys - 1; otherwise a description of what breaks that.  The GPU tests launch out-of-range indices only after this
    holds, so that a clamp regression fails a test instead of reading out of bounds on the device."""
    text = strip_comments(source("mlkem_kernels.cuh"))
    if KEY_ROW not in text:
        return "key_row not found"
    lo, hi = function_body(text, KEY_ROW)
    if CLAMP not in text[lo:hi]:
        return f"key_row does not clamp with {CLAMP}"
    outside = [text.count("\n", 0, m.start()) + 1 for m in re.finditer(r"(\.|->)\s*index\b", text) if not lo <= m.start() < hi]
    if outside:
        return f"KeySel index read outside key_row at mlkem_kernels.cuh lines {outside}"
    return None


def test_geometry_constants_match_the_sources():
    kernels, host = strip_comments(source("mlkem_kernels.cuh")), strip_comments(source("mlkem_b200.cu"))
    for name in ("kHashTPB", "kNoiseTPB", "kWarpTPB", "kMatTableTPB", "kWarpHashTPB", "kWarpHashMaxItems", "kPrimTPB"):
        found = re.findall(rf"constexpr int {name} = (\d+);", kernels)
        assert found == [str(GEOMETRY[name])], (name, found)

    def one(pattern, what, count=1):
        hits = re.findall(pattern, host)
        assert len(hits) == count, (what, pattern, hits)

    one(r"inline unsigned warp_grid\(size_t items, int warps_per_block\) \{[^}]*const size_t cap = 148 \* 16;", "warp_grid cap")
    one(r"list_grid = std::min<unsigned>\(blocks, 148 \* 4\);", "k_sample_matvec_list grid cap")
    one(r"inline unsigned prim_grid\(size_t n_polys\) \{[^}]*size_t cap = 148 \* 8 \* 4;", "prim_grid cap")
    one(r"if \(grid > 148 \* 32\) grid = 148 \* 32;", "k_compress_batch / k_poly_addsub grid cap", count=2)
    one(r"if \(a\.group_limit >= 168 && rows > 32\)", "the fused kernel's row threshold")
    one(r"on_device \? \(env_chunk > 0 \? \(size_t\)env_chunk : \(size_t\)1 << 18\) : \(env_hchunk > 0 \? \(size_t\)env_hchunk : \(size_t\)1 << 16\)",
        "default chunks")
    one(r"if \(chunk > \(\(size_t\)1 << 26\)\) chunk = \(size_t\)1 << 26;", "chunk_items clamp")
    one(r"n >= \(\(size_t\)1 << 16\) && nchunks < 2 && g_streams\.load\(\) > 1\) \{\s*chunk = \(\(n \+ 1\) / 2 \+ 1023\) & ~\(size_t\)1023;",
        "the automatic two-chunk split")
    one(r"if \(oo\.chunk_items <= 0\) oo\.chunk_items = 1 << 16;", "primitive default chunk", count=3)
    # the persistent kernels and k_matvec_table take warp_grid(); the hashes cdiv(n, kHashTPB) or warp_hash_grid()
    one(r"LAUNCH\(\(k_encrypt_v<P, (?:true|false)>\), warp_grid\(n, kWarpTPB / 32\), kWarpTPB", "k_encrypt_v grid", count=2)
    assert len(re.findall(r"LAUNCH\(\(k_decrypt<P>\), warp_grid\(c?n, kWarpTPB / 32\), kWarpTPB", host)) == 2
    one(r"const unsigned tgrid = warp_grid\(\(size_t\)n \* K, kMatTableTPB / 32\);", "k_matvec_table grid")
    assert re.search(r"int warp_hash_max\(\) \{\s*static const int v = env_int\(\"MLKEM_B200_WARP_HASH_MAX\", kWarpHashMaxItems\);", host)
    assert (PERSISTENT_WARPS, LIST_ROWS_PER_PASS, PRIM_POLYS_PER_PASS, VECTORS_PER_PASS) == (9472, 18944, 37888, 1212416)


def test_key_index_is_read_only_through_the_clamp():
    assert key_index_confined() is None, key_index_confined()


def test_key_index_check_sees_a_stray_read():
    """The check itself: a second, unclamped read of the index outside key_row is reported, and so is a key_row without
    the clamp."""
    text = source("mlkem_kernels.cuh")
    stray = text + "\n__device__ uint32_t raw_row(const KeySel &k, int i) { return k.index[i]; }\n"
    unclamped = text.replace(CLAMP, "__ldg(k.index + item)")
    assert unclamped != text
    real = source
    try:
        globals()["source"] = lambda name: stray
        assert "outside key_row" in key_index_confined()
        globals()["source"] = lambda name: unclamped
        assert "does not clamp" in key_index_confined()
    finally:
        globals()["source"] = real
    assert key_index_confined() is None
