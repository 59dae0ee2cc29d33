"""CPU tests of build/libref_dropin.so (oracle/ref_shim.c built against the drop-in, Makefile target `dropin`) and of the
drop-in's host-only functions.  The GPU side is tests/test_dropin_api_gpu.py."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN_SO = os.path.join(ROOT, "build", "libref_dropin.so")
LIB_SO = os.path.join(ROOT, "crystals-kyber_b200", "libmlkem_b200.so")

# sha256 of oracle/ref_shim.c, the file that recorded tests/golden/ref_vectors*.json and sha_examples.json from the
# reference.  The drop-in tests replay those generators through this same file, so it must not drift from them.
REF_SHIM_SHA256 = "192d51f29905bd17b8361ddd4e22fa57800baebf544e390cb81e43122e9c8c57"

# what ref_shim.c calls from include/ml_kem.h and include/sha3.h
SHIM_CALLS = {"init", "BitRev7", "Compress", "Decompress", "ByteEncode", "ByteDecode", "SampleNTT", "SamplePolyCBD", "NTT",
              "InverseNTT", "BaseCaseMultiply", "MultiplyNTTs", "PKE_KeyGen", "PKE_Encrypt", "PKE_Decrypt", "KeyGen_internal",
              "Encaps_internal", "Decaps_internal", "KEM_KeyGen", "KEM_Encaps", "KEM_Decaps", "sha3_b", "sha3_s"}
# what the seven stand-ins of tests/csrc/dropin/ml_kem.c call
STAND_IN_CALLS = {"mlkem_b200_poly_add_batch", "mlkem_b200_poly_sub_batch", "mlkem_b200_vector_multiply_batch",
                  "mlkem_b200_sha3_bits_batch"}
LIBC = {"malloc", "calloc", "free", "memcpy", "memset", "clock_gettime", "pthread_create", "pthread_join", "__stack_chk_fail"}


@pytest.fixture(scope="module")
def dropin():
    if not os.path.exists(DROPIN_SO):
        subprocess.run(["make", "-C", ROOT, "dropin"], check=True, stdout=subprocess.DEVNULL)
    from oracle.oracle import Reference

    return Reference(DROPIN_SO)


def test_ref_shim_is_the_one_that_recorded_the_goldens():
    with open(os.path.join(ROOT, "oracle", "ref_shim.c"), "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == REF_SHIM_SHA256
    if os.path.isdir(os.path.join(ROOT, ".git")):
        assert subprocess.run(["git", "-C", ROOT, "diff", "--quiet", "HEAD", "--", "oracle/ref_shim.c"]).returncode == 0


def test_dropin_builds_with_werror(tmp_path):
    """The Makefile's recipe (-Wall -Werror) compiles the unmodified shim against the drop-in headers."""
    so = tmp_path / "libref_dropin.so"
    out = subprocess.run(["make", "-C", ROOT, "dropin", f"DROPIN_SO={so}"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    assert "-Wall -Werror" in out and "oracle/ref_shim.c" in out and "-Itests/csrc/dropin" in out, out
    assert so.exists()


def test_undefined_symbols_are_the_dropin_functions_the_shim_calls(dropin):
    """Nothing the shim needs is left to the stand-ins but the seven reference-internal helpers, which stay inside the
    .so: its undefined symbols are the 23 drop-in functions, ml_errno, the four batched calls the stand-ins make and libc."""
    out = subprocess.run(["nm", "-D", "--undefined-only", DROPIN_SO], stdout=subprocess.PIPE, check=True).stdout.decode()
    undef = {line.split()[-1].split("@")[0] for line in out.splitlines() if line.split() and line.split()[0] == "U"}
    assert len(SHIM_CALLS) == 23
    assert undef == SHIM_CALLS | {"ml_errno"} | STAND_IN_CALLS | LIBC
    out = subprocess.run(["nm", "-D", "--defined-only", DROPIN_SO], stdout=subprocess.PIPE, check=True).stdout.decode()
    defined = {line.split()[-1] for line in out.splitlines() if line.split()}
    assert all(name.startswith("ref_") for name in defined - {"_init", "_fini"}), sorted(defined)


def test_host_only_calls_through_the_dropin(dropin):
    with open(os.path.join(ROOT, "tests", "golden", "ref_vectors.json")) as f:
        v = json.load(f)
    assert dropin.sizes() == v["sizes"]
    for ps in (512, 768, 1024):
        assert dropin.init(ps) == (0, tuple(v["init"][str(ps)]))
    assert dropin.init(999)[0] == v["init_bad"] == -1
    assert [dropin.bitrev7(i) for i in range(128)] == v["bitrev7"]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB_SO):
        subprocess.run(["make", "-C", ROOT, "lib"], check=True, stdout=subprocess.DEVNULL)
    lib = C.CDLL(LIB_SO)
    for name in ("h2b", "b2h", "BitsToBytes", "BytesToBits"):
        getattr(lib, name).restype = C.c_void_p
    lib.h2b.argtypes = [C.c_void_p, C.c_uint, C.c_uint]
    for name in ("b2h", "BitsToBytes", "BytesToBits"):
        getattr(lib, name).argtypes = [C.c_void_p, C.c_uint]
    return lib


_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]


def take(ptr, n):
    assert ptr
    a = np.frombuffer((C.c_uint32 * n).from_address(ptr), np.uint32).copy() if n else np.zeros(0, np.uint32)
    _libc.free(ptr)
    return a


def with_upper_bits(rng, vals, width):
    """The cells as a caller may hand them over: random bits above the field, which the reference leaves unspecified."""
    junk = rng.integers(0, 1 << 32, len(vals), dtype=np.uint64).astype(np.uint32) & np.uint32((0xFFFFFFFF << width) & 0xFFFFFFFF)
    return np.ascontiguousarray(np.asarray(vals, np.uint32) | junk)


def test_h2b_b2h_against_fips202_appendix_b1(lib):
    """h2b (sha3.c:329) and b2h (sha3.c:367) against FIPS 202 Appendix B.1, restated below, for every m <= 200 and every
    n <= 8m, on hex digits / bits whose cells carry junk above their 4-bit / 1-bit field."""
    rng = np.random.default_rng(31)
    for m in range(201):
        digits = rng.integers(0, 16, 2 * m, dtype=np.uint8)
        # B.1 h2b: h_i = 16 H[2i] + H[2i+1]; T[8i + j] = bit j of h_i; S = Trunc_n(T)
        T = np.unpackbits((16 * digits[0::2] + digits[1::2]).astype(np.uint8), bitorder="little")
        H = with_upper_bits(rng, digits, 4)
        S = rng.integers(0, 2, 8 * m, dtype=np.uint8)
        Sc = with_upper_bits(rng, S, 1)
        for n in range(8 * m + 1):
            got = take(lib.h2b(H.ctypes.data, m, n), n) & 1
            assert (got == T[:n]).all(), (m, n)
            # B.1 b2h: pad S to 8 ceil(n/8) bits with zeros; h_i = sum_j S[8i + j] 2^j; H[2i] = h_i div 16, H[2i+1] = h_i mod 16
            h = np.packbits(S[:n], bitorder="little")
            want = np.stack([h >> 4, h & 15], axis=1).ravel()
            assert (take(lib.b2h(Sc.ctypes.data, n), len(want)) & 15 == want).all(), (m, n)


def test_bytes_to_bits_and_back(lib):
    rng = np.random.default_rng(32)
    for L in range(0, 201):
        B = rng.integers(0, 256, L, dtype=np.uint8)
        Bc = with_upper_bits(rng, B, 8)
        bits = take(lib.BytesToBits(Bc.ctypes.data, L), 8 * L) & 1  # ml_kem.c:62
        assert (bits == np.unpackbits(B, bitorder="little")).all(), L
        bits_c = with_upper_bits(rng, bits, 1)
        back = take(lib.BitsToBytes(bits_c.ctypes.data, 8 * L), L) & 0xFF  # ml_kem.c:47
        assert (back == B).all(), L
