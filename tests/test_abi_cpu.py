"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol the headers declare
(no compute calls -- there is no GPU here), and refuses to compute without a device instead of falling back."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import crystals_kyber_b200 as ck

    if not os.path.exists(ck.LIB_PATH):
        import subprocess

        subprocess.run(["make", "-C", ROOT, "lib"], check=True, stdout=subprocess.DEVNULL)
    return ck.load()


def declared_functions(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    txt = re.sub(r"^\s*#.*$", "", txt, flags=re.M)  # drop preprocessor lines (macros with parenthesised values)
    return sorted(set(re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{()]*\)\s*;", txt)))


def test_batched_header_symbols_exported(lib):
    from crystals_kyber_b200.lib import SIGNATURES

    names = [n for n in declared_functions("mlkem_b200.h") if n.startswith("mlkem_b200_")]
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mlkem_b200.h but not exported"
        assert n in SIGNATURES, f"{n} has no ctypes signature in lib.py"
    assert set(SIGNATURES) == set(names)


def test_reference_header_symbols_exported(lib):
    from crystals_kyber_b200.lib import COMPAT_SYMBOLS

    names = declared_functions("ml_kem.h") + declared_functions("sha3.h")
    expect = {"h2b", "b2h", "sha3_b", "sha3_h", "sha3_s","init", "KEM_KeyGen", "KEM_Encaps", "KEM_Decaps", "SampleNTT", "SamplePolyCBD", "NTT", "InverseNTT", "BitRev7",
              "BitsToBytes", "BytesToBits", "Compress", "Decompress", "ByteEncode", "ByteDecode", "BaseCaseMultiply",
              "MultiplyNTTs", "PKE_KeyGen", "PKE_Encrypt", "PKE_Decrypt", "KeyGen_internal", "Encaps_internal", "Decaps_internal"}
    assert expect <= set(names)
    for n in expect:
        assert hasattr(lib, n)
    assert set(COMPAT_SYMBOLS) == expect | {"ml_errno"}
    assert C.c_int.in_dll(lib, "ml_errno").value == 0


def test_batched_header_is_valid_c99():
    """include/mlkem_b200.h is a C header (cgo / JNI / plain C callers): gcc -std=c99 must accept it, and the plain-C example
    that uses the keyed entry points must compile against it."""
    import subprocess

    src = '#include "mlkem_b200.h"\nint main(void) { mlkem_b200_opts o = {0, MLKEM_B200_MEM_HOST, 0, 0, 0, MLKEM_B200_FLAG_ASYNC}; return o.device; }\n'
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c", "-"],
                   input=src.encode(), check=True)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "keyed_server.c")], check=True)


def test_sizes_match_reference_formulas(lib):
    for ps, (k, du, dv) in {512: (2, 10, 4), 768: (3, 10, 4), 1024: (4, 11, 5)}.items():
        assert lib.mlkem_b200_ek_bytes(ps) == 384 * k + 32       # ml_kem.c:730
        assert lib.mlkem_b200_dkpke_bytes(ps) == 384 * k         # ml_kem.c:731
        assert lib.mlkem_b200_dk_bytes(ps) == 768 * k + 96       # ml_kem.c:1050
        assert lib.mlkem_b200_ct_bytes(ps) == 32 * (du * k + dv)  # ml_kem.c:1105
    assert lib.mlkem_b200_ek_bytes(999) == 0


def test_host_side_helpers_without_gpu(lib):
    """Pure layout helpers of the reference-signature API need no device."""
    class U(C.Structure):
        _fields_ = [("v", C.c_uint)]

    lib.BitRev7.restype, lib.BitRev7.argtypes = U, [U]
    assert [lib.BitRev7(U(i)).v & 0x7F for i in (0, 1, 2, 3, 64, 127)] == [0, 64, 32, 96, 1, 127]  # ml_kem.c:26
    lib.BitsToBytes.restype, lib.BitsToBytes.argtypes = C.POINTER(C.c_uint), [C.POINTER(C.c_uint), C.c_uint]
    bits = (C.c_uint * 8)(*[i % 2 for i in range(8)])  # BitsAndBytes_test02.c: 01010101 -> 170
    out = lib.BitsToBytes(bits, 8)
    assert out[0] & 0xFF == 170
    C.CDLL(None).free(out)


def test_no_cpu_fallback(lib):
    """Without a CUDA device every compute entry point must fail loudly (MLKEM_B200_ERR_CUDA), never compute."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    f = np.zeros((1, 256), np.uint16)
    out = np.full((1, 256), 0xABCD, np.uint16)
    rc = lib.mlkem_b200_ntt_batch(1, C.c_void_p(f.ctypes.data), C.c_void_p(out.ctypes.data), None)
    assert rc == -10 and (out == 0xABCD).all()
    assert b"failed" in lib.mlkem_b200_last_error()
    assert lib.mlkem_b200_device_count() == 0
    import crystals_kyber_b200 as ck

    with pytest.raises(ck.MlKemB200Error):
        ck.MLKEM().keygen(768, np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8))
    # round-2 entry points: a key table cannot be built, the cell-layout calls and the copy probe refuse as well
    handle = C.c_void_p(123)
    dk = np.zeros((1, 2400), np.uint8)
    assert lib.mlkem_b200_keys_load(768, 1, C.c_void_p(dk.ctypes.data), None, None, C.byref(handle)) == -10 and not handle.value
    with pytest.raises(ck.MlKemB200Error):
        ck.MLKEM().keys_load(768, dk=dk)
    cells = np.zeros((1, 2400), np.uint32)
    with pytest.raises(ck.MlKemB200Error):
        ck.MLKEM().decaps_cells(768, cells, np.zeros((1, 1088), np.uint32))
    assert lib.mlkem_b200_keys_count(None) == 0
    lib.mlkem_b200_keys_free(None)  # a no-op


def test_product_does_not_import_oracle():
    """The shipped package must never import, include, link or dlopen anything under oracle/."""
    pkg = os.path.join(ROOT, "crystals-kyber_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            path = os.path.join(dirpath, fn)
            if fn.endswith(".py"):
                for line in open(path):
                    assert not re.match(r"\s*(from|import)\s+oracle\b", line), f"{path}: {line.strip()}"
                    assert "libmlkem_oracle" not in line and "libref_mlkem" not in line, f"{path}: {line.strip()}"
            if fn.endswith((".cu", ".cuh", ".inl", ".h")):
                for line in open(path):
                    if line.lstrip().startswith("#include"):
                        assert "oracle" not in line and "reference" not in line, f"{path}: {line.strip()}"
    mk = open(os.path.join(ROOT, "Makefile")).read()
    lib_rule = mk[mk.index("$(LIB):"):].split("\n\n")[0]
    assert "oracle" not in lib_rule


def test_arithmetic_lemmas():
    """Exhaustive checks of the integer identities the kernels rely on (csrc/mlkem_device.cuh, mlkem_kernels.cuh).
    The reference's own formulas are ml_kem.c:83 (Compress) and the plain `% q` of its ring arithmetic."""
    q = 3329
    M = 1290168  # ceil(2^32 / q)
    u = lambda a: np.asarray(a, dtype=np.uint64)
    mulhi = lambda a, b: (u(a) * u(b)) >> np.uint64(32)
    # canon_fma: x - floor(x M / 2^32) q == x mod q for x < 2^21
    x = np.arange(1 << 21, dtype=np.uint64)
    assert (x - mulhi(x, M) * u(q) == x % u(q)).all()
    # the rejection bit of the three-block sampler: floor(d M / 2^32) == (d >= q) for every 12-bit d
    d = np.arange(4096, dtype=np.uint64)
    assert (mulhi(d, M) == (d >= q)).all()
    # Shoup multiplication with the quotient by multiply-high: result congruent and < 2q for any 32-bit a
    rng = np.random.default_rng(5)
    a = np.concatenate([np.arange(1 << 17, dtype=np.uint64), rng.integers(0, 1 << 32, 1 << 18, dtype=np.uint64)])
    for w in (1, 17, 1729, 3303, 3328):
        w32 = (w << 32) // q
        r = a * u(w) - mulhi(a, w32) * u(q)
        assert (r < 2 * q).all() and (r % u(q) == a * u(w) % u(q)).all()
    # Compress_d by one multiply-high: canonical inputs for the d of the parameter sets (compress_canon) ...
    xc = np.arange(q, dtype=np.uint64)
    for dd, c, m in ((1, 1665, 1290167), (4, 1665, 1290167), (5, 1665, 1290167), (10, 1664, 1290168), (11, 1664, 1290168)):
        want = ((xc << np.uint64(dd)) + u(1664)) // u(q) % u(1 << dd)
        assert (mulhi((xc << np.uint64(dd)) + u(c), m) % u(1 << dd) == want).all()
    # ... and any residue below 4q for d <= 5 (compress_resid); the same form is NOT exact for d = 10, 11
    xr = np.arange(4 * q, dtype=np.uint64)
    for dd in (1, 4, 5, 10, 11):
        want = (((xr % u(q)) << np.uint64(dd)) + u(1664)) // u(q) % u(1 << dd)
        exact = (mulhi((xr << np.uint64(dd)) + u(1664), M) % u(1 << dd) == want).all()
        assert exact == (dd <= 5)
    # the literal NTT butterfly for inputs >= q (ct_bfly_exact): Shoup product with the 16-bit quotient, one conditional
    # subtraction, for every 12-bit operand and every zeta; and canon16 on sums below 4096 + q
    zetas = np.array([pow(17, int(f"{i:07b}"[::-1], 2), q) for i in range(128)], dtype=np.uint64)
    bb = np.arange(4096, dtype=np.uint64)[:, None]
    wy = (zetas << np.uint64(16)) // u(q)
    r = bb * zetas - ((bb * wy) >> np.uint64(16)) * u(q)
    assert (r < 2 * q).all() and (np.where(r >= q, r - u(q), r) == bb * zetas % u(q)).all()
    # barrett16 (32-bit product, shift 27) on every x < 2^16: congruent, in [0, q + 1]; q + 1 at exactly three inputs, all
    # above 16q = 53264, the bound of the sums that the balanced inverse transform reduces with barrett16 alone
    barrett16 = lambda x: x - (((x * u(40317)) & u(0xFFFFFFFF)) >> np.uint64(27)) * u(q)
    xs = np.arange(1 << 16, dtype=np.uint64)
    b16 = barrett16(xs)
    assert (b16 % u(q) == xs % u(q)).all() and (b16 <= q + 1).all()
    assert np.flatnonzero(b16 == q + 1).tolist() == [56594, 59923, 63252]
    assert (b16[:16 * q] <= q).all()
    # canon16 = csubq(barrett16) on every x < 2^17: exact exactly up to 106529 (where x 40317 still fits 32 bits), which
    # covers its callers: 4096 + 14q = 50702 (ntt_warp), 16 (q - 1) = 53248 (k_vecmul_batch at k = 16), 2 * 4095 (poly_add)
    x17 = np.arange(1 << 17, dtype=np.uint64)
    b = barrett16(x17)
    c16 = np.minimum(b, b - u(q))  # csubq: a wrapped r - q is large
    exact = c16 == x17 % u(q)
    assert exact[:106530].all() and not exact[106530]
    assert max(4096 + 14 * q, 16 * (q - 1), 2 * 4095) <= 106529
    # mul_shoup (16-bit Shoup word) on every a < 2^16 with every zeta and both inverse-last words: congruent, < 2q
    a16 = np.arange(1 << 16, dtype=np.uint64)[:, None]
    ws = np.concatenate([zetas, u([zetas[1] * u(3303) % u(q), 3303])])
    r = (a16 * ws - ((a16 * ((ws << np.uint64(16)) // u(q))) >> np.uint64(16)) * u(q)) & u(0xFFFFFFFF)
    assert (r < 2 * q).all() and (r % u(q) == a16 * ws % u(q)).all()
    # nibble j of a word by multiply (2^(28-4j)) and multiply-high (2^4)
    w = rng.integers(0, 1 << 32, 4096, dtype=np.uint64)
    for j in range(8):
        top = (w << np.uint64(28 - 4 * j)) & u(0xFFFFFFFF)
        assert (mulhi(top, 16) == (w >> np.uint64(4 * j)) & u(15)).all()


def test_algorithmic_work_model_matches_the_scope_table():
    """SURVEY.md 8(d): the per-operation work the roofline is computed from (bench.py uses workload.op_counts)."""
    from crystals_kyber_b200 import workload as wl

    kc = wl.keccak_calls(3, 2, 10, 4)
    assert (kc["keygen"], kc["encaps"], kc["decaps"]) == (43, 44, 42)
    ops = wl.op_counts(3, 2, 10, 4)
    assert (ops["keygen"], ops["encaps"], ops["decaps"]) == (232_224, 250_624, 267_200)
    assert ops["encaps"] + ops["decaps"] == 517_824 and ops["matvec_encrypt"] == 151_968


def test_warp_keccak_model():
    """The one-sponge-per-warp Keccak of the small-batch hash kernels (keccak_f1600_warp, mlkem_device.cuh): a numpy model of its
    32 lanes -- same shuffle sources, rho offsets, funnel-shift rotate and pad placement -- reproduces hashlib's SHA3-256,
    SHA3-512, SHAKE128 and SHAKE256 on ML-KEM-sized messages, and the rho constants packed in the CUDA source are the model's."""
    import re

    import warp_keccak_model as model

    assert model.check_against_hashlib()
    src = open(os.path.join(ROOT, "crystals-kyber_b200", "csrc", "mlkem_device.cuh")).read()
    body = re.search(r"constexpr uint32_t kRho\[7\] = \{(.*?)\};", src, re.S).group(1)
    words = [eval(w.replace("u", "")) for w in body.replace("\n", " ").split(",")]  # "27u | 36u << 8 | ..." -> int
    assert len(words) == 7
    assert [(words[l >> 2] >> (8 * (l & 3))) & 63 for l in range(25)] == model.RHO
    # the shuffle sources the kernel computes, restated from the source text's formulas, are permutations of the 25 lanes
    for name in ("s5", "s10", "s15", "s20", "pi_src"):
        assert sorted(getattr(model, name)[:25]) == list(range(25)), name
