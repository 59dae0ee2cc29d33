"""The drop-in API (include/ml_kem.h, include/sha3.h) function by function on the GPU (-m gpu).

Most of it drives the library through build/libref_dropin.so: the unmodified oracle/ref_shim.c, the code that recorded
tests/golden/*.json from the reference, built against libmlkem_b200.so (Makefile target `dropin`).  Replaying the golden
generators through it must give back every recorded reference output byte for byte; nothing here needs the reference's
sources.  Seven reference-internal helpers the shim calls (PolyAddition, PolySubtraction, VectorMultiply, H, G, J, PRF)
are not part of the drop-in: tests/csrc/dropin/ml_kem.c stands them in over the batched entry points, so the golden
entries "addsub", "vector_multiply", "hash" and the "ring" add / sub fields check those entry points, not ml_kem.h.

The ref_* wrappers dereference what the drop-in returns, so a NULL from a broken drop-in function would kill the
process: every group of calls runs in a child process (this file run as a script) and a crash shows as a failed test
with the child's exit status.  The parts that call the library directly through ctypes (upper cell bits, the public
wrappers, the error paths, the SHA-3 sweep) run the same way, so that stderr is the child's own.
"""
import ctypes as C
import hashlib
import importlib.util
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
DROPIN_SO = os.path.join(ROOT, "build", "libref_dropin.so")
LIB_SO = os.path.join(ROOT, "crystals-kyber_b200", "libmlkem_b200.so")
SETS = (512, 768, 1024)
Q = 3329

pytestmark = pytest.mark.gpu


# ================================================================== parent side: one child process per group of calls
@pytest.fixture(scope="module")
def dropin(oracle):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if not os.path.exists(DROPIN_SO):
        subprocess.run(["make", "-C", ROOT, "dropin"], check=True, stdout=subprocess.DEVNULL)
    return DROPIN_SO


def child(group, *args, timeout=1200):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), group]
    r = subprocess.run(cmd + [str(a) for a in args], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout)
    assert r.returncode == 0, (f"child `{group} {' '.join(map(str, args))}` exited with status {r.returncode}\n"
                               + r.stderr.decode(errors="replace")[-6000:])
    return r


def test_round1_golden_generator_replayed_through_the_dropin(dropin):
    """make_golden.ref_vectors() run on the drop-in (its own assertions included) returns ref_vectors.json exactly."""
    child("golden_r01")


def test_round2_goldens_through_the_dropin(dropin):
    child("golden_r02")


def test_sha3_goldens_through_sha3_b_and_sha3_s(dropin):
    child("sha_goldens")


def test_archive_drivers_through_the_dropin(dropin):
    """The 9 deterministic Test_Archive drivers (tests/archive_drivers.py) on single drop-in calls hash to archive_stdout.json."""
    child("archive")


@pytest.mark.parametrize("ps", SETS)
def test_kem_functions_vs_oracle(dropin, ps):
    child("kem_vs_oracle", ps)


def test_ring_sampler_codec_functions_vs_oracle(dropin):
    child("primitives_vs_oracle")


def test_basecase_multiply_vs_oracle(dropin):
    child("basecase")


@pytest.mark.parametrize("ps", SETS)
def test_upper_cell_bits_are_ignored(dropin, ps):
    child("upper_bits", ps)


@pytest.mark.parametrize("ps", SETS)
def test_public_wrappers(dropin, ps):
    child("wrappers", ps)


@pytest.mark.parametrize("ps", SETS)
def test_error_paths(dropin, ps):
    child("errors", ps)


@pytest.mark.parametrize("name", ["SHA3-224", "SHA3-256", "SHA3-384", "SHA3-512", "SHAKE128", "SHAKE256"])
def test_sha3_bit_length_sweep(dropin, name):
    child("sha3_sweep", name)


# ================================================================== child side
def h2a(hexstr, dtype):
    return np.frombuffer(bytes.fromhex(hexstr), dtype=dtype)


def golden(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def sizes(ps):
    k, du, dv = {512: (2, 10, 4), 768: (3, 10, 4), 1024: (4, 11, 5)}[ps]
    return {"k": k, "ek": 384 * k + 32, "dk": 768 * k + 96, "c": 32 * (du * k + dv), "dk_pke": 384 * k, "c1": 32 * du * k}


def dropin_ref():
    from oracle.oracle import Reference

    return Reference(DROPIN_SO)


def first_difference(got, want, path="$"):
    """Path of the first entry where two JSON values differ, or None."""
    if type(got) is not type(want):
        return path
    if isinstance(want, dict):
        if sorted(got) != sorted(want):
            return f"{path} keys {sorted(set(got) ^ set(want))}"
        for k in sorted(want):
            d = first_difference(got[k], want[k], f"{path}.{k}")
            if d:
                return d
        return None
    if isinstance(want, list):
        if len(got) != len(want):
            return f"{path} length {len(got)} != {len(want)}"
        for i, (g, w) in enumerate(zip(got, want)):
            d = first_difference(g, w, f"{path}[{i}]")
            if d:
                return d
        return None
    return None if got == want else f"{path}: {got!r} != {want!r}"


def child_golden_r01():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    got = json.loads(json.dumps(mg.ref_vectors(dropin_ref())))
    diff = first_difference(got, golden("ref_vectors.json"))
    assert diff is None, f"first differing entry: {diff}"


def child_golden_r02():
    r, v = dropin_ref(), golden("ref_vectors_r02.json")
    for i, rec in enumerate(v["ntt12"]):
        assert r.ntt(h2a(rec["f"], np.uint16)).tobytes().hex() == rec["ntt_f"], f"ntt12[{i}]"
    for i, rec in enumerate(v["decaps_random"]):  # intt12_undefined is undefined behaviour in the reference: not replayed
        ps, dk, c = rec["set"], bytes.fromhex(rec["dk"]), bytes.fromhex(rec["c"])
        assert r.decaps_internal(ps, dk, c).hex() == rec["K"], f"decaps_random[{i}].K"
        assert r.pke_decrypt(ps, dk[: sizes(ps)["dk_pke"]], c).hex() == rec["m"], f"decaps_random[{i}].m"
    for i, rec in enumerate(v["addsub"]):
        u, w = h2a(rec["u"], np.uint16), h2a(rec["v"], np.uint16)
        assert r.poly_add(u, w).tobytes().hex() == rec["add"], f"addsub[{i}].add"
        assert r.poly_sub(u, w).tobytes().hex() == rec["sub"], f"addsub[{i}].sub"
    for i, rec in enumerate(v["vector_multiply"]):
        u, w = h2a(rec["u"], np.uint16), h2a(rec["v"], np.uint16)
        assert r.vector_multiply(u, w, rec["k"]).tobytes().hex() == rec["w"], f"vector_multiply[{i}]"


def child_sha_goldens():
    r, v = dropin_ref(), golden("sha_examples.json")
    assert len(v["examples"]) == 16 and len(v["boundary"]) == 54 and any(b["quirk"] for b in v["boundary"])
    for ex in v["examples"]:
        got = r.sha3_bits([int(b) for b in ex["bits"]], ex["sfx"], ex["c"], ex["d"])
        assert np.packbits(got, bitorder="little").tobytes().hex() == ex["hex"], ex["name"]
    for i, b in enumerate(v["boundary"]):
        got = r.sha3_bits([int(x) for x in b["bits"]], b["sfx"], b["c"], b["d"])
        assert hashlib.sha256(got.tobytes()).hexdigest() == b["out_bits_sha256"], f"boundary[{i}] ({len(b['bits'])} bits)"
    for rec in v["sha3_s"]:
        assert r.sha3_s(rec["text"].encode(), [0, 1, 0, 0], 512, 256).hex() == rec["hex"], rec["text"]


class DropinImpl:
    """tests/archive_drivers.py's batched numpy interface on single drop-in calls."""

    def __init__(self, r, zeta):
        self.r, self.zeta = r, zeta

    def bitrev7(self, i):
        return self.r.bitrev7(int(i))

    def byte_encode(self, F, d):
        return np.stack([self.r.byte_encode(f, d) for f in np.asarray(F, np.uint16).reshape(-1, 256)])

    def byte_decode(self, B, d):
        return np.stack([self.r.byte_decode(b, d) for b in np.asarray(B, np.uint8).reshape(-1, 32 * d)])

    def compress(self, x, d):
        return np.array([self.r.compress(int(v), d) for v in np.ravel(x)], np.uint16)

    def decompress(self, y, d):
        return np.array([self.r.decompress(int(v), d) for v in np.ravel(y)], np.uint16)

    def sample_ntt(self, seeds):
        return np.stack([self.r.sample_ntt(s.tobytes())[0] for s in np.asarray(seeds, np.uint8).reshape(-1, 34)])

    def cbd(self, B, eta):
        return np.stack([self.r.sample_cbd(b.tobytes(), eta) for b in np.asarray(B, np.uint8).reshape(-1, 64 * eta)])

    def ntt(self, f):
        return np.stack([self.r.ntt(x) for x in np.asarray(f, np.uint16).reshape(-1, 256)])

    def intt(self, f):
        return np.stack([self.r.intt(x) for x in np.asarray(f, np.uint16).reshape(-1, 256)])

    def zeta_table(self):
        return self.zeta

    def pke_keygen(self, ps, d):
        ek, dk = self.r.pke_keygen(ps, np.asarray(d, np.uint8).tobytes())
        return np.frombuffer(ek, np.uint8)[None], np.frombuffer(dk, np.uint8)[None]

    def pke_encrypt(self, ps, ek, m, rr):
        b = lambda a: np.asarray(a, np.uint8).tobytes()
        return np.frombuffer(self.r.pke_encrypt(ps, b(ek), b(m), b(rr)), np.uint8)[None]

    def pke_decrypt(self, ps, dk, c):
        b = lambda a: np.asarray(a, np.uint8).tobytes()
        return np.frombuffer(self.r.pke_decrypt(ps, b(dk), b(c)), np.uint8)[None]


def child_archive():
    from archive_drivers import DRIVERS

    r = dropin_ref()
    zeta, gamma = np.zeros(128, np.uint16), np.zeros(128, np.uint16)
    assert C.CDLL(LIB_SO).mlkem_b200_tables(C.c_void_p(zeta.ctypes.data), C.c_void_p(gamma.ctypes.data)) == 0
    want = golden("archive_stdout.json")
    assert len(DRIVERS) == 9
    for name, fn in sorted(DRIVERS.items()):
        out = fn(DropinImpl(r, zeta)).encode()
        assert hashlib.sha256(out).hexdigest() == want[name]["sha256"], (name, out[:300])


def child_kem_vs_oracle(ps):
    """KeyGen_internal / Encaps_internal / Decaps_internal and the K-PKE functions, one drop-in call per item, against the
    oracle; Decaps on valid ciphertexts and with one bit flipped at the start, middle and last byte of c1 and of c2."""
    from oracle.oracle import Oracle

    ps = int(ps)
    r, orc, sz = dropin_ref(), Oracle(), sizes(ps)
    rng = np.random.default_rng(7000 + ps)
    n = 200
    d, z, m, rr = (rng.integers(0, 256, (n, 32), dtype=np.uint8) for _ in range(4))
    oek, odk = orc.keygen(ps, d, z)
    oc, oK = orc.encaps(ps, oek, m)
    c1 = sz["c1"]
    flips = (0, c1 // 2, c1 - 1, c1, (c1 + sz["c"]) // 2, sz["c"] - 1)
    bad = np.repeat(oc[:, None, :], len(flips), axis=1)
    for j, pos in enumerate(flips):
        bad[np.arange(n), j, pos] ^= (1 << rng.integers(0, 8, n)).astype(np.uint8)
    oKbad = orc.decaps(ps, np.repeat(odk, len(flips), axis=0), bad.reshape(-1, sz["c"])).reshape(n, len(flips), 32)
    assert (oKbad != oK[:, None, :]).any(axis=2).all()  # every flip takes the rejection path
    for i in range(n):
        ek, dk = r.keygen_internal(ps, d[i].tobytes(), z[i].tobytes())
        assert ek == oek[i].tobytes() and dk == odk[i].tobytes(), f"KeyGen_internal item {i}"
        c, K = r.encaps_internal(ps, ek, m[i].tobytes())
        assert c == oc[i].tobytes() and K == oK[i].tobytes(), f"Encaps_internal item {i}"
        assert r.decaps_internal(ps, dk, c) == K, f"Decaps_internal item {i}"
        for j, pos in enumerate(flips):
            assert r.decaps_internal(ps, dk, bad[i, j].tobytes()) == oKbad[i, j].tobytes(), f"Decaps_internal item {i}, flip in byte {pos}"
    # K-PKE, plus keys and ciphertexts made of all-0x00 / all-0xFF bytes
    pek, pdk = orc.pke_keygen(ps, d)
    pc = orc.pke_encrypt(ps, pek, m, rr)
    for i in range(n // 2):
        ek, dk = r.pke_keygen(ps, d[i].tobytes())
        assert ek == pek[i].tobytes() and dk == pdk[i].tobytes(), f"PKE_KeyGen item {i}"
        assert r.pke_encrypt(ps, ek, m[i].tobytes(), rr[i].tobytes()) == pc[i].tobytes(), f"PKE_Encrypt item {i}"
        assert r.pke_decrypt(ps, dk, pc[i].tobytes()) == m[i].tobytes(), f"PKE_Decrypt item {i}"
    for fill in (0x00, 0xFF):
        ek = np.full((1, sz["ek"]), fill, np.uint8)
        assert r.pke_encrypt(ps, ek.tobytes(), m[0].tobytes(), rr[0].tobytes()) == orc.pke_encrypt(ps, ek, m[:1], rr[:1]).tobytes()
        dkp = np.full((1, sz["dk_pke"]), fill, np.uint8)
        for c in (pc[:1], np.full((1, sz["c"]), fill, np.uint8), np.full((1, sz["c"]), 0xFF - fill, np.uint8)):
            assert r.pke_decrypt(ps, dkp.tobytes(), c.tobytes()) == orc.pke_decrypt(ps, dkp, c).tobytes(), f"PKE_Decrypt fill {fill:#x}"
            assert r.pke_decrypt(ps, pdk[0].tobytes(), c.tobytes()) == orc.pke_decrypt(ps, pdk[:1], c).tobytes()


def child_primitives_vs_oracle():
    """NTT, InverseNTT, MultiplyNTTs, SampleNTT, SamplePolyCBD, ByteEncode / ByteDecode: one drop-in call per item."""
    from oracle.oracle import Oracle

    r, orc = dropin_ref(), Oracle()
    rng = np.random.default_rng(7001)
    n = 300
    f12 = rng.integers(0, 4096, (n, 256), dtype=np.uint16)
    f12[0], f12[1] = 4095, 3329
    fq = rng.integers(0, Q, (n, 256), dtype=np.uint16)
    fq[0], fq[1] = Q - 1, 0
    g12 = rng.integers(0, 4096, (n, 256), dtype=np.uint16)
    want_ntt, want_intt, want_mul = orc.ntt(f12), orc.intt(fq), orc.multiply_ntts(f12, g12)
    for i in range(n):
        assert (r.ntt(f12[i]) == want_ntt[i]).all(), f"NTT item {i}"
        assert (r.intt(fq[i]) == want_intt[i]).all(), f"InverseNTT item {i}"
        assert (r.multiply_ntts(f12[i], g12[i]) == want_mul[i]).all(), f"MultiplyNTTs item {i}"
    seeds = rng.integers(0, 256, (n, 34), dtype=np.uint8)
    want_a, want_after = orc.sample_ntt_with_seeds(seeds)
    for i in range(n):
        a, after = r.sample_ntt(seeds[i].tobytes())
        assert (a == want_a[i]).all() and after == want_after[i].tobytes(), f"SampleNTT item {i}"
    for eta in (2, 3):
        B = rng.integers(0, 256, (n, 64 * eta), dtype=np.uint8)
        B[0] = 0xFF
        want = orc.cbd(B, eta)
        for i in range(n):
            assert (r.sample_cbd(B[i].tobytes(), eta) == want[i]).all(), f"SamplePolyCBD eta={eta} item {i}"
    for d in (1, 4, 5, 10, 11, 12):
        F = rng.integers(0, 1 << d, (n, 256), dtype=np.uint16)
        B = rng.integers(0, 256, (n, 32 * d), dtype=np.uint8)
        want_B, want_F = orc.byte_encode(F, d), orc.byte_decode(B, d)
        for i in range(n):
            assert (r.byte_encode(F[i], d) == want_B[i]).all(), f"ByteEncode d={d} item {i}"
            assert (r.byte_decode(B[i], d) == want_F[i]).all(), f"ByteDecode d={d} item {i}"


def child_basecase():
    """BaseCaseMultiply (its own one-thread kernel) against orc_basecase_multiply: every gamma in [0, q), each with operand
    tuples from {0, 1, q-1, q, 4095} (the 625 tuples cycle over the gammas), and random 12-bit tuples.  gamma >= q is left
    out: the shim passes gamma in the 24-bit .l field, and nothing pins the reference's result there."""
    from oracle.oracle import Oracle

    r, orc = dropin_ref(), Oracle()
    ofn = orc.fn("basecase_multiply")
    edge = (0, 1, Q - 1, Q, 4095)
    tuples = [(a0, a1, b0, b1) for a0 in edge for a1 in edge for b0 in edge for b1 in edge]
    rng = np.random.default_rng(7002)
    cases = [(*tuples[(2 * g + j) % len(tuples)], g) for g in range(Q) for j in range(2)]
    cases += [tuple(int(x) for x in rng.integers(0, 4096, 4)) + (int(rng.integers(0, Q)),) for _ in range(2000)]
    out = (C.c_uint16 * 2)()
    for a0, a1, b0, b1, g in cases:
        ofn(*(C.c_uint16(x) for x in (a0, a1, b0, b1, g)), out)
        assert r.basecase_multiply(a0, a1, b0, b1, g) == (out[0], out[1]), (a0, a1, b0, b1, g)


# ------------------------------------------------------------------ direct ctypes calls on libmlkem_b200.so
class PARAMS(C.Structure):
    _fields_ = [("k", C.c_uint32), ("n1", C.c_uint32), ("n2", C.c_uint32), ("du", C.c_uint32), ("dv", C.c_uint32)]


class PKE(C.Structure):
    _fields_ = [("ek", C.c_void_p), ("dk", C.c_void_p), ("ek_len", C.c_uint), ("dk_len", C.c_uint)]


class KEM(C.Structure):
    _fields_ = [("K", C.c_uint32 * 32), ("c", C.c_void_p), ("c_len", C.c_uint)]


class Opts(C.Structure):  # mlkem_b200_opts
    _fields_ = [("device", C.c_int), ("mem", C.c_int), ("stream", C.c_void_p), ("chunk_items", C.c_int),
                ("sample_group_limit", C.c_int), ("flags", C.c_int)]


def dropin_lib():
    """libmlkem_b200.so with the ml_kem.h / sha3.h prototypes (cells as uint32 words, by-value unions as uint32)."""
    lib = C.CDLL(LIB_SO)
    vp, u, P = C.c_void_p, C.c_uint, C.POINTER(PARAMS)
    sig = {"init": (PARAMS, [C.c_int]), "SampleNTT": (vp, [vp]), "SamplePolyCBD": (vp, [vp, u]), "NTT": (vp, [vp]),
           "InverseNTT": (vp, [vp]), "MultiplyNTTs": (vp, [vp, vp]), "BitRev7": (C.c_uint32, [C.c_uint32]),
           "Compress": (C.c_uint32, [C.c_uint32, u]), "Decompress": (C.c_uint32, [C.c_uint32, u]),
           "ByteEncode": (vp, [vp, u]), "ByteDecode": (vp, [vp, u]), "BaseCaseMultiply": (vp, [C.c_uint32] * 5),
           "BitsToBytes": (vp, [vp, u]), "BytesToBits": (vp, [vp, u]), "PKE_KeyGen": (PKE, [P, vp]),
           "PKE_Encrypt": (vp, [P, vp, vp, vp]), "PKE_Decrypt": (vp, [P, vp, vp]), "KeyGen_internal": (PKE, [P, vp, vp]),
           "Encaps_internal": (KEM, [P, vp, vp]), "Decaps_internal": (vp, [P, vp, vp]), "KEM_KeyGen": (PKE, [P]),
           "KEM_Encaps": (KEM, [P, vp, u]), "KEM_Decaps": (vp, [P, vp, u, vp, u]), "h2b": (vp, [vp, u, u]),
           "b2h": (vp, [vp, u]), "sha3_b": (vp, [vp, u, u, u, vp]), "sha3_h": (vp, [vp, u, u, u, vp]),
           "sha3_s": (vp, [C.c_char_p, u, u, u, vp])}
    for name, (res, args) in sig.items():
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]


def cells(a):
    """A uint32 cell array and the pointer to pass for it (the pointer keeps the array alive)."""
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a, a.ctypes.data_as(C.c_void_p)


def take(ptr, n, what):
    """Copy n returned cells out of a malloc'ed array and free it; a NULL return fails the test."""
    assert ptr, f"{what} returned NULL"
    a = np.frombuffer((C.c_uint32 * n).from_address(ptr), np.uint32).copy()
    _libc.free(ptr)
    return a


def dirty(rng, vals, width):
    """vals with random bits above the low `width` bits (the bits a cell leaves unspecified)."""
    vals = np.asarray(vals, np.uint32)
    return vals | (rng.integers(0, 1 << 32, vals.shape, dtype=np.uint64).astype(np.uint32) & np.uint32(~((1 << width) - 1) & 0xFFFFFFFF))


def child_upper_bits(ps):
    """Every input cell with random bits above its field (union byte: 8-31, union integer: 12-31 for .t and 24-31 for the
    gamma .l, union bit: 1-31, union hex: 4-31): each function returns what it returns for clean cells."""
    from oracle.oracle import Oracle

    ps = int(ps)
    lib, orc, sz = dropin_lib(), Oracle(), sizes(ps)
    rng = np.random.default_rng(7100 + ps)
    p = lib.init(ps)
    P = C.byref(p)
    B8, T12, L24 = 8, 12, 24

    def both(fn, n_out, mask, *inputs):
        """fn on clean and on dirty cells; inputs are (values, width) pairs; returns the clean result's fields."""
        res = []
        for messy in (False, True):
            arrs = [cells(dirty(rng, v, w) if messy else v) for v, w in inputs]
            res.append(take(fn(*[pp for _, pp in arrs]), n_out, fn.__name__) & mask)
        assert (res[0] == res[1]).all(), f"{fn.__name__}: upper cell bits change the result"
        return res[0]

    # ring, samplers, codec
    f12 = rng.integers(0, 4096, 256, dtype=np.uint16)
    fq = rng.integers(0, Q, 256, dtype=np.uint16)
    g12 = rng.integers(0, 4096, 256, dtype=np.uint16)
    assert (both(lib.NTT, 256, 0xFFF, (f12, T12)) == orc.ntt(f12)[0]).all()
    assert (both(lib.InverseNTT, 256, 0xFFF, (fq, T12)) == orc.intt(fq)[0]).all()
    assert (both(lib.MultiplyNTTs, 256, 0xFFF, (f12, T12), (g12, T12)) == orc.multiply_ntts(f12, g12)[0]).all()
    for eta in (2, 3):
        B = rng.integers(0, 256, 64 * eta, dtype=np.uint8)
        assert (both(lambda b: lib.SamplePolyCBD(b, eta), 256, 0xFFF, (B, B8)) == orc.cbd(B, eta)[0]).all()
    for d in (1, 4, 5, 10, 11, 12):
        F = rng.integers(0, 1 << d, 256, dtype=np.uint16)
        Bd = rng.integers(0, 256, 32 * d, dtype=np.uint8)
        assert (both(lambda f: lib.ByteEncode(f, d), 32 * d, 0xFF, (F, T12)) == orc.byte_encode(F, d)[0]).all()
        assert (both(lambda b: lib.ByteDecode(b, d), 256, 0xFFF, (Bd, B8)) == orc.byte_decode(Bd, d)[0]).all()
    for d in range(1, 13):
        for x in rng.integers(0, 4096, 16):
            x, y = int(x), int(x) & ((1 << d) - 1)
            assert lib.Compress(x, d) & 0xFFF == orc.compress(x, d)[0] == lib.Compress(int(dirty(rng, x, T12)), d) & 0xFFF
            assert lib.Decompress(y, d) & 0xFFF == orc.decompress(y, d)[0] == lib.Decompress(int(dirty(rng, y, T12)), d) & 0xFFF
    for i in range(128):
        assert lib.BitRev7(i) & 0x7F == lib.BitRev7(int(dirty(rng, i, B8))) & 0x7F == orc.bitrev7(i)
    a0, a1, b0, b1 = (int(x) for x in rng.integers(0, 4096, 4))
    for g in (0, 17, Q - 1):
        out = (C.c_uint16 * 2)()
        orc.fn("basecase_multiply")(*(C.c_uint16(x) for x in (a0, a1, b0, b1, g)), out)
        args = [int(dirty(rng, x, T12)) for x in (a0, a1, b0, b1)] + [int(dirty(rng, g, L24))]
        assert list(take(lib.BaseCaseMultiply(a0, a1, b0, b1, g), 2, "BaseCaseMultiply") & 0xFFF) == list(out)
        assert list(take(lib.BaseCaseMultiply(*args), 2, "BaseCaseMultiply") & 0xFFF) == list(out)
    bits = rng.integers(0, 2, 80, dtype=np.uint8)
    assert (both(lambda b: lib.BitsToBytes(b, 80), 10, 0xFF, (bits, 1)) == np.packbits(bits, bitorder="little")).all()
    by = rng.integers(0, 256, 10, dtype=np.uint8)
    assert (both(lambda b: lib.BytesToBits(b, 10), 80, 1, (by, B8)) == np.unpackbits(by, bitorder="little")).all()
    # SampleNTT writes at most B[32].e and B[33].e: every other bit of the caller's 34 cells stays as it was
    for _ in range(8):
        seed = rng.integers(0, 256, 34, dtype=np.uint8)
        want_a, want_after = orc.sample_ntt_with_seeds(seed[None])
        for messy in (False, True):
            B, pB = cells(dirty(rng, seed, B8) if messy else seed)
            before = B.copy()
            a = take(lib.SampleNTT(pB), 256, "SampleNTT") & 0xFFF
            assert (a == want_a[0]).all()
            assert (B[:32] == before[:32]).all() and (B[32:] >> 8 == before[32:] >> 8).all()
            assert ((B[32:] & 0xFF) == want_after[0, 32:]).all()
    # K-PKE and ML-KEM internal
    d, z, m, rr = (rng.integers(0, 256, 32, dtype=np.uint8) for _ in range(4))
    oek, odk = orc.keygen(ps, d[None], z[None])
    pek, pdk = orc.pke_keygen(ps, d[None])
    oc, oK = orc.encaps(ps, oek, m[None])
    pc = orc.pke_encrypt(ps, pek, m[None], rr[None])
    for messy in (False, True):
        cv = lambda v: cells(dirty(rng, v, B8) if messy else v)
        (_, pd), (_, pz), (_, pm), (_, pr) = cv(d), cv(z), cv(m), cv(rr)
        k = lib.KeyGen_internal(P, pd, pz)
        assert k.ek_len == sz["ek"] and k.dk_len == sz["dk"]
        assert (take(k.ek, sz["ek"], "KeyGen_internal") & 0xFF == oek[0]).all()
        assert (take(k.dk, sz["dk"], "KeyGen_internal") & 0xFF == odk[0]).all()
        k = lib.PKE_KeyGen(P, pd)
        assert (take(k.ek, sz["ek"], "PKE_KeyGen") & 0xFF == pek[0]).all()
        assert (take(k.dk, sz["dk_pke"], "PKE_KeyGen") & 0xFF == pdk[0]).all()
        (_, pe), (_, pdkc), (_, pcc), (_, ppc), (_, ppdk) = cv(oek[0]), cv(odk[0]), cv(oc[0]), cv(pc[0]), cv(pdk[0])
        e = lib.Encaps_internal(P, pe, pm)
        assert e.c_len == sz["c"] and (take(e.c, sz["c"], "Encaps_internal") & 0xFF == oc[0]).all()
        assert (np.array(e.K, np.uint32) & 0xFF == oK[0]).all()
        assert (take(lib.Decaps_internal(P, pdkc, pcc), 32, "Decaps_internal") & 0xFF == oK[0]).all()
        assert (take(lib.PKE_Encrypt(P, pe, pm, pr), sz["c"], "PKE_Encrypt") & 0xFF == pc[0]).all()
        assert (take(lib.PKE_Decrypt(P, ppdk, ppc), 32, "PKE_Decrypt") & 0xFF == m).all()
        # the public wrappers: KEM_Decaps exactly, KEM_Encaps (random m) by decapsulating its result
        assert (take(lib.KEM_Decaps(P, pdkc, sz["dk"], pcc, sz["c"]), 32, "KEM_Decaps") & 0xFF == oK[0]).all()
        e = lib.KEM_Encaps(P, pe, sz["ek"])
        c = take(e.c, sz["c"], "KEM_Encaps") & 0xFF
        assert (orc.decaps(ps, odk, c.astype(np.uint8)[None])[0] == np.array(e.K, np.uint32) & 0xFF).all()
    # the SHA-3 front end
    sfx_hash, sfx_xof = (C.c_uint32 * 4)(0, 1, 0, 0), (C.c_uint32 * 4)(1, 1, 1, 1)
    for n in (0, 5, 1080, 1087):
        bits = rng.integers(0, 2, n, dtype=np.uint8)
        want = orc.sha3_bits(bits, [0, 1, 0, 0], 512, 256)
        assert (both(lambda b: lib.sha3_b(b, n, 256, 512, sfx_hash), 256, 1, (bits, 1)) == want).all()
        assert (both(lambda b: lib.sha3_b(b, n, 300, 256, sfx_xof), 300, 1, (bits, 1)) == orc.sha3_bits(bits, [1, 1, 1, 1], 256, 300)).all()
    msg = rng.integers(0, 256, 150, dtype=np.uint8)
    hexd = np.stack([msg >> 4, msg & 15], axis=1).ravel()
    want = np.frombuffer(hashlib.sha3_256(msg.tobytes()).digest(), np.uint8)
    assert (both(lambda h: lib.sha3_h(h, 150, 256, 512, sfx_hash), 64, 0xF, (hexd, 4)) == np.stack([want >> 4, want & 15], 1).ravel()).all()
    assert (both(lambda h: lib.h2b(h, 150, 1200), 1200, 1, (hexd, 4)) == np.unpackbits(msg, bitorder="little")).all()
    assert (both(lambda b: lib.b2h(b, 1200), 300, 0xF, (np.unpackbits(msg, bitorder="little"), 1)) == hexd).all()


def child_wrappers(ps):
    """KEM_KeyGen -> KEM_Encaps -> KEM_Decaps: K agrees, the oracle decapsulates to K, dk = dk_pke || ek || H(ek) || z."""
    from oracle.oracle import Oracle

    ps = int(ps)
    lib, orc, sz, k = dropin_lib(), Oracle(), sizes(ps), sizes(ps)["k"]
    errno = C.c_int.in_dll(lib, "ml_errno")
    p = lib.init(ps)
    assert (p.k & 0xFF, p.du & 0xFF, p.dv & 0xFF) == (k, {512: 10, 768: 10, 1024: 11}[ps], {512: 4, 768: 4, 1024: 5}[ps])
    seen = set()
    for _ in range(4):
        keys = lib.KEM_KeyGen(C.byref(p))
        assert keys.ek_len == sz["ek"] and keys.dk_len == sz["dk"]
        ek = (take(keys.ek, sz["ek"], "KEM_KeyGen") & 0xFF).astype(np.uint8)
        dk = (take(keys.dk, sz["dk"], "KEM_KeyGen") & 0xFF).astype(np.uint8)
        assert (dk[384 * k : 768 * k + 32] == ek).all()
        assert dk[768 * k + 32 : 768 * k + 64].tobytes() == hashlib.sha3_256(ek.tobytes()).digest()
        ekc, pe = cells(ek)
        e = lib.KEM_Encaps(C.byref(p), pe, sz["ek"])
        assert e.c_len == sz["c"]
        c = (take(e.c, sz["c"], "KEM_Encaps") & 0xFF).astype(np.uint8)
        K = bytes(x & 0xFF for x in e.K)
        dkc, pd = cells(dk)
        cc, pc = cells(c)
        Kd = take(lib.KEM_Decaps(C.byref(p), pd, sz["dk"], pc, sz["c"]), 32, "KEM_Decaps") & 0xFF
        assert bytes(Kd.astype(np.uint8)) == K == orc.decaps(ps, dk[None], c[None])[0].tobytes()
        seen.add(K)
    assert len(seen) == 4 and errno.value == 0


class StderrCapture:
    """Everything written to file descriptor 2 (the C library's stderr) inside the block."""

    def __enter__(self):
        self.f = tempfile.TemporaryFile()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode()
        self.f.close()


def child_errors(ps):
    """Each error of the public wrappers: the reference's ml_errno, a NULL / zeroed result and its stderr lines
    ("ERROR: ml_kem.c - <line>\\n\\t<message>\\n\\n", the reference's ERR_MSG).  The reference never clears ml_errno, so a
    successful call after an error leaves it as it was."""
    ps = int(ps)
    lib, sz = dropin_lib(), sizes(ps)
    errno = C.c_int.in_dll(lib, "ml_errno")
    p = lib.init(ps)
    P = C.byref(p)
    keys = lib.KEM_KeyGen(P)
    ek = take(keys.ek, sz["ek"], "KEM_KeyGen")
    dk = take(keys.dk, sz["dk"], "KEM_KeyGen")
    (_, pe), (_, pd) = cells(ek), cells(dk)
    e = lib.KEM_Encaps(P, pe, sz["ek"])
    c = take(e.c, sz["c"], "KEM_Encaps")
    _, pc = cells(c)
    assert errno.value == 0

    def expect(code, line, msg, call):
        errno.value = 0
        with StderrCapture() as cap:
            r = call()
        assert errno.value == code, (msg, errno.value)
        assert cap.text == f"ERROR: ml_kem.c - {line}\n\t{msg}\n\n", (msg, cap.text)
        # a later successful call leaves ml_errno alone
        with StderrCapture() as cap:
            K = take(lib.KEM_Decaps(P, pd, sz["dk"], pc, sz["c"]), 32, "KEM_Decaps")
        assert errno.value == code and cap.text == "" and (K & 0xFF == np.array(e.K, np.uint32) & 0xFF).all()
        return r

    bad = expect(-1, 1390, "init() :: Invalid paramater set provided", lambda: lib.init(999))
    assert (bad.k, bad.n1, bad.n2, bad.du, bad.dv) == (0, 0, 0, 0, 0)
    for ek_len in (sz["ek"] - 1, sz["ek"] + 1, 0):
        r = expect(-3, 1268, "KEM_Encaps() :: Type check failed", lambda: lib.KEM_Encaps(P, pe, ek_len))
        assert not r.c and r.c_len == 0 and not any(r.K)
    for c_len in (sz["c"] - 1, sz["c"] + 32):
        assert not expect(-3, 1322, "KEM_Decaps() :: Ciphertext type check failed",
                          lambda: lib.KEM_Decaps(P, pd, sz["dk"], pc, c_len))
    for dk_len in (sz["dk"] - 1, sz["dk"] + 1):
        assert not expect(-3, 1330, "KEM_Decaps() :: Decapsulation key type check failed",
                          lambda: lib.KEM_Decaps(P, pd, dk_len, pc, sz["c"]))
    k = sz["k"]
    for pos in (768 * k + 32, 768 * k + 63, 384 * k):  # the stored H(ek), and ek itself
        bad_dk = dk.copy()
        bad_dk[pos] ^= 0x10
        _, pbad = cells(bad_dk)
        assert not expect(-5, 1346, "KEM_Decaps() :: Hash check failed", lambda: lib.KEM_Decaps(P, pbad, sz["dk"], pc, sz["c"]))


SHA3 = {  # name: (suffix bits, capacity, default output bits, hashlib constructor, is_xof)
    "SHA3-224": ([0, 1, 0, 0], 448, 224, hashlib.sha3_224, False),
    "SHA3-256": ([0, 1, 0, 0], 512, 256, hashlib.sha3_256, False),
    "SHA3-384": ([0, 1, 0, 0], 768, 384, hashlib.sha3_384, False),
    "SHA3-512": ([0, 1, 0, 0], 1024, 512, hashlib.sha3_512, False),
    "SHAKE128": ([1, 1, 1, 1], 256, 256, hashlib.shake_128, True),
    "SHAKE256": ([1, 1, 1, 1], 512, 512, hashlib.shake_256, True),
}


def child_sha3_sweep(name):
    """mlkem_b200_sha3_bits_batch at every message bit length 0 .. 2r + 16, five messages per call in chunks of 2 items,
    against oracle.sha3_bits; byte-aligned lengths also against hashlib; XOF output lengths across the squeeze blocks;
    then sha3_b / sha3_h / sha3_s as single calls on a sample of the lengths."""
    from oracle.oracle import Oracle

    lib, orc = dropin_lib(), Oracle()
    sfx, c, d0, hfn, xof = SHA3[name]
    r = 1600 - c
    slen = 4 if xof else 2
    rng = np.random.default_rng(7200 + c + slen)
    opts = Opts(-1, 0, None, 2, 0, 0)
    sf = np.asarray(sfx, np.uint8)

    def batch(msgs_bits, nbits, d):
        packed = np.packbits(msgs_bits, axis=1, bitorder="little") if nbits else np.zeros((len(msgs_bits), 1), np.uint8)
        packed = np.ascontiguousarray(packed)
        out = np.full((len(msgs_bits), (d + 7) // 8), 0xA5, np.uint8)
        rc = lib.mlkem_b200_sha3_bits_batch(C.c_size_t(len(msgs_bits)), C.c_void_p(packed.ctypes.data), C.c_size_t(nbits),
                                            C.c_void_p(sf.ctypes.data), C.c_uint(c), C.c_size_t(d),
                                            C.c_void_p(out.ctypes.data), C.byref(opts))
        assert rc == 0, (name, nbits, d, rc)
        if d % 8:
            assert (out[:, -1] >> (d % 8) == 0).all(), f"{name}: bits above d = {d} not zero"
        return out

    quirks = 0
    for nbits in range(0, 2 * r + 17):
        msgs = rng.integers(0, 2, (5, nbits), dtype=np.uint8)
        out = batch(msgs, nbits, d0)
        quirks += (nbits + slen + 2) % r == 0
        for i in range(5):
            want = orc.sha3_bits(msgs[i], sfx, c, d0)
            assert (np.unpackbits(out[i], bitorder="little")[:d0] == want).all(), (name, nbits, i)
        if nbits % 8 == 0:
            assert (nbits + slen + 2) % r != 0  # the reference's padding deviation never falls on a byte-aligned length
            for i in range(5):
                msg = np.packbits(msgs[i], bitorder="little").tobytes() if nbits else b""
                h = hfn(msg)
                assert out[i].tobytes() == (h.digest(d0 // 8) if xof else h.digest()), (name, nbits, i, "hashlib")
    assert quirks == 2
    if xof:
        for nbits in (0, 7, 8, r - slen - 2, r - slen - 1, r, 2 * r - slen - 2, 2 * r + 16):
            msgs = rng.integers(0, 2, (5, nbits), dtype=np.uint8)
            for d in (1, 7, 8, r - 1, r, r + 1, 2 * r, 3 * r + 5):
                out = batch(msgs, nbits, d)
                for i in range(5):
                    want = orc.sha3_bits(msgs[i], sfx, c, d)
                    assert (np.unpackbits(out[i], bitorder="little")[:d] == want).all(), (name, nbits, d, i)
    # the reference-signature front end, one call per message
    sfc = (C.c_uint32 * 4)(*sfx)
    for nbits in sorted({0, 1, 8, r - slen - 2, r - slen - 1, r - 8, r, r + 3, 2 * r - slen - 2, 2 * r + 16}):
        bits = rng.integers(0, 2, nbits, dtype=np.uint8)
        _, pb = cells(bits)
        got = take(lib.sha3_b(pb, nbits, d0, c, sfc), d0, "sha3_b") & 1
        assert (got == orc.sha3_bits(bits, sfx, c, d0)).all(), (name, "sha3_b", nbits)
    for nbytes in (0, 1, r // 8 - 1, r // 8, r // 8 + 1, 2 * r // 8 + 2):
        msg = rng.integers(0, 256, nbytes, dtype=np.uint8)
        h = hfn(msg.tobytes())
        want = np.frombuffer(h.digest(d0 // 8) if xof else h.digest(), np.uint8)
        _, ph = cells(np.stack([msg >> 4, msg & 15], axis=1).ravel())
        got = take(lib.sha3_h(ph, nbytes, d0, c, sfc), d0 // 4, "sha3_h") & 0xF
        assert (got == np.stack([want >> 4, want & 15], axis=1).ravel()).all(), (name, "sha3_h", nbytes)
        s = lib.sha3_s(msg.tobytes(), nbytes, d0, c, sfc)
        assert s, "sha3_s returned NULL"
        got = C.string_at(s, d0 // 8)
        _libc.free(s)
        assert got == want.tobytes(), (name, "sha3_s", nbytes)


if __name__ == "__main__":
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    globals()["child_" + sys.argv[1]](*sys.argv[2:])
