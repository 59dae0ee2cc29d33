"""CPU tests of X25519 and the X25519MLKEM768 hybrid: the independent Python X25519 the GPU tests compare against, pinned to
RFC 7748's vectors (and to `cryptography` where it is installed); the wire-format sizes the header exports; and that without a
device every new entry point refuses (MLKEM_B200_ERR_CUDA) without writing anything."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 2 ** 255 - 19
A24 = 121665


# ------------------------------------------------------------------ RFC 7748 section 5, straight from the text
def decode_scalar(k: bytes) -> int:
    b = bytearray(k)
    b[0] &= 248
    b[31] &= 127
    b[31] |= 64
    return int.from_bytes(b, "little")


def decode_u(u: bytes) -> int:
    return int.from_bytes(u, "little") & ((1 << 255) - 1)  # bit 255 ignored; values >= p accepted


def x25519_ref(k: bytes, u: bytes) -> bytes:
    """X25519(k, u): the Montgomery ladder of RFC 7748 section 5 on Python integers."""
    k, x1 = decode_scalar(k), decode_u(u)
    x2, z2, x3, z3, swap = 1, 0, x1, 1, 0
    for t in range(254, -1, -1):
        kt = (k >> t) & 1
        swap ^= kt
        if swap:
            x2, x3, z2, z3 = x3, x2, z3, z2
        swap = kt
        A, B, C_, D = (x2 + z2) % P, (x2 - z2) % P, (x3 + z3) % P, (x3 - z3) % P
        AA, BB, DA, CB = A * A % P, B * B % P, D * A % P, C_ * B % P
        E = (AA - BB) % P
        x3, z3 = (DA + CB) ** 2 % P, x1 * (DA - CB) ** 2 % P
        x2, z2 = AA * BB % P, E * (AA + A24 * E) % P
    if swap:
        x2, z2 = x3, z3
    return (x2 * pow(z2, P - 2, P) % P).to_bytes(32, "little")


BASE = (9).to_bytes(32, "little")
RFC_5_2 = [
    ("a546e36bf0527c9d3b16154b82465edd62144c0ac1fc5a18506a2244ba449ac4",
     "e6db6867583030db3594c1a424b15f7c726624ec26b3353b10a903a6d0ab1c4c",
     "c3da55379de9c6908e94ea4df28d084f32eccf03491c71f754b4075577a28552"),
    ("4b66e9d4d1b4673c5ad22691957d6af5c11b6421e0ea01d42ca4169e7918ba0d",
     "e5210f12786811d3f4b7959d0538ae2c31dbe7106fc03c3efc4cd549c715a493",
     "95cbde9476e8907d7aade45cb4b873f88b595a68799fa152e6f8f7647aac7957"),
]
ITER_1 = "422c8e7a6227d7bca1350b3e2bb7279f7897b87bb6854b783c60e80311ae3079"
ITER_1000 = "684cf59ba83309552800ef566f2f4d3c1c3887c49360e3875f2eb94d99532c51"
ALICE = ("77076d0a7318a57d3c16c17251b26645df4c2f87ebc0992ab177fba51db92c2a",
         "8520f0098930a754748b7ddcb43ef75a0dbf3a0d26381af4eba4a98eaa9b4e6a")
BOB = ("5dab087e624a8a4b79e17f8b83800ee66f3bb1292618b6fd1c2f8b27ff88e0eb",
       "de9edb7d7b7dc1b4d35b61c2ece435373f8343c85b78674dadfc7e146f882b4f")
SHARED = "4a5d9d5ba4ce2de1728e3bf480350f25e07e21c947d19e3376f09b3c1e161742"


def small_order_points():
    """u-coordinates of the points of order 1, 2, 4 and 8 on the curve and its twist, as canonical integers: 0 (order 2),
    1 and p - 1 (order 4), and the two of order 8 (the x-only doubling of each is 1 or p - 1).  Checked below by the ladder:
    every clamped scalar is a multiple of 8, so each of them maps to 0."""
    order8 = [325606250916557431795983626356110631294008115727848805560023387167927233504,
              39382357235489614581723060781553021112529911719440698176882885853963445705823]
    for u in order8:  # x(2 P) = (u^2 - 1)^2 / (4 u (u^2 + 486662 u + 1)) is +-1, of order 4
        dbl = (u * u - 1) ** 2 * pow(4 * u * (u * u + 486662 * u + 1), P - 2, P) % P
        assert dbl in (1, P - 1)
    return [0, 1, P - 1] + order8


def test_rfc7748_section_5_2_vectors():
    for k, u, out in RFC_5_2:
        assert x25519_ref(bytes.fromhex(k), bytes.fromhex(u)).hex() == out
    # the second u has bit 255 set: the same u with the bit cleared gives the same output
    k, u, out = RFC_5_2[1]
    ub = bytearray(bytes.fromhex(u))
    assert ub[31] & 0x80
    ub[31] &= 0x7F
    assert x25519_ref(bytes.fromhex(k), bytes(ub)).hex() == out


def test_rfc7748_iterated_vector():
    k = u = BASE
    for i in range(1, 1001):
        k, u = x25519_ref(k, u), k
        if i == 1:
            assert k.hex() == ITER_1
    assert k.hex() == ITER_1000


def test_rfc7748_section_6_1_diffie_hellman():
    a, b = bytes.fromhex(ALICE[0]), bytes.fromhex(BOB[0])
    assert x25519_ref(a, BASE).hex() == ALICE[1]
    assert x25519_ref(b, BASE).hex() == BOB[1]
    assert x25519_ref(a, bytes.fromhex(BOB[1])).hex() == SHARED == x25519_ref(b, bytes.fromhex(ALICE[1])).hex()


def test_small_order_points_give_zero():
    """Every u derived by small_order_points() is of small order: any clamped scalar maps it to 0."""
    rng = np.random.default_rng(7)
    pts = small_order_points()
    for u in pts:
        for _ in range(3):
            k = bytes(rng.integers(0, 256, 32, dtype=np.uint8))
            assert x25519_ref(k, u.to_bytes(32, "little")) == bytes(32), u
    # the same u plus p (a non-canonical encoding below 2^255) too
    for u in pts:
        if u + P < 2 ** 255:
            assert x25519_ref(bytes(range(32)), (u + P).to_bytes(32, "little")) == bytes(32)


def test_against_cryptography():
    x = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.x25519")
    from cryptography.hazmat.primitives import serialization

    rng = np.random.default_rng(11)
    raw = serialization.Encoding.Raw, serialization.PublicFormat.Raw
    for _ in range(64):
        k, u = (bytes(rng.integers(0, 256, 32, dtype=np.uint8)) for _ in range(2))
        sk = x.X25519PrivateKey.from_private_bytes(k)
        assert sk.public_key().public_bytes(*raw) == x25519_ref(k, BASE)
        try:
            want = sk.exchange(x.X25519PublicKey.from_public_bytes(u))
        except ValueError:  # an all-zero result: cryptography refuses it
            want = bytes(32)
        assert want == x25519_ref(k, u)


# ------------------------------------------------------------------ the C ABI without a device
def test_header_wire_format_sizes():
    txt = open(os.path.join(ROOT, "include", "mlkem_b200.h")).read()
    defs = dict(re.findall(r"#define (MLKEM_B200_X25519MLKEM768_\w+|MLKEM_B200_ERR_X25519_ZERO) \(?(-?\d+)\)?", txt))
    assert {k: int(v) for k, v in defs.items()} == {
        "MLKEM_B200_X25519MLKEM768_CLIENT_SHARE_BYTES": 1184 + 32,
        "MLKEM_B200_X25519MLKEM768_CLIENT_SECRET_BYTES": 2400 + 32,
        "MLKEM_B200_X25519MLKEM768_SERVER_SHARE_BYTES": 1088 + 32,
        "MLKEM_B200_X25519MLKEM768_SHARED_SECRET_BYTES": 32 + 32,
        "MLKEM_B200_ERR_X25519_ZERO": -6,
    }
    for v in (1216, 2432, 1120, 64, 1184, 2400, 1088):
        assert v % 16 == 0


@pytest.fixture(scope="module")
def lib():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import crystals_kyber_b200 as ck

    if not os.path.exists(ck.LIB_PATH):
        import subprocess

        subprocess.run(["make", "-C", ROOT, "lib"], check=True, stdout=subprocess.DEVNULL)
    return ck.load()


def test_entry_points_refuse_without_device(lib):
    n = 3
    buf = lambda size, fill: np.full((n, size), fill, np.uint8)
    ptr = lambda a: C.c_void_p(a.ctypes.data)
    ins = {w: buf(w, 0x11) for w in (32, 1216, 2432, 1120)}
    outs = {w: buf(w, 0xA5) for w in (32, 1216, 2432, 1120, 64)}
    status = np.full(n, 0x5A5A5A5A, np.int32)
    seed = C.c_char_p(bytes(32))
    rcs = [
        lib.mlkem_b200_x25519_batch(n, ptr(ins[32]), None, ptr(outs[32]), None),
        lib.mlkem_b200_x25519_batch(n, ptr(ins[32]), ptr(ins[32]), ptr(outs[32]), None),
        lib.mlkem_b200_x25519mlkem768_keygen_batch(n, ptr(ins[32]), ptr(ins[32]), ptr(ins[32]), ptr(outs[1216]), ptr(outs[2432]), None),
        lib.mlkem_b200_x25519mlkem768_encaps_batch(n, ptr(ins[1216]), ptr(ins[32]), ptr(ins[32]), ptr(outs[1120]), ptr(outs[64]),
                                                   ptr(status), None),
        lib.mlkem_b200_x25519mlkem768_decaps_batch(n, ptr(ins[2432]), ptr(ins[1120]), ptr(outs[64]), ptr(status), None),
        lib.mlkem_b200_x25519mlkem768_keygen_seeded_batch(n, seed, ptr(outs[1216]), ptr(outs[2432]), None),
        lib.mlkem_b200_x25519mlkem768_encaps_seeded_batch(n, ptr(ins[1216]), seed, ptr(outs[1120]), ptr(outs[64]), ptr(status), None),
        lib.mlkem_b200_x25519mlkem768_keygen_seeded_batch(n, None, ptr(outs[1216]), ptr(outs[2432]), None),
    ]
    assert rcs == [-10] * len(rcs)
    assert all((o == 0xA5).all() for o in outs.values()) and (status == 0x5A5A5A5A).all()
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM()
    z32 = np.zeros((1, 32), np.uint8)
    for call in (lambda: kem.x25519(z32), lambda: kem.x25519(z32, z32), lambda: kem.x25519mlkem768_keygen(z32, z32, z32),
                 lambda: kem.x25519mlkem768_encaps(np.zeros((1, 1216), np.uint8), z32, z32),
                 lambda: kem.x25519mlkem768_decaps(np.zeros((1, 2432), np.uint8), np.zeros((1, 1120), np.uint8)),
                 lambda: kem.x25519mlkem768_keygen_seeded(1, seed=bytes(32)),
                 lambda: kem.x25519mlkem768_encaps_seeded(np.zeros((1, 1216), np.uint8), seed=bytes(32))):
        with pytest.raises(ck.MlKemB200Error):
            call()
