"""CPU tests of P-256 and the SecP256r1MLKEM768 hybrid: the independent Python P-256 the GPU tests compare against (affine
arithmetic on Python integers, straight from FIPS 186-5 / SP 800-186), pinned to `cryptography`; the wire-format sizes and
status codes the header exports; and that without a device every new entry point refuses (MLKEM_B200_ERR_CUDA) without writing
anything."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 2 ** 256 - 2 ** 224 + 2 ** 192 + 2 ** 96 - 1
A = P - 3
B = 0x5AC635D8AA3A93E7B3EBBD55769886BC651D06B0CC53B0F63BCE3C3E27D2604B
N = 0xFFFFFFFF00000000FFFFFFFFFFFFFFFFBCE6FAADA7179E84F3B9CAC2FC632551
GX = 0x6B17D1F2E12C4247F8BCE6E563A440F277037D812DEB33A0F4A13945D898C296
GY = 0x4FE342E2FE1A7F9B8EE7EB4A7C0F9E162BCE33576B315ECECBB6406837BF51F5
G = (GX, GY)
SHARE, SECRET, SERVER, SS, POINT = 1249, 2432, 1153, 64, 65


# ------------------------------------------------------------------ P-256 on Python integers (None is the identity)
def on_curve(pt) -> bool:
    x, y = pt
    return (y * y - (x * x * x + A * x + B)) % P == 0


def add(p1, p2):
    if p1 is None:
        return p2
    if p2 is None:
        return p1
    (x1, y1), (x2, y2) = p1, p2
    if x1 == x2 and (y1 + y2) % P == 0:
        return None
    if p1 == p2:
        lam = (3 * x1 * x1 + A) * pow(2 * y1, -1, P) % P
    else:
        lam = (y2 - y1) * pow(x2 - x1, -1, P) % P
    x3 = (lam * lam - x1 - x2) % P
    return x3, (lam * (x1 - x3) - y1) % P


def mul(k: int, pt=G):
    r = None
    for bit in bin(k)[2:] if k > 0 else "":
        r = add(r, r)
        if bit == "1":
            r = add(r, pt)
    return r


def encode(pt) -> bytes:
    return b"\x04" + pt[0].to_bytes(32, "big") + pt[1].to_bytes(32, "big")


def decode(b: bytes):
    """SP 800-56A partial public-key validation of a 65-byte UncompressedPointRepresentation: the point, or None."""
    if len(b) != 65 or b[0] != 4:
        return None
    x, y = int.from_bytes(b[1:33], "big"), int.from_bytes(b[33:], "big")
    if x >= P or y >= P or not on_curve((x, y)):
        return None
    return x, y


def public(k: bytes):
    """The 65-byte public key of a 32-byte big-endian scalar, or None when it is outside [1, n - 1]."""
    d = int.from_bytes(k, "big")
    return encode(mul(d)) if 1 <= d < N else None


def ecdh(k: bytes, peer: bytes):
    """X of d Q (32 bytes), or the status that rejects it: -7 (scalar outside [1, n - 1]) before -8 (invalid point)."""
    d = int.from_bytes(k, "big")
    if not 1 <= d < N:
        return -7
    q = decode(peer)
    if q is None:
        return -8
    return mul(d, q)[0].to_bytes(32, "big")


def seed_scalar(r: bytes) -> bytes:
    """FIPS 186-5 A.2.1: d = (c mod (n - 1)) + 1 for c = the big-endian integer of r[0..40)."""
    return ((int.from_bytes(r[:40], "big") % (N - 1)) + 1).to_bytes(32, "big")


def invalid_points():
    """One of every kind of invalid 65-byte point: (name, bytes)."""
    g = encode(G)
    out = [("prefix 0", b"\x00" + g[1:]), ("prefix 2", b"\x02" + g[1:]), ("prefix 3", b"\x03" + g[1:]),
           ("prefix 5", b"\x05" + g[1:]), ("prefix ff", b"\xff" + g[1:])]
    out += [("x = p", b"\x04" + P.to_bytes(32, "big") + g[33:]), ("x = 2^256 - 1", b"\x04" + b"\xff" * 32 + g[33:])]
    out += [("y = p", g[:33] + P.to_bytes(32, "big")), ("y = 2^256 - 1", g[:33] + b"\xff" * 32)]
    # x + p, for a curve point with a small x: the same residue as a valid point, rejected for its encoding alone
    x0, y0 = small_x_point()
    out += [("x + p", b"\x04" + (x0 + P).to_bytes(32, "big") + y0.to_bytes(32, "big"))]
    out += [("off curve", g[:64] + bytes([g[64] ^ 1])), ("zero", b"\x04" + bytes(64)), ("all zero", bytes(65)),
            ("(0, 1)", b"\x04" + bytes(32) + (1).to_bytes(32, "big"))]
    return out


def small_x_point():
    """The curve point with the smallest x >= 1 (p = 3 mod 4: the square root is a power)."""
    for x in range(1, 100):
        rhs = (x ** 3 + A * x + B) % P
        y = pow(rhs, (P + 1) // 4, P)
        if y * y % P == rhs:
            return x, y


def test_generator_multiples():
    assert on_curve(G)
    assert encode(mul(1)) == b"\x04" + bytes.fromhex("6b17d1f2e12c4247f8bce6e563a440f277037d812deb33a0f4a13945d898c296"
                                                   "4fe342e2fe1a7f9b8ee7eb4a7c0f9e162bce33576b315ececbb6406837bf51f5")
    assert mul(N - 1) == (GX, (-GY) % P) and mul(N) is None and add(mul(N - 1), G) is None
    assert mul(2) == add(G, G)
    # the modular square root used by invalid_points() is right: p = 3 mod 4
    assert P % 4 == 3


def test_against_cryptography():
    ec = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ec")
    from cryptography.hazmat.primitives import serialization

    def pub_of(d):
        return ec.derive_private_key(d, ec.SECP256R1()).public_key().public_bytes(serialization.Encoding.X962,
                                                                                    serialization.PublicFormat.UncompressedPoint)

    for d in (1, 2, N - 1):
        assert pub_of(d) == public(d.to_bytes(32, "big"))
    rng = np.random.default_rng(256)
    for _ in range(1000):
        a, b = (bytes(rng.integers(0, 256, 32, dtype=np.uint8)) for _ in range(2))
        da, db = int.from_bytes(a, "big"), int.from_bytes(b, "big")
        if not (1 <= da < N and 1 <= db < N):
            continue
        ka, kb = ec.derive_private_key(da, ec.SECP256R1()), ec.derive_private_key(db, ec.SECP256R1())
        pa = pub_of(da)
        assert pa == public(a)
        want = ka.exchange(ec.ECDH(), ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), pub_of(db)))
        assert want == ecdh(a, public(b)) == ecdh(b, pa)
    # out-of-range scalars: cryptography refuses them too
    for d in (0, N, 2 ** 256 - 1):
        with pytest.raises(ValueError):
            ec.derive_private_key(d, ec.SECP256R1())
        assert public(d.to_bytes(32, "big")) is None and ecdh(d.to_bytes(32, "big"), encode(G)) == -7
    for name, pt in invalid_points():
        assert decode(pt) is None, name
        with pytest.raises(ValueError):
            ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), pt)


def test_seed_scalar_reduction():
    for c, want in ((0, 1), (N - 2, N - 1), (N - 1, 1), (2 ** 320 - 1, (2 ** 320 - 1) % (N - 1) + 1)):
        assert int.from_bytes(seed_scalar(c.to_bytes(40, "big")), "big") == want
    rng = np.random.default_rng(5)
    for _ in range(200):
        d = int.from_bytes(seed_scalar(bytes(rng.integers(0, 256, 64, dtype=np.uint8))), "big")
        assert 1 <= d <= N - 1


# ------------------------------------------------------------------ the C ABI without a device
def test_header_constants():
    txt = open(os.path.join(ROOT, "include", "mlkem_b200.h")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define (MLKEM_B200_\w+) \(?(-?\d+)\)?", txt)}
    assert {k: v for k, v in defs.items() if "SECP256R1" in k or "P256" in k or k.startswith("MLKEM_B200_ERR_EC")} == {
        "MLKEM_B200_P256_POINT_BYTES": 65,
        "MLKEM_B200_SECP256R1MLKEM768_CLIENT_SHARE_BYTES": 65 + 1184,
        "MLKEM_B200_SECP256R1MLKEM768_CLIENT_SECRET_BYTES": 2400 + 32,
        "MLKEM_B200_SECP256R1MLKEM768_SERVER_SHARE_BYTES": 65 + 1088,
        "MLKEM_B200_SECP256R1MLKEM768_SHARED_SECRET_BYTES": 32 + 32,
        "MLKEM_B200_ERR_EC_SCALAR": -7,
        "MLKEM_B200_ERR_EC_POINT": -8,
    }
    codes = [v for k, v in defs.items() if k.startswith("MLKEM_B200_ERR_")]
    assert len(codes) == len(set(codes)), "two error codes share a value"


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
    ins = {w: buf(w, 0x11) for w in (32, 65, SHARE, SECRET, SERVER)}
    outs = {w: buf(w, 0xA5) for w in (32, 65, SHARE, SECRET, SERVER, SS)}
    status = np.full(n, 0x5A5A5A5A, np.int32)
    seed = C.c_char_p(bytes(32))
    rcs = [
        lib.mlkem_b200_p256_public_batch(n, ptr(ins[32]), ptr(outs[65]), ptr(status), None),
        lib.mlkem_b200_p256_ecdh_batch(n, ptr(ins[32]), ptr(ins[65]), ptr(outs[32]), ptr(status), None),
        lib.mlkem_b200_secp256r1mlkem768_keygen_batch(n, ptr(ins[32]), ptr(ins[32]), ptr(ins[32]), ptr(outs[SHARE]), ptr(outs[SECRET]),
                                                      ptr(status), None),
        lib.mlkem_b200_secp256r1mlkem768_encaps_batch(n, ptr(ins[SHARE]), ptr(ins[32]), ptr(ins[32]), ptr(outs[SERVER]), ptr(outs[SS]),
                                                      ptr(status), None),
        lib.mlkem_b200_secp256r1mlkem768_decaps_batch(n, ptr(ins[SECRET]), ptr(ins[SERVER]), ptr(outs[SS]), ptr(status), None),
        lib.mlkem_b200_secp256r1mlkem768_keygen_seeded_batch(n, seed, ptr(outs[SHARE]), ptr(outs[SECRET]), None),
        lib.mlkem_b200_secp256r1mlkem768_encaps_seeded_batch(n, ptr(ins[SHARE]), seed, ptr(outs[SERVER]), ptr(outs[SS]), ptr(status), None),
        lib.mlkem_b200_secp256r1mlkem768_keygen_seeded_batch(n, None, ptr(outs[SHARE]), ptr(outs[SECRET]), None),
    ]
    assert rcs == [-10] * len(rcs)
    assert all((o == 0xA5).all() for o in outs.values()) and (status == 0x5A5A5A5A).all()
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM()
    z32, z65 = np.zeros((1, 32), np.uint8), np.zeros((1, 65), np.uint8)
    for call in (lambda: kem.p256_public(z32), lambda: kem.p256_ecdh(z32, z65),
                 lambda: kem.secp256r1mlkem768_keygen(z32, z32, z32),
                 lambda: kem.secp256r1mlkem768_encaps(np.zeros((1, SHARE), np.uint8), z32, z32),
                 lambda: kem.secp256r1mlkem768_decaps(np.zeros((1, SECRET), np.uint8), np.zeros((1, SERVER), np.uint8)),
                 lambda: kem.secp256r1mlkem768_keygen_seeded(1, seed=bytes(32)),
                 lambda: kem.secp256r1mlkem768_encaps_seeded(np.zeros((1, SHARE), np.uint8), seed=bytes(32))):
        with pytest.raises(ck.MlKemB200Error):
            call()
