"""GPU tests of P-256 (mlkem_b200_p256_*_batch) and the SecP256r1MLKEM768 hybrid key exchange (include/mlkem_b200.h).

References that share no code with the kernels: the Python P-256 of test_secp256r1mlkem768_cpu.py (pinned there to
`cryptography`), `cryptography`'s P-256 ECDH and ML-KEM-768 for bulk and interoperability, and the oracle in FIPS 203 mode for
ML-KEM.  The wire order is ECDH first: client share = point || ek, server share = point || c, ss = ECDH || K.
"""
import ctypes as C
import hashlib
import struct

import numpy as np
import pytest

from test_launch_geometry_gpu import Guarded, call
from test_secp256r1mlkem768_cpu import GX, GY, N, P, encode, ecdh, invalid_points, mul, public, seed_scalar

pytestmark = pytest.mark.gpu

OK, ERR_ARG, ERR_MODULUS, ERR_SCALAR, ERR_POINT = 0, -11, -4, -7, -8
CS, SEC, SS_, SSEC, PT = 1249, 2432, 1153, 64, 65
SEED = bytes.fromhex("c0ffee00000102030405060708090a0b0c0d0e0f101112131415161718191a1b")
TAG_KEYGEN, TAG_ENCAPS, TAG_EC_KEYGEN, TAG_EC_ENCAPS = 1, 2, 5, 6


@pytest.fixture(scope="module")
def kem():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


@pytest.fixture(scope="module")
def lib(kem):
    return kem.lib


@pytest.fixture
def fips_oracle(oracle, kem):
    oracle.set_fips(True)
    yield oracle
    oracle.set_fips(False)


def rand(rng, n, w):
    return rng.integers(0, 256, (n, w), dtype=np.uint8)


def scalars(rng, n):
    """n random in-range P-256 scalars, 32 bytes big-endian (a row >= n is redrawn)."""
    k = rand(rng, n, 32)
    k[:, 0] &= 0x7F  # < 2^255 < n: always in range, and 0 has probability 2^-255
    return k


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    import torch

    if isinstance(t, torch.Tensor):
        torch.cuda.synchronize()
        return t.cpu().numpy()
    return t


def ec_public_many(k):
    from cryptography.hazmat.primitives import serialization
    from cryptography.hazmat.primitives.asymmetric import ec

    enc = serialization.Encoding.X962, serialization.PublicFormat.UncompressedPoint
    return np.array([np.frombuffer(ec.derive_private_key(int.from_bytes(bytes(r), "big"), ec.SECP256R1()).public_key().public_bytes(*enc), np.uint8)
                     for r in k]).reshape(len(k), PT)


def ec_ecdh_many(k, q):
    from cryptography.hazmat.primitives.asymmetric import ec

    out = np.empty((len(k), 32), np.uint8)
    for i in range(len(k)):
        sk = ec.derive_private_key(int.from_bytes(bytes(k[i]), "big"), ec.SECP256R1())
        out[i] = np.frombuffer(sk.exchange(ec.ECDH(), ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), bytes(q[i]))), np.uint8)
    return out


def derive(seed, n, tag, width=32):
    return np.frombuffer(b"".join(hashlib.shake_256(seed + struct.pack("<QQ", j, tag)).digest(width) for j in range(n)),
                         np.uint8).reshape(n, width).copy()


def derive_scalars(seed, n, tag):
    return np.array([np.frombuffer(seed_scalar(bytes(r)), np.uint8) for r in derive(seed, n, tag, 64)]).reshape(n, 32)


# ------------------------------------------------------------------ the P-256 primitive
@pytest.mark.parametrize("device", [False, True])
def test_random_pairs(kem, device):
    pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ec")
    rng = np.random.default_rng(200 + device)
    n = 1 << 16
    a, b = scalars(rng, n), scalars(rng, n)
    conv = cuda if device else (lambda x: x)
    pub_b, st = (host(t) for t in kem.p256_public(conv(b)))
    assert (st == 0).all()
    assert (pub_b[:4096] == ec_public_many(b[:4096])).all()
    ss, st = (host(t) for t in kem.p256_ecdh(conv(a), conv(pub_b)))
    assert (st == 0).all() and (ss == ec_ecdh_many(a, pub_b)).all()


def test_scalar_edges(kem):
    ks = [0, 1, 2, N - 1, N, 2 ** 256 - 1, N + 1, 2 ** 255]
    k = np.array([np.frombuffer(v.to_bytes(32, "big"), np.uint8) for v in ks])
    pub, st = kem.p256_public(k)
    ss, st2 = kem.p256_ecdh(k, np.tile(np.frombuffer(encode(mul(7)), np.uint8), (len(ks), 1)))
    for i, v in enumerate(ks):
        if 1 <= v < N:
            assert st[i] == 0 and st2[i] == 0
            assert bytes(pub[i]) == public(v.to_bytes(32, "big"))
            assert bytes(ss[i]) == ecdh(v.to_bytes(32, "big"), encode(mul(7)))
        else:
            assert st[i] == ERR_SCALAR and st2[i] == ERR_SCALAR and (pub[i] == 0).all() and (ss[i] == 0).all()
    assert bytes(pub[1]) == encode((GX, GY)) and int.from_bytes(bytes(pub[3][1:33]), "big") == GX


@pytest.mark.parametrize("device", [False, True])
def test_invalid_points_mixed_batch(kem, device):
    """Every kind of invalid point gives -8 and zero output; the valid items between them are unaffected."""
    rng = np.random.default_rng(33 + device)
    bad = [np.frombuffer(b, np.uint8) for _, b in invalid_points()]
    n = 4 * len(bad) + 5
    k = scalars(rng, n)
    good_pts = np.array([np.frombuffer(encode(mul(int(j) + 2)), np.uint8) for j in range(8)])
    q = good_pts[np.arange(n) % 8].copy()
    bad_rows = list(range(1, n, 4))[:len(bad)]
    for r, b in zip(bad_rows, bad):
        q[r] = b
    k[n - 1] = 0  # a bad scalar with a bad point: -7 wins
    q[n - 1] = bad[0]
    conv = cuda if device else (lambda x: x)
    ss, st = (host(t) for t in kem.p256_ecdh(conv(k), conv(q)))
    want = np.zeros(n, np.int32)
    want[bad_rows] = ERR_POINT
    want[n - 1] = ERR_SCALAR
    assert (st == want).all()
    assert (ss[want != 0] == 0).all()
    good = want == 0
    assert (ss[good] == np.array([np.frombuffer(ecdh(bytes(k[i]), bytes(q[i])), np.uint8) for i in np.nonzero(good)[0]])).all()


# ------------------------------------------------------------------ the hybrid against an independent composition
def compose_keygen(orc, d, z, sk):
    ek, dk = orc.keygen(768, d, z)
    return np.hstack([ec_public_many(sk), ek]), np.hstack([dk, sk])


def compose_encaps(orc, share, m, e):
    c, K = orc.encaps(768, share[:, PT:], m)
    return np.hstack([ec_public_many(e), c]), np.hstack([ec_ecdh_many(e, share[:, :PT]), K])


def compose_decaps(orc, secret, share):
    K = orc.decaps(768, secret[:, :2400], share[:, PT:])
    return np.hstack([ec_ecdh_many(secret[:, 2400:], share[:, :PT]), K])


@pytest.mark.parametrize("n,device,chunk,streams", [(1, False, 0, 0), (33, True, 0, 0), (1024, False, 7, 0), (1025, True, 0, 1),
                                                    (2500, False, 0, 0), (2500, True, 7, 0), (1025, False, 0, 1), (33, True, 7, 1)])
def test_hybrid_against_composition(fips_oracle, n, device, chunk, streams):
    pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ec")
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM(chunk_items=chunk)  # no FIPS flag: the hybrid runs ML-KEM in FIPS 203 mode regardless; chunk 7 -> 16
    if streams:
        kem.set_streams(streams)
    try:
        rng = np.random.default_rng(n * 7 + chunk + device)
        d, z, m = (rand(rng, n, 32) for _ in range(3))
        x, e = scalars(rng, n), scalars(rng, n)
        conv = cuda if device else (lambda a: a)
        cs, sec, st0 = (host(t) for t in kem.secp256r1mlkem768_keygen(conv(d), conv(z), conv(x)))
        wcs, wsec = compose_keygen(fips_oracle, d, z, x)
        assert (st0 == 0).all() and (cs == wcs).all() and (sec == wsec).all()
        share, ss, st = (host(t) for t in kem.secp256r1mlkem768_encaps(conv(cs), conv(m), conv(e)))
        wshare, wss = compose_encaps(fips_oracle, cs, m, e)
        assert (st == 0).all() and (share == wshare).all() and (ss == wss).all()
        ss2, st2 = (host(t) for t in kem.secp256r1mlkem768_decaps(conv(sec), conv(share)))
        assert (st2 == 0).all() and (ss2 == ss).all()
        assert (ss2 == compose_decaps(fips_oracle, sec, share)).all()
    finally:
        kem.set_streams(0)


def test_hybrid_equals_existing_calls_at_2_20(kem):
    """At 2^20 items the hybrid's outputs are the existing FIPS-mode GPU calls and the p256_* primitives, assembled in torch."""
    import crystals_kyber_b200 as ck

    fk = ck.MLKEM(fips203=True)
    rng = np.random.default_rng(2021)
    n = 1 << 20
    d, z, m = (cuda(rand(rng, n, 32)) for _ in range(3))
    x, e = cuda(scalars(rng, n)), cuda(scalars(rng, n))
    cs, sec, st0 = kem.secp256r1mlkem768_keygen(d, z, x)
    ek, dk = fk.keygen(768, d, z)
    px, _ = kem.p256_public(x)
    assert host((st0 == 0).all()) and host((cs[:, PT:] == ek).all()) and host((cs[:, :PT] == px).all())
    assert host((sec[:, :2400] == dk).all()) and host((sec[:, 2400:] == x).all())
    share, ss, st = kem.secp256r1mlkem768_encaps(cs, m, e)
    c, K = fk.encaps(768, ek, m)
    pe, _ = kem.p256_public(e)
    ee, _ = kem.p256_ecdh(e, cs[:, :PT])
    assert host((st == 0).all())
    assert host((share[:, PT:] == c).all()) and host((share[:, :PT] == pe).all())
    assert host((ss[:, 32:] == K).all()) and host((ss[:, :32] == ee).all())
    ss2, st2 = kem.secp256r1mlkem768_decaps(sec, share)
    assert host((st2 == 0).all()) and host((ss2[:, 32:] == fk.decaps(768, dk, c)).all()) and host((ss2 == ss).all())


# ------------------------------------------------------------------ interoperability with cryptography
def test_interop_cryptography_client_gpu_server(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    from cryptography.hazmat.primitives import serialization
    from cryptography.hazmat.primitives.asymmetric import ec

    enc = serialization.Encoding.X962, serialization.PublicFormat.UncompressedPoint
    rng = np.random.default_rng(19)
    n = 16
    clients, shares = [], []
    for _ in range(n):
        mk = mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(rand(rng, 1, 64)[0]))
        xk = ec.generate_private_key(ec.SECP256R1())
        clients.append((mk, xk))
        shares.append(np.frombuffer(xk.public_key().public_bytes(*enc) + mk.public_key().public_bytes_raw(), np.uint8))
    server_share, ss, st = kem.secp256r1mlkem768_encaps_seeded(np.array(shares), seed=SEED)
    assert (st == 0).all()
    for i, (mk, xk) in enumerate(clients):
        peer = ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), bytes(server_share[i, :PT]))
        want = xk.exchange(ec.ECDH(), peer) + mk.decapsulate(bytes(server_share[i, PT:]))
        assert bytes(ss[i]) == want


def test_interop_gpu_client_cryptography_server(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    from cryptography.hazmat.primitives import serialization
    from cryptography.hazmat.primitives.asymmetric import ec

    enc = serialization.Encoding.X962, serialization.PublicFormat.UncompressedPoint
    n = 16
    cs, sec = kem.secp256r1mlkem768_keygen_seeded(n, seed=SEED)
    dz = derive(SEED, n, TAG_KEYGEN, 64)
    shares, wants = [], []
    for i in range(n):
        pk = mlkem.MLKEM768PublicKey.from_public_bytes(bytes(cs[i, PT:]))
        K, c = pk.encapsulate()
        xe = ec.generate_private_key(ec.SECP256R1())
        shares.append(np.frombuffer(xe.public_key().public_bytes(*enc) + c, np.uint8))
        wants.append(xe.exchange(ec.ECDH(), ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), bytes(cs[i, :PT]))) + K)
        # cryptography's own keys from the same seeds are the GPU's
        assert mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(dz[i])).public_key().public_bytes_raw() == bytes(cs[i, PT:])
        assert ec.derive_private_key(int.from_bytes(bytes(sec[i, 2400:]), "big"), ec.SECP256R1()).public_key().public_bytes(*enc) == bytes(cs[i, :PT])
    ss, st = kem.secp256r1mlkem768_decaps(sec, np.array(shares))
    assert (st == 0).all() and [bytes(r) for r in ss] == wants


# ------------------------------------------------------------------ per-item status
@pytest.mark.parametrize("device", [False, True])
def test_status_precedence(kem, fips_oracle, device):
    pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ec")
    rng = np.random.default_rng(54 + device)
    n = 64
    d, z, m = (rand(rng, n, 32) for _ in range(3))
    x, e = scalars(rng, n), scalars(rng, n)
    conv = cuda if device else (lambda a: a)
    # keygen: an out-of-range scalar zeroes the item's share and secret
    xb = x.copy()
    xb[3] = 0
    xb[4] = np.frombuffer(N.to_bytes(32, "big"), np.uint8)
    cs_b, sec_b, stk = (host(t) for t in kem.secp256r1mlkem768_keygen(conv(d), conv(z), conv(xb)))
    want_k = np.zeros(n, np.int32)
    want_k[[3, 4]] = ERR_SCALAR
    assert (stk == want_k).all() and (cs_b[[3, 4]] == 0).all() and (sec_b[[3, 4]] == 0).all()
    cs, sec, _ = kem.secp256r1mlkem768_keygen(d, z, x)
    assert (cs_b[5:] == cs[5:]).all() and (sec_b[5:] == sec[5:]).all()
    # encaps: -7 (own scalar) before -4 (ek modulus) before -8 (peer point)
    bad = cs.copy()
    eb = e.copy()
    bad[5, PT], bad[5, PT + 1] = 0xFF, bad[5, PT + 1] | 0x0F  # coefficient 0 of item 5 = 0xFFF >= q
    bad[9, 0] = 0x02  # point prefix
    bad[10, 1:33] = 0xFF  # X >= p
    bad[11, 64] ^= 1  # off the curve
    bad[20, 0] = 0x05
    bad[20, PT], bad[20, PT + 1] = 0xFF, 0xFF  # modulus and point: -4
    eb[21] = 0  # scalar and point and modulus: -7
    bad[21, 0] = 0x00
    bad[21, PT], bad[21, PT + 1] = 0xFF, 0xFF
    eb[22] = np.frombuffer((2 ** 256 - 1).to_bytes(32, "big"), np.uint8)  # scalar only: -7
    share, ss, st = (host(t) for t in kem.secp256r1mlkem768_encaps(conv(bad), conv(m), conv(eb)))
    want = np.zeros(n, np.int32)
    want[[5, 20]] = ERR_MODULUS
    want[[9, 10, 11]] = ERR_POINT
    want[[21, 22]] = ERR_SCALAR
    assert (st == want).all()
    failed = want != 0
    assert (share[failed] == 0).all() and (ss[failed] == 0).all()
    good = ~failed
    wshare, wss = compose_encaps(fips_oracle, cs[good], m[good], e[good])
    assert (share[good] == wshare).all() and (ss[good] == wss).all()
    # decaps: -7 for a stored scalar out of range, -8 for a bad server point, a tampered ciphertext gives status 0
    share_ok, ss_ok, _ = kem.secp256r1mlkem768_encaps(cs, m, e)
    srv, secb = share_ok.copy(), sec.copy()
    srv[3, 0] = 0x03
    srv[7, 100] ^= 0x40
    secb[12, 2400:] = 0xFF
    ss2, st2 = (host(t) for t in kem.secp256r1mlkem768_decaps(conv(secb), conv(srv)))
    want2 = np.zeros(n, np.int32)
    want2[3], want2[12] = ERR_POINT, ERR_SCALAR
    assert (st2 == want2).all() and (ss2[[3, 12]] == 0).all()
    keep = want2 == 0
    assert (ss2[keep] == compose_decaps(fips_oracle, secb[keep], srv[keep])).all()
    assert (ss2[7, 32:] != ss_ok[7, 32:]).any() and (ss2[7, :32] == ss_ok[7, :32]).all()


def test_tampered_ciphertext_matches_cryptography_rejection(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    rng = np.random.default_rng(13)
    d, z, m = (rand(rng, 4, 32) for _ in range(3))
    x, e = scalars(rng, 4), scalars(rng, 4)
    cs, sec, _ = kem.secp256r1mlkem768_keygen(d, z, x)
    share, ss, _ = kem.secp256r1mlkem768_encaps(cs, m, e)
    share[:, 500] ^= 1
    ss2, st2 = kem.secp256r1mlkem768_decaps(sec, share)
    assert (st2 == 0).all()
    for i in range(4):
        sk = mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(d[i]) + bytes(z[i]))
        assert bytes(ss2[i, 32:]) == sk.decapsulate(bytes(share[i, PT:])) != bytes(ss[i, 32:])


# ------------------------------------------------------------------ seeded calls
@pytest.mark.parametrize("device", [False, True])
def test_seeded(kem, fips_oracle, device):
    pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ec")
    import crystals_kyber_b200 as ck

    n = 300
    cs, sec = (host(t) for t in kem.secp256r1mlkem768_keygen_seeded(n, seed=SEED, device=device))
    dz = derive(SEED, n, TAG_KEYGEN, 64)
    xs = derive_scalars(SEED, n, TAG_EC_KEYGEN)
    wcs, wsec = compose_keygen(fips_oracle, dz[:, :32], dz[:, 32:], xs)
    assert (cs == wcs).all() and (sec == wsec).all()
    fk = ck.MLKEM(fips203=True)
    ek, dk = fk.kem_keygen_seeded(768, n, seed=SEED)
    assert (cs[:, PT:] == ek).all() and (sec[:, :2400] == dk).all()
    share, ss, st = (host(t) for t in kem.secp256r1mlkem768_encaps_seeded(cuda(cs) if device else cs, seed=SEED))
    ms, es = derive(SEED, n, TAG_ENCAPS), derive_scalars(SEED, n, TAG_EC_ENCAPS)
    wshare, wss = compose_encaps(fips_oracle, cs, ms, es)
    assert (st == 0).all() and (share == wshare).all() and (ss == wss).all()
    rc, c, K = fk.kem_encaps_seeded(768, ek, seed=SEED)
    assert rc == 0 and (share[:, PT:] == c).all() and (ss[:, 32:] == K).all()
    # NULL seed: fresh entropy per call, every item differs
    a, _ = kem.secp256r1mlkem768_keygen_seeded(n, device=device)
    b, _ = kem.secp256r1mlkem768_keygen_seeded(n, device=device)
    assert (host(a) != host(b)).any(axis=1).all()
    s1, q1, _ = kem.secp256r1mlkem768_encaps_seeded(cuda(cs) if device else cs)
    s2, q2, _ = kem.secp256r1mlkem768_encaps_seeded(cuda(cs) if device else cs)
    assert (host(s1) != host(s2)).any(axis=1).all() and (host(q1) != host(q2)).any(axis=1).all()


def test_seeded_synchronous_with_async_flag(lib):
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    n = 5000
    cs = np.zeros((n, CS), np.uint8)
    sec = np.zeros((n, SEC), np.uint8)
    o = Opts(-1, MEM_HOST, None, 1024, 0, 2)  # MLKEM_B200_FLAG_ASYNC, pageable buffers, several chunks
    assert lib.mlkem_b200_secp256r1mlkem768_keygen_seeded_batch(n, C.c_char_p(SEED), C.c_void_p(cs.ctypes.data), C.c_void_p(sec.ctypes.data),
                                                                C.byref(o)) == OK
    xs = derive_scalars(SEED, n, TAG_EC_KEYGEN)
    assert (sec[:, 2400:] == xs).all() and (cs[:, 0] == 4).all()
    share = np.zeros((n, SS_), np.uint8)
    ss = np.zeros((n, SSEC), np.uint8)
    st = np.full(n, 99, np.int32)
    assert lib.mlkem_b200_secp256r1mlkem768_encaps_seeded_batch(n, C.c_void_p(cs.ctypes.data), C.c_char_p(SEED), C.c_void_p(share.ctypes.data),
                                                                C.c_void_p(ss.ctypes.data), C.c_void_p(st.ctypes.data), C.byref(o)) == OK
    assert (st == 0).all() and (share[:, 0] == 4).all() and (ss != 0).any(axis=1).all()


# ------------------------------------------------------------------ guard bands, sizes, errors
GUARD_SIZES = [1, 15, 16, 17, 127, 128, 129, 1024, 1025]


@pytest.fixture(scope="module")
def guarded_case(kem):
    """Inputs of the largest case and their expected outputs (the calls themselves, each pinned above, are the oracle here)."""
    rng = np.random.default_rng(78)
    n = max(GUARD_SIZES) + 1
    d, z, m = (rand(rng, n, 32) for _ in range(3))
    x, e = scalars(rng, n), scalars(rng, n)
    cs, sec, _ = kem.secp256r1mlkem768_keygen(d, z, x)
    share, ss, _ = kem.secp256r1mlkem768_encaps(cs, m, e)
    ss2, _ = kem.secp256r1mlkem768_decaps(sec, share)
    pub, _ = kem.p256_public(x)
    xss, _ = kem.p256_ecdh(x, share[:, :PT])
    return dict(d=d, z=z, x=x, m=m, e=e, cs=cs, sec=sec, share=share, ss=ss, ss2=ss2, pub=pub, xss=xss, pts=np.ascontiguousarray(share[:, :PT]))


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("n", GUARD_SIZES)
def test_guard_bands(lib, guarded_case, device, n):
    g = guarded_case
    conv = (lambda a: cuda(np.ascontiguousarray(a).reshape(-1).view(np.uint8))) if device else \
        (lambda a: np.ascontiguousarray(a).reshape(-1).view(np.uint8))
    zero4 = np.zeros(n, np.int32)
    chunk = n - 1 if n > 1 else 0  # a one-item last chunk (rounded up to a multiple of 16)
    errors = []
    cases = [
        ("mlkem_b200_p256_public_batch", lambda G: (n, G.inp(conv(g["x"][:n]), 32), G.out(conv(g["pub"][:n]), PT), G.out(conv(zero4), 4))),
        ("mlkem_b200_p256_ecdh_batch", lambda G: (n, G.inp(conv(g["x"][:n]), 32), G.inp(conv(g["pts"][:n]), PT), G.out(conv(g["xss"][:n]), 32),
                                                  G.out(conv(zero4), 4))),
        ("mlkem_b200_secp256r1mlkem768_keygen_batch", lambda G: (n, G.inp(conv(g["d"][:n]), 32), G.inp(conv(g["z"][:n]), 32),
                                                                 G.inp(conv(g["x"][:n]), 32), G.out(conv(g["cs"][:n]), CS),
                                                                 G.out(conv(g["sec"][:n]), SEC), G.out(conv(zero4), 4))),
        ("mlkem_b200_secp256r1mlkem768_encaps_batch", lambda G: (n, G.inp(conv(g["cs"][:n]), CS), G.inp(conv(g["m"][:n]), 32),
                                                                 G.inp(conv(g["e"][:n]), 32), G.out(conv(g["share"][:n]), SS_),
                                                                 G.out(conv(g["ss"][:n]), SSEC), G.out(conv(zero4), 4))),
        ("mlkem_b200_secp256r1mlkem768_decaps_batch", lambda G: (n, G.inp(conv(g["sec"][:n]), SEC), G.inp(conv(g["share"][:n]), SS_),
                                                                 G.out(conv(g["ss2"][:n]), SSEC), G.out(conv(zero4), 4))),
    ]
    for salt, (fname, make) in enumerate(cases):
        for ch in sorted({0, chunk}):
            G = Guarded(device, salt=salt * 1000 + n)
            args = make(G)
            G.seal()
            rc = call(lib, fname, args, device, chunk=ch)
            errors += [f"{fname} rc={rc}"] if rc != OK else G.check(f"{fname} n={n} chunk={ch}")
    assert not errors, errors


@pytest.mark.parametrize("device", [False, True])
def test_errors(lib, device):
    import torch

    n = 4
    mk = (lambda w, fill=0x33: torch.full((n * w + 16,), fill, dtype=torch.uint8, device="cuda")) if device else \
        (lambda w, fill=0x33: np.full(n * w + 16, fill, np.uint8))
    ptr = (lambda a, off=0: C.c_void_p(a.data_ptr() + off)) if device else (lambda a, off=0: C.c_void_p(a.ctypes.data + off))
    ins = {w: mk(w, 0x11) for w in (32, PT, CS, SEC, SS_)}
    outs = {w: mk(w) for w in (32, PT, CS, SEC, SS_, SSEC, 4)}
    snap = {w: (o.clone() if device else o.copy()) for w, o in outs.items()}

    def unchanged():
        if device:
            torch.cuda.synchronize()
        return all((o == snap[w]).all() for w, o in outs.items())

    i, o = lambda w: ptr(ins[w]), lambda w: ptr(outs[w])
    null_cases = [
        ("mlkem_b200_p256_public_batch", (n, i(32), o(PT), None)),
        ("mlkem_b200_p256_public_batch", (n, None, o(PT), o(4))),
        ("mlkem_b200_p256_ecdh_batch", (n, i(32), i(PT), o(32), None)),
        ("mlkem_b200_p256_ecdh_batch", (n, i(32), None, o(32), o(4))),
        ("mlkem_b200_secp256r1mlkem768_keygen_batch", (n, i(32), i(32), i(32), o(CS), o(SEC), None)),
        ("mlkem_b200_secp256r1mlkem768_keygen_batch", (n, i(32), i(32), None, o(CS), o(SEC), o(4))),
        ("mlkem_b200_secp256r1mlkem768_encaps_batch", (n, i(CS), i(32), i(32), o(SS_), o(SSEC), None)),
        ("mlkem_b200_secp256r1mlkem768_encaps_batch", (n, None, i(32), i(32), o(SS_), o(SSEC), o(4))),
        ("mlkem_b200_secp256r1mlkem768_decaps_batch", (n, i(SEC), i(SS_), o(SSEC), None)),
        ("mlkem_b200_secp256r1mlkem768_decaps_batch", (n, i(SEC), None, o(SSEC), o(4))),
        ("mlkem_b200_secp256r1mlkem768_keygen_seeded_batch", (n, C.c_char_p(SEED), o(CS), None)),
        ("mlkem_b200_secp256r1mlkem768_encaps_seeded_batch", (n, i(CS), C.c_char_p(SEED), o(SS_), o(SSEC), None)),
    ]
    for fname, args in null_cases:
        assert call(lib, fname, args, device) == ERR_ARG, fname
        assert unchanged(), fname
    if device:  # misaligned device pointers
        mis = [("mlkem_b200_p256_ecdh_batch", (n, i(32), ptr(ins[PT], 1), o(32), o(4))),
               ("mlkem_b200_p256_public_batch", (n, i(32), ptr(outs[PT], 8), o(4))),
               ("mlkem_b200_secp256r1mlkem768_encaps_batch", (n, ptr(ins[CS], 1), i(32), i(32), o(SS_), o(SSEC), o(4))),
               ("mlkem_b200_secp256r1mlkem768_decaps_batch", (n, i(SEC), ptr(ins[SS_], 8), o(SSEC), o(4)))]
        for fname, args in mis:
            assert call(lib, fname, args, device) == ERR_ARG, fname
            assert unchanged(), fname
    zero = [("mlkem_b200_p256_public_batch", (0, i(32), o(PT), o(4))),
            ("mlkem_b200_p256_ecdh_batch", (0, i(32), i(PT), o(32), o(4))),
            ("mlkem_b200_secp256r1mlkem768_keygen_batch", (0, i(32), i(32), i(32), o(CS), o(SEC), o(4))),
            ("mlkem_b200_secp256r1mlkem768_encaps_batch", (0, i(CS), i(32), i(32), o(SS_), o(SSEC), o(4))),
            ("mlkem_b200_secp256r1mlkem768_decaps_batch", (0, i(SEC), i(SS_), o(SSEC), o(4))),
            ("mlkem_b200_secp256r1mlkem768_keygen_seeded_batch", (0, C.c_char_p(SEED), o(CS), o(SEC))),
            ("mlkem_b200_secp256r1mlkem768_encaps_seeded_batch", (0, i(CS), C.c_char_p(SEED), o(SS_), o(SSEC), o(4)))]
    for fname, args in zero:
        assert call(lib, fname, args, device) == OK, fname
        assert unchanged(), fname
