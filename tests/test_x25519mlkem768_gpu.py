"""GPU tests of X25519 (mlkem_b200_x25519_batch) and the X25519MLKEM768 hybrid key exchange (include/mlkem_b200.h).

References that share no code with the kernels: the Python RFC 7748 ladder of test_x25519mlkem768_cpu.py (pinned there to the
RFC's vectors), `cryptography`'s X25519 and ML-KEM-768 where installed, and the oracle in FIPS 203 mode for ML-KEM.
"""
import ctypes as C
import hashlib
import struct

import numpy as np
import pytest

from test_launch_geometry_gpu import Guarded, call
from test_x25519mlkem768_cpu import (ALICE, BASE, BOB, ITER_1, ITER_1000, P, RFC_5_2, SHARED, small_order_points,
                                     x25519_ref)

pytestmark = pytest.mark.gpu

OK, ERR_ARG, ERR_MODULUS, ERR_ZERO = 0, -11, -4, -6
CS, SEC, SS_, SSEC = 1216, 2432, 1120, 64
SEED = bytes.fromhex("f00dfeed000102030405060708090a0b0c0d0e0f101112131415161718191a1b")
TAG_KEYGEN, TAG_ENCAPS, TAG_X_KEYGEN, TAG_X_ENCAPS = 1, 2, 3, 4


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


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    import torch

    if isinstance(t, torch.Tensor):
        torch.cuda.synchronize()
        return t.cpu().numpy()
    return t


def x25519_many(k, u=None):
    """X25519 row by row: cryptography where installed (all-zero results, which it refuses, via the Python ladder), else the ladder."""
    try:
        from cryptography.hazmat.primitives.asymmetric import x25519 as cx
    except ImportError:
        cx = None
    out = np.empty((len(k), 32), np.uint8)
    for i in range(len(k)):
        kb = bytes(k[i])
        ub = BASE if u is None else bytes(u[i])
        r = None
        if cx is not None:
            try:
                sk = cx.X25519PrivateKey.from_private_bytes(kb)
                r = sk.exchange(cx.X25519PublicKey.from_public_bytes(ub))
            except ValueError:
                r = None
        out[i] = np.frombuffer(r if r is not None else x25519_ref(kb, ub), np.uint8)
    return out


def derive(seed, n, tag, width=32):
    return np.frombuffer(b"".join(hashlib.shake_256(seed + struct.pack("<QQ", j, tag)).digest(width) for j in range(n)),
                         np.uint8).reshape(n, width).copy()


# ------------------------------------------------------------------ the X25519 primitive
def test_rfc7748_vectors(kem):
    k = np.array([np.frombuffer(bytes.fromhex(v[0]), np.uint8) for v in RFC_5_2] + [np.frombuffer(bytes.fromhex(ALICE[0]), np.uint8)])
    u = np.array([np.frombuffer(bytes.fromhex(v[1]), np.uint8) for v in RFC_5_2] + [np.frombuffer(bytes.fromhex(BOB[1]), np.uint8)])
    out = kem.x25519(k, u)
    assert [bytes(r).hex() for r in out] == [RFC_5_2[0][2], RFC_5_2[1][2], SHARED]
    pub = kem.x25519(np.array([np.frombuffer(bytes.fromhex(x[0]), np.uint8) for x in (ALICE, BOB)]))
    assert [bytes(r).hex() for r in pub] == [ALICE[1], BOB[1]]
    # bit 255 of u is ignored
    u2 = u[1:2].copy()
    u2[0, 31] &= 0x7F
    assert bytes(kem.x25519(k[1:2], u2)[0]).hex() == RFC_5_2[1][2]


def test_iterated_vector_single_item_calls(kem):
    k = u = np.frombuffer(BASE, np.uint8).reshape(1, 32).copy()
    for i in range(1, 1001):
        k, u = kem.x25519(k, u), k
        if i == 1:
            assert bytes(k[0]).hex() == ITER_1
    assert bytes(k[0]).hex() == ITER_1000


@pytest.mark.parametrize("device", [False, True])
def test_random_pairs(kem, device):
    rng = np.random.default_rng(100 + device)
    n = 1 << 16
    k, u = rand(rng, n, 32), rand(rng, n, 32)
    got = host(kem.x25519(cuda(k), cuda(u))) if device else kem.x25519(k, u)
    assert (got == x25519_many(k, u)).all()
    got_pub = host(kem.x25519(cuda(k[:4096]))) if device else kem.x25519(k[:4096])
    assert (got_pub == x25519_many(k[:4096])).all()


def test_edge_inputs(kem):
    rng = np.random.default_rng(3)
    us = []
    for v in (P, P + 1, P + 9, 2 ** 255 - 1, 2 ** 255 - 20, 9 + 2 ** 255, 2 ** 256 - 1):  # non-canonical and bit 255 set
        us.append(np.frombuffer((v % 2 ** 256).to_bytes(32, "little"), np.uint8))
    small = [np.frombuffer(v.to_bytes(32, "little"), np.uint8) for v in small_order_points()]
    small += [np.frombuffer((v + P).to_bytes(32, "little"), np.uint8) for v in small_order_points() if v + P < 2 ** 255]
    small += [np.frombuffer((v + 2 ** 255).to_bytes(32, "little"), np.uint8) for v in small_order_points()]  # bit 255 set
    u = np.array(us + small)
    k = rand(rng, len(u), 32)
    k[0], k[1] = 0x00, 0xFF  # scalars before clamping of all-0x00 and all-0xFF
    out = kem.x25519(k, u)
    want = np.array([np.frombuffer(x25519_ref(bytes(k[i]), bytes(u[i])), np.uint8) for i in range(len(u))])
    assert (out == want).all()
    assert (out[len(us):] == 0).all()
    k2 = np.array([[0x00] * 32, [0xFF] * 32], np.uint8)
    assert (kem.x25519(k2) == np.array([np.frombuffer(x25519_ref(bytes(r), BASE), np.uint8) for r in k2])).all()


# ------------------------------------------------------------------ the hybrid against an independent composition
def compose_keygen(orc, d, z, x):
    ek, dk = orc.keygen(768, d, z)
    return np.hstack([ek, x25519_many(x)]), np.hstack([dk, x])


def compose_encaps(orc, share, m, x):
    c, K = orc.encaps(768, share[:, :1184], m)
    xss = x25519_many(x, share[:, 1184:])
    return np.hstack([c, x25519_many(x)]), np.hstack([K, xss])


def compose_decaps(orc, secret, share):
    K = orc.decaps(768, secret[:, :2400], share[:, :1088])
    return np.hstack([K, x25519_many(secret[:, 2400:], share[:, 1088:])])


@pytest.mark.parametrize("n,device,chunk,streams", [(1, False, 0, 0), (33, True, 0, 0), (1024, False, 7, 0), (1025, True, 0, 1),
                                                    (2500, False, 0, 0), (2500, True, 7, 0), (1025, False, 0, 1), (33, True, 7, 1)])
def test_hybrid_against_composition(fips_oracle, n, device, chunk, streams):
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM(chunk_items=chunk)  # no FIPS flag: the hybrid runs ML-KEM in FIPS 203 mode regardless
    if streams:
        kem.set_streams(streams)
    try:
        rng = np.random.default_rng(n * 7 + chunk + device)
        d, z, x, m, e = (rand(rng, n, 32) for _ in range(5))
        conv = cuda if device else (lambda a: a)
        cs, sec = (host(t) for t in kem.x25519mlkem768_keygen(conv(d), conv(z), conv(x)))
        wcs, wsec = compose_keygen(fips_oracle, d, z, x)
        assert (cs == wcs).all() and (sec == wsec).all()
        share, ss, st = (host(t) for t in kem.x25519mlkem768_encaps(conv(cs), conv(m), conv(e)))
        wshare, wss = compose_encaps(fips_oracle, cs, m, e)
        assert (st == 0).all() and (share == wshare).all() and (ss == wss).all()
        ss2, st2 = (host(t) for t in kem.x25519mlkem768_decaps(conv(sec), conv(share)))
        assert (st2 == 0).all() and (ss2 == ss).all()
        assert (ss2 == compose_decaps(fips_oracle, sec, share)).all()
    finally:
        kem.set_streams(0)


def test_hybrid_equals_existing_calls_at_2_20(kem):
    """At 2^20 items the hybrid's outputs are the existing FIPS-mode GPU calls and x25519_batch, assembled in numpy."""
    import crystals_kyber_b200 as ck

    fk = ck.MLKEM(fips203=True)
    rng = np.random.default_rng(2020)
    n = 1 << 20
    d, z, x, m, e = (cuda(rand(rng, n, 32)) for _ in range(5))
    cs, sec = kem.x25519mlkem768_keygen(d, z, x)
    ek, dk = fk.keygen(768, d, z)
    assert host((cs[:, :1184] == ek).all()) and host((cs[:, 1184:] == kem.x25519(x)).all())
    assert host((sec[:, :2400] == dk).all()) and host((sec[:, 2400:] == x).all())
    share, ss, st = kem.x25519mlkem768_encaps(cs, m, e)
    c, K = fk.encaps(768, ek, m)
    assert host((st == 0).all())
    assert host((share[:, :1088] == c).all()) and host((share[:, 1088:] == kem.x25519(e)).all())
    assert host((ss[:, :32] == K).all()) and host((ss[:, 32:] == kem.x25519(e, cs[:, 1184:])).all())
    ss2, st2 = kem.x25519mlkem768_decaps(sec, share)
    assert host((st2 == 0).all()) and host((ss2[:, :32] == fk.decaps(768, dk, c)).all()) and host((ss2 == ss).all())


# ------------------------------------------------------------------ interoperability with cryptography
def test_interop_cryptography_client_gpu_server(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    from cryptography.hazmat.primitives.asymmetric import x25519 as cx

    rng = np.random.default_rng(9)
    n = 16
    clients, shares = [], []
    for _ in range(n):
        mk = mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(rand(rng, 1, 64)[0]))
        xk = cx.X25519PrivateKey.from_private_bytes(bytes(rand(rng, 1, 32)[0]))
        clients.append((mk, xk))
        shares.append(np.frombuffer(mk.public_key().public_bytes_raw() + xk.public_key().public_bytes_raw(), np.uint8))
    server_share, ss, st = kem.x25519mlkem768_encaps_seeded(np.array(shares), seed=SEED)
    assert (st == 0).all()
    for i, (mk, xk) in enumerate(clients):
        want = mk.decapsulate(bytes(server_share[i, :1088])) + xk.exchange(cx.X25519PublicKey.from_public_bytes(bytes(server_share[i, 1088:])))
        assert bytes(ss[i]) == want


def test_interop_gpu_client_cryptography_server(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    from cryptography.hazmat.primitives.asymmetric import x25519 as cx

    rng = np.random.default_rng(10)
    n = 16
    d, z, x = (rand(rng, n, 32) for _ in range(3))
    cs, sec = kem.x25519mlkem768_keygen(d, z, x)
    shares, wants = [], []
    for i in range(n):
        pk = mlkem.MLKEM768PublicKey.from_public_bytes(bytes(cs[i, :1184]))
        K, c = pk.encapsulate()
        xe = cx.X25519PrivateKey.from_private_bytes(bytes(rand(rng, 1, 32)[0]))
        shares.append(np.frombuffer(c + xe.public_key().public_bytes_raw(), np.uint8))
        wants.append(K + xe.exchange(cx.X25519PublicKey.from_public_bytes(bytes(cs[i, 1184:]))))
        # cryptography's own key from the same seed is the GPU's ek
        assert mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(d[i]) + bytes(z[i])).public_key().public_bytes_raw() == bytes(cs[i, :1184])
    ss, st = kem.x25519mlkem768_decaps(sec, np.array(shares))
    assert (st == 0).all() and [bytes(r) for r in ss] == wants


# ------------------------------------------------------------------ per-item status
@pytest.mark.parametrize("device", [False, True])
def test_status_modulus_and_small_order(kem, fips_oracle, device):
    rng = np.random.default_rng(44 + device)
    n = 64
    d, z, x, m, e = (rand(rng, n, 32) for _ in range(5))
    cs, sec = kem.x25519mlkem768_keygen(d, z, x)
    bad = cs.copy()
    bad[5, 0], bad[5, 1] = 0xFF, bad[5, 1] | 0x0F  # coefficient 0 of item 5 = 0xFFF >= q
    small = small_order_points()
    for j, i in enumerate((9, 10, 11, 12, 13)):  # X25519 keys of small order
        bad[i, 1184:] = np.frombuffer(small[j].to_bytes(32, "little"), np.uint8)
    bad[20, 1184:] = bad[9, 1184:]
    bad[20, 0], bad[20, 1] = 0xFF, 0xFF  # both checks fail: the modulus check wins
    conv = cuda if device else (lambda a: a)
    share, ss, st = (host(t) for t in kem.x25519mlkem768_encaps(conv(bad), conv(m), conv(e)))
    want_st = np.zeros(n, np.int32)
    want_st[5] = want_st[20] = ERR_MODULUS
    want_st[[9, 10, 11, 12, 13]] = ERR_ZERO
    assert (st == want_st).all()
    failed = want_st != 0
    assert (share[failed] == 0).all() and (ss[failed] == 0).all()
    good = ~failed
    wshare, wss = compose_encaps(fips_oracle, cs[good], m[good], e[good])
    assert (share[good] == wshare).all() and (ss[good] == wss).all()
    # decaps: a small-order server key gives -6; a tampered ciphertext gives status 0 and the implicit-rejection key
    share_ok, ss_ok, _ = kem.x25519mlkem768_encaps(cs, m, e)
    srv = share_ok.copy()
    srv[3, 1088:] = np.frombuffer(small[1].to_bytes(32, "little"), np.uint8)
    srv[7, 100] ^= 0x40
    ss2, st2 = (host(t) for t in kem.x25519mlkem768_decaps(conv(sec), conv(srv)))
    want2 = np.zeros(n, np.int32)
    want2[3] = ERR_ZERO
    assert (st2 == want2).all() and (ss2[3] == 0).all()
    keep = np.arange(n) != 3
    assert (ss2[keep] == compose_decaps(fips_oracle, sec[keep], srv[keep])).all()
    assert (ss2[7, :32] != ss_ok[7, :32]).any() and (ss2[7, 32:] == ss_ok[7, 32:]).all()


def test_tampered_ciphertext_matches_cryptography_rejection(kem):
    mlkem = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.mlkem")
    rng = np.random.default_rng(12)
    d, z, x, m, e = (rand(rng, 4, 32) for _ in range(5))
    cs, sec = kem.x25519mlkem768_keygen(d, z, x)
    share, ss, _ = kem.x25519mlkem768_encaps(cs, m, e)
    share[:, 500] ^= 1
    ss2, st2 = kem.x25519mlkem768_decaps(sec, share)
    assert (st2 == 0).all()
    for i in range(4):
        sk = mlkem.MLKEM768PrivateKey.from_seed_bytes(bytes(d[i]) + bytes(z[i]))
        assert bytes(ss2[i, :32]) == sk.decapsulate(bytes(share[i, :1088])) != bytes(ss[i, :32])


# ------------------------------------------------------------------ seeded calls
@pytest.mark.parametrize("device", [False, True])
def test_seeded(kem, fips_oracle, device):
    import crystals_kyber_b200 as ck

    n = 300
    cs, sec = (host(t) for t in kem.x25519mlkem768_keygen_seeded(n, seed=SEED, device=device))
    dz = derive(SEED, n, TAG_KEYGEN, 64)
    xs = derive(SEED, n, TAG_X_KEYGEN)
    wcs, wsec = compose_keygen(fips_oracle, dz[:, :32], dz[:, 32:], xs)
    assert (cs == wcs).all() and (sec == wsec).all()
    fk = ck.MLKEM(fips203=True)
    ek, dk = fk.kem_keygen_seeded(768, n, seed=SEED)
    assert (cs[:, :1184] == ek).all() and (sec[:, :2400] == dk).all()
    share, ss, st = (host(t) for t in kem.x25519mlkem768_encaps_seeded(cuda(cs) if device else cs, seed=SEED))
    ms, es = derive(SEED, n, TAG_ENCAPS), derive(SEED, n, TAG_X_ENCAPS)
    wshare, wss = compose_encaps(fips_oracle, cs, ms, es)
    assert (st == 0).all() and (share == wshare).all() and (ss == wss).all()
    rc, c, K = fk.kem_encaps_seeded(768, ek, seed=SEED)
    assert rc == 0 and (share[:, :1088] == c).all() and (ss[:, :32] == K).all()
    # NULL seed: fresh entropy per call, every item differs
    a, _ = kem.x25519mlkem768_keygen_seeded(n, device=device)
    b, _ = kem.x25519mlkem768_keygen_seeded(n, device=device)
    assert (host(a) != host(b)).any(axis=1).all()
    s1, q1, _ = kem.x25519mlkem768_encaps_seeded(cuda(cs) if device else cs)
    s2, q2, _ = kem.x25519mlkem768_encaps_seeded(cuda(cs) if device else cs)
    assert (host(s1) != host(s2)).any(axis=1).all() and (host(q1) != host(q2)).any(axis=1).all()


def test_seeded_synchronous_with_async_flag(lib):
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    n = 5000
    cs = np.zeros((n, CS), np.uint8)
    sec = np.zeros((n, SEC), np.uint8)
    o = Opts(-1, MEM_HOST, None, 1024, 0, 2)  # MLKEM_B200_FLAG_ASYNC, pageable buffers, several chunks
    assert lib.mlkem_b200_x25519mlkem768_keygen_seeded_batch(n, C.c_char_p(SEED), C.c_void_p(cs.ctypes.data), C.c_void_p(sec.ctypes.data),
                                                             C.byref(o)) == OK
    xs = derive(SEED, n, TAG_X_KEYGEN)
    assert (sec[:, 2400:] == xs).all() and (cs[:, 1184:] != 0).any(axis=1).all()


# ------------------------------------------------------------------ guard bands, sizes, errors
GUARD_SIZES = [1, 127, 128, 129, 1024, 1025]


@pytest.fixture(scope="module")
def guarded_case(kem):
    """Inputs of the largest case and their expected outputs (numpy composition of existing calls is the oracle here: the
    primitives the hybrid is built on, each pinned above)."""
    rng = np.random.default_rng(77)
    n = max(GUARD_SIZES) + 1
    d, z, x, m, e = (rand(rng, n, 32) for _ in range(5))
    cs, sec = kem.x25519mlkem768_keygen(d, z, x)
    share, ss, st = kem.x25519mlkem768_encaps(cs, m, e)
    ss2, _ = kem.x25519mlkem768_decaps(sec, share)
    pub = kem.x25519(x)
    return dict(d=d, z=z, x=x, m=m, e=e, cs=cs, sec=sec, share=share, ss=ss, ss2=ss2, pub=pub, xss=kem.x25519(x, share[:, 1088:]))


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("n", GUARD_SIZES)
def test_guard_bands(lib, guarded_case, device, n):
    import torch

    g = guarded_case
    conv = (lambda a: torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()) if device else \
        (lambda a: np.ascontiguousarray(a).reshape(-1).view(np.uint8))
    zero4 = np.zeros(n, np.int32)
    chunk = n - 1 if n > 1 else 0  # a one-item last chunk
    errors = []
    cases = [
        ("mlkem_b200_x25519_batch", lambda G: (n, G.inp(conv(g["x"][:n]), 32), None, G.out(conv(g["pub"][:n]), 32))),
        ("mlkem_b200_x25519_batch", lambda G: (n, G.inp(conv(g["x"][:n]), 32), G.inp(conv(g["share"][:n, 1088:]), 32),
                                               G.out(conv(g["xss"][:n]), 32))),
        ("mlkem_b200_x25519mlkem768_keygen_batch", lambda G: (n, G.inp(conv(g["d"][:n]), 32), G.inp(conv(g["z"][:n]), 32),
                                                              G.inp(conv(g["x"][:n]), 32), G.out(conv(g["cs"][:n]), CS),
                                                              G.out(conv(g["sec"][:n]), SEC))),
        ("mlkem_b200_x25519mlkem768_encaps_batch", lambda G: (n, G.inp(conv(g["cs"][:n]), CS), G.inp(conv(g["m"][:n]), 32),
                                                              G.inp(conv(g["e"][:n]), 32), G.out(conv(g["share"][:n]), SS_),
                                                              G.out(conv(g["ss"][:n]), SSEC), G.out(conv(zero4), 4))),
        ("mlkem_b200_x25519mlkem768_decaps_batch", lambda G: (n, G.inp(conv(g["sec"][:n]), SEC), G.inp(conv(g["share"][:n]), SS_),
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
    ins = {w: mk(w, 0x11) for w in (32, CS, SEC, SS_)}
    outs = {w: mk(w) for w in (32, CS, SEC, SS_, SSEC, 4)}
    snap = {w: (o.clone() if device else o.copy()) for w, o in outs.items()}

    def unchanged():
        if device:
            torch.cuda.synchronize()
        return all((o == snap[w]).all() for w, o in outs.items())

    i, o = lambda w: ptr(ins[w]), lambda w: ptr(outs[w])
    null_cases = [
        ("mlkem_b200_x25519_batch", (n, None, i(32), o(32))),
        ("mlkem_b200_x25519_batch", (n, i(32), i(32), None)),
        ("mlkem_b200_x25519mlkem768_keygen_batch", (n, i(32), i(32), None, o(CS), o(SEC))),
        ("mlkem_b200_x25519mlkem768_keygen_batch", (n, i(32), i(32), i(32), o(CS), None)),
        ("mlkem_b200_x25519mlkem768_encaps_batch", (n, i(CS), i(32), i(32), o(SS_), o(SSEC), None)),
        ("mlkem_b200_x25519mlkem768_encaps_batch", (n, None, i(32), i(32), o(SS_), o(SSEC), o(4))),
        ("mlkem_b200_x25519mlkem768_decaps_batch", (n, i(SEC), i(SS_), o(SSEC), None)),
        ("mlkem_b200_x25519mlkem768_decaps_batch", (n, i(SEC), None, o(SSEC), o(4))),
        ("mlkem_b200_x25519mlkem768_keygen_seeded_batch", (n, C.c_char_p(SEED), o(CS), None)),
        ("mlkem_b200_x25519mlkem768_encaps_seeded_batch", (n, i(CS), C.c_char_p(SEED), o(SS_), o(SSEC), None)),
    ]
    for fname, args in null_cases:
        assert call(lib, fname, args, device) == ERR_ARG, fname
        assert unchanged(), fname
    if device:  # misaligned device pointers
        mis = [("mlkem_b200_x25519_batch", (n, ptr(ins[32], 8), None, o(32))),
               ("mlkem_b200_x25519mlkem768_encaps_batch", (n, i(CS), i(32), i(32), o(SS_), o(SSEC), ptr(outs[4], 4))),
               ("mlkem_b200_x25519mlkem768_decaps_batch", (n, ptr(ins[SEC], 8), i(SS_), o(SSEC), o(4)))]
        for fname, args in mis:
            assert call(lib, fname, args, device) == ERR_ARG, fname
            assert unchanged(), fname
    zero = [("mlkem_b200_x25519_batch", (0, i(32), None, o(32))),
            ("mlkem_b200_x25519mlkem768_keygen_batch", (0, i(32), i(32), i(32), o(CS), o(SEC))),
            ("mlkem_b200_x25519mlkem768_encaps_batch", (0, i(CS), i(32), i(32), o(SS_), o(SSEC), o(4))),
            ("mlkem_b200_x25519mlkem768_decaps_batch", (0, i(SEC), i(SS_), o(SSEC), o(4))),
            ("mlkem_b200_x25519mlkem768_keygen_seeded_batch", (0, C.c_char_p(SEED), o(CS), o(SEC))),
            ("mlkem_b200_x25519mlkem768_encaps_seeded_batch", (0, i(CS), C.c_char_p(SEED), o(SS_), o(SSEC), o(4)))]
    for fname, args in zero:
        assert call(lib, fname, args, device) == OK, fname
        assert unchanged(), fname
