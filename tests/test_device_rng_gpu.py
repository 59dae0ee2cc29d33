"""GPU tests of the seeded calls: randomness expanded on the device from one 32-byte call seed (include/mlkem_b200.h).

Item j of a call gets R_j = SHAKE256(seed || LE64(j) || LE64(tag)) -- tag 1: (d_j, z_j) = R_j[0:32], R_j[32:64]; tag 2:
m_j = R_j[0:32] -- recomputed here with hashlib, and each seeded call must return byte for byte what the oracle and the
existing calls return with that randomness.  With seed=None the calls draw 32 bytes of host entropy per call.
"""
import ctypes as C
import hashlib
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SETS = (512, 768, 1024)
ERR_ARG = -11
TAG_KEYGEN, TAG_ENCAPS = 1, 2
SEED = bytes.fromhex("000102030405060708090a0b0c0d0e0f101112131415161718191a1b1c1d1e1f")


def derive(seed, n, tag):
    """R_j[0:64] (KeyGen: (d, z)) or R_j[0:32] (Encaps: m) for j < n."""
    width = 64 if tag == TAG_KEYGEN else 32
    out = np.frombuffer(b"".join(hashlib.shake_256(seed + struct.pack("<QQ", j, tag)).digest(width) for j in range(n)), np.uint8)
    out = out.reshape(n, width)
    return (out[:, :32].copy(), out[:, 32:].copy()) if tag == TAG_KEYGEN else out.copy()


@pytest.fixture(scope="module")
def mlkem():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


def kem(**kw):
    import crystals_kyber_b200 as ck

    return ck.MLKEM(**kw)


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    import torch

    torch.cuda.current_stream().synchronize()
    return t.cpu().numpy()


def tamper(c):
    """Item i is tampered iff i % 10 == 3: flip bit (i % 8) of byte (i * 7919) % len."""
    c = c.copy()
    n, L = c.shape
    sel = np.arange(n)[np.arange(n) % 10 == 3]
    c[sel, (sel * 7919) % L] ^= (1 << (sel % 8)).astype(np.uint8)
    return c


def seed_of(i):
    return hashlib.sha256(b"seed %d" % i).digest()


# ---------------------------------------------------------------------------------------------------------------- KeyGen
@pytest.mark.parametrize("ps", SETS)
def test_keygen_seeded_equals_oracle(mlkem, oracle, ps):
    """n = 2000 with a fixed seed: the oracle's keygen on the hashlib-derived (d_j, z_j), in host and device memory, with the
    default chunking and with chunks of 600 items (4 chunks: item j of chunk c is item 600 c + j of the call)."""
    n = 2000
    seed = seed_of(ps)
    d, z = derive(seed, n, TAG_KEYGEN)
    oek, odk = oracle.keygen(ps, d, z)
    for k in (mlkem, kem(chunk_items=600)):
        ek, dk = k.kem_keygen_seeded(ps, n, seed)
        assert (ek == oek).all() and (dk == odk).all()
        tek, tdk = k.kem_keygen_seeded(ps, n, np.frombuffer(seed, np.uint8), device=True)
        assert (host(tek) == oek).all() and (host(tdk) == odk).all()


@pytest.mark.parametrize("ps", SETS)
def test_keygen_seeded_large_equals_keygen_batch(mlkem, ps):
    """2^18 items: the GPU's keygen_batch on the same derived seeds, device memory (several chunks on the forked streams) and,
    for ML-KEM-768, host memory (4 staged chunks)."""
    import torch

    n = 1 << 18
    seed = seed_of(ps + 18)
    d, z = derive(seed, n, TAG_KEYGEN)
    ek, dk = mlkem.keygen(ps, cuda(d), cuda(z))
    sek, sdk = mlkem.kem_keygen_seeded(ps, n, seed, device=True)
    torch.cuda.synchronize()
    assert torch.equal(sek, ek) and torch.equal(sdk, dk)
    sek, sdk = kem(chunk_items=50000).kem_keygen_seeded(ps, n, seed, device=True)
    assert torch.equal(sek, ek) and torch.equal(sdk, dk)
    if ps == 768:
        hek, hdk = mlkem.kem_keygen_seeded(ps, n, seed)
        assert (hek == ek.cpu().numpy()).all() and (hdk == dk.cpu().numpy()).all()


def test_keygen_seeded_fips_equals_keygen_batch(oracle):
    """The derivation does not depend on MLKEM_B200_FLAG_FIPS203; KeyGen does: FIPS-mode results equal the FIPS oracle."""
    fk = kem(fips203=True)
    n = 700
    d, z = derive(SEED, n, TAG_KEYGEN)
    oracle.set_fips(True)
    try:
        for ps in SETS:
            oek, odk = oracle.keygen(ps, d, z)
            ek, dk = fk.kem_keygen_seeded(ps, n, SEED)
            assert (ek == oek).all() and (dk == odk).all()
    finally:
        oracle.set_fips(False)


# ---------------------------------------------------------------------------------------------------------------- Encaps
def keys_for(oracle, ps, n, salt=0):
    d, z = derive(seed_of(1000 + ps + salt), n, TAG_KEYGEN)
    return oracle.keygen(ps, d, z)


@pytest.mark.parametrize("ps", SETS)
def test_encaps_seeded_equals_oracle(mlkem, oracle, ps):
    """kem_encaps_seeded = the oracle's encaps with m_j, host and device memory, one chunk and several; decaps gives K back."""
    n = 2000
    ek, dk = keys_for(oracle, ps, n)
    seed = seed_of(ps + 2)
    m = derive(seed, n, TAG_ENCAPS)
    oc, oK = oracle.encaps(ps, ek, m)
    for k in (mlkem, kem(chunk_items=512)):
        rc, c, K = k.kem_encaps_seeded(ps, ek, seed)
        assert rc == 0 and (c == oc).all() and (K == oK).all()
        rc, tc, tK = k.kem_encaps_seeded(ps, cuda(ek), seed)
        assert rc == 0 and (host(tc) == oc).all() and (host(tK) == oK).all()
    assert (oracle.decaps(ps, dk, oc) == oK).all()


def test_encaps_seeded_checks(mlkem, oracle):
    """-3 for a bad ek_len and -1 for an unknown set; in FIPS mode an ek with a coefficient >= q gives -4 (host and device
    memory) while reference mode encapsulates it; FIPS-mode results equal the oracle in FIPS mode."""
    n = 300
    ek, _ = keys_for(oracle, 768, n)
    assert mlkem.kem_encaps_seeded(768, ek, SEED, ek_len=1183)[0] == -3
    assert mlkem.kem_encaps_seeded(768, cuda(ek), SEED, ek_len=1185)[0] == -3
    assert mlkem.kem_encaps_seeded(999, ek, SEED)[0] == -1
    bad = ek.copy()
    bad[123, 0], bad[123, 1] = 0xFF, bad[123, 1] | 0x0F  # first coefficient of item 123 = 4095 >= q
    fk = kem(fips203=True)
    assert fk.kem_encaps_seeded(768, bad, SEED)[0] == -4
    assert fk.kem_encaps_seeded(768, cuda(bad), SEED)[0] == -4
    rc, c, K = mlkem.kem_encaps_seeded(768, bad, SEED)
    m = derive(SEED, n, TAG_ENCAPS)
    oc, oK = oracle.encaps(768, bad, m)
    assert rc == 0 and (c == oc).all() and (K == oK).all()
    oracle.set_fips(True)
    try:
        for ps in SETS:
            fek, fdk = keys_for(oracle, ps, n, salt=7)
            oc, oK = oracle.encaps(ps, fek, m)
            rc, c, K = fk.kem_encaps_seeded(ps, fek, SEED)
            assert rc == 0 and (c == oc).all() and (K == oK).all()
            rc, tc, tK = fk.kem_encaps_seeded(ps, cuda(fek), SEED)
            assert rc == 0 and (host(tc) == oc).all() and (host(tK) == oK).all()
            assert (oracle.decaps(ps, fdk, oc) == oK).all()
    finally:
        oracle.set_fips(False)


# ---------------------------------------------------------------------------------------------------------------- keyed
def load(k, ps, kind, d, z, ek, dk, expand):
    if kind == "dk":
        return k.keys_load(ps, dk=dk, expand=expand)
    if kind == "seeds":
        return k.keys_load(ps, seeds=(d, z), expand=expand)
    return k.keys_load(ps, ek=ek, expand=expand)


@pytest.mark.parametrize("expand", [False, True], ids=["plain", "expanded"])
@pytest.mark.parametrize("kind", ["dk", "seeds", "ek"])
@pytest.mark.parametrize("ps", SETS)
def test_encaps_keyed_seeded(mlkem, oracle, ps, kind, expand):
    """kem_encaps_keyed = encaps_keyed_batch with m_j = the oracle's encaps on the selected ek rows, key_index NULL and explicit,
    host and device memory, one chunk and several; keyed Decaps gives K back; a host index >= n_keys is rejected."""
    nk, n = 37, 1500
    d, z = derive(seed_of(ps + 3), nk, TAG_KEYGEN)
    ek, dk = oracle.keygen(ps, d, z)
    seed = seed_of(ps + 4 + expand)
    m = derive(seed, n, TAG_ENCAPS)
    rng = np.random.default_rng(ps + len(kind) + expand)
    idx = rng.permutation(np.arange(n) % nk).astype(np.uint32)
    for k in (mlkem, kem(chunk_items=400)):
        table = load(k, ps, kind, d, z, ek, dk, expand)
        for key_index, rows in ((None, np.arange(n) % nk), (idx, idx)):
            oc, oK = oracle.encaps(ps, ek[rows], m)
            bc, bK = k.encaps_keyed(table, key_index, m)
            assert (bc == oc).all() and (bK == oK).all()
            c, K = k.kem_encaps_keyed(table, n, key_index, seed)
            assert (c == oc).all() and (K == oK).all()
            tc, tK = k.kem_encaps_keyed(table, n, None if key_index is None else cuda(key_index.astype(np.int32)), seed, device=True)
            assert (host(tc) == oc).all() and (host(tK) == oK).all()
            if kind != "ek":
                assert (k.decaps_keyed(table, key_index, c) == K).all()
                bad = tamper(c)
                assert (k.decaps_keyed(table, key_index, bad) == oracle.decaps(ps, dk[rows], bad)).all()
    P = lambda a: C.c_void_p(a.ctypes.data)
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    o = Opts(-1, MEM_HOST, None, 0, 0, 0)
    wild = idx.copy()
    wild[n // 2] = nk
    out = np.full((n, mlkem.lib.mlkem_b200_ct_bytes(ps)), 0xAB, np.uint8)
    Kout = np.full((n, 32), 0xAB, np.uint8)
    assert mlkem.lib.mlkem_b200_kem_encaps_keyed_batch(table.handle, n, P(wild), seed, P(out), P(Kout), C.byref(o)) == ERR_ARG
    assert (out == 0xAB).all() and (Kout == 0xAB).all()


# ---------------------------------------------------------------------------------------------------------------- tables
@pytest.mark.parametrize("fips", [False, True], ids=["reference", "fips203"])
@pytest.mark.parametrize("expand", [False, True], ids=["plain", "expanded"])
@pytest.mark.parametrize("ps", SETS)
def test_keys_generate_equals_oracle(oracle, ps, expand, fips):
    """keys_generate(seed): export_ek = the oracle's ek of the derived (d_j, z_j); keyed Decaps of untampered and tampered
    ciphertexts = the oracle's decaps with its dk (FIPS mode: the oracle in FIPS mode)."""
    k = kem(fips203=fips)
    nk, n = 45, 900
    seed = seed_of(ps * 4 + 2 * expand + fips)
    d, z = derive(seed, nk, TAG_KEYGEN)
    oracle.set_fips(fips)
    try:
        ek, dk = oracle.keygen(ps, d, z)
        table = k.keys_generate(ps, nk, seed, expand=expand)
        assert len(table) == nk
        assert (table.export_ek() == ek).all()
        rng = np.random.default_rng(ps + expand)
        idx = rng.permutation(np.arange(n) % nk).astype(np.uint32)
        m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        oc, oK = oracle.encaps(ps, ek[idx], m)
        c, K = k.encaps_keyed(table, idx, m)
        assert (c == oc).all() and (K == oK).all()
        bad = tamper(oc)
        assert (k.decaps_keyed(table, idx, oc) == oK).all()
        assert (k.decaps_keyed(table, idx, bad) == oracle.decaps(ps, dk[idx], bad)).all()
    finally:
        oracle.set_fips(False)


@pytest.mark.parametrize("ps", SETS)
def test_keys_replace_generate(mlkem, oracle, ps):
    """regenerate(slots, seed): the listed slots equal replace(slots, seeds=derived), slot[j] taking R_j; the other slots are
    unchanged; keyed calls on both tables agree with the oracle."""
    nk, n = 40, 800
    d, z = derive(seed_of(ps + 5), nk, TAG_KEYGEN)
    ek, dk = oracle.keygen(ps, d, z)
    for expand in (False, True):
        ta = mlkem.keys_generate(ps, nk, seed_of(ps + 5), expand=expand)
        tb = mlkem.keys_load(ps, dk=dk, expand=expand)
        slots = np.array([39, 0, 17, 5, 22], np.uint32)
        seed = seed_of(ps + 6 + expand)
        ta.regenerate(slots, seed)
        d2, z2 = derive(seed, len(slots), TAG_KEYGEN)
        tb.replace(slots, seeds=(d2, z2))
        ek2, dk2 = oracle.keygen(ps, d2, z2)
        cur_ek, cur_dk = ek.copy(), dk.copy()
        cur_ek[slots], cur_dk[slots] = ek2, dk2
        assert (ta.export_ek() == cur_ek).all() and (tb.export_ek() == cur_ek).all()
        rng = np.random.default_rng(ps)
        idx = rng.permutation(np.arange(n) % nk).astype(np.uint32)
        m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        oc, oK = oracle.encaps(ps, cur_ek[idx], m)
        bad = tamper(oc)
        want = oracle.decaps(ps, cur_dk[idx], bad)
        for t in (ta, tb):
            c, K = mlkem.encaps_keyed(t, idx, m)
            assert (c == oc).all() and (K == oK).all()
            assert (mlkem.decaps_keyed(t, idx, bad) == want).all()


def test_rejected_regenerate_leaves_the_table_untouched(mlkem, oracle):
    """A slot out of range, a slot listed twice, a NULL table or slot list, a table of ek only: MLKEM_B200_ERR_ARG and the
    table byte-identical.  n = 0 is a successful no-op."""
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    lib = mlkem.lib
    nk, n = 16, 320
    table = mlkem.keys_generate(768, nk, SEED, expand=True)
    d, z = derive(SEED, nk, TAG_KEYGEN)
    ek, dk = oracle.keygen(768, d, z)
    t_ek = mlkem.keys_load(768, ek=ek)
    rng = np.random.default_rng(3)
    idx = rng.permutation(np.arange(n) % nk).astype(np.uint32)
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    oc, oK = oracle.encaps(768, ek[idx], m)
    bad = tamper(oc)
    want = oracle.decaps(768, dk[idx], bad)

    def untouched():
        for t in (table, t_ek):
            assert (t.export_ek() == ek).all()
            c, K = mlkem.encaps_keyed(t, idx, m)
            assert (c == oc).all() and (K == oK).all()
        assert (mlkem.decaps_keyed(table, idx, bad) == want).all()

    P = lambda a: C.c_void_p(a.ctypes.data)
    o = Opts(-1, MEM_HOST, None, 0, 0, 0)
    s = seed_of(99)
    calls = {
        "slot out of range": lambda: lib.mlkem_b200_keys_replace_generate(table.handle, 2, P(np.array([3, nk], np.uint32)), s, C.byref(o)),
        "slot twice": lambda: lib.mlkem_b200_keys_replace_generate(table.handle, 2, P(np.array([5, 5], np.uint32)), s, C.byref(o)),
        "NULL table": lambda: lib.mlkem_b200_keys_replace_generate(None, 2, P(np.array([1, 2], np.uint32)), s, C.byref(o)),
        "NULL slot": lambda: lib.mlkem_b200_keys_replace_generate(table.handle, 2, None, s, C.byref(o)),
        "ek table": lambda: lib.mlkem_b200_keys_replace_generate(t_ek.handle, 2, P(np.array([1, 2], np.uint32)), s, C.byref(o)),
        "ek table, entropy": lambda: lib.mlkem_b200_keys_replace_generate(t_ek.handle, 2, P(np.array([1, 2], np.uint32)), None, C.byref(o)),
    }
    for what, call in calls.items():
        assert call() == ERR_ARG, what
    assert lib.mlkem_b200_keys_replace_generate(table.handle, 0, None, None, C.byref(o)) == 0
    untouched()


@pytest.mark.parametrize("single_stream", [False, True], ids=["forked", "one-stream"])
def test_regenerate_is_ordered_after_device_calls_in_flight(oracle, single_stream):
    """Keyed Decaps of 2^18 items under slot s enqueued on torch stream A (not waited for), then regenerate(s) on stream C, then
    keyed Decaps on stream B: the first result is the old key's, the second the new key's."""
    import torch

    k = kem(chunk_items=1 << 18) if single_stream else kem()
    nk, s, n = 8, 5, 1 << 18
    table = k.keys_generate(768, nk, SEED)
    seed = seed_of(18 + single_stream)
    d2, z2 = derive(seed, 1, TAG_KEYGEN)
    d, z = derive(SEED, nk, TAG_KEYGEN)
    d[s], z[s] = d2[0], z2[0]
    t_new = k.keys_load(768, seeds=(d, z))
    idx = cuda(np.full(n, s, np.int32))
    rng = np.random.default_rng(5)
    m = cuda(rng.integers(0, 256, (n, 32), dtype=np.uint8))
    c, K_old = k.encaps_keyed(table, idx, m)
    K_new = k.decaps_keyed(t_new, idx, c)
    torch.cuda.synchronize()
    sa, sb, sc = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        K1 = k.decaps_keyed(table, idx, c)
    with torch.cuda.stream(sc):
        table.regenerate(np.array([s], np.uint32), seed)
    with torch.cuda.stream(sb):
        K2 = k.decaps_keyed(table, idx, c)
    torch.cuda.synchronize()
    assert (K1 == K_old).all().item()
    assert (K2 == K_new).all().item() and (K2 != K_old).any().item()
    _, dk_new = oracle.keygen(768, d2, z2)
    assert (K2[:64].cpu().numpy() == oracle.decaps(768, np.repeat(dk_new, 64, axis=0), c[:64].cpu().numpy())).all()


# ---------------------------------------------------------------------------------------------------------------- seed=None
def test_entropy_calls_differ(mlkem, oracle):
    """Two calls without a seed differ in every item, in every entry point; what they return is still consistent:
    decaps(dk, c) == K."""
    n = 1000
    ek1, dk1 = mlkem.kem_keygen_seeded(768, n)
    ek2, dk2 = mlkem.kem_keygen_seeded(768, n, device=True)
    ek2, dk2 = host(ek2), host(dk2)
    assert (dk1[:, -32:] != dk2[:, -32:]).any(axis=1).all() and (ek1[:, -32:] != ek2[:, -32:]).any(axis=1).all()
    assert (oracle.keygen(768, np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8))[0] != ek1[:1]).any()
    # known keys
    ek, dk = keys_for(oracle, 768, n)
    rc1, c1, K1 = mlkem.kem_encaps_seeded(768, ek)
    rc2, c2, K2 = mlkem.kem_encaps_seeded(768, cuda(ek))
    c2, K2 = host(c2), host(K2)
    assert rc1 == 0 and rc2 == 0 and (K1 != K2).any(axis=1).all() and (c1 != c2).any(axis=1).all()
    assert (oracle.decaps(768, dk, c1) == K1).all() and (oracle.decaps(768, dk, c2) == K2).all()
    table = mlkem.keys_load(768, dk=dk[:50])
    kc1, kK1 = mlkem.kem_encaps_keyed(table, n)
    kc2, kK2 = mlkem.kem_encaps_keyed(table, n, device=True)
    kK2 = host(kK2)
    assert (kK1 != kK2).any(axis=1).all()
    assert (mlkem.decaps_keyed(table, None, kc1) == kK1).all()
    assert (oracle.decaps(768, dk[np.arange(n) % 50], kc1) == kK1).all()
    ta, tb = mlkem.keys_generate(768, 64), mlkem.keys_generate(768, 64)
    ea, eb = ta.export_ek(), tb.export_ek()
    assert (ea != eb).any(axis=1).all()
    ta.regenerate(np.arange(64, dtype=np.uint32))
    assert (ta.export_ek() != ea).any(axis=1).all()


def test_entropy_keygen_distinct_and_uniform(mlkem):
    """One call of 2^20 KeyGens without a seed: all z distinct, all rho distinct, and the 2^25 bytes of z pass a chi-square test
    of uniformity (255 degrees of freedom) at p > 1e-6."""
    from scipy.stats import chi2

    n = 1 << 20
    ek, dk = mlkem.kem_keygen_seeded(512, n, device=True)
    z = host(dk[:, -32:].contiguous())
    rho = host(ek[:, -32:].contiguous())
    del ek, dk
    for name, a in (("z", z), ("rho", rho)):
        rows = np.ascontiguousarray(a).view(np.dtype((np.void, 32))).ravel()
        assert np.unique(rows).size == n, name
    counts = np.bincount(z.ravel(), minlength=256).astype(np.float64)
    expected = z.size / 256
    stat = float(((counts - expected) ** 2 / expected).sum())
    assert chi2.sf(stat, 255) > 1e-6, stat


# ---------------------------------------------------------------------------------------------------------------- synchrony
def test_seeded_host_calls_are_synchronous_with_async_flag(mlkem, oracle):
    """With MLKEM_B200_FLAG_ASYNC set, host-memory (pinned) outputs are complete when a seeded call returns."""
    import torch

    from crystals_kyber_b200.lib import MEM_HOST, Opts

    lib = mlkem.lib
    n = 1 << 18
    o = Opts(-1, MEM_HOST, None, 0, 0, 2)  # MLKEM_B200_FLAG_ASYNC
    P = lambda t: C.c_void_p(t.data_ptr())
    pinned = lambda shape: torch.full(shape, 0xAB, dtype=torch.uint8).pin_memory()
    ek, dk = pinned((n, 1184)), pinned((n, 2400))
    assert lib.mlkem_b200_kem_keygen_seeded_batch(768, n, SEED, P(ek), P(dk), C.byref(o)) == 0
    got_ek, got_dk = ek.numpy().copy(), dk.numpy().copy()
    want_ek, want_dk = mlkem.kem_keygen_seeded(768, n, SEED)
    assert (got_ek == want_ek).all() and (got_dk == want_dk).all()
    c, K = pinned((n, 1088)), pinned((n, 32))
    src = torch.from_numpy(want_ek).pin_memory()
    assert lib.mlkem_b200_kem_encaps_seeded_batch(768, n, P(src), 1184, SEED, P(c), P(K), C.byref(o)) == 0
    got_c, got_K = c.numpy().copy(), K.numpy().copy()
    wc, wK = mlkem.encaps(768, want_ek, derive(SEED, n, TAG_ENCAPS))
    assert (got_c == wc).all() and (got_K == wK).all()
    table = mlkem.keys_load(768, dk=want_dk[:100])
    c.fill_(0xAB)
    K.fill_(0xAB)
    assert lib.mlkem_b200_kem_encaps_keyed_batch(table.handle, n, None, SEED, P(c), P(K), C.byref(o)) == 0
    got_c, got_K = c.numpy().copy(), K.numpy().copy()
    assert (mlkem.decaps_keyed(table, None, got_c) == got_K).all()
    assert (got_K == mlkem.kem_encaps_keyed(table, n, seed=SEED)[1]).all()
