"""Implicit rejection at every ciphertext bit, SampleNTT's block boundaries and extreme input bytes, on every Decaps path.

Decaps returns the real shared key only when re-encrypting m' reproduces the received ciphertext bit for bit, and the
rejection key J(z || c) otherwise (ml_kem.c:1206-1221).  The compare and the select exist in several places:
- the u rows in matvec_row_tail: the fused k_sample_matvec, the general k_sample_matvec_list (deferred rows, batches of
  at most 32 rows, lowered group limits) and k_matvec_table (expanded key tables);
- v in k_encrypt_v<P, true>;
- the select in k_decaps_J_select (chunks of more than 1024 items) and k_decaps_J_select_warp, each with SHAKE128 and with
  the FIPS 203 SHAKE256.
The tests below flip every bit of a ciphertext and run the batch through each of those paths, checking the path itself in
the library's per-kernel profile.

The fused kernel samples exactly three SHAKE128 blocks (168 three-byte groups, 336 candidates) per matrix entry, so an entry
completes there iff its 256th accepted candidate, at 1-based index T, has T <= 336; other rows are deferred to the general
kernel.  With a lowered group limit L the reference gives up and restarts an entry whose group ceil(T / 2) exceeds L
(ml_kem.c:221-242).  The key search below finds keys whose entries sit on each side of those edges, so that the suite tests
them on purpose instead of by chance.  The search needs no GPU; every test that does is marked `gpu`.
"""
import contextlib
import hashlib

import numpy as np
import pytest

from oracle.oracle import sizes

SETS = (512, 768, 1024)
Q = 3329
SEARCH_BLOCK = 1024     # keys per step of the edge-key search
SEARCH_LIMIT = 1 << 14  # a class not found among this many keys fails the search


@pytest.fixture(scope="module")
def mlkem():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


@contextlib.contextmanager
def oracle_mode(oracle, fips=False, limit=0):
    """The oracle in FIPS 203 mode and / or with a lowered SampleNTT group limit; both global hooks are reset on the way out."""
    try:
        oracle.set_fips(fips)
        oracle.set_sample_group_limit(limit)
        yield
    finally:
        oracle.set_fips(False)
        oracle.set_sample_group_limit(0)


# ------------------------------------------------------------------ 1. SampleNTT edges, found on the CPU
def _candidates(seeds34):
    """d1, d2, d1, d2, ... of the first five SHAKE128 blocks of each 34-byte seed (ml_kem.c:201-216): shape (n, 560)."""
    seeds = np.ascontiguousarray(seeds34, np.uint8).reshape(-1, 34)
    xof = b"".join(hashlib.shake_128(s.tobytes()).digest(5 * 168) for s in seeds)
    g = np.frombuffer(xof, np.uint8).reshape(len(seeds), 280, 3).astype(np.uint16)
    d1 = g[..., 0] | (g[..., 1] & 15) << 8
    d2 = g[..., 1] >> 4 | g[..., 2] << 4
    return np.stack([d1, d2], -1).reshape(len(seeds), 560)


def completion_indices(seeds34):
    """T of each seed: the 1-based index of its 256th candidate < q (0 if five blocks do not hold 256)."""
    accepted = np.cumsum(_candidates(seeds34) < Q, axis=1)
    return np.where(accepted[:, -1] >= 256, (accepted >= 256).argmax(axis=1) + 1, 0)


def completion_index(seed34):
    return int(completion_indices(np.frombuffer(bytes(seed34), np.uint8))[0])


def parse_ntt(seeds34):
    """SampleNTT without a group limit: the first 256 candidates < q of each seed."""
    return np.stack([c[c < Q][:256] for c in _candidates(seeds34)]).astype(np.uint16)


def matrix_seeds(rho, k):
    """The seeds rho || j || i of A[i][j] (ml_kem.c:686-693, oracle/mlkem_oracle.c:475-478), k * k per key in (i, j) order."""
    rho = np.ascontiguousarray(rho, np.uint8).reshape(-1, 32)
    ji = np.array([(j, i) for i in range(k) for j in range(k)], np.uint8)
    return np.concatenate([np.repeat(rho, k * k, 0), np.tile(ji, (len(rho), 1))], 1)


def key_seeds(counters):
    """KeyGen_internal inputs of the search: d = LE64(counter) || 0^24, z = SHA3-256(d)."""
    c = np.asarray(counters, np.uint64).reshape(-1)
    d = np.zeros((c.size, 32), np.uint8)
    d[:, :8] = c.astype("<u8").view(np.uint8).reshape(-1, 8)
    z = np.frombuffer(b"".join(hashlib.sha3_256(r.tobytes()).digest() for r in d), np.uint8).reshape(-1, 32)
    return d, z


def group(T):
    return (T + 1) // 2


# class -> which keys have it, from T of shape (keys, k, k).  Candidate 2g - 1 is d1 of group g, 2g is its d2.
CLASSES = {
    "T335": lambda T: (T == 335).any((1, 2)) & (T.max((1, 2)) <= 336),  # d1 of group 168 completes: its d2 must be dropped
    "T336": lambda T: (T == 336).any((1, 2)) & (T.max((1, 2)) <= 336),  # the last candidate of block 3, all rows fused
    "T337": lambda T: (T == 337).any((1, 2)),  # the first group of block 4: the row is deferred
    "T338": lambda T: (T == 338).any((1, 2)),
    "group170": lambda T: (group(T) == 170).any((1, 2)),  # the last group a run may consume under limit 170
    "group171": lambda T: (group(T) == 171).any((1, 2)),  # the first one it may not: restart
    "fast": lambda T: T.max((1, 2)) <= 336,  # every entry complete in the fused kernel
}
_found = {}


def find_keys(oracle, ps, fips):
    """Walk the counters 0, 1, 2, ... in steps of SEARCH_BLOCK until each class of CLASSES has a key.  rho is read from the
    ek the oracle computes in the mode under test.  Returns {class: counter} -- the first key of each class, a "fast" key
    that is none of the others, and the keys with the largest and the smallest T of the walked range -- and T of every
    walked key."""
    if (ps, fips) in _found:
        return _found[(ps, fips)]
    k = sizes(ps)["k"]
    Ts = []
    with oracle_mode(oracle, fips=fips):
        for start in range(0, SEARCH_LIMIT, SEARCH_BLOCK):
            d, z = key_seeds(np.arange(start, start + SEARCH_BLOCK))
            ek, _ = oracle.keygen(ps, d, z)
            Ts.append(completion_indices(matrix_seeds(ek[:, -32:], k)).reshape(-1, k, k))
            T = np.concatenate(Ts)
            hits = {name: np.nonzero(pred(T))[0] for name, pred in CLASSES.items()}
            if all(h.size for h in hits.values()) and hits["fast"].size > len(CLASSES):
                break
        else:
            missing = sorted(name for name, h in hits.items() if not h.size)
            pytest.fail(f"ML-KEM-{ps} (fips={fips}): no key of class {missing} among the first {SEARCH_LIMIT} counters")
    assert (T > 0).all()
    keys = {name: int(h[0]) for name, h in hits.items() if name != "fast"}
    keys["fast"] = int(next(i for i in hits["fast"] if i not in keys.values()))
    keys["max"] = int(T.max((1, 2)).argmax())
    keys["min"] = int(T.min((1, 2)).argmin())
    _found[(ps, fips)] = keys, T
    return keys, T


@pytest.mark.parametrize("ps", SETS)
def test_edge_key_search(oracle, ps):
    """The parser behind T equals the oracle's SampleNTT; the search finds every class well within its bound; and the
    oracle's give-up rule under a lowered limit L is exactly 'restart iff group ceil(T / 2) > L'."""
    k = sizes(ps)["k"]
    rng = np.random.default_rng(ps)
    seeds = rng.integers(0, 256, (200, 34), dtype=np.uint8)
    assert (parse_ntt(seeds) == oracle.sample_ntt(seeds)).all()
    assert [completion_index(s) for s in seeds[:5]] == list(completion_indices(seeds[:5]))
    for fips in (False, True):
        keys, T = find_keys(oracle, ps, fips)
        assert set(keys) == set(CLASSES) | {"max", "min"}
        assert len({keys["T336"], keys["T337"], keys["fast"]}) == 3
        for name, pred in CLASSES.items():
            assert pred(T[keys[name]][None])[0], name
        assert T[keys["max"]].max() == T.max() > 342 and T[keys["min"]].min() == T.min() < 300
        counters = sorted(set(keys.values()))
        with oracle_mode(oracle, fips=fips):
            ek, _ = oracle.keygen(ps, *key_seeds(counters))
        edge = matrix_seeds(ek[:, -32:], k)
        assert (completion_indices(edge).reshape(-1, k, k) == T[counters]).all()
        assert (parse_ntt(edge) == oracle.sample_ntt(edge)).all()
        Te = completion_indices(edge)
        for limit in (168, 170):
            with oracle_mode(oracle, limit=limit):
                _, after = oracle.sample_ntt_with_seeds(edge)
            assert ((after != edge).any(1) == (group(Te) > limit)).all(), limit


# ------------------------------------------------------------------ 2. every single-bit flip, every Decaps path
def single_bit_flips(c):
    """For each row of c and each bit p in [0, 8 L): c with bit p flipped, then c untouched.  Returns the batch, the row
    (key) of each item and its flipped bit (-1: untouched)."""
    nk, L = c.shape
    p = np.arange(8 * L)
    batch = np.broadcast_to(c[:, None, None, :], (nk, 8 * L, 2, L)).copy()
    batch[:, p, 0, p // 8] ^= (1 << (p % 8)).astype(np.uint8)
    bit = np.tile(np.stack([p, np.full_like(p, -1)], 1).ravel(), nk)
    return batch.reshape(-1, L), np.repeat(np.arange(nk), 16 * L), bit


def host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def mismatch(got, want, key_of, bit, what):
    """None if got == want, else which items differ, by key and flipped bit."""
    bad = np.nonzero((host(got) != want).any(1))[0]
    if bad.size:
        first = [(int(key_of[i]), int(bit[i])) for i in bad[:8]]
        return f"{what}: {bad.size} of {len(want)} items differ; first (key, flipped bit or -1): {first}"
    return None


def profiled(kem, call):
    """Runs call() with the per-kernel profile on; returns its result and the names of the kernels it launched, as the
    LAUNCH macro spells them (for instance 'k_decaps_J_select<P, kRateSha3_256>')."""
    kem.profile(True)
    try:
        out = call()
    finally:
        kem.profile(False)
    return out, {name.strip("()") for name in kem.profile_report()}


def bases(names):
    """Kernel names without template arguments: 'k_sample_matvec' and 'k_sample_matvec_list' stay apart."""
    return {n.split("<")[0] for n in names}


MODES = {"reference": dict(fips=False, limit=0), "fips203": dict(fips=True, limit=0), "limit168": dict(fips=False, limit=168)}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("ps", SETS)
def test_every_single_bit_flip_is_rejected(mlkem, oracle, ps, mode):
    """Three keys -- one with a T = 336 entry, one with a T = 337 entry (its rows are compared in the general kernel, and
    under limit 168 they restart there), one with every T <= 336 -- and one valid c each.  The batch holds, per key, c with
    each of its 8 L bits flipped, each followed by the untouched c.  Every path must return the K of Encaps for each untouched
    item and J(z || c') -- SHAKE128, or SHAKE256 in FIPS 203 mode -- for each flipped one, which is never K.  Every path is
    run and checked before the test fails, so that a failure names each path that accepts a modified ciphertext."""
    import torch

    import crystals_kyber_b200 as ck

    fips, limit = MODES[mode]["fips"], MODES[mode]["limit"]
    keys, _ = find_keys(oracle, ps, fips)
    d, z = key_seeds([keys["T336"], keys["T337"], keys["fast"]])
    m = np.random.default_rng(ps).integers(0, 256, (3, 32), dtype=np.uint8)
    with oracle_mode(oracle, fips=fips, limit=limit):
        ek, dk = oracle.keygen(ps, d, z)
        c, K = oracle.encaps(ps, ek, m)
        batch, key_of, bit = single_bit_flips(c)
        per_key = len(batch) // 3
        want_oracle = np.concatenate([oracle.decaps(ps, np.repeat(dk[i:i + 1], per_key, 0), batch[i * per_key:(i + 1) * per_key])
                                      for i in range(3)])
    J = hashlib.shake_256 if fips else hashlib.shake_128
    want = K[key_of]
    flipped = np.nonzero(bit >= 0)[0]
    want[flipped] = np.frombuffer(b"".join(J(z[key_of[i]].tobytes() + batch[i].tobytes()).digest(32) for i in flipped),
                                  np.uint8).reshape(-1, 32)
    assert (want[flipped] != K[key_of[flipped]]).any(1).all()
    assert mismatch(want_oracle, want, key_of, bit, "oracle") is None
    if limit:
        with oracle_mode(oracle, fips=fips):
            ek_278, _ = oracle.keygen(ps, d, z)
        assert (ek_278[1] != ek[1]).any() and (ek_278[[0, 2]] == ek[[0, 2]]).all(), "the T = 337 key must restart under limit 168"

    wrong = []
    check = lambda got, what, sel=slice(None): wrong.append(mismatch(got, want[sel], key_of[sel], bit[sel], what))
    dk_of = dk[key_of]
    edge = key_of < 2  # the two edge keys' items
    kem = ck.MLKEM(fips203=fips, sample_group_limit=limit)
    small = ck.MLKEM(chunk_items=1000, fips203=fips, sample_group_limit=limit)
    tiny = ck.MLKEM(chunk_items=8, fips203=fips, sample_group_limit=limit)
    J_thread = "k_decaps_J_select<P, kRateSha3_256>" if fips else "k_decaps_J_select<P>"
    J_warp = "k_decaps_J_select_warp<P, kRateSha3_256>" if fips else "k_decaps_J_select_warp<P>"

    Kd, names = profiled(kem, lambda: kem.decaps(ps, dk_of, batch))
    check(Kd, "host memory")
    assert {"k_sample_matvec", "k_sample_matvec_list", "k_encrypt_v"} <= bases(names) and J_thread in names, names
    assert "k_decaps_J_select_warp" not in bases(names), names
    if mode != "limit168":
        Kd, names = profiled(small, lambda: small.decaps(ps, dk_of, batch))
        check(Kd, "chunks of 1000 items")
        assert "k_sample_matvec" in bases(names) and J_warp in names and "k_decaps_J_select" not in bases(names), names
    if mode != "fips203":
        Kd, names = profiled(tiny, lambda: tiny.decaps(ps, dk_of[edge], batch[edge]))
        check(Kd, "chunks of 8 items", edge)
        assert "k_sample_matvec_list" in bases(names) and "k_sample_matvec" not in bases(names), names
    if fips:
        table = kem.keys_load(ps, dk=dk, expand=True)
        Kd, names = profiled(kem, lambda: kem.decaps_keyed(table, key_of, batch))
        check(Kd, "expanded key table")
        assert "k_matvec_table" in bases(names) and not bases(names) & {"k_sample_matvec", "k_sample_matvec_list"}, names
        table.free()
    if mode == "reference":
        tdk, tbatch, tkey = (torch.from_numpy(a).cuda() for a in (dk_of, batch, key_of.astype(np.int32)))
        Kd, names = profiled(kem, lambda: kem.decaps(ps, tdk, tbatch))
        check(Kd, "device memory")
        assert "k_sample_matvec" in bases(names) and J_thread in names, names
        del tdk
        for expand in (False, True):
            table = kem.keys_load(ps, dk=dk, expand=expand)
            Kd, names = profiled(kem, lambda: kem.decaps_keyed(table, key_of, batch))
            check(Kd, f"key table (expand={expand}), host memory")
            assert ("k_matvec_table" in bases(names)) == expand and ("k_sample_matvec" in bases(names)) != expand, names
            check(kem.decaps_keyed(table, tkey, tbatch), f"key table (expand={expand}), device memory")
            table.free()
        one = key_of == 1  # the T = 337 key: the public wrapper and the reference's cell layout
        rc, Kd, status = kem.kem_decaps(ps, dk[1:2].repeat(one.sum(), 0), batch[one])
        assert rc == 0 and (status == 0).all()
        check(Kd, "kem_decaps", one)
        check(kem.decaps_cells(ps, dk[1:2].repeat(one.sum(), 0).astype(np.uint32), batch[one].astype(np.uint32)), "decaps_cells", one)
    wrong = [w for w in wrong if w]
    assert not wrong, "\n".join(wrong)


# ------------------------------------------------------------------ 3. SampleNTT boundary corpus through the whole KEM
def tamper(c):
    """The benchmark's rule: item i is tampered iff i % 10 == 3, by flipping bit (i % 8) of byte (i * 7919) % len."""
    c = c.copy()
    n, L = c.shape
    idx = np.arange(n)
    sel = idx[idx % 10 == 3]
    c[sel, (sel * 7919) % L] ^= (1 << (sel % 8)).astype(np.uint8)
    return c, sel


@pytest.mark.gpu
@pytest.mark.parametrize("ps", SETS)
def test_sample_ntt_boundary_corpus(mlkem, oracle, ps):
    """Every edge key of the search, each at 37 consecutive item positions (every row offset within the fused kernel's
    32-row blocks), padded with random keys to 2500 items, and each edge key as a batch of one: KeyGen, Encaps, Decaps,
    key tables from seeds with expanded matrices, and SampleNTT with its post-restart seeds, bit-exact against the oracle
    at group limits 278 (the reference's), 168 and 170 on both sides."""
    import crystals_kyber_b200 as ck

    k, n, reps = sizes(ps)["k"], 2500, 37
    keys, _ = find_keys(oracle, ps, False)
    edge = sorted(set(keys.values()))
    rng = np.random.default_rng(ps + 2026)
    de, ze = key_seeds(edge)
    d = np.concatenate([np.repeat(de, reps, 0), rng.integers(0, 256, (n - reps * len(edge), 32), dtype=np.uint8)])
    z = np.concatenate([np.repeat(ze, reps, 0), rng.integers(0, 256, (n - reps * len(edge), 32), dtype=np.uint8)])
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    for limit in (0, 168, 170):
        with oracle_mode(oracle, limit=limit):
            oek, odk = oracle.keygen(ps, d, z)
            oc, oK = oracle.encaps(ps, oek, m)
            bad, sel = tamper(oc)
            oKd = oracle.decaps(ps, odk, bad)
            seeds = matrix_seeds(oek[:, -32:], k)
            oa, oafter = oracle.sample_ntt_with_seeds(seeds)
        # the corpus must hold each edge that applies under this limit, or the test would pass without testing it
        T, restarted = completion_indices(seeds), (oafter != seeds).any(1)
        assert (restarted == (group(T) > (limit or 278))).all()
        if limit == 0:
            assert {335, 336, 337, 338} <= set(T.tolist()) and not restarted.any()
        elif limit == 168:
            assert {336, 337} <= set(T.tolist())
        else:
            assert {170, 171} <= set(group(T).tolist())
        assert (np.delete(oKd, sel, 0) == np.delete(oK, sel, 0)).all() and (oKd[sel] != oK[sel]).any(1).all()

        gpu = ck.MLKEM(sample_group_limit=limit)
        ek, dk = gpu.keygen(ps, d, z)
        assert (ek == oek).all() and (dk == odk).all(), limit
        c, K = gpu.encaps(ps, oek, m)
        assert (c == oc).all() and (K == oK).all(), limit
        assert (gpu.decaps(ps, odk, bad) == oKd).all(), limit
        table = gpu.keys_load(ps, seeds=(d, z), expand=True)
        c, K = gpu.encaps_keyed(table, None, m)
        assert (c == oc).all() and (K == oK).all(), limit
        assert (gpu.decaps_keyed(table, None, bad) == oKd).all(), limit
        table.free()
        a, after = gpu.sample_ntt(seeds, return_seeds=True)
        assert (a == oa).all() and (after == oafter).all(), limit
        for e in range(len(edge)):
            i = slice(reps * e, reps * e + 1)
            ek, dk = gpu.keygen(ps, d[i], z[i])
            assert (ek == oek[i]).all() and (dk == odk[i]).all(), (limit, edge[e])
            c, K = gpu.encaps(ps, oek[i], m[i])
            assert (c == oc[i]).all() and (K == oK[i]).all(), (limit, edge[e])
            assert (gpu.decaps(ps, odk[i], oc[i]) == oK[i]).all(), (limit, edge[e])
            flip = oc[i].copy()
            flip[0, -1] ^= 0x80
            assert gpu.decaps(ps, odk[i], flip)[0].tobytes() == hashlib.shake_128(z[i].tobytes() + flip.tobytes()).digest(32)


# ------------------------------------------------------------------ 4. extreme bytes
@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 1000, 8])
@pytest.mark.parametrize("ps", SETS)
def test_extreme_bytes(mlkem, oracle, ps, chunk):
    """ek, dk and c of all 0x00 and all 0xFF bytes among valid ones.  An all-0xFF ek decodes to t^ = 4095 with rho = 0xFF...
    (ByteDecode12 does not reduce, D4); an all-0xFF dk gives s^ = 4095, the largest operands basemul_acc's lazy sums in
    k_decrypt see.  Encaps, Decaps, PKE_Decrypt and the keyed calls on tables of those keys (plain and expanded), from host
    and device memory, all equal the oracle.  Both extreme dk fail the hash check (-5) and are loaded all the same."""
    import torch

    import crystals_kyber_b200 as ck

    sz, n = sizes(ps), 1100  # more than 1024 items: the default options take the thread form of the hashes
    rng = np.random.default_rng(ps * 10 + chunk)
    d, z = (rng.integers(0, 256, (6, 32), dtype=np.uint8) for _ in range(2))
    ek_v, dk_v = oracle.keygen(ps, d, z)
    pool_ek = np.concatenate([np.zeros((1, sz["ek"]), np.uint8), np.full((1, sz["ek"]), 0xFF, np.uint8), ek_v])
    pool_dk = np.concatenate([np.zeros((1, sz["dk"]), np.uint8), np.full((1, sz["dk"]), 0xFF, np.uint8), dk_v])
    idx = (np.arange(n) % len(pool_ek)).astype(np.uint32)
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    k = sz["k"]
    ek_in_dk = pool_dk[:, 384 * k: 768 * k + 32]
    c = oracle.encaps(ps, ek_in_dk[idx], m)[0]  # valid for the item's own key, then every third c all 0x00, every third all 0xFF
    c[1::3], c[2::3] = 0x00, 0xFF
    oc, oK = oracle.encaps(ps, pool_ek[idx], m)
    oKd = oracle.decaps(ps, pool_dk[idx], c)
    om = oracle.pke_decrypt(ps, pool_dk[idx], c, dk_stride=sz["dk"])
    status_want = [0 if hashlib.sha3_256(e.tobytes()).digest() == h.tobytes() else -5 for e, h in zip(ek_in_dk, pool_dk[:, -64:-32])]
    assert status_want == [-5, -5] + [0] * len(dk_v)

    gpu = ck.MLKEM(chunk_items=chunk)
    for dev in (False, True):
        up = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if dev else (lambda a: a)
        where = "device" if dev else "host"
        c_, K_ = gpu.encaps(ps, up(pool_ek[idx]), up(m))
        assert (host(c_) == oc).all() and (host(K_) == oK).all(), where
        assert (host(gpu.decaps(ps, up(pool_dk[idx]), up(c))) == oKd).all(), where
        assert (host(gpu.pke_decrypt(ps, up(pool_dk[idx]), up(c), dk_stride=sz["dk"])) == om).all(), where
        kidx = up(idx.astype(np.int32)) if dev else idx
        for expand in (False, True):
            table = gpu.keys_load(ps, ek=up(pool_ek), expand=expand)
            c_, K_ = gpu.encaps_keyed(table, kidx, up(m))
            assert (host(c_) == oc).all() and (host(K_) == oK).all(), (where, expand)
            table.free()
            table, status = gpu.keys_load(ps, dk=up(pool_dk), return_status=True, expand=expand)
            assert list(status) == status_want, (where, expand)
            assert (host(gpu.decaps_keyed(table, kidx, up(c))) == oKd).all(), (where, expand)
            table.free()
