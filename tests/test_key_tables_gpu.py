"""GPU tests of key rotation on resident key tables: mlkem_b200_keys_replace / _replace_ek / _replace_from_seeds and
mlkem_b200_keys_export_ek.

After a replace, keyed Encaps / Decaps must return exactly what the unkeyed calls return on the expected key list (new keys
in the replaced slots, old keys elsewhere), checked against the oracle; a rejected call must leave the table byte for byte as
it was; and a replace must be ordered after keyed calls already in flight on other streams.  All comparisons are bit-exact.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SETS = (512, 768, 1024)
ERR_ARG = -11


@pytest.fixture(scope="module")
def mlkem():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


def tamper(c):
    """Item i is tampered iff i % 10 == 3 (10 %): flip bit (i % 8) of byte (i * 7919) % len."""
    c = c.copy()
    n, L = c.shape
    sel = np.arange(n)[np.arange(n) % 10 == 3]
    c[sel, (sel * 7919) % L] ^= (1 << (sel % 8)).astype(np.uint8)
    return c, sel


def seeds(rng, n):
    return rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (n, 32), dtype=np.uint8)


def every_slot(rng, nk, n):
    """n key indices that cover every slot of a table of nk keys, shuffled."""
    return rng.permutation(np.arange(n) % nk).astype(np.uint32)


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def load(kem, ps, kind, d, z, ek, dk, expand, device=None):
    if kind == "dk":
        return kem.keys_load(ps, dk=dk, expand=expand, device=device)
    if kind == "seeds":
        return kem.keys_load(ps, seeds=(d, z), expand=expand, device=device)
    return kem.keys_load(ps, ek=ek, expand=expand, device=device)


def replace(table, kind, slots, d, z, ek, dk, on_device):
    up = cuda if on_device else (lambda a: np.ascontiguousarray(a))
    if kind == "dk":
        table.replace(slots, dk=up(dk[slots]))
    elif kind == "seeds":
        table.replace(slots, seeds=(up(d[slots]), up(z[slots])))
    else:
        table.replace(slots, ek=up(ek[slots]))


@pytest.mark.parametrize("expand", [False, True], ids=["plain", "expanded"])
@pytest.mark.parametrize("kind", ["dk", "seeds", "ek"])
@pytest.mark.parametrize("ps", SETS)
def test_replace_equals_unkeyed(mlkem, oracle, ps, kind, expand):
    """Scattered, unsorted slots (the first, the last, middle ones) replaced from host and then from device memory; keyed calls
    over every slot equal the oracle and the unkeyed calls on the expected key list, and rejection uses the new z."""
    rng = np.random.default_rng(ps * 10 + len(kind) + expand)
    nk, n = 41, 820
    d, z = seeds(rng, nk)
    ek, dk = oracle.keygen(ps, d, z)
    table = load(mlkem, ps, kind, d, z, ek, dk, expand)
    d2, z2 = seeds(rng, nk)
    ek2, dk2 = oracle.keygen(ps, d2, z2)
    cur_ek, cur_dk = ek.copy(), dk.copy()
    host_slots = np.array([nk - 1, 0, 17, 5], np.uint32)
    dev_slots = np.array([23, 8, 30, 2, 39], np.uint32)
    for slots, on_device in ((host_slots, False), (dev_slots, True)):
        replace(table, kind, slots, d2, z2, ek2, dk2, on_device)
        cur_ek[slots], cur_dk[slots] = ek2[slots], dk2[slots]
    replaced = np.concatenate([host_slots, dev_slots])
    assert (table.export_ek() == cur_ek).all()

    idx = every_slot(rng, nk, n)
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    c, K = mlkem.encaps(ps, cur_ek[idx], m)
    oc, oK = oracle.encaps(ps, cur_ek[idx], m)
    assert (c == oc).all() and (K == oK).all()
    kc, kK = mlkem.encaps_keyed(table, idx, m)
    assert (kc == c).all() and (kK == K).all()
    if kind == "ek":
        return
    bad, sel = tamper(c)
    Kd = mlkem.decaps(ps, cur_dk[idx], bad)
    assert (Kd == oracle.decaps(ps, cur_dk[idx], bad)).all()
    assert (mlkem.decaps_keyed(table, idx, bad) == Kd).all()
    assert (mlkem.decaps_keyed(table, cuda(idx.astype(np.int32)), cuda(bad)).cpu().numpy() == Kd).all()
    # implicit rejection (J(z || c)) under a replaced slot uses the NEW z: the new key with the old z gives other keys
    rej = sel[np.isin(idx[sel], replaced)]
    assert rej.size > 0
    old_z = cur_dk[idx[rej]].copy()
    old_z[:, -32:] = dk[idx[rej], -32:]
    assert (oracle.decaps(ps, old_z, bad[rej]) != Kd[rej]).any(axis=1).all()


@pytest.mark.parametrize("fips", [False, True], ids=["reference", "fips203"])
def test_replace_from_seeds_equals_replace_from_dk(mlkem, oracle, fips):
    """_replace_from_seeds(d, z) and _replace(KeyGen_internal(d, z).dk) leave identical tables: the same export_ek and the same
    keyed outputs, equal to the unkeyed calls of the same mode (FIPS mode: the unkeyed FIPS calls)."""
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM(fips203=fips)
    rng = np.random.default_rng(1034 + fips)
    nk, n = 33, 660
    for ps in SETS:
        d, z = seeds(rng, nk)
        ek, dk = kem.keygen(ps, d, z)
        ta = kem.keys_load(ps, seeds=(d, z), expand=True)
        tb = kem.keys_load(ps, seeds=(d, z), expand=True)
        slots = np.array([20, 0, nk - 1, 7, 11], np.uint32)
        d2, z2 = seeds(rng, len(slots))
        ek2, dk2 = kem.keygen(ps, d2, z2)
        ta.replace(slots, seeds=(d2, z2))
        tb.replace(slots, dk=dk2)
        ek[slots], dk[slots] = ek2, dk2
        assert (ta.export_ek() == tb.export_ek()).all() and (ta.export_ek() == ek).all()
        idx = every_slot(rng, nk, n)
        m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        c, K = kem.encaps(ps, ek[idx], m)
        bad, _ = tamper(c)
        Kd = kem.decaps(ps, dk[idx], bad)
        for t in (ta, tb):
            kc, kK = kem.encaps_keyed(t, idx, m)
            assert (kc == c).all() and (kK == K).all()
            assert (kem.decaps_keyed(t, idx, bad) == Kd).all()
        if not fips:
            assert (ek2 == oracle.keygen(ps, d2, z2)[0]).all()
        else:
            assert (ek2 != oracle.keygen(ps, d2, z2)[0]).any()  # FIPS mode really is another function


@pytest.mark.parametrize("ps", SETS)
def test_export_ek(mlkem, oracle, ps):
    """export_ek of a table built from seeds is KeyGen's ek (no second KeyGen needed): all rows and sub-ranges, host and device
    destinations, for every kind of table, and again after a replace."""
    import torch

    rng = np.random.default_rng(ps + 1050)
    nk = 300
    d, z = seeds(rng, nk)
    ek, dk = mlkem.keygen(ps, d, z)
    assert (ek == oracle.keygen(ps, d, z)[0]).all()
    t = mlkem.keys_load(ps, seeds=(d, z))
    assert (t.export_ek() == ek).all()
    got = t.export_ek(device=True)
    assert got.device.type == "cuda"
    torch.cuda.current_stream().synchronize()
    assert (got.cpu().numpy() == ek).all()
    for first, cnt in ((0, 1), (5, 7), (nk - 1, 1), (128, 100), (nk, 0)):
        assert (t.export_ek(first, cnt) == ek[first:first + cnt]).all()
        assert (t.export_ek(first, cnt, device=True).cpu().numpy() == ek[first:first + cnt]).all()
    assert (t.export_ek(250) == ek[250:]).all()
    for other in (mlkem.keys_load(ps, dk=dk), mlkem.keys_load(ps, ek=ek), mlkem.keys_load(ps, ek=ek, expand=True)):
        assert (other.export_ek() == ek).all() and (other.export_ek(17, 3) == ek[17:20]).all()
    slots = np.array([299, 3, 150], np.uint32)
    d2, z2 = seeds(rng, 3)
    t.replace(slots, seeds=(d2, z2))
    ek[slots] = oracle.keygen(ps, d2, z2)[0]
    assert (t.export_ek() == ek).all()
    assert (t.export_ek(140, 20, device=True).cpu().numpy() == ek[140:160]).all()


def test_replace_reports_the_hash_check(mlkem, oracle):
    """status of a replace: a dk whose stored H(ek) is wrong is reported (-5) and written all the same, and the keyed Decaps on
    it equals the unkeyed Decaps (Decaps_internal does not validate, ml_kem.c:1136)."""
    rng = np.random.default_rng(1347)
    nk = 24
    d, z = seeds(rng, nk)
    _, dk = oracle.keygen(768, d, z)
    table = mlkem.keys_load(768, dk=dk, expand=True)
    d2, z2 = seeds(rng, 4)
    ek2, dk2 = oracle.keygen(768, d2, z2)
    dk2[2, 768 * 3 + 40] ^= 0x10  # the stored hash H(ek) of the third new key
    slots = np.array([9, 1, 23, 14], np.uint32)
    for src in (dk2, cuda(dk2)):
        status = table.replace(slots, dk=src, return_status=True)
        assert list(status) == [0, 0, -5, 0]
    dk[slots] = dk2
    assert (table.export_ek()[slots] == ek2).all()
    idx = every_slot(rng, nk, 480)
    m = rng.integers(0, 256, (480, 32), dtype=np.uint8)
    c, _ = mlkem.encaps(768, dk[idx, 1152:2336], m)
    bad, _ = tamper(c)
    want = oracle.decaps(768, dk[idx], bad)
    assert (mlkem.decaps_keyed(table, idx, bad) == want).all()


def test_rejected_calls_leave_the_table_untouched(mlkem, oracle):
    """Every rejected replace / export returns MLKEM_B200_ERR_ARG and writes nothing: a slot out of range, a slot twice, NULL
    pointers, the wrong kind of table, another device's ordinal, a range past the end.  n = 0 is a successful no-op."""
    import torch

    from crystals_kyber_b200.lib import MEM_HOST, Opts

    dev = torch.cuda.current_device()
    lib = mlkem.lib
    rng = np.random.default_rng(11)
    nk, n = 16, 320
    d, z = seeds(rng, nk)
    ek, dk = oracle.keygen(768, d, z)
    t_dk = mlkem.keys_load(768, dk=dk, expand=True, device=dev)
    t_ek = mlkem.keys_load(768, ek=ek, device=dev)
    d2, z2 = seeds(rng, 2)
    ek2, dk2 = oracle.keygen(768, d2, z2)
    idx = every_slot(rng, nk, n)
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    c, K = mlkem.encaps(768, ek[idx], m)
    bad, _ = tamper(c)
    Kd = mlkem.decaps(768, dk[idx], bad)

    def untouched():
        for t in (t_dk, t_ek):
            assert (t.export_ek() == ek).all()
            kc, kK = mlkem.encaps_keyed(t, idx, m)
            assert (kc == c).all() and (kK == K).all()
        assert (mlkem.decaps_keyed(t_dk, idx, bad) == Kd).all()

    P = lambda a: C.c_void_p(a.ctypes.data)
    o = Opts(-1, MEM_HOST, None, 0, 0, 0)
    other = Opts(dev + 1, MEM_HOST, None, 0, 0, 0)
    ok_slots = np.array([4, 11], np.uint32)
    out = np.zeros((nk, ek.shape[1]), np.uint8)
    st = np.zeros(2, np.int32)
    calls = {
        "slot out of range": lambda: lib.mlkem_b200_keys_replace(t_dk.handle, 2, P(np.array([3, nk], np.uint32)), P(dk2), P(st), C.byref(o)),
        "slot twice": lambda: lib.mlkem_b200_keys_replace(t_dk.handle, 2, P(np.array([5, 5], np.uint32)), P(dk2), P(st), C.byref(o)),
        "slot twice (ek)": lambda: lib.mlkem_b200_keys_replace_ek(t_ek.handle, 2, P(np.array([7, 7], np.uint32)), P(ek2), C.byref(o)),
        "NULL table": lambda: lib.mlkem_b200_keys_replace(None, 2, P(ok_slots), P(dk2), P(st), C.byref(o)),
        "NULL slot": lambda: lib.mlkem_b200_keys_replace(t_dk.handle, 2, None, P(dk2), P(st), C.byref(o)),
        "NULL dk": lambda: lib.mlkem_b200_keys_replace(t_dk.handle, 2, P(ok_slots), None, P(st), C.byref(o)),
        "NULL ek": lambda: lib.mlkem_b200_keys_replace_ek(t_ek.handle, 2, P(ok_slots), None, C.byref(o)),
        "NULL z": lambda: lib.mlkem_b200_keys_replace_from_seeds(t_dk.handle, 2, P(ok_slots), P(d2), None, C.byref(o)),
        "dk into an ek table": lambda: lib.mlkem_b200_keys_replace(t_ek.handle, 2, P(ok_slots), P(dk2), P(st), C.byref(o)),
        "seeds into an ek table": lambda: lib.mlkem_b200_keys_replace_from_seeds(t_ek.handle, 2, P(ok_slots), P(d2), P(z2), C.byref(o)),
        "ek into a dk table": lambda: lib.mlkem_b200_keys_replace_ek(t_dk.handle, 2, P(ok_slots), P(ek2), C.byref(o)),
        "another device": lambda: lib.mlkem_b200_keys_replace(t_dk.handle, 2, P(ok_slots), P(dk2), P(st), C.byref(other)),
        "another device (seeds)": lambda: lib.mlkem_b200_keys_replace_from_seeds(t_dk.handle, 2, P(ok_slots), P(d2), P(z2), C.byref(other)),
        "export past the end": lambda: lib.mlkem_b200_keys_export_ek(t_dk.handle, nk - 2, 3, P(out), C.byref(o)),
        "export start past the end": lambda: lib.mlkem_b200_keys_export_ek(t_ek.handle, nk + 1, 0, P(out), C.byref(o)),
        "export NULL": lambda: lib.mlkem_b200_keys_export_ek(t_dk.handle, 0, 2, None, C.byref(o)),
        "export on another device": lambda: lib.mlkem_b200_keys_export_ek(t_dk.handle, 0, 2, P(out), C.byref(other)),
    }
    for what, call in calls.items():
        assert call() == ERR_ARG, what
    untouched()
    assert lib.mlkem_b200_keys_replace(t_dk.handle, 0, None, None, None, C.byref(o)) == 0
    assert lib.mlkem_b200_keys_replace_from_seeds(t_dk.handle, 0, None, None, None, C.byref(o)) == 0
    assert lib.mlkem_b200_keys_replace_ek(t_ek.handle, 0, None, None, C.byref(o)) == 0
    assert lib.mlkem_b200_keys_export_ek(t_dk.handle, nk, 0, None, C.byref(o)) == 0
    untouched()
    # and a valid call after all that
    assert lib.mlkem_b200_keys_replace(t_dk.handle, 2, P(ok_slots), P(dk2), P(st), C.byref(o)) == 0
    assert (st == 0).all() and (t_dk.export_ek()[ok_slots] == ek2).all()


@pytest.mark.parametrize("single_stream", [False, True], ids=["forked", "one-stream"])
def test_replace_is_ordered_after_device_calls_in_flight(mlkem, oracle, single_stream):
    """Keyed Decaps of 2^18 items under slot s enqueued on torch stream A (not waited for), then a replace of s from device memory
    on stream C, then keyed Decaps on stream B: the first result is the old key's, the second the new key's.  'forked' lets the
    first call spread its chunks over the library's streams, 'one-stream' keeps it on stream A."""
    import torch

    import crystals_kyber_b200 as ck

    kem = ck.MLKEM(chunk_items=1 << 18) if single_stream else ck.MLKEM()
    rng = np.random.default_rng(18 + single_stream)
    nk, s, n = 8, 5, 1 << 18
    d, z = seeds(rng, nk)
    ek, dk = oracle.keygen(768, d, z)
    table = kem.keys_load(768, dk=dk)
    d2, z2 = seeds(rng, 1)
    _, dk_new = oracle.keygen(768, d2, z2)
    new_list = dk.copy()
    new_list[s] = dk_new[0]
    t_new = kem.keys_load(768, dk=new_list)
    idx = cuda(np.full(n, s, np.int32))
    m = cuda(rng.integers(0, 256, (n, 32), dtype=np.uint8))
    c, K_old = kem.encaps_keyed(table, idx, m)
    K_new = kem.decaps_keyed(t_new, idx, c)
    src = cuda(dk_new)
    torch.cuda.synchronize()
    sa, sb, sc = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        K1 = kem.decaps_keyed(table, idx, c)
    with torch.cuda.stream(sc):
        table.replace(np.array([s], np.uint32), dk=src)
    with torch.cuda.stream(sb):
        K2 = kem.decaps_keyed(table, idx, c)
    torch.cuda.synchronize()
    assert (K1 == K_old).all().item()
    assert (K2 == K_new).all().item() and (K2 != K_old).any().item()
    hc = c[:64].cpu().numpy()
    assert (K2[:64].cpu().numpy() == oracle.decaps(768, np.repeat(dk_new, 64, axis=0), hc)).all()


def test_replace_is_ordered_after_async_host_calls(mlkem, oracle):
    """The same with MLKEM_B200_FLAG_ASYNC host-memory keyed Decaps on pinned buffers, a replace from host memory in between, and
    one mlkem_b200_synchronize at the end."""
    import torch

    import crystals_kyber_b200 as ck
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    kem = ck.MLKEM()
    lib = kem.lib
    dev = torch.cuda.current_device()
    rng = np.random.default_rng(2718)
    nk, s, n = 8, 2, 1 << 18
    d, z = seeds(rng, nk)
    ek, dk = oracle.keygen(768, d, z)
    table = kem.keys_load(768, dk=dk, device=dev)
    d2, z2 = seeds(rng, 1)
    _, dk_new = oracle.keygen(768, d2, z2)
    new_list = dk.copy()
    new_list[s] = dk_new[0]
    t_new = kem.keys_load(768, dk=new_list, device=dev)
    idx = np.full(n, s, np.uint32)
    m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    c, K_old = kem.encaps_keyed(table, idx, m)
    K_new = kem.decaps_keyed(t_new, idx, c)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    hidx, hc = pin(idx), pin(c)
    K1 = torch.zeros((n, 32), dtype=torch.uint8, pin_memory=True)
    K2 = torch.zeros((n, 32), dtype=torch.uint8, pin_memory=True)
    P = lambda t: C.c_void_p(t.data_ptr())
    o = Opts(dev, MEM_HOST, None, 0, 0, 2)  # MLKEM_B200_FLAG_ASYNC
    assert lib.mlkem_b200_decaps_keyed_batch(table.handle, n, P(hidx), P(hc), P(K1), C.byref(o)) == 0
    table.replace(np.array([s], np.uint32), dk=dk_new)
    assert lib.mlkem_b200_decaps_keyed_batch(table.handle, n, P(hidx), P(hc), P(K2), C.byref(o)) == 0
    assert lib.mlkem_b200_synchronize(dev, None) == 0
    assert (K1.numpy() == K_old).all()
    assert (K2.numpy() == K_new).all() and (K2.numpy() != K_old).any()


def test_replace_keeps_the_tables_group_limit(mlkem, oracle):
    """An expanded table loaded with a lowered sample_group_limit (the restart path, ml_kem.c:221-242) keeps that limit: slots
    replaced with default-limit options (from dk, and from seeds whose KeyGen runs at the call's limit) get matrices sampled at
    the table's limit, so keyed Encaps equals unkeyed Encaps at that limit."""
    import crystals_kyber_b200 as ck
    from crystals_kyber_b200.lib import MEM_HOST, Opts

    lib = mlkem.lib
    rng = np.random.default_rng(158)
    nk, n = 64, 640
    d, z = seeds(rng, nk)
    dn, zn = seeds(rng, 8)  # new keys from seeds: KeyGen at the default limit (the replacing call's)
    ek_seeds, dk_seeds = oracle.keygen(768, dn, zn)
    lim = ck.MLKEM(sample_group_limit=158)
    oracle.set_sample_group_limit(158)
    try:
        ek, dk = oracle.keygen(768, d, z)
        table = lim.keys_load(768, dk=dk, expand=True)
        dd, zd = seeds(rng, 8)
        ek_dk, dk_dk = oracle.keygen(768, dd, zd)
        s_dk = np.array([63, 0, 31, 12, 40, 7, 50, 22], np.uint32)
        s_seeds = np.array([1, 62, 30, 13, 41, 8, 51, 23], np.uint32)
        o = Opts(-1, MEM_HOST, None, 0, 0, 0)  # default options: sample_group_limit 0 = the reference's 278
        P = lambda a: C.c_void_p(a.ctypes.data)
        assert lib.mlkem_b200_keys_replace(table.handle, len(s_dk), P(s_dk), P(dk_dk), None, C.byref(o)) == 0
        assert lib.mlkem_b200_keys_replace_from_seeds(table.handle, len(s_seeds), P(s_seeds), P(dn), P(zn), C.byref(o)) == 0
        ek[s_dk], ek[s_seeds] = ek_dk, ek_seeds
        dk[s_dk], dk[s_seeds] = dk_dk, dk_seeds
        idx = every_slot(rng, nk, n)
        m = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        oc, oK = oracle.encaps(768, ek[idx], m)
        c, K = lim.encaps_keyed(table, idx, m)
        assert (c == oc).all() and (K == oK).all()
        bad, _ = tamper(oc)
        assert (lim.decaps_keyed(table, idx, bad) == oracle.decaps(768, dk[idx], bad)).all()
    finally:
        oracle.set_sample_group_limit(0)
    on_new = np.isin(idx, np.concatenate([s_dk, s_seeds]))
    assert (oracle.encaps(768, ek[idx][on_new], m[on_new])[0] != oc[on_new]).any(), \
        "the lowered limit must change some matrix entries of the new keys for the test to mean anything"
