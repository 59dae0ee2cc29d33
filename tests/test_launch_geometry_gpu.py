"""Every batched entry point at the batch sizes where its launch geometry changes, with guard bands around every buffer.

Batched kernels go wrong in *which items* they write as much as in what they compute: a tail block that stores one item too
many, a grid-stride loop that stops one pass early, a persistent warp whose 3rd item reuses a buffer, a call whose chunks
take different paths.  The tests below call the C ABI directly with every input and output placed inside a larger
allocation: a region at a 16-byte but not 256-byte aligned address, with at least 4 KiB of guard before and after it.
Guards and output regions are filled with a seeded pseudo-random pattern first.  After every call every guard byte and
every input byte must be unchanged and every output byte must equal the oracle's, so a stray write shows up in a guard
and an item left unwritten shows up as the pattern.  Inputs sit inside allocations the test owns too, so a stray read
stays in memory the test owns.

The batch sizes come from the launch-geometry constants that tests/test_launch_geometry_cpu.py checks against the
sources.  Each case is a prefix of one input set per parameter set, run once through the oracle.  The per-kernel profile
confirms that each case ran the kernels it was chosen for.
"""
import ctypes as C
import hashlib
import math
import os
import struct

import numpy as np
import pytest

from oracle.oracle import sizes
from test_launch_geometry_cpu import (GEOMETRY, LIST_ROWS_PER_PASS, PERSISTENT_WARPS, PRIM_POLYS_PER_PASS,
                                      VECTORS_PER_PASS, key_index_confined)

pytestmark = pytest.mark.gpu

SETS = (512, 768, 1024)
Q = 3329
OK, ERR_ARG = 0, -11
GUARD = 4096
MISALIGN = 48  # every region starts 48 bytes past a 256-byte boundary: 16-byte aligned (the documented minimum), no more
SEED = bytes.fromhex("8f0e1d2c3b4a59687786950a1b2c3d4e5f60718293a4b5c6d7e8f90112233445")
TAG_KEYGEN, TAG_ENCAPS = 1, 2
N_MAX = 65537
PW = PERSISTENT_WARPS  # 9 472 warps: a warp's 2nd item is item PW, its 3rd (buffer 0 again) 2 PW, its 4th (buffer 1 again) 3 PW
SIZES = sorted({1, 2, 3, 4, 5,  # warp-per-item blocks of 4
                8, 9, 10, 11, 16, 17,  # rows = n K crosses 32 (K = 4, 3, 2): general kernel alone -> fused + clean-up
                31, 32, 33, 127, 128, 129,  # 128-thread hash and noise blocks
                1024, 1025,  # warp-form -> thread-form hashing
                PW, PW + 1, 2 * PW + 1, 3 * PW + 1,  # persistent warps: 1st, 2nd, 3rd, 4th item
                65536, 65537})  # host: a 1-item last chunk; device: the automatic two-way split
WARP_MAX = int(os.environ.get("MLKEM_B200_WARP_HASH_MAX", GEOMETRY["kWarpHashMaxItems"]))
STREAMS = int(os.environ.get("MLKEM_B200_STREAMS", "0") or 0)
DEFAULT_STREAMS = 4 if STREAMS < 1 else min(STREAMS, 4)


@pytest.fixture(scope="module")
def lib():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.load()


@pytest.fixture(scope="module")
def kem(lib):
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


# ------------------------------------------------------------------------------------------------ guarded buffers
_POOL = np.frombuffer(np.random.default_rng(20261021).bytes((1 << 24) + 61), np.uint8)  # host pattern source


def _host_pattern(total, salt):
    out = np.empty(total, np.uint8)
    at = (salt * 7919 + 13) % len(_POOL)
    done = 0
    while done < total:
        take = min(total - done, len(_POOL) - at)
        out[done:done + take] = _POOL[at:at + take]
        done, at = done + take, 0
    return out


class Guarded:
    """The buffers of one call.  inp() and out() return the pointer of a region inside a fresh allocation; check() lists
    every guard, input or output byte that is not what it must be."""

    def __init__(self, device, salt=0):
        self.device, self.salt, self.bufs = device, salt, []

    def _region(self, nbytes):
        total = GUARD + 256 + nbytes + GUARD
        salt = self.salt * 131 + len(self.bufs)
        if self.device:
            import torch

            g = torch.Generator(device="cuda")
            g.manual_seed(salt)
            a = torch.randint(0, 256, (total,), dtype=torch.uint8, device="cuda", generator=g)
            ptr = a.data_ptr()
        else:
            a = _host_pattern(total, salt)
            ptr = a.ctypes.data
        off = GUARD + (MISALIGN - ptr - GUARD) % 256
        assert (ptr + off) % 16 == 0 and (ptr + off) % 256 != 0 and total - off - nbytes >= GUARD
        return a, off, ptr + off

    def inp(self, data, item=1, name="in"):
        """An input: `data` (uint8, numpy for host memory, torch CUDA for device memory) copied into its region."""
        a, off, p = self._region(len(data))
        a[off:off + len(data)] = data
        self.bufs.append([name, a, off, len(data), None, item])
        return C.c_void_p(p)

    def out(self, expect, item=1, name="out"):
        """An output region left as the pattern; afterwards it must hold `expect` (uint8; an int stands for that many
        bytes that must keep the pattern: nothing may be written)."""
        n = expect if isinstance(expect, int) else len(expect)
        a, off, p = self._region(n)
        self.bufs.append([name, a, off, n, None if isinstance(expect, int) else expect, item])
        return C.c_void_p(p)

    def seal(self):
        """Take the reference copy of every allocation: call after the last inp() / out(), before the launch."""
        for b in self.bufs:
            a = b[1]
            b.append(a.clone() if self.device else a.copy())

    def check(self, what):
        import torch

        if self.device:
            torch.cuda.synchronize()
        errors = []
        for name, a, off, n, expect, item, ref in self.bufs:
            eq = torch.equal if self.device else np.array_equal
            if not eq(a[:off], ref[:off]):
                errors.append(f"{what}: {name}: guard before the region changed")
            if not eq(a[off + n:], ref[off + n:]):
                errors.append(f"{what}: {name}: guard after the region changed")
            want = ref[off:off + n] if expect is None else expect
            got = a[off:off + n]
            if not eq(got, want):
                bad = (got != want).nonzero().reshape(-1).cpu().numpy() if self.device else np.nonzero(got != want)[0]
                items = np.unique(bad // item)
                kind = "input changed" if expect is None and name.startswith("in") else "differs"
                errors.append(f"{what}: {name} {kind}: {len(items)} of {n // item} items, first {items[:6].tolist()}")
        return errors


def call(lib, fname, args, device, chunk=0, limit=0, stream=None):
    """fname(*args, &opts) with the memory space `device` selects; returns the return code."""
    import torch

    from crystals_kyber_b200.lib import MEM_DEVICE, MEM_HOST, Opts

    if device:
        o = Opts(torch.cuda.current_device(), MEM_DEVICE, torch.cuda.current_stream().cuda_stream, chunk, limit, 0)
    else:
        o = Opts(-1, MEM_HOST, None, chunk, limit, 0)
    return getattr(lib, fname)(*args, C.byref(o))


def chunk_sizes(n, device, chunk=0, streams=None):
    """The chunks drive() cuts a batch of n items into (mlkem_b200.cu): the kernels of each chunk see only its size."""
    streams = DEFAULT_STREAMS if streams is None else streams
    c = chunk or (GEOMETRY["device_chunk"] if device else GEOMETRY["host_chunk"])
    c = min(c, n)
    if device and not chunk and n >= GEOMETRY["split_min"] and -(-n // c) < 2 and streams > 1:
        c = ((n + 1) // 2 + 1023) & ~1023
    return [min(c, n - i) for i in range(0, n, c)]


def profiled(kem, fn):
    kem.profile(True)
    try:
        out = fn()
    finally:
        kem.profile(False)
    return out, {name.strip("()").split("<")[0] for name in kem.profile_report()}


HASH_STEM = {"keygen": "k_keygen_H", "encaps": "k_encaps_HG", "decaps": "k_decaps_J_select", "check_dk": "k_check_dk_hash"}


def path_errors(entry, names, chunks, k, limit=0):
    """The kernels `entry` must have run for these chunks: the fused matrix kernel iff some chunk has more than 32 rows
    (at the reference's group limit), the warp form of its hash iff some chunk has at most WARP_MAX items, the thread form
    iff some chunk has more."""
    errs = []
    if entry in ("keygen", "encaps", "decaps"):
        fused = limit == 0 and any(cn * k > GEOMETRY["fused_min_rows"] for cn in chunks)
        if ("k_sample_matvec" in names) != fused or "k_sample_matvec_list" not in names:
            errs.append(f"{entry} {chunks}: fused kernel {'missing' if fused else 'ran'}: {sorted(names)}")
    stem = HASH_STEM[entry]
    warp, thread = any(cn <= WARP_MAX for cn in chunks), any(cn > WARP_MAX for cn in chunks)
    if (stem + "_warp" in names) != warp or (stem in names) != thread:
        errs.append(f"{entry} {chunks}: warp form {warp}, thread form {thread} expected: {sorted(names)}")
    return errs


# ------------------------------------------------------------------------------------------------ the input set
def derive(seed, n, tag):
    width = 64 if tag == TAG_KEYGEN else 32
    out = np.frombuffer(b"".join(hashlib.shake_256(seed + struct.pack("<QQ", j, tag)).digest(width) for j in range(n)), np.uint8)
    return out.reshape(n, width)


def tamper(c):
    """Item i is tampered iff i % 10 == 3: flip bit (i % 8) of byte (i * 7919) % len."""
    c = c.copy()
    n, L = c.shape
    sel = np.arange(n)[np.arange(n) % 10 == 3]
    c[sel, (sel * 7919) % L] ^= (1 << (sel % 8)).astype(np.uint8)
    return c


class Data:
    """One input set of N_MAX items for a parameter set and its oracle results.  (d, z) and m are the R_j of the seeded
    calls for SEED, so the seeded calls share the expected values of the plain ones.  Arrays are numpy, item-major;
    dev(name) is the same bytes on the GPU (uploaded once)."""

    def __init__(self, oracle, ps, n=N_MAX, limit=0):
        self.ps, self.sz, self._dev = ps, sizes(ps), {}
        k, dkp = self.sz["k"], self.sz["dk_pke"]
        R = derive(SEED, n, TAG_KEYGEN)
        self.d, self.z = R[:, :32].copy(), R[:, 32:].copy()
        self.m = derive(SEED, n, TAG_ENCAPS).copy()
        try:
            oracle.set_sample_group_limit(limit)
            self.ek, self.dk = oracle.keygen(ps, self.d, self.z)
            self.c, self.K = oracle.encaps(ps, self.ek, self.m)
            self.ct = tamper(self.c)
            self.Kd = oracle.decaps(ps, self.dk, self.ct)
        finally:
            oracle.set_sample_group_limit(0)
        if limit:
            return
        # K-PKE from the same run: ek = ek_pke, dk = dk_pke || ..., (K, r) = G(m || H(ek)), c = PKE_Encrypt(ek, m, r)
        G = [hashlib.sha3_512(mi.tobytes() + hi.tobytes()).digest() for mi, hi in zip(self.m, self.dk[:, -64:-32])]
        self.r = np.frombuffer(b"".join(g[32:] for g in G), np.uint8).reshape(n, 32).copy()
        assert np.array_equal(np.frombuffer(b"".join(g[:32] for g in G), np.uint8).reshape(n, 32), self.K)
        self.dk_pke = np.ascontiguousarray(self.dk[:, :dkp])
        pad = np.random.default_rng(ps).integers(0, 256, (n, 16), dtype=np.uint8)
        self.dk_pad = np.ascontiguousarray(np.concatenate([self.dk_pke, pad], 1))  # dk_stride = DK_PKE + 16
        probe = slice(0, 64)
        pek, pdk = oracle.pke_keygen(ps, self.d[probe])
        assert np.array_equal(pek, self.ek[probe]) and np.array_equal(pdk, self.dk_pke[probe])
        assert np.array_equal(oracle.pke_encrypt(ps, self.ek[probe], self.m[probe], self.r[probe]), self.c[probe])
        # dk hash check: every item with i % 10 == 7 gets a wrong H(ek) (-5 from check_dk; KEM_Decaps zeroes its key)
        self.dk_bad = self.dk.copy()
        bad = np.arange(n) % 10 == 7
        self.dk_bad[bad, -64] ^= 1
        self.status = np.where(bad, -5, 0).astype(np.int32)
        self.Kd_bad = np.where(bad[:, None], 0, self.Kd).astype(np.uint8)

    def b(self, name, n, device):
        """The bytes of items [0, n) of array `name`."""
        a = getattr(self, name)
        w = a[0].nbytes
        if not device:
            return a[:n].reshape(-1).view(np.uint8)
        if name not in self._dev:
            import torch

            self._dev[name] = torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()
        return self._dev[name][:n * w]

    def cells(self, name, n, device, poison_high=False):
        """The same bytes in the reference's cell layout (one per uint32); inputs carry junk in the upper 24 bits, which
        the calls ignore."""
        a = self.b(name, n, device)
        if device:
            import torch

            t = a.to(torch.int32)
            return (t | 0x5A5A5A00 if poison_high else t).view(torch.uint8)
        t = a.astype(np.uint32)
        return (t | 0x5A5A5A00 if poison_high else t).view(np.uint8)


_data = {}


def data(oracle, ps):
    if ps not in _data:
        _data[ps] = Data(oracle, ps)
    return _data[ps]


def entries(D, n, device):
    """(entry, function, args builder) for every batched entry point; the builder takes a Guarded and returns the argument
    list of the C call."""
    from crystals_kyber_b200.api import _seed_ptr

    ps, sz = D.ps, D.sz
    b = lambda name, nn=n: D.b(name, nn, device)
    dkp = sz["dk_pke"]
    yield "keygen", "mlkem_b200_keygen_batch", lambda g: [ps, n, g.inp(b("d"), 32, "in d"), g.inp(b("z"), 32, "in z"),
                                                           g.out(b("ek"), sz["ek"], "ek"), g.out(b("dk"), sz["dk"], "dk")]
    yield "encaps", "mlkem_b200_encaps_batch", lambda g: [ps, n, g.inp(b("ek"), sz["ek"], "in ek"), g.inp(b("m"), 32, "in m"),
                                                           g.out(b("c"), sz["c"], "c"), g.out(b("K"), 32, "K")]
    yield "decaps", "mlkem_b200_decaps_batch", lambda g: [ps, n, g.inp(b("dk"), sz["dk"], "in dk"), g.inp(b("ct"), sz["c"], "in c"),
                                                           g.out(b("Kd"), 32, "K")]
    yield "check_dk", "mlkem_b200_check_dk_batch", lambda g: [ps, n, g.inp(b("dk_bad"), sz["dk"], "in dk"),
                                                               g.out(b("status"), 4, "status")]
    yield "pke_keygen", "mlkem_b200_pke_keygen_batch", lambda g: [ps, n, g.inp(b("d"), 32, "in d"), g.out(b("ek"), sz["ek"], "ek"),
                                                                   g.out(b("dk_pke"), dkp, "dk_pke")]
    yield "pke_encrypt", "mlkem_b200_pke_encrypt_batch", lambda g: [ps, n, g.inp(b("ek"), sz["ek"], "in ek"), g.inp(b("m"), 32, "in m"),
                                                                     g.inp(b("r"), 32, "in r"), g.out(b("c"), sz["c"], "c")]
    for src, stride in (("dk_pke", dkp), ("dk", sz["dk"]), ("dk_pad", dkp + 16)):
        yield f"pke_decrypt/{stride}", "mlkem_b200_pke_decrypt_batch", \
            lambda g, src=src, stride=stride: [ps, n, g.inp(b(src), stride, "in dk"), stride, g.inp(b("c"), sz["c"], "in c"),
                                               g.out(b("m"), 32, "m")]
    cl = lambda name, poison=False: D.cells(name, n, device, poison)
    yield "keygen_cells", "mlkem_b200_keygen_cells_batch", lambda g: [ps, n, g.inp(cl("d", True), 128, "in d"), g.inp(cl("z", True), 128, "in z"),
                                                                       g.out(cl("ek"), 4 * sz["ek"], "ek"), g.out(cl("dk"), 4 * sz["dk"], "dk")]
    yield "encaps_cells", "mlkem_b200_encaps_cells_batch", lambda g: [ps, n, g.inp(cl("ek", True), 4 * sz["ek"], "in ek"),
                                                                       g.inp(cl("m", True), 128, "in m"), g.out(cl("c"), 4 * sz["c"], "c"),
                                                                       g.out(cl("K"), 128, "K")]
    yield "decaps_cells", "mlkem_b200_decaps_cells_batch", lambda g: [ps, n, g.inp(cl("dk", True), 4 * sz["dk"], "in dk"),
                                                                       g.inp(cl("ct", True), 4 * sz["c"], "in c"), g.out(cl("Kd"), 128, "K")]
    yield "kem_keygen_seeded", "mlkem_b200_kem_keygen_seeded_batch", lambda g: [ps, n, _seed_ptr(SEED), g.out(b("ek"), sz["ek"], "ek"),
                                                                                 g.out(b("dk"), sz["dk"], "dk")]
    yield "kem_encaps_seeded", "mlkem_b200_kem_encaps_seeded_batch", lambda g: [ps, n, g.inp(b("ek"), sz["ek"], "in ek"), sz["ek"],
                                                                                 _seed_ptr(SEED), g.out(b("c"), sz["c"], "c"),
                                                                                 g.out(b("K"), 32, "K")]
    yield "kem_decaps", "mlkem_b200_kem_decaps_batch", lambda g: [ps, n, g.inp(b("dk_bad"), sz["dk"], "in dk"), sz["dk"],
                                                                   g.inp(b("ct"), sz["c"], "in c"), sz["c"], g.out(b("Kd_bad"), 32, "K"),
                                                                   g.out(b("status"), 4, "status")]


def run_entry(lib, kem, D, entry, fname, build, n, device, chunk=0, limit=0, streams=None, salt=0):
    """One guarded call; returns the list of what went wrong (empty: nothing)."""
    g = Guarded(device, salt)
    args = build(g)
    g.seal()
    what = f"ML-KEM-{D.ps} {entry} n={n} {'device' if device else 'host'}" + (f" chunk={chunk}" if chunk else "")
    if entry in HASH_STEM:
        rc, names = profiled(kem, lambda: call(lib, fname, args, device, chunk, limit))
    else:
        rc, names = call(lib, fname, args, device, chunk, limit), None
    if rc != OK:
        return [f"{what}: rc={rc} {lib.mlkem_b200_last_error().decode()}"]
    errs = g.check(what)
    if names is not None:
        errs += [f"{what}: {e}" for e in path_errors(entry, names, chunk_sizes(n, device, chunk, streams), D.sz["k"], limit)]
    return errs


# ------------------------------------------------------------------------------------------------ 1. the size table
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("ps", SETS)
def test_every_entry_point_at_every_geometry_boundary(lib, kem, oracle, ps, device):
    """Every batched entry point at every size of SIZES, in guarded buffers: keygen, encaps, decaps (the i % 10 == 3 tamper
    rule), check_dk (a wrong H(ek) at i % 10 == 7), the three pke_* calls (pke_decrypt at dk_stride DK_PKE, DK and
    DK_PKE + 16), the three *_cells calls, the seeded KeyGen / Encaps and the public KEM_Decaps batch with its status words.
    Sizes that differ only in which item of a persistent warp or which tail block is last are all here, so a kernel that
    skips or adds one item's store fails at the size that reaches it."""
    D = data(oracle, ps)
    errors = []
    for n in SIZES:
        for entry, fname, build in entries(D, n, device):
            errors += run_entry(lib, kem, D, entry, fname, build, n, device, salt=n)
    assert not errors, "\n".join(errors[:40])


CHUNKINGS = [(9, 1), (50, 7), (2051, 1025)]  # 2 051 at 1 025: thread, thread, then warp + general kernel only


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("ps", SETS)
def test_explicit_chunkings(lib, kem, oracle, ps, device):
    """Chunks of 1 item, of 7 and of 1 025 items (the last call's final chunk of one item takes the warp-form hashes and the
    general matrix kernel alone while the two before it take the thread form and the fused kernel), and in device memory
    65 537 items with the default streams (a two-way split) and after set_streams(1) (one chunk)."""
    D = data(oracle, ps)
    errors = []
    for n, chunk in CHUNKINGS:
        for entry, fname, build in entries(D, n, device):
            errors += run_entry(lib, kem, D, entry, fname, build, n, device, chunk=chunk, salt=7 * n + chunk)
    assert chunk_sizes(2051, device, 1025) == [1025, 1025, 1]
    if device:
        assert len(chunk_sizes(N_MAX, True)) == (2 if DEFAULT_STREAMS > 1 else 1)
        kem.set_streams(1)
        try:
            for entry, fname, build in entries(D, N_MAX, device):
                if entry in ("keygen", "encaps", "decaps", "check_dk", "kem_decaps"):
                    errors += run_entry(lib, kem, D, entry, fname, build, N_MAX, device, streams=1, salt=99)
        finally:
            kem.set_streams(0)
    assert not errors, "\n".join(errors[:40])


# ------------------------------------------------------------------------------------------------ 2. list-kernel stride passes
LIMIT = 158  # below 168: every row goes through k_sample_matvec_list


@pytest.mark.parametrize("ps", SETS)
def test_list_kernel_stride_passes(lib, kem, oracle, ps):
    """With a lowered group limit every row goes through k_sample_matvec_list, 18 944 rows per grid-stride pass: KeyGen,
    Encaps and Decaps at ceil(18 944 / K) + 1 and ceil(2 * 18 944 / K) + 1 items (2 and 3 passes), in both memory spaces,
    against the oracle at the same limit."""
    k = sizes(ps)["k"]
    sizes_ = [math.ceil(LIST_ROWS_PER_PASS / k) + 1, math.ceil(2 * LIST_ROWS_PER_PASS / k) + 1]
    D = Data(oracle, ps, n=sizes_[-1], limit=LIMIT)
    errors = []
    for n in sizes_:
        assert -(-n * k // LIST_ROWS_PER_PASS) == sizes_.index(n) + 2
        for device in (False, True):
            for entry, fname, build in entries(D, n, device):
                if entry in ("keygen", "encaps", "decaps"):
                    errors += run_entry(lib, kem, D, entry, fname, build, n, device, limit=LIMIT, salt=n)
    assert not errors, "\n".join(errors[:40])


# ------------------------------------------------------------------------------------------------ 3. keyed calls
KEYED_SIZES = [PW, PW + 1, 2 * PW + 1, 3 * PW + 1]
NULL_CHUNK = 20000  # not a multiple of 37: the first key of each chunk (first % n_keys) moves


class Keyed:
    """Tables of 1 and of 37 keys of a Data set and the oracle results of keyed Encaps / Decaps under three index patterns:
    a random index array, NULL with 37 keys (key i % 37) and NULL with one key."""

    def __init__(self, oracle, D, n):
        rng = np.random.default_rng(D.ps + 37)
        self.idx = {"random": rng.integers(0, 37, n).astype(np.uint32), "mod37": (np.arange(n) % 37).astype(np.uint32),
                    "one": np.zeros(n, np.uint32)}
        self.want = {}
        for pat, idx in self.idx.items():
            c, K = oracle.encaps(D.ps, D.ek[idx], D.m[:n])
            ct = tamper(c)
            self.want[pat] = dict(c=c, K=K, ct=ct, Kd=oracle.decaps(D.ps, D.dk[idx], ct))


def keyed_calls(D, want, idx, n, device, handle):
    """encaps_keyed, decaps_keyed and kem_encaps_keyed of n items in guarded buffers; idx None = the NULL index."""
    from crystals_kyber_b200.api import _seed_ptr

    import torch

    sz = D.sz
    up = (lambda a: torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()) if device else \
        (lambda a: np.ascontiguousarray(a).reshape(-1).view(np.uint8))
    ix = lambda g: None if idx is None else g.inp(up(idx[:n]), 4, "in key_index")
    yield "encaps_keyed", "mlkem_b200_encaps_keyed_batch", lambda g: [handle, n, ix(g), g.inp(up(D.m[:n]), 32, "in m"),
                                                                       g.out(up(want["c"][:n]), sz["c"], "c"), g.out(up(want["K"][:n]), 32, "K")]
    yield "decaps_keyed", "mlkem_b200_decaps_keyed_batch", lambda g: [handle, n, ix(g), g.inp(up(want["ct"][:n]), sz["c"], "in c"),
                                                                       g.out(up(want["Kd"][:n]), 32, "K")]
    yield "kem_encaps_keyed", "mlkem_b200_kem_encaps_keyed_batch", lambda g: [handle, n, ix(g), _seed_ptr(SEED),
                                                                               g.out(up(want["c"][:n]), sz["c"], "c"),
                                                                               g.out(up(want["K"][:n]), 32, "K")]


def run_keyed(lib, kem, D, calls, n, device, chunk=0, expanded=False, what=""):
    errors = []
    for entry, fname, build in calls:
        g = Guarded(device, n)
        args = build(g)
        g.seal()
        label = f"ML-KEM-{D.ps} {entry} {what} n={n} {'device' if device else 'host'}"
        rc, names = profiled(kem, lambda: call(lib, fname, args, device, chunk))
        if rc != OK:
            errors.append(f"{label}: rc={rc} {lib.mlkem_b200_last_error().decode()}")
            continue
        errors += g.check(label)
        if ("k_matvec_table" in names) != expanded:
            errors.append(f"{label}: k_matvec_table {'missing' if expanded else 'ran'}: {sorted(names)}")
    return errors


@pytest.mark.parametrize("ps", SETS)
def test_keyed_calls_at_persistent_warp_sizes(lib, kem, oracle, ps):
    """encaps_keyed, decaps_keyed and kem_encaps_keyed at 9 472, 9 473, 18 945 and 28 417 items -- the 1st to 4th item of a
    persistent warp, and of a k_matvec_table row slot -- on tables of 37 keys and of 1 key, plain and expanded: a random
    device index array, the NULL index at chunks of 20 000 items (37 does not divide it, so the first key of each chunk
    moves) in both memory spaces, and the NULL index on the 1-key table.  Against the oracle on dk[index]."""
    D = data(oracle, ps)
    KY = Keyed(oracle, D, KEYED_SIZES[-1])
    errors = []
    for expand in (False, True):
        t37 = kem.keys_load(ps, dk=D.dk[:37], expand=expand)
        t1 = kem.keys_load(ps, dk=D.dk[:1], expand=expand)
        try:
            for n in KEYED_SIZES:
                tag = f"expand={expand}"
                errors += run_keyed(lib, kem, D, keyed_calls(D, KY.want["random"], KY.idx["random"], n, True, t37.handle), n, True,
                                    expanded=expand, what=f"37 keys random index {tag}")
                for device in (False, True):
                    errors += run_keyed(lib, kem, D, keyed_calls(D, KY.want["mod37"], None, n, device, t37.handle), n, device,
                                        chunk=NULL_CHUNK, expanded=expand, what=f"37 keys NULL index chunk={NULL_CHUNK} {tag}")
                errors += run_keyed(lib, kem, D, keyed_calls(D, KY.want["one"], None, n, True, t1.handle), n, True,
                                    expanded=expand, what=f"1 key NULL index {tag}")
        finally:
            t37.free()
            t1.free()
    assert not errors, "\n".join(errors[:40])


OUT_OF_RANGE = np.array([37, 38, 1 << 31, (1 << 32) - 1], np.uint32)  # n_keys, n_keys + 1, 2^31, int32 -1


@pytest.mark.parametrize("ps", SETS)
def test_key_index_out_of_range(lib, kem, oracle, ps):
    """Indices n_keys, n_keys + 1, 2^31 and 2^32 - 1 among valid ones.  In device memory every keyed call clamps them and
    returns exactly what index n_keys - 1 gives; in host memory the call returns -11, writes nothing and leaves the table
    as it was.  Nothing is launched with such an index unless the source check shows that the kernels read the index only
    through the clamp in key_row."""
    problem = key_index_confined()
    if problem:
        pytest.fail(f"not launching out-of-range key indices: {problem}")
    D = data(oracle, ps)
    n = 2051
    idx = np.random.default_rng(ps).integers(0, 37, n).astype(np.uint32)
    idx[::5] = np.resize(OUT_OF_RANGE, len(idx[::5]))
    idx[-1] = OUT_OF_RANGE[-1]
    clamped = np.minimum(idx, 36)
    c, K = oracle.encaps(ps, D.ek[clamped], D.m[:n])
    ct = tamper(c)
    want = dict(c=c, K=K, ct=ct, Kd=oracle.decaps(ps, D.dk[clamped], ct))
    errors = []
    for expand in (False, True):
        table = kem.keys_load(ps, dk=D.dk[:37], expand=expand)
        try:
            ek_before = table.export_ek()
            errors += run_keyed(lib, kem, D, keyed_calls(D, want, idx, n, True, table.handle), n, True, expanded=expand,
                                what=f"clamped expand={expand}")
            for entry, fname, build in keyed_calls(D, want, idx, n, False, table.handle):
                g = Guarded(False, 5)
                args = build(g)
                for b in g.bufs:  # outputs must keep the pattern
                    if b[4] is not None:
                        b[4] = None
                g.seal()
                rc = call(lib, fname, args, False)
                if rc != ERR_ARG:
                    errors.append(f"ML-KEM-{ps} {entry} host: rc={rc}, not {ERR_ARG}")
                errors += g.check(f"ML-KEM-{ps} {entry} host, rejected index")
            if not np.array_equal(table.export_ek(), ek_before):
                errors.append(f"ML-KEM-{ps} expand={expand}: a rejected call changed the table")
        finally:
            table.free()
    assert not errors, "\n".join(errors[:40])


# ------------------------------------------------------------------------------------------------ 4. primitives
PRIM_SIZES = [1, 7, 8, 9, PRIM_POLYS_PER_PASS, PRIM_POLYS_PER_PASS + 1, 2 * PRIM_POLYS_PER_PASS + 1]
CODEC_D = (1, 11, 12)


class Prims:
    """Inputs of the stand-alone primitives for the largest size and their oracle results."""

    def __init__(self, oracle, n):
        rng = np.random.default_rng(2026)
        u16 = lambda hi, shape: rng.integers(0, hi, shape, dtype=np.uint16)
        self.f, self.g = u16(Q, (n, 256)), u16(Q, (n, 256))
        self.a12, self.b12 = u16(4096, (n, 256)), u16(4096, (n, 256))
        self.u3, self.v3 = u16(Q, (n, 3, 256)), u16(Q, (n, 3, 256))
        self.cbd_in = {eta: rng.integers(0, 256, (n, 64 * eta), dtype=np.uint8) for eta in (2, 3)}
        self.prf_s, self.prf_b = rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, n, dtype=np.uint8)
        self.seeds = rng.integers(0, 256, (n, 34), dtype=np.uint8)
        self.low = {d: u16(1 << d, (n, 256)) for d in CODEC_D}
        self.enc_in = {d: rng.integers(0, 256, (n, 32 * d), dtype=np.uint8) for d in CODEC_D}
        self.want = {
            "ntt": oracle.ntt(self.f), "intt": oracle.intt(self.f), "mul": oracle.multiply_ntts(self.a12, self.b12),
            "vec": oracle.vector_multiply(self.u3, self.v3, 3), "add": oracle.poly_add(self.f, self.g),
            "sub": oracle.poly_sub(self.f, self.g),
            **{f"cbd{eta}": oracle.cbd(self.cbd_in[eta], eta) for eta in (2, 3)},
            **{f"prf{eta}": oracle.prf_cbd(self.prf_s, self.prf_b, eta) for eta in (2, 3)},
            **{f"enc{d}": oracle.byte_encode(self.low[d], d) for d in CODEC_D},
            **{f"dec{d}": oracle.byte_decode(self.enc_in[d], d) for d in CODEC_D},
            **{f"cenc{d}": oracle.byte_encode(oracle.compress(self.f, d).reshape(n, 256), d) for d in CODEC_D},
            **{f"ddec{d}": oracle.decompress(oracle.byte_decode(self.enc_in[d], d), d).reshape(n, 256) for d in CODEC_D},
        }
        self.want["sample"], self.want["after"] = oracle.sample_ntt_with_seeds(self.seeds)


def prim_calls(P, n, device):
    import torch

    up = (lambda a: torch.from_numpy(np.ascontiguousarray(a[:n]).reshape(-1).view(np.uint8)).cuda()) if device else \
        (lambda a: np.ascontiguousarray(a[:n]).reshape(-1).view(np.uint8))
    W = P.want
    poly = 512
    yield "ntt", lambda g: ["mlkem_b200_ntt_batch", n, g.inp(up(P.f), poly), g.out(up(W["ntt"]), poly)]
    yield "intt", lambda g: ["mlkem_b200_intt_batch", n, g.inp(up(P.f), poly), g.out(up(W["intt"]), poly)]
    yield "multiply_ntts", lambda g: ["mlkem_b200_multiply_ntts_batch", n, g.inp(up(P.a12), poly), g.inp(up(P.b12), poly),
                                      g.out(up(W["mul"]), poly)]
    yield "vector_multiply", lambda g: ["mlkem_b200_vector_multiply_batch", 3, n, g.inp(up(P.u3), 3 * poly), g.inp(up(P.v3), 3 * poly),
                                        g.out(up(W["vec"]), poly)]
    yield "poly_add", lambda g: ["mlkem_b200_poly_add_batch", n, g.inp(up(P.f), poly), g.inp(up(P.g), poly), g.out(up(W["add"]), poly)]
    yield "poly_sub", lambda g: ["mlkem_b200_poly_sub_batch", n, g.inp(up(P.f), poly), g.inp(up(P.g), poly), g.out(up(W["sub"]), poly)]
    for eta in (2, 3):
        yield f"cbd{eta}", lambda g, eta=eta: ["mlkem_b200_cbd_batch", eta, n, g.inp(up(P.cbd_in[eta]), 64 * eta),
                                               g.out(up(W[f"cbd{eta}"]), poly)]
        yield f"prf_cbd{eta}", lambda g, eta=eta: ["mlkem_b200_prf_cbd_batch", eta, n, g.inp(up(P.prf_s), 32), g.inp(up(P.prf_b), 1),
                                                   g.out(up(W[f"prf{eta}"]), poly)]
    yield "sample_ntt", lambda g: ["mlkem_b200_sample_ntt_batch", n, g.inp(up(P.seeds), 34), g.out(up(W["sample"]), poly),
                                   g.out(up(W["after"]), 34, "seeds_after")]
    for d in CODEC_D:
        yield f"byte_encode{d}", lambda g, d=d: ["mlkem_b200_byte_encode_batch", d, n, g.inp(up(P.low[d]), poly), g.out(up(W[f"enc{d}"]), 32 * d)]
        yield f"byte_decode{d}", lambda g, d=d: ["mlkem_b200_byte_decode_batch", d, n, g.inp(up(P.enc_in[d]), 32 * d), g.out(up(W[f"dec{d}"]), poly)]
        yield f"compress_encode{d}", lambda g, d=d: ["mlkem_b200_compress_encode_batch", d, n, g.inp(up(P.f), poly),
                                                     g.out(up(W[f"cenc{d}"]), 32 * d)]
        yield f"decode_decompress{d}", lambda g, d=d: ["mlkem_b200_decode_decompress_batch", d, n, g.inp(up(P.enc_in[d]), 32 * d),
                                                       g.out(up(W[f"ddec{d}"]), poly)]


_prims = []


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_primitives_at_grid_stride_boundaries(lib, oracle, device):
    """ntt, intt, multiply_ntts, vector_multiply (k = 3), poly_add, poly_sub, cbd and prf_cbd (eta = 2, 3), sample_ntt with
    seeds_after and the four codec calls at d = 1, 11, 12, at 1, 7, 8, 9, 37 888, 37 889 and 75 777 polynomials: prim_grid()
    caps at 37 888 polynomials per pass, so the last three sizes take a second pass in some chunk."""
    if not _prims:
        _prims.append(Prims(oracle, PRIM_SIZES[-1]))
    P = _prims[0]
    errors = []
    for n in PRIM_SIZES:
        for name, build in prim_calls(P, n, device):
            g = Guarded(device, n)
            fname, *args = build(g)
            g.seal()
            what = f"{name} n={n} {'device' if device else 'host'}"
            rc = call(lib, fname, args, device)
            errors += [f"{what}: rc={rc}"] if rc != OK else g.check(what)
    assert not errors, "\n".join(errors[:40])


BIG_CHUNK = 1 << 21  # in 16-byte vectors: one chunk holds more than the 1 212 416 vectors one grid pass covers


def test_vector_kernels_take_a_second_pass(lib, oracle):
    """k_compress_batch and k_poly_addsub cap their grids at 1 212 416 16-byte vectors.  Default chunks never get there;
    chunks of 2^21 vectors do: compress / decompress at 8, 9 699 328 (exactly one pass) and 9 699 336 coefficients (one
    vector more), poly_add / poly_sub at 37 889 polynomials, in device memory, against the oracle."""
    import torch

    rng = np.random.default_rng(5)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()
    errors = []
    x = rng.integers(0, Q, 8 * (VECTORS_PER_PASS + 1), dtype=np.uint16)
    y = {d: rng.integers(0, 1 << d, x.size, dtype=np.uint16) for d in (1, 11)}
    for ncoef in (8, 8 * VECTORS_PER_PASS, 8 * (VECTORS_PER_PASS + 1)):
        for d in (1, 11):
            for fname, src, want in (("mlkem_b200_compress_batch", x, oracle.compress(x[:ncoef], d)),
                                     ("mlkem_b200_decompress_batch", y[d], oracle.decompress(y[d][:ncoef], d))):
                g = Guarded(True, ncoef + d)
                args = [d, ncoef, g.inp(up(src[:ncoef]), 16), g.out(up(want), 16)]
                g.seal()
                what = f"{fname} d={d} n_coeffs={ncoef}"
                rc = call(lib, fname, args, True, chunk=BIG_CHUNK)
                errors += [f"{what}: rc={rc}"] if rc != OK else g.check(what)
    n = PRIM_POLYS_PER_PASS + 1
    assert n * 32 > VECTORS_PER_PASS
    u, v = rng.integers(0, Q, (n, 256), dtype=np.uint16), rng.integers(0, Q, (n, 256), dtype=np.uint16)
    for fname, want in (("mlkem_b200_poly_add_batch", oracle.poly_add(u, v)), ("mlkem_b200_poly_sub_batch", oracle.poly_sub(u, v))):
        g = Guarded(True, 3)
        args = [n, g.inp(up(u), 512), g.inp(up(v), 512), g.out(up(want), 512)]
        g.seal()
        rc = call(lib, fname, args, True, chunk=BIG_CHUNK)
        errors += [f"{fname}: rc={rc}"] if rc != OK else g.check(f"{fname} n={n}")
    assert not errors, "\n".join(errors)


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_hash_batch_and_cell_conversion_tails(lib, oracle, device):
    """hash_batch at 127, 128 and 129 messages (one 128-thread block, and one item past it) for every `which`, at lengths
    of 8, 32, 40 and 136 bytes (three of them 8 mod 16: the chunk starts then sit 8 bytes off a 16-byte boundary); and
    cells_from_bytes / cells_to_bytes at 4, 1 020, 1 024 and 1 028 bytes."""
    import torch

    rng = np.random.default_rng(128)
    up = (lambda a: torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()) if device else \
        (lambda a: np.ascontiguousarray(a).reshape(-1).view(np.uint8))
    errors = []
    for n in (127, 128, 129):
        for which in range(4):
            for length in (8, 32, 40, 136):
                msgs = rng.integers(0, 256, (n, length), dtype=np.uint8)
                want = oracle.hash_batch(which, msgs, length) if which != 3 else np.frombuffer(
                    b"".join(hashlib.shake_256(m.tobytes()).digest(32) for m in msgs), np.uint8).reshape(n, 32).copy()
                if which == 2:
                    assert np.array_equal(want[:1], np.frombuffer(hashlib.shake_128(msgs[0].tobytes()).digest(32), np.uint8)[None])
                g = Guarded(device, n * 10 + which)
                args = [which, n, length, g.inp(up(msgs), length), g.out(up(want), want.shape[1])]
                g.seal()
                what = f"hash_batch which={which} n={n} len={length}"
                rc = call(lib, "mlkem_b200_hash_batch", args, device)
                errors += [f"{what}: rc={rc}"] if rc != OK else g.check(what)
    for nbytes in (4, 1020, 1024, 1028):
        b = rng.integers(0, 256, nbytes, dtype=np.uint8)
        cells = b.astype(np.uint32)
        junk = cells | (rng.integers(1, 1 << 24, nbytes, dtype=np.uint32) << 8)  # upper bits are ignored on input
        for fname, src, want, item in (("mlkem_b200_cells_from_bytes", b, cells, 4), ("mlkem_b200_cells_to_bytes", junk, b, 1)):
            g = Guarded(device, nbytes)
            args = [nbytes, g.inp(up(src), 4 // item), g.out(up(want), item)]
            g.seal()
            rc = call(lib, fname, args, device)
            errors += [f"{fname} {nbytes}: rc={rc}"] if rc != OK else g.check(f"{fname} {nbytes} bytes")
    assert not errors, "\n".join(errors)


# ------------------------------------------------------------------------------------------------ 5. one chunk past 4 GiB
HUGE = 1 << 21


def test_one_chunk_past_4_gib(lib, oracle):
    """ML-KEM-1024 KeyGen, Encaps and Decaps on 2^21 items in ONE chunk: the noise workspace alone is 8 GiB, so every
    per-item offset of the workspace and of the outputs passes 2^32 bytes.  The results equal, byte for byte, those of
    the default chunking (which the whole-batch tests tie to the oracle), and the last 2 048 items and 2 048 random ones
    equal the oracle.  Needs about 35 GB of device memory (computed, not measured): skipped below 48 GB free."""
    import torch

    import crystals_kyber_b200 as ck

    free, _ = torch.cuda.mem_get_info()
    if free < 48 << 30:
        pytest.skip(f"needs about 35 GB of device memory, {free / 2**30:.1f} GiB free")
    ps = 1024
    gen = torch.Generator(device="cuda")
    gen.manual_seed(21)
    d, z, m = (torch.randint(0, 256, (HUGE, 32), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(3))
    dev = torch.cuda.current_device()
    results = {}
    try:
        for label, chunk in (("default", 0), ("one chunk", HUGE)):
            gpu = ck.MLKEM(chunk_items=chunk)
            ek, dk = gpu.keygen(ps, d, z)
            c, K = gpu.encaps(ps, ek, m)
            L = c.shape[1]
            sel = torch.arange(3, HUGE, 10, device="cuda")
            ct = c.clone()
            ct[sel, (sel * 7919) % L] ^= (torch.ones_like(sel) << (sel % 8)).to(torch.uint8)
            Kd = gpu.decaps(ps, dk, ct)
            del ct
            torch.cuda.synchronize()
            results[label] = dict(ek=ek, dk=dk, c=c, K=K, Kd=Kd)
        step = 1 << 18
        for name in ("ek", "dk", "c", "K", "Kd"):
            a, b = results["default"][name], results["one chunk"][name]
            for i in range(0, HUGE, step):
                assert torch.equal(a[i:i + step], b[i:i + step]), (name, i)
        pick = np.concatenate([np.arange(HUGE - 2048, HUGE), np.random.default_rng(4).choice(HUGE - 2048, 2048, replace=False)])
        tp = torch.from_numpy(pick).cuda()
        hd, hz, hm = (t[tp].cpu().numpy() for t in (d, z, m))
        oek, odk = oracle.keygen(ps, hd, hz)
        oc, oK = oracle.encaps(ps, oek, hm)
        oKd = oracle.decaps(ps, odk, tamper_at(oc, pick))
        got = {name: results["one chunk"][name][tp].cpu().numpy() for name in ("ek", "dk", "c", "K", "Kd")}
        for name, want in (("ek", oek), ("dk", odk), ("c", oc), ("K", oK), ("Kd", oKd)):
            assert np.array_equal(got[name], want), name
    finally:
        results.clear()
        torch.cuda.synchronize()
        lib.mlkem_b200_release(dev)
        torch.cuda.empty_cache()


def tamper_at(c, index):
    """tamper() for items whose batch positions are `index`."""
    c = c.copy()
    L = c.shape[1]
    for row, i in enumerate(index):
        if i % 10 == 3:
            c[row, (i * 7919) % L] ^= 1 << (i % 8)
    return c
