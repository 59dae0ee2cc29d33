"""The device functions of mlkem_device.cuh, one at a time, across their documented input domains (-m gpu), and the
stand-alone ring entry points across theirs, against exact references.

The KEM path sees most of these functions only through Compress, which hides an error in the last bits of a coefficient
most of the time, and its callers feed them narrower inputs than their comments promise.  Here each one runs alone, through
the test-only harness tests/csrc/device_contracts.cu (`make contracts`; it #includes mlkem_device.cuh and builds its tables
with the library's own mlkem_tables.inl), on every input where that is cheap and on edge families elsewhere.

The references share no code with the kernels or the oracle: a numpy int64 NTT / InverseNTT written from FIPS 203
Algorithms 9 and 10 with its own zeta table, plain `%` for the scalars, and 64-bit `%` on the device for the sweeps too large
to copy back (all 2^32 inputs of barrett32 / canon32, 2^17 + 2^24 inputs of mul_shoup_fma times 258 table words).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "build", "libmlkem_b200_contracts.so")
Q = 3329
BIG = 1 << 20  # polynomials in each random family


# ------------------------------------------------------------------ FIPS 203 reference (numpy, int64)
def bitrev7(i):
    return int(f"{i:07b}"[::-1], 2)


ZETAS = np.array([pow(17, bitrev7(i), Q) for i in range(128)], np.int64)          # FIPS 203 Appendix A
GAMMAS = np.array([pow(17, 2 * bitrev7(i) + 1, Q) for i in range(128)], np.int64)  # FIPS 203 (4.8), Algorithm 11


def ref_ntt(f):
    """FIPS 203 Algorithm 9 on each row of f (n x 256), after reducing the input mod q; output canonical."""
    f = np.asarray(f, np.int64).reshape(-1, 256) % Q
    i, length = 1, 128
    while length >= 2:
        nb = 128 // length
        g = f.reshape(-1, nb, 2, length)  # a view: block `start / (2 len)`, halves j and j + len
        t = ZETAS[i:i + nb, None] * g[:, :, 1] % Q
        g[:, :, 1] = (g[:, :, 0] - t) % Q
        g[:, :, 0] = (g[:, :, 0] + t) % Q
        i, length = i + nb, length // 2
    return f


def ref_intt(f):
    """FIPS 203 Algorithm 10 on each row of f (n x 256), after reducing the input mod q; output canonical."""
    f = np.asarray(f, np.int64).reshape(-1, 256) % Q
    i, length = 127, 2
    while length <= 128:
        nb = 128 // length
        g = f.reshape(-1, nb, 2, length)
        z = ZETAS[i - nb + 1:i + 1][::-1, None]  # i counts down from 127, one zeta per block
        t = g[:, :, 0].copy()
        g[:, :, 0] = (t + g[:, :, 1]) % Q
        g[:, :, 1] = z * (g[:, :, 1] - t) % Q
        i, length = i - nb, length * 2
    return f * 3303 % Q


def as_matrix(fn):
    """fn (a map that is linear mod q) applied as x @ fn(I) in float64: exact, since every sum is < 256 q^2 < 2^53, and
    BLAS-fast for the 2^20-polynomial families."""
    m = fn(np.eye(256, dtype=np.int64)).astype(np.float64)
    return lambda x: ((np.asarray(x, np.int64).reshape(-1, 256) % Q).astype(np.float64) @ m % Q).astype(np.int64)


NTT_BY_MATRIX, INTT_BY_MATRIX = as_matrix(ref_ntt), as_matrix(ref_intt)


def compress_ref(x, d):
    """FIPS 203 (4.7): round(2^d x / q) mod 2^d, rounding halves up, for canonical x."""
    x = np.asarray(x, np.int64)
    return ((x << (d + 1)) + Q) // (2 * Q) % (1 << d)


# ------------------------------------------------------------------ the harness
@pytest.fixture(scope="module")
def harness():
    """The harness library; built with `make contracts` when it is missing (a failing build fails the tests)."""
    if not os.path.exists(HARNESS):
        subprocess.run(["make", "-C", ROOT, "contracts"], check=True, stdout=subprocess.DEVNULL)
    lib = C.CDLL(HARNESS)
    lib.contracts_tables.restype, lib.contracts_tables.argtypes = C.c_longlong, [C.c_void_p, C.c_size_t, C.c_void_p]
    lib.contracts_init.restype, lib.contracts_init.argtypes = C.c_int, []
    lib.contracts_transform.restype = C.c_int
    lib.contracts_transform.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.contracts_basemul.restype = C.c_int
    lib.contracts_basemul.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.contracts_scalar.restype = C.c_int
    lib.contracts_scalar.argtypes = [C.c_int, C.c_longlong, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    lib.contracts_sweep.restype = C.c_int
    lib.contracts_sweep.argtypes = [C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def harness_tables(lib):
    """TwiddleTables as a dict of (rows x 2) uint32 arrays {w, Shoup word}, and the 24 round constants as uint64."""
    tw = np.zeros(4 * 1024, np.uint32)  # > sizeof(TwiddleTables)
    rc = np.zeros(48, np.uint32)
    size = lib.contracts_tables(tw.ctypes.data, tw.nbytes, rc.ctypes.data)
    rows = {"zeta": 128, "zeta_inv_last": 2, "gamma": 128, "gamma32": 128, "zeta32": 128, "zeta_inv_last32": 2}
    assert size == 8 * sum(rows.values())
    out, at = {}, 0
    for name, n in rows.items():
        out[name] = tw[at:at + 2 * n].reshape(n, 2).astype(np.int64)
        at += 2 * n
    out["rc"] = rc[0::2].astype(np.uint64) | (rc[1::2].astype(np.uint64) << np.uint64(32))
    return out


class Device:
    """The harness's entry points on torch CUDA tensors, launched on the current stream."""

    NTT_FMA, NTT_BALANCED, NTT_EXACT, INTT_FMA_LAZY, INTT_BALANCED, ROUND_TRIP_FMA = range(6)
    BARRETT16, CANON16, CANON_FMA, COMPRESS, COMPRESS_CANON, COMPRESS_RESID, DECOMPRESS, MUL_SHOUP, NOISE_CODE, ADD_NOISE_CODE, \
        NIBBLE = range(11)
    SWEEP_BARRETT32, SWEEP_MUL_SHOUP_FMA = range(2)

    def __init__(self, lib):
        import torch

        self.torch, self.lib = torch, lib
        assert lib.contracts_init() == 0

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def _dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def transform(self, which, x):
        t = self._dev(np.asarray(x, np.uint16).reshape(-1, 256))
        out = self.torch.empty_like(t)
        assert self.lib.contracts_transform(which, t.shape[0], t.data_ptr(), out.data_ptr(), self._stream()) == 0
        return out.cpu().numpy()

    def basemul(self, a, b):
        """a, b: n x k x 256.  Returns (raw, barrett32, canon32), each n x 256 int64."""
        n, k, _ = a.shape
        ta, tb = self._dev(a.astype(np.uint16)), self._dev(b.astype(np.uint16))
        out = self.torch.empty((n, 3, 256), dtype=self.torch.int32, device="cuda")
        assert self.lib.contracts_basemul(n, k, ta.data_ptr(), tb.data_ptr(), out.data_ptr(), self._stream()) == 0
        o = out.cpu().numpy().view(np.uint32).astype(np.int64)
        return o[:, 0], o[:, 1], o[:, 2]

    def scalar(self, op, x, y0=0, ny=1):
        """op(x_i, y0 + j) as an ny x len(x) int64 array; x an int (range(x)) or an array."""
        if isinstance(x, int):
            nx, xs = x, None
        else:
            xs = self._dev(np.asarray(x, np.uint32).view(np.int32))
            nx = xs.numel()
        out = self.torch.empty(nx * ny, dtype=self.torch.int32, device="cuda")
        ptr = None if xs is None else xs.data_ptr()
        assert self.lib.contracts_scalar(op, nx, ptr, y0, ny, out.data_ptr(), self._stream()) == 0
        return out.cpu().numpy().view(np.uint32).astype(np.int64).reshape(ny, nx)

    def sweep(self, op, a=None):
        """(failures, first failing index) of a device-side check."""
        res = self._dev(np.array([0, -1], np.int64))  # {failures, first failing index = ~0}
        ta = None if a is None else self._dev(np.asarray(a, np.uint32).view(np.int32))
        n = 0 if ta is None else ta.numel()
        assert self.lib.contracts_sweep(op, n, None if ta is None else ta.data_ptr(), res.data_ptr(), self._stream()) == 0
        r = res.cpu().numpy().view(np.uint64)
        return int(r[0]), int(r[1])


@pytest.fixture(scope="module")
def dev(harness):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return Device(harness)


@pytest.fixture(scope="module")
def mlkem():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import crystals_kyber_b200 as ck

    return ck.MLKEM()


# ------------------------------------------------------------------ input families of the transforms
FAMILIES = ["zero", "all bound-1 / all q-1", "every constant", "spikes", "uniform", "edge values"]


def family(name, bound):
    """Polynomials (uint16, n x 256) of one input family, every coefficient below `bound`."""
    rng = np.random.default_rng([bound, FAMILIES.index(name) if name in FAMILIES else 99])
    edges = [v for v in (1, Q - 1, Q, 2 * Q - 1, bound - 1) if v < bound]
    if name == "zero":
        x = np.zeros((1, 256), np.uint16)
    elif name == "all bound-1 / all q-1":
        x = np.stack([np.full(256, bound - 1), np.full(256, Q - 1)]).astype(np.uint16)
    elif name == "every constant":
        x = np.repeat(np.arange(bound, dtype=np.uint16)[:, None], 256, axis=1)
    elif name == "spikes":  # v e_i for every position i
        x = np.concatenate([v * np.eye(256, dtype=np.uint16) for v in edges])
    elif name == "uniform":
        x = rng.integers(0, bound, (BIG, 256), dtype=np.uint16)
    elif name == "edge values":
        x = np.array([0] + edges, np.uint16)[rng.integers(0, len(edges) + 1, (BIG, 256))]
    else:  # "noise residues": what k_noise hands ntt_warp<kFmaPipe>, CBD samples as the residues q-3 .. q+3
        x = rng.integers(Q - 3, Q + 4, (1 << 16, 256), dtype=np.uint16)
    assert int(x.max(initial=0)) < bound
    return x


def mismatch(name, family, got, want, exact=False, below=None, first=0):
    """Message for the first coefficient where got is not congruent to want (equal to it when exact) or not below `below`;
    `first` is the index of got's first polynomial in the family."""
    got = got.astype(np.int64)
    bad = got != want if exact else got % Q != want
    if below is not None:
        bad |= got >= below
    if not bad.any():
        return None
    p, c = np.argwhere(bad)[0]
    rule = "equal" if exact else "congruent" + (f", below {below}" if below else "")
    return (f"{name} on '{family}': {int(bad.sum())} coefficients wrong; first: polynomial {first + p} coefficient {c}: "
            f"got {got[p, c]}, want {want[p, c]} ({rule})")


CHUNK = 1 << 15


@pytest.mark.gpu
@pytest.mark.parametrize("fam", FAMILIES + ["noise residues"])
def test_forward_transforms(dev, oracle, fam):
    """ntt_warp<kFmaPipe>, ntt_warp<kBalanced>: inputs < 4096 taken as residues, output canonical.  ntt_warp_exact: the
    reference's literal result (oracle.ntt) on [0, 4096).  ntt_warp<kFmaPipe> -> intt_warp<kFmaPipe, false>: the input
    back, in [0, 2q)."""
    x = family(fam, 4096)
    got = {name: dev.transform(which, x) for name, which in (("ntt_warp<kFmaPipe>", dev.NTT_FMA), ("ntt_warp<kBalanced>", dev.NTT_BALANCED),
                                                             ("ntt_warp_exact", dev.NTT_EXACT), ("round trip (kFmaPipe)", dev.ROUND_TRIP_FMA))}
    errors = []
    for s in range(0, len(x), CHUNK):
        xc = x[s:s + CHUNK]
        want = NTT_BY_MATRIX(xc)
        for name in ("ntt_warp<kFmaPipe>", "ntt_warp<kBalanced>"):
            errors.append(mismatch(name, fam, got[name][s:s + CHUNK], want, below=Q, first=s))
        errors.append(mismatch("ntt_warp_exact", fam, got["ntt_warp_exact"][s:s + CHUNK], oracle.ntt(xc).astype(np.int64), exact=True, first=s))
        errors.append(mismatch("round trip (kFmaPipe)", fam, got["round trip (kFmaPipe)"][s:s + CHUNK], xc.astype(np.int64) % Q, below=2 * Q,
                               first=s))
    errors = [e for e in errors if e]
    assert not errors, "\n".join(errors[:8])


@pytest.mark.gpu
@pytest.mark.parametrize("fam", FAMILIES)
def test_inverse_transforms(dev, fam):
    """intt_warp<kBalanced, true> on inputs < 4096 -> canonical; intt_warp<kFmaPipe, false> on inputs < 8192 -> [0, 2q),
    the whole domain its comment promises (the KEM path only feeds it values < 2q)."""
    errors = []
    for name, which, bound, below in (("intt_warp<kBalanced, true>", dev.INTT_BALANCED, 4096, Q),
                                      ("intt_warp<kFmaPipe, false>", dev.INTT_FMA_LAZY, 8192, 2 * Q)):
        x = family(fam, bound)
        got = dev.transform(which, x)
        for s in range(0, len(x), CHUNK):
            errors.append(mismatch(name, fam, got[s:s + CHUNK], INTT_BY_MATRIX(x[s:s + CHUNK]), below=below, first=s))
    errors = [e for e in errors if e]
    assert not errors, "\n".join(errors[:8])


# ------------------------------------------------------------------ base-case products
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_basemul_acc_accumulators(dev, harness, k):
    """basemul_acc summed over k rows (what matvec_row_tail, k_encrypt_v and k_decrypt accumulate): the 32-bit accumulator
    equals the exact integer sum -- no wrap even for all-4095 operands (the 0xFF key) -- and barrett32 / canon32 of it meet
    their ranges."""
    g32 = harness_tables(harness)["gamma32"]
    rng = np.random.default_rng(k)
    n = 2048
    cases = {
        "all 4095 x all q-1": (np.full((1, k, 256), 4095), np.full((1, k, 256), Q - 1)),
        "all 4095 x all 4095": (np.full((1, k, 256), 4095), np.full((1, k, 256), 4095)),
        "random 12-bit": (rng.integers(0, 4096, (n, k, 256)), rng.integers(0, 4096, (n, k, 256))),
    }
    for case, (a, b) in cases.items():
        raw, bar, can = dev.basemul(a, b)
        a, b = a.astype(np.int64), b.astype(np.int64)
        a0, a1, b0, b1 = a[..., 0::2], a[..., 1::2], b[..., 0::2], b[..., 1::2]
        # the kernel's a1 gamma: mul_shoup_fma(a1, gamma32), a representative below 2q (its range is checked in
        # test_mul_shoup_fma_domain); with it the accumulation is plain integer arithmetic
        w, w32 = g32[:, 0], g32[:, 1]
        a1g = a1 * w - ((a1 * w32) >> 32) * Q
        assert (a1g >= 0).all() and (a1g < 2 * Q).all() and (a1g % Q == a1 * GAMMAS % Q).all()
        exact = np.empty(raw.shape, np.int64)
        exact[:, 0::2] = (a0 * b0 + a1g * b1).sum(axis=1)
        exact[:, 1::2] = (a0 * b1 + a1 * b0).sum(axis=1)
        math = np.empty(raw.shape, np.int64)  # BaseCaseMultiply (FIPS 203 Algorithm 12), summed
        math[:, 0::2] = (a0 * b0 + a1 * b1 % Q * GAMMAS).sum(axis=1) % Q
        math[:, 1::2] = (a0 * b1 + a1 * b0).sum(axis=1) % Q
        assert exact.max() < 2**32
        assert (raw == exact).all(), f"{case}, k={k}: raw accumulator differs from the exact sum"
        assert (exact % Q == math).all()
        assert (bar < 2 * Q).all() and (bar % Q == math).all(), f"{case}, k={k}: barrett32"
        assert (can == math).all(), f"{case}, k={k}: canon32"


# ------------------------------------------------------------------ scalars on their whole domains
@pytest.mark.gpu
def test_reductions_on_their_domains(dev):
    """barrett16 / canon16 on every x < 2^16, canon_fma on every x < 2^21, barrett32 / canon32 on all 2^32 inputs."""
    x = np.arange(1 << 16, dtype=np.int64)
    b16 = dev.scalar(dev.BARRETT16, 1 << 16)[0]
    assert (b16 % Q == x % Q).all() and (b16 <= Q + 1).all()
    assert np.flatnonzero(b16 == Q + 1).tolist() == [56594, 59923, 63252]  # the only results above q
    assert (dev.scalar(dev.CANON16, 1 << 16)[0] == x % Q).all()
    x21 = np.arange(1 << 21, dtype=np.int64)
    assert (dev.scalar(dev.CANON_FMA, 1 << 21)[0] == x21 % Q).all()
    assert dev.sweep(dev.SWEEP_BARRETT32) == (0, 2**64 - 1)


@pytest.mark.gpu
def test_mul_shoup_domain(dev, harness):
    """mul_shoup on every a < 2^16 with each of the 130 words of the balanced table (zeta, zeta_inv_last): congruent, < 2q."""
    t = harness_tables(harness)
    w = np.concatenate([t["zeta"][:, 0], t["zeta_inv_last"][:, 0]])
    got = dev.scalar(dev.MUL_SHOUP, 1 << 16, 0, 130)
    a = np.arange(1 << 16, dtype=np.int64)
    bad = (got >= 2 * Q) | (got % Q != a[None, :] * w[:, None] % Q)
    assert not bad.any(), "word %d, a = %d" % tuple(np.argwhere(bad)[0])


@pytest.mark.gpu
def test_mul_shoup_fma_domain(dev):
    """mul_shoup_fma on every a < 2^17 and 2^24 random 32-bit a, with each of the 258 words of the FMA tables (zeta32,
    gamma32, zeta_inv_last32): congruent and < 2q, checked on the device against 64-bit arithmetic."""
    rng = np.random.default_rng(258)
    a = np.concatenate([np.arange(1 << 17, dtype=np.uint32), rng.integers(0, 1 << 32, 1 << 24, dtype=np.uint32)])
    bad, first = dev.sweep(dev.SWEEP_MUL_SHOUP_FMA, a)
    assert bad == 0, f"{bad} failures; first: a = {a[first % len(a)]}, word {first // len(a)}"


@pytest.mark.gpu
def test_compress_decompress_domains(dev, oracle):
    """compress<D> on every x < 4096 (the reference's Compress, any 12-bit x), compress_canon<D> on every x < q and
    compress_resid<D> on every x < 4q (Compress of x mod q), decompress<D> on every y < 2^D."""
    x = np.arange(4096)
    got = dev.scalar(dev.COMPRESS, 4096, 1, 11)
    for d in range(1, 12):
        assert (got[d - 1] == oracle.compress(x, d)).all(), f"compress<{d}>"
        assert (got[d - 1, :Q] == compress_ref(x[:Q], d)).all(), f"compress<{d}>"
    for d in (1, 4, 5, 10, 11):
        assert (dev.scalar(dev.COMPRESS_CANON, Q, d)[0] == compress_ref(np.arange(Q), d)).all(), f"compress_canon<{d}>"
    for d in (1, 4, 5):
        assert (dev.scalar(dev.COMPRESS_RESID, 4 * Q, d)[0] == compress_ref(np.arange(4 * Q) % Q, d)).all(), f"compress_resid<{d}>"
    for d in range(1, 12):
        y = np.arange(1 << d)
        got = dev.scalar(dev.DECOMPRESS, 1 << d, d)[0]
        assert (got == oracle.decompress(y, d)).all(), f"decompress<{d}>"
        assert (got == (Q * y * 2 + (1 << d)) // (1 << (d + 1))).all(), f"decompress<{d}>"  # round(q y / 2^d), halves up


@pytest.mark.gpu
def test_noise_codes_and_nibbles(dev):
    """noise_code_to_coeff on every code 0..6, add_noise_code on every (canonical x, code), nibble_fma at every position
    with every nibble value."""
    assert (dev.scalar(dev.NOISE_CODE, 7)[0] == (np.arange(7) - 3) % Q).all()
    got = dev.scalar(dev.ADD_NOISE_CODE, Q, 0, 7)
    assert (got == (np.arange(Q)[None, :] + np.arange(7)[:, None] - 3) % Q).all()
    rng = np.random.default_rng(4)
    w = rng.integers(0, 1 << 32, 1 << 16, dtype=np.uint64)
    for j in range(8):  # every value at every nibble, under random neighbours
        ww = (w[:4096] & ~np.uint64(15 << (4 * j))) | (np.arange(4096, dtype=np.uint64) % np.uint64(16)) << np.uint64(4 * j)
        w = np.concatenate([w, ww])
    got = dev.scalar(dev.NIBBLE, w, 0, 8)
    want = np.stack([(w >> np.uint64(4 * j)) & np.uint64(15) for j in range(8)]).astype(np.int64)
    assert (got == want).all()


# ------------------------------------------------------------------ the stand-alone ABI on its documented domains
def both_memories(fn, *arrays):
    """fn on host arrays and on torch CUDA tensors; both results as numpy."""
    import torch

    host = fn(*arrays)
    devr = fn(*[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]).cpu().numpy()
    return host, devr


@pytest.mark.gpu
def test_intt_batch_takes_residues(mlkem, oracle):
    """mlkem_b200_intt_batch: any 12-bit coefficients are residues mod q and the output is canonical; where the reference's
    arithmetic is defined (every first-layer pair has f[j] - f[j+2] <= q), the result is the reference's bit for bit."""
    rng = np.random.default_rng(336)
    f = np.concatenate([rng.integers(0, 4096, (1 << 16, 256), dtype=np.uint16), np.full((1, 256), 4095, np.uint16)])
    want = INTT_BY_MATRIX(f)
    for got in both_memories(mlkem.intt, f):
        assert mismatch("intt_batch", "12-bit", got, want, exact=True) is None
    # defined for the reference: f[j] <= f[j+2] + q in each (j, j+2) pair of the first layer
    g = rng.integers(0, 4096, (1 << 14, 256)).reshape(-1, 64, 2, 2)
    g[:, :, 0] = rng.integers(0, np.minimum(4096, g[:, :, 1] + Q + 1))
    g = g.reshape(-1, 256).astype(np.uint16)
    pairs = g.reshape(-1, 64, 2, 2)
    assert (g >= Q).mean() > 0.1 and ((pairs[:, :, 0] >= Q) & (pairs[:, :, 0] > pairs[:, :, 1])).any()
    assert (pairs[:, :, 0].astype(np.int64) - pairs[:, :, 1] <= Q).all()
    want = oracle.intt(g)
    assert (want == ref_intt(g)).all()
    for got in both_memories(mlkem.intt, g):
        assert mismatch("intt_batch", "reference-defined 12-bit", got, want.astype(np.int64), exact=True) is None


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(1, 17))
def test_vector_multiply_every_k(mlkem, oracle, k):
    """mlkem_b200_vector_multiply_batch for every 1 <= k <= 16: all-4095 u against all-3328 v (the largest sums the final
    canon16 sees, 16 * 3328 at k = 16) and random 12-bit operands, against the oracle."""
    rng = np.random.default_rng(618 + k)
    u = np.concatenate([np.full((1, k, 256), 4095), rng.integers(0, 4096, (255, k, 256))]).astype(np.uint16)
    v = np.concatenate([np.full((1, k, 256), Q - 1), rng.integers(0, 4096, (255, k, 256))]).astype(np.uint16)
    want = oracle.vector_multiply(u, v, k)
    for got in both_memories(lambda a, b: mlkem.vector_multiply(a, b, k), u, v):
        assert (got == want).all()


@pytest.mark.gpu
def test_poly_add_sub_every_pair(mlkem, oracle):
    """mlkem_b200_poly_add_batch / _poly_sub_batch on all 2^24 pairs of 12-bit coefficients."""
    u = np.repeat(np.arange(4096, dtype=np.uint16), 4096).reshape(-1, 256)
    v = np.tile(np.arange(4096, dtype=np.uint16), 4096).reshape(-1, 256)
    for fn, want in ((mlkem.poly_add, oracle.poly_add(u, v)), (mlkem.poly_sub, oracle.poly_sub(u, v))):
        for got in both_memories(fn, u, v):
            assert (got == want).all()


@pytest.mark.gpu
def test_multiply_ntts_every_constant_term_and_extreme_pairs(mlkem, oracle):
    """mlkem_b200_multiply_ntts_batch on every (a0, b0) in [0, 4096)^2 with a1 = b1 = 0, and on every combination of
    extreme values of (a0, a1, b0, b1) at each of the 128 gamma positions."""
    a0 = np.repeat(np.arange(4096, dtype=np.uint16), 4096)
    b0 = np.tile(np.arange(4096, dtype=np.uint16), 4096)
    f = np.stack([a0, np.zeros_like(a0)], axis=1).reshape(-1, 256)
    g = np.stack([b0, np.zeros_like(b0)], axis=1).reshape(-1, 256)
    want = oracle.multiply_ntts(f, g)
    assert (want[:, 0::2] == (a0.astype(np.int64) * b0 % Q).reshape(-1, 128)).all()
    for got in both_memories(mlkem.multiply_ntts, f, g):
        assert (got == want).all()
    ext = np.array([0, 1, Q - 1, Q, 4095], np.uint16)
    combos = np.stack(np.meshgrid(ext, ext, ext, ext, indexing="ij"), -1).reshape(-1, 4)  # (a0, a1, b0, b1)
    f = np.tile(combos[:, None, 0:2], (1, 128, 1)).reshape(-1, 256)
    g = np.tile(combos[:, None, 2:4], (1, 128, 1)).reshape(-1, 256)
    want = oracle.multiply_ntts(f, g)
    for got in both_memories(mlkem.multiply_ntts, f, g):
        assert (got == want).all()


# ------------------------------------------------------------------ CPU: the references and the harness's tables
def test_reference_transforms_match_the_oracle(oracle):
    """The numpy FIPS 203 transforms equal the oracle's on canonical inputs, and invert each other."""
    rng = np.random.default_rng(9)
    f = np.concatenate([rng.integers(0, Q, (2048, 256)), np.full((1, 256), Q - 1), np.eye(256, dtype=np.int64) * (Q - 1)]).astype(np.uint16)
    assert (ref_ntt(f) == oracle.ntt(f)).all()
    assert (ref_intt(f) == oracle.intt(f)).all()
    assert (ref_intt(ref_ntt(f)) == f).all()
    assert (ref_ntt(f + Q) == ref_ntt(f)).all()  # residue semantics
    g = np.concatenate([f, rng.integers(0, 8192, (2048, 256)).astype(np.uint16)])
    assert (NTT_BY_MATRIX(g) == ref_ntt(g)).all() and (INTT_BY_MATRIX(g) == ref_intt(g)).all()


def test_harness_tables_match_fips(harness):
    """The tables the harness (and the library, through the same mlkem_tables.inl) builds: zeta, gamma, both Shoup words,
    both inverse-last entries, and the Keccak round constants recomputed with the FIPS 202 LFSR (Algorithms 5 and 6)."""
    t = harness_tables(harness)
    sh16 = lambda w: (w << 16) // Q
    sh32 = lambda w: (w << 32) // Q
    assert (t["zeta"][:, 0] == ZETAS).all() and (t["zeta"][:, 1] == sh16(ZETAS)).all()
    assert (t["zeta32"][:, 0] == ZETAS).all() and (t["zeta32"][:, 1] == sh32(ZETAS)).all()
    assert (t["gamma"][:, 0] == GAMMAS).all() and (t["gamma"][:, 1] == sh16(GAMMAS)).all()
    assert (t["gamma32"][:, 0] == GAMMAS).all() and (t["gamma32"][:, 1] == sh32(GAMMAS)).all()
    inv_last = np.array([ZETAS[1] * 3303 % Q, 3303], np.int64)  # 3303 = 128^-1 mod q folded into the last layer
    assert pow(128, -1, Q) == 3303
    assert (t["zeta_inv_last"][:, 0] == inv_last).all() and (t["zeta_inv_last"][:, 1] == sh16(inv_last)).all()
    assert (t["zeta_inv_last32"][:, 0] == inv_last).all() and (t["zeta_inv_last32"][:, 1] == sh32(inv_last)).all()

    def rc_bit(tt):  # FIPS 202 Algorithm 5
        if tt % 255 == 0:
            return 1
        r = [1, 0, 0, 0, 0, 0, 0, 0]
        for _ in range(tt % 255):
            r = [0] + r
            r[0] ^= r[8]
            r[4] ^= r[8]
            r[5] ^= r[8]
            r[6] ^= r[8]
            r = r[:8]
        return r[0]

    rcs = [sum(rc_bit(j + 7 * ir) << ((1 << j) - 1) for j in range(7)) for ir in range(24)]  # Algorithm 6
    assert rcs[0] == 1 and rcs[23] == 0x8000000080008008
    assert t["rc"].tolist() == rcs
