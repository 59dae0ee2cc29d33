"""The field, point and scalar functions of p256_device.cuh, one at a time, at their documented input bounds and on 2^20 random
inputs within them, against Python integers (-m gpu).

A carry slip in a 256-bit chain shows up about once in 2^32 random inputs, so random values alone are not enough: every
function also runs on the values where its final subtraction changes its mind (p - 1, p, p + 1, 2^256 - 1, the Montgomery
images of 0, 1 and -1) and with operands at the top of their accepted range.  The harness tests/csrc/p256_contracts.cu
(`make contracts`) #includes p256_device.cuh unchanged.

Bounds (p256_device.cuh): field elements are 8 little-endian words in [0, p), Montgomery domain (x R mod p, R = 2^256).
fe_add / fe_sub / fe_sqr / fe_inv / fe_from_mont: [0, p) -> [0, p); fe_mul: a < 2^256 when b < p -> [0, p); fe_canon /
fe_to_mont: any 256-bit value -> [0, p).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_secp256r1mlkem768_cpu import GX, GY, N, P, add, decode, encode, invalid_points, mul, seed_scalar, small_x_point

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "build", "libp256_contracts.so")
R = 2 ** 256
RINV = pow(R, -1, P)
(ADD, SUB, MUL, SQR, CANON, INV, TO_MONT, FROM_MONT, PT_ADD, PT_DBL, SEED, SCALAR_OK, DECODE, MUL_POINT) = range(14)
RANDOM = 1 << 20


def run_with(lib, device):
    """run(op, a, b, out_words): a, b are (n, words) uint32 arrays; returns the (n, out_words) uint32 output."""

    def run(op, a, b=None, ow=8):
        a = np.ascontiguousarray(a, np.uint32)
        b = a if b is None else np.ascontiguousarray(b, np.uint32)
        n = a.shape[0]
        if device:
            import torch

            ta, tb = torch.from_numpy(a.view(np.int32)).cuda(), torch.from_numpy(b.view(np.int32)).cuda()
            out = torch.empty((n, ow), dtype=torch.int32, device="cuda")
            s = torch.cuda.current_stream()
            assert lib.p256_op(op, n, ta.data_ptr(), a.shape[1], tb.data_ptr(), b.shape[1], out.data_ptr(), ow, C.c_void_p(s.cuda_stream)) == 0
            return out.cpu().numpy().view(np.uint32)
        out = np.empty((n, ow), np.uint32)
        assert lib.p256_op(op, n, a.ctypes.data, a.shape[1], b.ctypes.data, b.shape[1], out.ctypes.data, ow, None) == 0
        return out

    return run


def load(path):
    lib = C.CDLL(path)
    lib.p256_op.restype = C.c_int
    lib.p256_op.argtypes = [C.c_int, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def run():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if not os.path.exists(HARNESS):
        subprocess.run(["make", "-C", ROOT, "contracts"], check=True, stdout=subprocess.DEVNULL)
    return run_with(load(HARNESS), True)


def rows(vals, width=32):
    """Python integers -> (n, width / 4) little-endian uint32 rows."""
    return np.frombuffer(b"".join(v.to_bytes(width, "little") for v in vals), "<u4").reshape(len(vals), width // 4).copy()


def ints(arr, words=8, first=0):
    return [int.from_bytes(r[first:first + words].tobytes(), "little") for r in np.asarray(arr, np.uint32)]


def be_rows(chunks, width):
    """Byte strings -> uint32 rows holding the bytes in memory order (zero padded to whole words)."""
    pad = -width % 4
    return np.frombuffer(b"".join(c + bytes(pad) for c in chunks), np.uint32).reshape(len(chunks), (width + pad) // 4).copy()


EDGE_FE = [0, 1, 2, 3, P - 3, P - 2, P - 1, R % P, (P - 1) * R % P, RINV, 2 ** 255, 2 ** 224, 2 ** 192 - 1, 2 ** 96, 2 ** 32 - 1, 2 ** 32,
           P - 2 ** 32, P - 2 ** 224]
EDGE_WIDE = EDGE_FE + [P, P + 1, P + 2, 2 ** 256 - 1, 2 ** 256 - 2, 2 ** 256 - 2 ** 224, 2 ** 256 - 2 ** 32]


def random_fe(n, seed, bound=P):
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64).astype(np.uint32)
    vals = ints(raw)
    return [v % bound for v in vals]


def pair_inputs(left, right, seed, lbound=P, rbound=P):
    a = [x for x in left for _ in right] + random_fe(RANDOM, seed, lbound)
    b = [y for _ in left for y in right] + random_fe(RANDOM, seed + 1, rbound)
    return a, b


def check_fe(out, want):
    got = ints(out)
    assert all(g < P for g in got), "output outside [0, p)"
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, f"{len(bad)} mismatches, first at row {bad[0]}"


@pytest.mark.parametrize("op", [ADD, SUB])
def test_add_sub(run, op):
    a, b = pair_inputs(EDGE_FE, EDGE_FE, 10 + op)
    out = run(op, rows(a), rows(b))
    check_fe(out, [(x + y) % P if op == ADD else (x - y) % P for x, y in zip(a, b)])


def test_mul_one_operand_wide(run):
    """fe_mul(a, b) with a anywhere in [0, 2^256) and b in [0, p): a b R^-1 mod p."""
    a, b = pair_inputs(EDGE_WIDE, EDGE_FE, 20, lbound=R)
    check_fe(run(MUL, rows(a), rows(b)), [x * y * RINV % P for x, y in zip(a, b)])
    check_fe(run(MUL, rows(b), rows(a)), [x * y * RINV % P for x, y in zip(a, b)])  # the wide operand second


def test_sqr(run):
    a = EDGE_FE + random_fe(RANDOM, 30)
    check_fe(run(SQR, rows(a)), [x * x * RINV % P for x in a])


@pytest.mark.parametrize("op", [CANON, TO_MONT])
def test_wide_inputs(run, op):
    a = EDGE_WIDE + random_fe(RANDOM, 40 + op, R) + [2 ** 256 - 1 - i for i in range(4096)] + [P + i for i in range(-2048, 2048)]
    check_fe(run(op, rows(a)), [x % P if op == CANON else x * R % P for x in a])


def test_canon_named_values(run):
    got = ints(run(CANON, rows([P - 1, P, P + 1, 2 ** 256 - 1])))
    assert got == [P - 1, 0, 1, 2 ** 256 - 1 - P]


def test_from_mont(run):
    a = EDGE_FE + random_fe(RANDOM, 50)
    check_fe(run(FROM_MONT, rows(a)), [x * RINV % P for x in a])


def test_inv(run):
    """In the Montgomery domain: A = a R -> a^-1 R; 0 -> 0."""
    a = EDGE_FE + random_fe(1 << 14, 60)  # 255 squarings per item: a smaller random set
    want = [pow(x * RINV % P, P - 2, P) * R % P for x in a]
    check_fe(run(INV, rows(a)), want)


# ------------------------------------------------------------------ points
def small_multiples(k):
    """[None, G, 2G, ..., kG] by repeated addition."""
    out, acc = [None], None
    for _ in range(k):
        acc = add(acc, (GX, GY))
        out.append(acc)
    return out


def projective(pts, zs):
    """Montgomery-domain projective rows (24 words) of affine points (None = the identity (0 : 1 : 0)) with the given Z."""
    vals = []
    for pt, z in zip(pts, zs):
        if pt is None:
            vals += [0, R % P, 0]
        else:
            vals += [pt[0] * z * R % P, pt[1] * z * R % P, z * R % P]
    return rows(vals).reshape(len(pts), 24)


def check_points(out, want):
    X, Y, Z = ints(out, 8, 0), ints(out, 8, 8), ints(out, 8, 16)
    bad = []
    for i, w in enumerate(want):
        if max(X[i], Y[i], Z[i]) >= P:
            bad.append(i)
        elif w is None:
            if Z[i] != 0 or X[i] != 0 or Y[i] == 0:
                bad.append(i)
        elif Z[i] == 0 or (X[i] - w[0] * Z[i]) % P or (Y[i] - w[1] * Z[i]) % P:
            bad.append(i)
    assert not bad, f"{len(bad)} mismatches, first at row {bad[0]}"


def test_point_add_and_double(run):
    """Complete formulas: random projective representatives of iG + jG, with the identity on either side, P = Q and P = -Q."""
    k = 64
    mults = small_multiples(2 * k)
    neg = lambda pt: None if pt is None else (pt[0], (-pt[1]) % P)
    rng = np.random.default_rng(70)
    i = rng.integers(0, k + 1, RANDOM)
    j = rng.integers(0, k + 1, RANDOM)
    zs = random_fe(2 * RANDOM, 71)
    zs = [z or 1 for z in zs]
    p1 = [mults[x] for x in i]
    p2 = [mults[y] for y in j]
    special = [(None, None), (None, mults[1]), (mults[1], None), (mults[5], mults[5]), (mults[7], neg(mults[7])),
               (neg(mults[3]), mults[3]), (mults[k], mults[k])]
    p1 += [s[0] for s in special]
    p2 += [s[1] for s in special]
    zs += [1, P - 1] * len(special)
    a, b = projective(p1, zs[0::2]), projective(p2, zs[1::2])
    check_points(run(PT_ADD, a, b, 24), [add(x, y) for x, y in zip(p1, p2)])
    check_points(run(PT_DBL, a, None, 24), [add(x, x) for x in p1])


def test_scalarmult(run):
    rng = np.random.default_rng(80)
    ks = [0, 1, 2, 3, N - 1, N, N + 1, 2 ** 256 - 1] + [int.from_bytes(bytes(rng.integers(0, 256, 32, dtype=np.uint8)), "big") for _ in range(24)]
    base = [(GX, GY)] * 8 + [mul(5)] * 24
    got = run(MUL_POINT, rows(ks), projective(base, [1] * len(ks)), 24)
    check_points(got, [mul(k % N, b) for k, b in zip(ks, base)])


# ------------------------------------------------------------------ scalars and encodings
def test_seed_scalar(run):
    cs = [0, 1, N - 2, N - 1, N, 2 * (N - 1) - 1, 2 * (N - 1), (N - 1) << 64, ((N - 1) << 64) - 1, 2 ** 256 - 1, (2 ** 256 - 1) << 64,
          2 ** 320 - 1]
    rng = np.random.default_rng(90)
    cs += [int.from_bytes(r.tobytes(), "big") for r in rng.integers(0, 256, (RANDOM, 40), dtype=np.uint8)]
    raw = [c.to_bytes(40, "big") for c in cs]
    got = ints(run(SEED, be_rows(raw, 40)))
    want = [int.from_bytes(seed_scalar(r), "big") for r in raw]
    assert want[:4] == [1, 2, N - 1, 1]
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, f"{len(bad)} mismatches, first at row {bad[0]}"


def test_scalar_range(run):
    ks = [0, 1, 2, N - 2, N - 1, N, N + 1, 2 ** 256 - 1, 2 ** 255, N - 2 ** 32, N + 2 ** 32]
    got = run(SCALAR_OK, rows(ks), None, 1)[:, 0].tolist()
    assert got == [0xFFFFFFFF if 1 <= k < N else 0 for k in ks]


def test_point_decode(run):
    x0, y0 = small_x_point()
    valid = [encode((GX, GY)), encode(mul(2)), encode(mul(N - 1)), encode((x0, y0)), encode((x0, (-y0) % P))]
    pts = valid + [b for _, b in invalid_points()]
    got = run(DECODE, be_rows(pts, 65), None, 25)
    assert got[:, 0].tolist() == [0xFFFFFFFF if decode(b) else 0 for b in pts]
    for i, b in enumerate(valid):
        pt = decode(b)
        assert ints(got[i:i + 1], 8, 1)[0] == pt[0] * R % P and ints(got[i:i + 1], 8, 9)[0] == pt[1] * R % P
        assert ints(got[i:i + 1], 8, 17)[0] == R % P
