"""The field arithmetic of x25519_device.cuh, one function at a time, at its documented limb bounds and on 2^20 random inputs within
them, against Python integers (-m gpu).

A carry-propagation slip shows up about once in 2^30 random inputs, so random values alone are not enough: every function is
also run with every limb at the maximum its comment allows, and on the values around p and 2^255 where the final reduction
changes its mind.  The harness tests/csrc/x25519_contracts.cu (`make contracts`) #includes x25519_device.cuh unchanged.

Bounds (x25519_device.cuh): T_i = 2^26 (i even) / 2^25 (i odd).  tight: limb_i < T_i, limb_1 < 2^25 + 2^18.  loose: limb_i <
3 T_i + 2^18.  fe_add / fe_sub: tight -> loose; fe_mul / fe_sq / fe_mul121665 / fe_carry: loose -> tight; fe_freeze: loose ->
the canonical value in [0, p).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "build", "libx25519_contracts.so")
P = 2 ** 255 - 19
OFF = [(51 * i + 1) // 2 for i in range(10)]  # ceil(25.5 i)
T = np.array([1 << (26 if i % 2 == 0 else 25) for i in range(10)], np.int64)
TIGHT = T.copy()
TIGHT[1] += 1 << 18
LOOSE = 3 * T + (1 << 18)
ADD, SUB, MUL, SQ, MUL121665, FREEZE, CARRY = range(7)
RANDOM = 1 << 20


@pytest.fixture(scope="module")
def field():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if not os.path.exists(HARNESS):
        subprocess.run(["make", "-C", ROOT, "contracts"], check=True, stdout=subprocess.DEVNULL)
    lib = C.CDLL(HARNESS)
    lib.x25519_contracts_field.restype = C.c_int
    lib.x25519_contracts_field.argtypes = [C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]

    def run(op, a, b=None):
        a = np.ascontiguousarray(a, np.uint32).reshape(-1, 10)
        b = a if b is None else np.ascontiguousarray(b, np.uint32).reshape(-1, 10)
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        out = torch.empty((a.shape[0], 8 if op == FREEZE else 10), dtype=torch.int32, device="cuda")
        s = torch.cuda.current_stream()
        assert lib.x25519_contracts_field(op, a.shape[0], ta.data_ptr(), tb.data_ptr(), out.data_ptr(), C.c_void_p(s.cuda_stream)) == 0
        return out.cpu().numpy().view(np.uint32)

    return run


def value(limbs):
    """Python integers (object array) of n x 10 limbs."""
    limbs = np.asarray(limbs, np.uint64).reshape(-1, 10)
    v = np.zeros(limbs.shape[0], object)
    for i in range(10):
        v = v + (limbs[:, i].astype(object) << OFF[i])
    return v


def words_value(words):
    words = np.asarray(words, np.uint64).reshape(-1, 8)
    v = np.zeros(words.shape[0], object)
    for i in range(8):
        v = v + (words[:, i].astype(object) << (32 * i))
    return v


def limbs_of(x):
    """The exact split of 0 <= x < 2^255 into limbs below T_i."""
    return [(x >> OFF[i]) & (int(T[i]) - 1) for i in range(10)]


def edge_inputs(bound):
    """Limb vectors at and around the bounds, plus the values where the reduction mod p turns over."""
    vals = [0, 1, 2, 18, 19, 20, P - 2, P - 1, P, P + 1, P + 18, 2 ** 255 - 1, 2 ** 255 - 2, 2 ** 254, 2 ** 254 - 1]
    rows = [limbs_of(v) for v in vals]
    top = (bound - 1).tolist()
    rows += [top, [0] * 10]
    for i in range(10):  # one limb at its maximum, the others zero or at theirs
        r = [0] * 10
        r[i] = top[i]
        rows.append(r)
        r = list(top)
        r[i] = 0
        rows.append(r)
    return np.array(rows, np.uint32)


def random_inputs(bound, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((n, 10)) * bound).astype(np.int64).astype(np.uint32)


def pairs(bound, seed):
    """Every pair of edge rows, then RANDOM random pairs within the bound."""
    e = edge_inputs(bound)
    ia, ib = np.meshgrid(np.arange(len(e)), np.arange(len(e)), indexing="ij")
    a = np.concatenate([e[ia.ravel()], random_inputs(bound, RANDOM, seed)])
    b = np.concatenate([e[ib.ravel()], random_inputs(bound, RANDOM, seed + 1)])
    return a, b


def check_bound(out, bound):
    assert (out.astype(np.int64) < bound).all(), "output limb above its documented bound"


@pytest.mark.parametrize("op", [ADD, SUB])
def test_add_sub_tight_to_loose(field, op):
    a, b = pairs(TIGHT, 10 + op)
    out = field(op, a, b)
    check_bound(out, LOOSE)
    va, vb, vo = value(a), value(b), value(out)
    want = (va + vb) if op == ADD else (va - vb)
    assert ((vo - want) % P == 0).all()


def test_mul_loose_to_tight(field):
    a, b = pairs(LOOSE, 20)
    out = field(MUL, a, b)
    check_bound(out, TIGHT)
    assert ((value(out) - value(a) * value(b)) % P == 0).all()


@pytest.mark.parametrize("op", [SQ, MUL121665, CARRY])
def test_unary_loose_to_tight(field, op):
    a = np.concatenate([edge_inputs(LOOSE), edge_inputs(TIGHT), random_inputs(LOOSE, RANDOM, 30 + op)])
    out = field(op, a)
    check_bound(out, TIGHT)
    va = value(a)
    want = {SQ: va * va, MUL121665: va * 121665, CARRY: va}[op]
    assert ((value(out) - want) % P == 0).all()


def test_freeze_canonical(field):
    a = np.concatenate([edge_inputs(LOOSE), edge_inputs(TIGHT), random_inputs(LOOSE, RANDOM, 40), random_inputs(TIGHT, RANDOM, 41)])
    out = field(FREEZE, a)
    assert (words_value(out) == value(a) % P).all()
