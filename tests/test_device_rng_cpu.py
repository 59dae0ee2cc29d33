"""CPU tests of the seeded calls (randomness expanded on the device, include/mlkem_b200.h): without a device they refuse to
compute, write nothing to their outputs, and the Python wrappers raise."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_CUDA, ERR_ARG = -10, -11


@pytest.fixture(scope="module")
def lib():
    import torch

    import crystals_kyber_b200 as ck

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    if not os.path.exists(ck.LIB_PATH):
        import subprocess

        subprocess.run(["make", "-C", ROOT, "lib"], check=True, stdout=subprocess.DEVNULL)
    return ck.load()


P = lambda a: C.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("seed", [None, bytes(range(32))], ids=["entropy", "fixed"])
def test_seeded_calls_refuse_without_a_device(lib, seed):
    from crystals_kyber_b200.lib import MEM_DEVICE, MEM_HOST, Opts

    n = 3
    for mem in (MEM_HOST, MEM_DEVICE):
        o = Opts(-1, mem, None, 0, 0, 0)
        ek = np.full((n, 1184), 0xAB, np.uint8)
        dk = np.full((n, 2400), 0xAB, np.uint8)
        assert lib.mlkem_b200_kem_keygen_seeded_batch(768, n, seed, P(ek), P(dk), C.byref(o)) == ERR_CUDA
        assert (ek == 0xAB).all() and (dk == 0xAB).all()
        c = np.full((n, 1088), 0xAB, np.uint8)
        K = np.full((n, 32), 0xAB, np.uint8)
        src = np.zeros((n, 1184), np.uint8)
        assert lib.mlkem_b200_kem_encaps_seeded_batch(768, n, P(src), 1184, seed, P(c), P(K), C.byref(o)) == ERR_CUDA
        assert (c == 0xAB).all() and (K == 0xAB).all()
        handle = C.c_void_p(123)
        assert lib.mlkem_b200_keys_generate(768, 4, seed, C.byref(o), C.byref(handle)) == ERR_CUDA
        assert not handle.value
        # no table can exist without a device: the keyed calls refuse a NULL one before touching anything
        assert lib.mlkem_b200_kem_encaps_keyed_batch(None, n, None, seed, P(c), P(K), C.byref(o)) == ERR_ARG
        assert (c == 0xAB).all() and (K == 0xAB).all()
        slots = np.array([0, 1], np.uint32)
        assert lib.mlkem_b200_keys_replace_generate(None, 2, P(slots), seed, C.byref(o)) == ERR_ARG
    # the checks that need no device come first, as in mlkem_b200_kem_encaps_batch
    o = Opts(-1, MEM_HOST, None, 0, 0, 0)
    assert lib.mlkem_b200_kem_keygen_seeded_batch(999, n, seed, P(ek), P(dk), C.byref(o)) == -1
    assert lib.mlkem_b200_kem_encaps_seeded_batch(999, n, P(src), 1184, seed, P(c), P(K), C.byref(o)) == -1
    assert lib.mlkem_b200_kem_encaps_seeded_batch(768, n, P(src), 1183, seed, P(c), P(K), C.byref(o)) == -3
    assert lib.mlkem_b200_kem_keygen_seeded_batch(768, 0, seed, None, None, C.byref(o)) == 0


def test_python_wrappers_raise_without_a_device(lib):
    import crystals_kyber_b200 as ck

    kem = ck.MLKEM()
    seed = bytes(32)
    with pytest.raises(ck.MlKemB200Error):
        kem.kem_keygen_seeded(768, 4, seed)
    with pytest.raises(ck.MlKemB200Error):
        kem.kem_keygen_seeded(768, 4)
    with pytest.raises(ck.MlKemB200Error):
        kem.keys_generate(768, 4, seed)
    with pytest.raises(ck.MlKemB200Error):
        kem.keys_generate(512, 4, expand=True)
    rc, c, K = kem.kem_encaps_seeded(768, np.zeros((2, 1184), np.uint8), seed)
    assert rc == ERR_CUDA
    with pytest.raises(ValueError):
        kem.kem_keygen_seeded(768, 4, bytes(31))
    from crystals_kyber_b200.api import KeyTable

    fake = KeyTable(kem, None, 768)
    with pytest.raises(ck.MlKemB200Error):
        kem.kem_encaps_keyed(fake, 4, seed=seed)
    with pytest.raises(ck.MlKemB200Error):
        fake.regenerate([0, 1], seed)
