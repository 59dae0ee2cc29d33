"""Host-side mirror of the batched ML-KEM API on numpy arrays / torch CUDA tensors.

`MLKEM` wraps the C ABI of libmlkem_b200.so.  Method names follow the reference's function names
(ml_kem.c) so that tests read like the reference's own drivers:

    keygen(KeyGen_internal)  encaps(Encaps_internal)  decaps(Decaps_internal)
    pke_keygen / pke_encrypt / pke_decrypt            ntt / intt / multiply_ntts
    sample_ntt / cbd / prf_cbd                        byte_encode / byte_decode / compress / decompress
    hash_batch (H, G, J)                              check_dk (the hash check of KEM_Decaps)

numpy inputs are treated as host memory (the library stages them through the GPU and returns numpy);
torch CUDA tensors are treated as device memory (kernels are enqueued on the current torch stream and
torch CUDA tensors are returned without synchronising).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .lib import MEM_DEVICE, MEM_HOST, MlKemB200Error, Opts, load

PARAMS = {512: (2, 3, 2, 10, 4), 768: (3, 2, 2, 10, 4), 1024: (4, 2, 2, 11, 5)}


def sizes(param_set: int):
    k, _, _, du, dv = PARAMS[param_set]
    return {"k": k, "ek": 384 * k + 32, "dk": 768 * k + 96, "dk_pke": 384 * k, "c": 32 * (du * k + dv)}


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _seed_ptr(seed):
    """The call seed of the seeded calls as a host pointer: 32 bytes (bytes or a uint8 array), or None = fresh host entropy.
    ctypes copies `bytes` into a buffer it owns for the duration of the call."""
    if seed is None:
        return None
    b = bytes(np.ascontiguousarray(seed, np.uint8).ravel()) if not isinstance(seed, (bytes, bytearray)) else bytes(seed)
    if len(b) != 32:
        raise ValueError(f"the call seed is 32 bytes, got {len(b)}")
    return C.c_char_p(b)


class KeyTable:
    """Owner of a mlkem_b200_keys handle (freed, and wiped, with the object)."""

    def __init__(self, kem, handle, ps, device=-1):
        self.kem, self.handle, self.ps, self.device = kem, handle, ps, device

    def __len__(self):
        return int(self.kem.lib.mlkem_b200_keys_count(self.handle))

    def replace(self, slots, dk=None, ek=None, seeds=None, return_status=False):
        """Overwrite the keys in `slots` in place with decapsulation keys `dk`, encapsulation keys `ek` (a table of
        encapsulation keys only) or the 64-byte seeds `(d, z)` (KeyGen_internal on the device): mlkem_b200_keys_replace /
        _replace_ek / _replace_from_seeds.  numpy key material goes through host memory, torch CUDA tensors through device memory
        on the current torch stream; `slots` is always a host list.  return_status=True (dk only) also returns the dk hash
        check per replaced key (0 / -5)."""
        kem = self.kem
        if _is_torch(slots):
            slots = slots.cpu().numpy()
        slots = np.ascontiguousarray(slots, np.uint32).ravel()
        n = slots.size
        prep = lambda a: a.contiguous() if _is_torch(a) else np.ascontiguousarray(a, np.uint8)
        ptr = lambda a: C.c_void_p(a.data_ptr() if _is_torch(a) else a.ctypes.data)
        sp = C.c_void_p(slots.ctypes.data)
        status = None
        if dk is not None:
            dk = prep(dk)
            o, _ = kem._src_opts(dk)
            status = np.empty(n, np.int32) if return_status else None
            rc = kem.lib.mlkem_b200_keys_replace(self.handle, n, sp, ptr(dk), None if status is None else C.c_void_p(status.ctypes.data),
                                                 C.byref(o))
            fname = "mlkem_b200_keys_replace"
        elif ek is not None:
            ek = prep(ek)
            o, _ = kem._src_opts(ek)
            rc = kem.lib.mlkem_b200_keys_replace_ek(self.handle, n, sp, ptr(ek), C.byref(o))
            fname = "mlkem_b200_keys_replace_ek"
        else:
            d, z = (prep(a) for a in seeds)
            o, _ = kem._src_opts(d, z)
            rc = kem.lib.mlkem_b200_keys_replace_from_seeds(self.handle, n, sp, ptr(d), ptr(z), C.byref(o))
            fname = "mlkem_b200_keys_replace_from_seeds"
        kem._check(rc, fname)
        return status if return_status else None

    def regenerate(self, slots, seed=None):
        """Overwrite the keys in `slots` in place with KeyGen_internal(d_j, z_j) expanded on the device from the 32-byte call
        seed (None: fresh host entropy) -- mlkem_b200_keys_replace_generate.  `slots` is a host list."""
        kem = self.kem
        if _is_torch(slots):
            slots = slots.cpu().numpy()
        slots = np.ascontiguousarray(slots, np.uint32).ravel()
        o = kem._opts(False, self.device)
        rc = kem.lib.mlkem_b200_keys_replace_generate(self.handle, slots.size, C.c_void_p(slots.ctypes.data), _seed_ptr(seed), C.byref(o))
        kem._check(rc, "mlkem_b200_keys_replace_generate")

    def export_ek(self, first=0, n=None, device=False):
        """Encapsulation keys of rows [first, first + n) (default: to the end) -- mlkem_b200_keys_export_ek.  Returns numpy, or
        with device=True a torch CUDA tensor on the table's device, filled on the current torch stream."""
        kem = self.kem
        ekb = sizes(self.ps)["ek"]
        n = max(len(self) - first, 0) if n is None else n
        if device:
            import torch

            dev = self.device if self.device >= 0 else torch.cuda.current_device()
            out = torch.empty((n, ekb), dtype=torch.uint8, device=f"cuda:{dev}")
            o = kem._opts(True, dev, torch.cuda.current_stream(dev).cuda_stream)
            p = C.c_void_p(out.data_ptr())
        else:
            out = np.empty((n, ekb), np.uint8)
            o = kem._opts(False)
            p = C.c_void_p(out.ctypes.data)
        kem._check(kem.lib.mlkem_b200_keys_export_ek(self.handle, first, n, p, C.byref(o)), "mlkem_b200_keys_export_ek")
        return out

    def free(self):
        if self.handle:
            self.kem.lib.mlkem_b200_keys_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class MLKEM:
    def __init__(self, chunk_items: int = 0, sample_group_limit: int = 0, fips203: bool = False):
        """fips203=True selects the conformant variant (SHAKE256 PRF/J, real modulus check) instead of the
        reference's behaviour -- see MLKEM_B200_FLAG_FIPS203 in include/mlkem_b200.h."""
        self.lib = load()
        self.chunk_items = chunk_items
        self.sample_group_limit = sample_group_limit
        self.flags = 1 if fips203 else 0

    # ------------------------------------------------------------------ plumbing
    def _opts(self, device_mem: bool, device: int = -1, stream=None):
        return Opts(device, MEM_DEVICE if device_mem else MEM_HOST, stream, self.chunk_items, self.sample_group_limit, self.flags)

    def _check(self, rc, what):
        if rc != 0:
            raise MlKemB200Error(f"{what} failed: rc={rc} {self.lib.mlkem_b200_last_error().decode()}")

    def _call(self, fname, pre, ins, outs, post=()):
        """ins: list of (array, dtype); outs: list of (shape, dtype).  Returns the outputs."""
        fn = getattr(self.lib, fname)
        on_dev = any(_is_torch(a) for a, _ in ins)
        if on_dev:
            import torch

            dev = next(a for a, _ in ins if _is_torch(a)).device
            tdt = {np.uint8: torch.uint8, np.uint16: torch.uint16, np.int32: torch.int32, np.uint32: torch.uint32}
            iarr = []
            for a, dt in ins:
                if a is None:
                    iarr.append(None)
                    continue
                if not _is_torch(a):
                    a = torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
                a = a.contiguous()
                assert a.dtype == tdt[dt], (a.dtype, dt)
                iarr.append(a)
            oarr = [torch.empty(shape, dtype=tdt[dt], device=dev) for shape, dt in outs]
            stream = torch.cuda.current_stream(dev).cuda_stream
            o = self._opts(True, dev.index if dev.index is not None else torch.cuda.current_device(), stream)
            ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        else:
            iarr = [None if a is None else np.ascontiguousarray(a, dtype=dt) for a, dt in ins]
            oarr = [np.empty(shape, dtype=dt) for shape, dt in outs]
            o = self._opts(False)
            ptr = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        rc = fn(*pre, *[ptr(a) for a in iarr], *[ptr(a) for a in oarr], *post, C.byref(o))
        self._check(rc, fname)
        return oarr[0] if len(oarr) == 1 else tuple(oarr)

    @staticmethod
    def _count(a, item_elems):
        n = (a.numel() if _is_torch(a) else np.asarray(a).size) // item_elems
        return n

    # ------------------------------------------------------------------ ML-KEM internal
    def keygen(self, ps, d, z):
        sz, n = sizes(ps), self._count(d, 32)
        return self._call("mlkem_b200_keygen_batch", (ps, n), [(d, np.uint8), (z, np.uint8)],
                          [((n, sz["ek"]), np.uint8), ((n, sz["dk"]), np.uint8)])

    def encaps(self, ps, ek, m):
        sz, n = sizes(ps), self._count(m, 32)
        return self._call("mlkem_b200_encaps_batch", (ps, n), [(ek, np.uint8), (m, np.uint8)],
                          [((n, sz["c"]), np.uint8), ((n, 32), np.uint8)])

    def decaps(self, ps, dk, c):
        sz = sizes(ps)
        n = self._count(c, sz["c"])
        return self._call("mlkem_b200_decaps_batch", (ps, n), [(dk, np.uint8), (c, np.uint8)], [((n, 32), np.uint8)])

    def check_dk(self, ps, dk):
        n = self._count(dk, sizes(ps)["dk"])
        return self._call("mlkem_b200_check_dk_batch", (ps, n), [(dk, np.uint8)], [((n,), np.int32)])

    # ------------------------------------------------------------------ the reference's cell layout (one byte per uint32 cell)
    def keygen_cells(self, ps, d, z):
        sz, n = sizes(ps), self._count(d, 32)
        return self._call("mlkem_b200_keygen_cells_batch", (ps, n), [(d, np.uint32), (z, np.uint32)],
                          [((n, sz["ek"]), np.uint32), ((n, sz["dk"]), np.uint32)])

    def encaps_cells(self, ps, ek, m):
        sz, n = sizes(ps), self._count(m, 32)
        return self._call("mlkem_b200_encaps_cells_batch", (ps, n), [(ek, np.uint32), (m, np.uint32)],
                          [((n, sz["c"]), np.uint32), ((n, 32), np.uint32)])

    def decaps_cells(self, ps, dk, c):
        sz = sizes(ps)
        n = self._count(c, sz["c"])
        return self._call("mlkem_b200_decaps_cells_batch", (ps, n), [(dk, np.uint32), (c, np.uint32)], [((n, 32), np.uint32)])

    def cells_from_bytes(self, b):
        n = self._count(b, 1)
        return self._call("mlkem_b200_cells_from_bytes", (n,), [(b, np.uint8)], [(tuple(b.shape), np.uint32)])

    def cells_to_bytes(self, c):
        n = self._count(c, 1)
        return self._call("mlkem_b200_cells_to_bytes", (n,), [(c, np.uint32)], [(tuple(c.shape), np.uint8)])

    # ------------------------------------------------------------------ resident key tables (keyed Encaps / Decaps)
    def _src_opts(self, *arrays, device=None):
        """Options describing where `arrays` live: torch CUDA tensors -> device memory on their device and the current
        torch stream; anything else -> host memory (on `device`, default: the current one)."""
        t = next((a for a in arrays if a is not None and _is_torch(a)), None)
        if t is not None:
            import torch

            return self._opts(True, t.device.index, torch.cuda.current_stream(t.device).cuda_stream), True
        return self._opts(False, -1 if device is None else device), False

    def keys_load(self, ps, dk=None, ek=None, seeds=None, device=None, return_status=False, expand=False):
        """A resident key table on the GPU from decapsulation keys `dk`, from encapsulation keys `ek` (Encaps only) or
        from the 64-byte seeds `(d, z)` (KeyGen_internal on the device).  expand=True also keeps every key's matrix A^
        (MLKEM_B200_FLAG_EXPAND_KEYS): keyed calls then skip the matrix expansion."""
        sz = sizes(ps)
        handle = C.c_void_p()
        prep = lambda a: a.contiguous() if _is_torch(a) else np.ascontiguousarray(a, np.uint8)
        ptr = lambda a: C.c_void_p(a.data_ptr() if _is_torch(a) else a.ctypes.data)
        status = None
        if dk is not None:
            dk = prep(dk)
            n = self._count(dk, sz["dk"])
            o, _ = self._src_opts(dk, device=device)
            o.flags |= 4 if expand else 0
            status = np.empty(n, np.int32)
            rc = self.lib.mlkem_b200_keys_load(ps, n, ptr(dk), C.c_void_p(status.ctypes.data), C.byref(o), C.byref(handle))
        elif ek is not None:
            ek = prep(ek)
            o, _ = self._src_opts(ek, device=device)
            o.flags |= 4 if expand else 0
            rc = self.lib.mlkem_b200_keys_load_ek(ps, self._count(ek, sz["ek"]), ptr(ek), C.byref(o), C.byref(handle))
        else:
            d, z = (prep(a) for a in seeds)
            o, _ = self._src_opts(d, z, device=device)
            o.flags |= 4 if expand else 0
            rc = self.lib.mlkem_b200_keys_from_seeds(ps, self._count(d, 32), ptr(d), ptr(z), C.byref(o), C.byref(handle))
        self._check(rc, "mlkem_b200_keys_load")
        table = KeyTable(self, handle, ps, o.device)
        return (table, status) if return_status else table

    def _keyed(self, fname, table, key_index, data, item_bytes, out_shapes):
        n = self._count(data, item_bytes)
        if _is_torch(data):
            import torch

            data = data.contiguous()
            idx = None if key_index is None else key_index.to(device=data.device, dtype=torch.int32).contiguous()
            outs = [torch.empty((n, w), dtype=torch.uint8, device=data.device) for w in out_shapes]
            o, _ = self._src_opts(data)
            ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        else:
            data = np.ascontiguousarray(data, np.uint8)
            idx = None if key_index is None else np.ascontiguousarray(key_index, np.uint32)
            outs = [np.empty((n, w), np.uint8) for w in out_shapes]
            o = self._opts(False)
            ptr = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        rc = getattr(self.lib, fname)(table.handle, n, ptr(idx), ptr(data), *[ptr(a) for a in outs], C.byref(o))
        self._check(rc, fname)
        return outs[0] if len(outs) == 1 else tuple(outs)

    def encaps_keyed(self, table, key_index, m):
        """Encaps_internal under table[key_index[i]] (key_index=None: key i mod n_keys).  Returns (c, K)."""
        return self._keyed("mlkem_b200_encaps_keyed_batch", table, key_index, m, 32, [sizes(table.ps)["c"], 32])

    def decaps_keyed(self, table, key_index, c):
        """Decaps_internal under table[key_index[i]].  Returns K."""
        return self._keyed("mlkem_b200_decaps_keyed_batch", table, key_index, c, sizes(table.ps)["c"], [32])

    # ------------------------------------------------------------------ public wrappers (entropy + checks), host memory
    def kem_keygen(self, ps, n):
        sz = sizes(ps)
        ek, dk = np.empty((n, sz["ek"]), np.uint8), np.empty((n, sz["dk"]), np.uint8)
        o = self._opts(False)
        self._check(self.lib.mlkem_b200_kem_keygen_batch(ps, n, C.c_void_p(ek.ctypes.data), C.c_void_p(dk.ctypes.data), C.byref(o)),
                    "mlkem_b200_kem_keygen_batch")
        return ek, dk

    def kem_encaps(self, ps, ek, ek_len=None):
        sz = sizes(ps if ps in PARAMS else 768)  # an unknown set is the library's error to report (-1)
        ek = np.ascontiguousarray(ek, np.uint8)
        n = ek.size // sz["ek"] if ek_len is None else ek.shape[0]
        c, K = np.empty((n, sz["c"]), np.uint8), np.empty((n, 32), np.uint8)
        o = self._opts(False)
        rc = self.lib.mlkem_b200_kem_encaps_batch(ps, n, C.c_void_p(ek.ctypes.data), sz["ek"] if ek_len is None else ek_len,
                                                  C.c_void_p(c.ctypes.data), C.c_void_p(K.ctypes.data), C.byref(o))
        return rc, c, K

    def kem_decaps(self, ps, dk, c, dk_len=None, c_len=None):
        sz = sizes(ps)
        dk, c = np.ascontiguousarray(dk, np.uint8), np.ascontiguousarray(c, np.uint8)
        n = c.size // sz["c"]
        K, status = np.empty((n, 32), np.uint8), np.empty(n, np.int32)
        o = self._opts(False)
        rc = self.lib.mlkem_b200_kem_decaps_batch(ps, n, C.c_void_p(dk.ctypes.data), sz["dk"] if dk_len is None else dk_len,
                                                  C.c_void_p(c.ctypes.data), sz["c"] if c_len is None else c_len,
                                                  C.c_void_p(K.ctypes.data), C.c_void_p(status.ctypes.data), C.byref(o))
        return rc, K, status

    # ------------------------------------------------------------------ randomness expanded on the device from a 32-byte call seed
    # seed: 32 bytes (bytes or uint8 array) makes a call deterministic (tests, known answers); None draws it from the host entropy
    # source.  Item j gets R_j = SHAKE256(seed || LE64(j) || LE64(tag)), see include/mlkem_b200.h.  Every call is synchronous.
    def _out_opts(self, device_mem, shapes, dev=None):
        """Empty outputs and options: numpy and host memory, or torch CUDA tensors on `dev` (default: the current device) and
        device memory on its current torch stream."""
        if device_mem:
            import torch

            dev = torch.cuda.current_device() if dev is None or dev < 0 else dev
            outs = [torch.empty(s, dtype=torch.uint8, device=f"cuda:{dev}") for s in shapes]
            return outs, self._opts(True, dev, torch.cuda.current_stream(dev).cuda_stream), lambda t: C.c_void_p(t.data_ptr())
        return [np.empty(s, np.uint8) for s in shapes], self._opts(False, -1 if dev is None else dev), lambda a: C.c_void_p(a.ctypes.data)

    def kem_keygen_seeded(self, ps, n, seed=None, device=False):
        """KEM_KeyGen with (d_j, z_j) expanded on the GPU -- mlkem_b200_kem_keygen_seeded_batch.  Returns (ek, dk): numpy, or with
        device=True torch CUDA tensors filled on the current torch stream."""
        sz = sizes(ps if ps in PARAMS else 768)
        (ek, dk), o, ptr = self._out_opts(device, [(n, sz["ek"]), (n, sz["dk"])])
        rc = self.lib.mlkem_b200_kem_keygen_seeded_batch(ps, n, _seed_ptr(seed), ptr(ek), ptr(dk), C.byref(o))
        self._check(rc, "mlkem_b200_kem_keygen_seeded_batch")
        return ek, dk

    def kem_encaps_seeded(self, ps, ek, seed=None, ek_len=None):
        """KEM_Encaps with m_j expanded on the GPU -- mlkem_b200_kem_encaps_seeded_batch.  A numpy ek is host memory, a torch ek
        device memory.  Returns (rc, c, K) like kem_encaps."""
        sz = sizes(ps if ps in PARAMS else 768)  # an unknown set is the library's error to report (-1)
        on_dev = _is_torch(ek)
        if on_dev:
            ek = ek.contiguous()
            n = ek.numel() // sz["ek"] if ek_len is None else ek.shape[0]
            (c, K), o, ptr = self._out_opts(True, [(n, sz["c"]), (n, 32)], ek.device.index)
        else:
            ek = np.ascontiguousarray(ek, np.uint8)
            n = ek.size // sz["ek"] if ek_len is None else ek.shape[0]
            (c, K), o, ptr = self._out_opts(False, [(n, sz["c"]), (n, 32)])
        rc = self.lib.mlkem_b200_kem_encaps_seeded_batch(ps, n, ptr(ek), sz["ek"] if ek_len is None else ek_len, _seed_ptr(seed),
                                                         ptr(c), ptr(K), C.byref(o))
        return rc, c, K

    def kem_encaps_keyed(self, table, n, key_index=None, seed=None, device=False):
        """KEM_Encaps under table[key_index[i]] (None: key i mod n_keys) with m_j expanded on the GPU --
        mlkem_b200_kem_encaps_keyed_batch.  Returns (c, K): numpy, or with device=True torch CUDA tensors on the table's device."""
        (c, K), o, ptr = self._out_opts(device, [(n, sizes(table.ps)["c"]), (n, 32)], table.device)
        idx = None
        if key_index is not None:
            if device:
                import torch

                idx = torch.as_tensor(key_index).to(device=c.device, dtype=torch.int32).contiguous()
            else:
                idx = np.ascontiguousarray(key_index.cpu().numpy() if _is_torch(key_index) else key_index, np.uint32)
        rc = self.lib.mlkem_b200_kem_encaps_keyed_batch(table.handle, n, None if idx is None else ptr(idx), _seed_ptr(seed), ptr(c), ptr(K),
                                                        C.byref(o))
        self._check(rc, "mlkem_b200_kem_encaps_keyed_batch")
        return c, K

    def keys_generate(self, ps, n_keys, seed=None, device=None, expand=False):
        """A resident key table of KeyGen_internal(d_j, z_j), j < n_keys, expanded on the GPU: its secrets never exist on the
        host -- mlkem_b200_keys_generate.  Publish its keys with KeyTable.export_ek()."""
        handle = C.c_void_p()
        o = self._opts(False, -1 if device is None else device)
        o.flags |= 4 if expand else 0
        rc = self.lib.mlkem_b200_keys_generate(ps, n_keys, _seed_ptr(seed), C.byref(o), C.byref(handle))
        self._check(rc, "mlkem_b200_keys_generate")
        return KeyTable(self, handle, ps, o.device)

    # ------------------------------------------------------------------ K-PKE
    def pke_keygen(self, ps, d):
        sz, n = sizes(ps), self._count(d, 32)
        return self._call("mlkem_b200_pke_keygen_batch", (ps, n), [(d, np.uint8)],
                          [((n, sz["ek"]), np.uint8), ((n, sz["dk_pke"]), np.uint8)])

    def pke_encrypt(self, ps, ek, m, r):
        sz, n = sizes(ps), self._count(m, 32)
        return self._call("mlkem_b200_pke_encrypt_batch", (ps, n), [(ek, np.uint8), (m, np.uint8), (r, np.uint8)],
                          [((n, sz["c"]), np.uint8)])

    def pke_decrypt(self, ps, dk, c, dk_stride=None):
        sz = sizes(ps)
        n = self._count(c, sz["c"])
        stride = dk_stride if dk_stride is not None else self._count(dk, 1) // n
        fn = self.lib.mlkem_b200_pke_decrypt_batch
        # dk_stride sits between the dk and c pointers in the C signature
        if _is_torch(c):
            import torch

            dk, c = dk.contiguous(), c.contiguous()
            out = torch.empty((n, 32), dtype=torch.uint8, device=c.device)
            o = self._opts(True, c.device.index, torch.cuda.current_stream(c.device).cuda_stream)
            rc = fn(ps, n, C.c_void_p(dk.data_ptr()), stride, C.c_void_p(c.data_ptr()), C.c_void_p(out.data_ptr()), C.byref(o))
        else:
            dk, c = np.ascontiguousarray(dk, np.uint8), np.ascontiguousarray(c, np.uint8)
            out = np.empty((n, 32), np.uint8)
            o = self._opts(False)
            rc = fn(ps, n, C.c_void_p(dk.ctypes.data), stride, C.c_void_p(c.ctypes.data), C.c_void_p(out.ctypes.data), C.byref(o))
        self._check(rc, "mlkem_b200_pke_decrypt_batch")
        return out

    # ------------------------------------------------------------------ ring arithmetic
    def ntt(self, f):
        n = self._count(f, 256)
        return self._call("mlkem_b200_ntt_batch", (n,), [(f, np.uint16)], [((n, 256), np.uint16)])

    def intt(self, f):
        n = self._count(f, 256)
        return self._call("mlkem_b200_intt_batch", (n,), [(f, np.uint16)], [((n, 256), np.uint16)])

    def multiply_ntts(self, f, g):
        n = self._count(f, 256)
        return self._call("mlkem_b200_multiply_ntts_batch", (n,), [(f, np.uint16), (g, np.uint16)], [((n, 256), np.uint16)])

    def poly_add(self, u, v):
        n = self._count(u, 256)
        return self._call("mlkem_b200_poly_add_batch", (n,), [(u, np.uint16), (v, np.uint16)], [((n, 256), np.uint16)])

    def poly_sub(self, u, v):
        n = self._count(u, 256)
        return self._call("mlkem_b200_poly_sub_batch", (n,), [(u, np.uint16), (v, np.uint16)], [((n, 256), np.uint16)])

    def vector_multiply(self, u, v, k):
        n = self._count(u, 256 * k)
        return self._call("mlkem_b200_vector_multiply_batch", (k, n), [(u, np.uint16), (v, np.uint16)], [((n, 256), np.uint16)])

    # ------------------------------------------------------------------ samplers
    def sample_ntt(self, seeds34, return_seeds=False):
        n = self._count(seeds34, 34)
        if return_seeds:
            return self._call("mlkem_b200_sample_ntt_batch", (n,), [(seeds34, np.uint8)],
                              [((n, 256), np.uint16), ((n, 34), np.uint8)])
        fn = self.lib.mlkem_b200_sample_ntt_batch
        if _is_torch(seeds34):
            import torch

            s = seeds34.contiguous()
            out = torch.empty((n, 256), dtype=torch.uint16, device=s.device)
            o = self._opts(True, s.device.index, torch.cuda.current_stream(s.device).cuda_stream)
            rc = fn(n, C.c_void_p(s.data_ptr()), C.c_void_p(out.data_ptr()), None, C.byref(o))
        else:
            s = np.ascontiguousarray(seeds34, np.uint8)
            out = np.empty((n, 256), np.uint16)
            o = self._opts(False)
            rc = fn(n, C.c_void_p(s.ctypes.data), C.c_void_p(out.ctypes.data), None, C.byref(o))
        self._check(rc, "mlkem_b200_sample_ntt_batch")
        return out

    def cbd(self, data, eta):
        n = self._count(data, 64 * eta)
        return self._call("mlkem_b200_cbd_batch", (eta, n), [(data, np.uint8)], [((n, 256), np.uint16)])

    def prf_cbd(self, seeds32, nonces, eta):
        n = self._count(nonces, 1)
        return self._call("mlkem_b200_prf_cbd_batch", (eta, n), [(seeds32, np.uint8), (nonces, np.uint8)], [((n, 256), np.uint16)])

    # ------------------------------------------------------------------ codec
    def byte_encode(self, F, d):
        n = self._count(F, 256)
        return self._call("mlkem_b200_byte_encode_batch", (d, n), [(F, np.uint16)], [((n, 32 * d), np.uint8)])

    def byte_decode(self, B, d):
        n = self._count(B, 32 * d)
        return self._call("mlkem_b200_byte_decode_batch", (d, n), [(B, np.uint8)], [((n, 256), np.uint16)])

    def compress_encode(self, F, d):
        n = self._count(F, 256)
        return self._call("mlkem_b200_compress_encode_batch", (d, n), [(F, np.uint16)], [((n, 32 * d), np.uint8)])

    def decode_decompress(self, B, d):
        n = self._count(B, 32 * d)
        return self._call("mlkem_b200_decode_decompress_batch", (d, n), [(B, np.uint8)], [((n, 256), np.uint16)])

    def _elementwise(self, fname, x, d):
        if _is_torch(x):
            n = x.numel()
            assert n % 8 == 0
            return self._call(fname, (d, n), [(x, np.uint16)], [(tuple(x.shape), np.uint16)])
        x = np.atleast_1d(np.asarray(x, dtype=np.uint16))
        n = x.size
        pad = (-n) % 8
        xp = np.concatenate([x.ravel(), np.zeros(pad, np.uint16)])
        y = self._call(fname, (d, xp.size), [(xp, np.uint16)], [((xp.size,), np.uint16)])
        return y[:n].reshape(x.shape)

    def compress(self, x, d):
        return self._elementwise("mlkem_b200_compress_batch", x, d)

    def decompress(self, x, d):
        return self._elementwise("mlkem_b200_decompress_batch", x, d)

    # ------------------------------------------------------------------ hashes / tables
    def hash_batch(self, which, data, length):
        n = self._count(data, length)
        return self._call("mlkem_b200_hash_batch", (which, n, length), [(data, np.uint8)], [((n, 64 if which == 1 else 32), np.uint8)])

    def sha3_bits(self, msgs_bits, sfx, c, d):
        """sha3_b (sha3.c:408) for a batch of equal-length bit strings: msgs_bits [n, nbits] of 0/1 -> [n, d] bits."""
        bits = np.atleast_2d(np.asarray(msgs_bits, dtype=np.uint8))
        n, nbits = bits.shape
        packed = np.packbits(bits, axis=1, bitorder="little") if nbits else np.zeros((n, 1), np.uint8)
        packed = np.ascontiguousarray(packed)
        out = np.zeros((n, (d + 7) // 8), np.uint8)
        sf = np.asarray(sfx, dtype=np.uint8)
        o = self._opts(False)
        rc = self.lib.mlkem_b200_sha3_bits_batch(n, C.c_void_p(packed.ctypes.data), nbits, C.c_void_p(sf.ctypes.data), c, d,
                                                 C.c_void_p(out.ctypes.data), C.byref(o))
        self._check(rc, "mlkem_b200_sha3_bits_batch")
        return np.unpackbits(out, axis=1, bitorder="little")[:, :d]

    def tables(self):
        z, g = np.empty(128, np.uint16), np.empty(128, np.uint16)
        self._check(self.lib.mlkem_b200_tables(C.c_void_p(z.ctypes.data), C.c_void_p(g.ctypes.data)), "mlkem_b200_tables")
        return z, g

    def zeta_table(self):
        return self.tables()[0]

    def gamma_table(self):
        return self.tables()[1]

    def bitrev7(self, r):
        """BitRev7 (ml_kem.c:26) through the library's exported reference-signature function."""
        class UByte(C.Structure):
            _fields_ = [("v", C.c_uint)]

        fn = self.lib.BitRev7
        fn.restype, fn.argtypes = UByte, [UByte]
        return fn(UByte(r & 0x7F)).v & 0x7F

    def launch_count(self):
        return int(self.lib.mlkem_b200_launch_count())

    # ------------------------------------------------------------------ measurement hooks
    def profile(self, enable: bool):
        self.lib.mlkem_b200_profile(1 if enable else 0)

    def set_streams(self, n: int):
        self.lib.mlkem_b200_set_streams(n)

    def profile_report(self):
        import json

        buf = C.create_string_buffer(1 << 16)
        n = self.lib.mlkem_b200_profile_report(buf, len(buf))
        return json.loads(buf.raw[:n].decode()) if n else {}

    def int32_peak(self):
        out = (C.c_double * 6)()
        self._check(self.lib.mlkem_b200_int32_peak(out), "mlkem_b200_int32_peak")
        return dict(zip(("lop3", "shf", "imad", "lop3+imad", "iadd3", "imad_hi"), [float(v) for v in out]))
