#!/usr/bin/env python3
"""What the randomized ML-KEM-768 calls cost when their randomness comes from the host entropy source versus when it is
expanded on the device from a 32-byte call seed (include/mlkem_b200.h, "randomness expanded on the device"):

  urandom      read rate of /dev/urandom on this host, from this process (1-second loops of 128 KB and of 32 MB reads);
  keygen       2^20 and 2^22 items, device memory and host memory (pinned buffers): mlkem_b200_kem_keygen_batch (host entropy),
               _kem_keygen_seeded_batch(NULL) and the ceiling _keygen_batch with its (d, z) already in the call's memory space
               (device memory: device-resident seeds);
  encaps       the same three for Encaps: _kem_encaps_batch, _kem_encaps_seeded_batch(NULL), _encaps_batch with m given;
  keyed        an expanded table of 2^16 keys, 2^22 items: _encaps_keyed_batch with m given vs _kem_encaps_keyed_batch(NULL), both
               memory spaces;
  tables       _keys_generate(NULL) vs _keys_from_seeds with host seeds, 2^16 keys, plain and expanded;
  profile      the share of k_expand_seed in the kernel time of each seeded call, from mlkem_b200_profile (a separate pass, one
               stream, after the timed ones).

Variants of one measurement alternate within each repetition.  Every call is timed with the host clock around the call and
a device synchronise.  One JSON object per line (GPU name, power limit and max SM clock in the first), to --out or stdout.
    python tools/time_device_rng.py --out profiles/device_rng_r03.jsonl
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import crystals_kyber_b200 as ck
from crystals_kyber_b200.lib import MEM_DEVICE, MEM_HOST, Opts

PS, EK, DK, CT = 768, 1184, 2400, 1088
NK = 1 << 16
FLAG_EXPAND = 4


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch": torch.__version__, "lib": os.path.relpath(ck.load()._name, ROOT)}


def urandom_rate(read_bytes, seconds=1.0):
    with open("/dev/urandom", "rb", buffering=0) as f:
        got, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            got += len(f.read(read_bytes))
        dt = time.perf_counter() - t0
    return got / dt


class Pinned:
    """Page-locked host buffer from mlkem_b200_host_alloc (exact size, freed with the object)."""

    def __init__(self, lib, shape):
        self.lib, self.size = lib, int(np.prod(shape))
        self.p = lib.mlkem_b200_host_alloc(self.size)
        if not self.p:
            raise MemoryError(f"mlkem_b200_host_alloc({self.size}) failed")
        self.a = np.ctypeslib.as_array((C.c_uint8 * self.size).from_address(self.p)).reshape(shape)

    def data_ptr(self):
        return self.p

    def __del__(self):
        if self.p:
            self.lib.mlkem_b200_host_free(self.p)
            self.p = None


def P(t):
    return C.c_void_p(t.data_ptr())


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: rc={rc} {ck.load().mlkem_b200_last_error().decode()}")


def race(variants, reps):
    """variants: name -> fn (returns when its work is done).  Warm each once, then `reps` rounds in alternation.  Returns
    name -> (median s, min s)."""
    for fn in variants.values():
        fn()
    ts = {k: [] for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[k].append(time.perf_counter() - t0)
    return {k: (statistics.median(v), min(v)) for k, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="20,22", help="log2 item counts of the unkeyed measurements")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the library has no CPU fallback")
    out = open(args.out, "w") if args.out else sys.stdout
    emit = lambda rec: (out.write(json.dumps(rec) + "\n"), out.flush())
    emit({"what": "setup", "param_set": PS, **gpu_info()})
    lib = ck.load()
    dev = torch.cuda.current_device()

    for rb in (128 << 10, 32 << 20):
        emit({"what": "urandom", "read_bytes": rb, "GB_per_s": round(urandom_rate(rb) / 1e9, 3)})

    def opts(mem, flags=0):
        return Opts(dev, mem, torch.cuda.current_stream().cuda_stream if mem == MEM_DEVICE else None, 0, 0, flags)

    def buf(shape, mem):
        if mem == MEM_DEVICE:
            return torch.empty(shape, dtype=torch.uint8, device="cuda")
        return Pinned(lib, shape)

    def rand(shape, mem, seed):
        if mem == MEM_DEVICE:
            g = torch.Generator(device="cuda").manual_seed(seed)
            return torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
        b = Pinned(lib, shape)
        b.a[...] = np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)
        return b

    def record(what, mem, items, res, base):
        for k, (med, mn) in res.items():
            emit({"what": what, "variant": k, "mem": "device" if mem == MEM_DEVICE else "host", "items": items, "reps": args.reps,
                  "median_ms": round(1e3 * med, 3), "min_ms": round(1e3 * mn, 3), "per_s_median": round(items / med),
                  "vs_ceiling": round(res[base][0] / med, 4)})

    # ---- unkeyed KeyGen / Encaps
    for lg in (int(s) for s in args.sizes.split(",")):
        n = 1 << lg
        for mem in (MEM_DEVICE, MEM_HOST):
            o = opts(mem)
            ek, dk = buf((n, EK), mem), buf((n, DK), mem)
            d, z = rand((n, 32), mem, 1), rand((n, 32), mem, 2)
            res = race({
                "kem_keygen_batch": lambda: check(lib.mlkem_b200_kem_keygen_batch(PS, n, P(ek), P(dk), C.byref(o)), "kem_keygen"),
                "kem_keygen_seeded": lambda: check(lib.mlkem_b200_kem_keygen_seeded_batch(PS, n, None, P(ek), P(dk), C.byref(o)), "seeded"),
                "keygen_batch": lambda: check(lib.mlkem_b200_keygen_batch(PS, n, P(d), P(z), P(ek), P(dk), C.byref(o)), "keygen"),
            }, args.reps)
            record("keygen", mem, n, res, "keygen_batch")
            del d, z, dk
            c, K, m = buf((n, CT), mem), buf((n, 32), mem), rand((n, 32), mem, 3)
            res = race({
                "kem_encaps_batch": lambda: check(lib.mlkem_b200_kem_encaps_batch(PS, n, P(ek), EK, P(c), P(K), C.byref(o)), "kem_encaps"),
                "kem_encaps_seeded": lambda: check(lib.mlkem_b200_kem_encaps_seeded_batch(PS, n, P(ek), EK, None, P(c), P(K), C.byref(o)),
                                                   "seeded"),
                "encaps_batch": lambda: check(lib.mlkem_b200_encaps_batch(PS, n, P(ek), P(m), P(c), P(K), C.byref(o)), "encaps"),
            }, args.reps)
            record("encaps", mem, n, res, "encaps_batch")
            del ek, c, K, m
            torch.cuda.empty_cache()

    # ---- keyed Encaps on an expanded table of 2^16 keys
    n = 1 << 22
    handle = C.c_void_p()
    check(lib.mlkem_b200_keys_generate(PS, NK, None, C.byref(Opts(dev, MEM_HOST, None, 0, 0, FLAG_EXPAND)), C.byref(handle)), "keys_generate")
    for mem in (MEM_DEVICE, MEM_HOST):
        o = opts(mem)
        c, K, m = buf((n, CT), mem), buf((n, 32), mem), rand((n, 32), mem, 4)
        res = race({
            "encaps_keyed_batch": lambda: check(lib.mlkem_b200_encaps_keyed_batch(handle, n, None, P(m), P(c), P(K), C.byref(o)), "keyed"),
            "kem_encaps_keyed": lambda: check(lib.mlkem_b200_kem_encaps_keyed_batch(handle, n, None, None, P(c), P(K), C.byref(o)), "seeded"),
        }, args.reps)
        record("keyed_encaps_expanded_table", mem, n, res, "encaps_keyed_batch")
        del c, K, m
    torch.cuda.empty_cache()

    # ---- key tables: generated on the device vs built from host seeds
    d, z = rand((NK, 32), MEM_HOST, 5), rand((NK, 32), MEM_HOST, 6)
    for flags, kind in ((0, "plain"), (FLAG_EXPAND, "expanded")):
        o = Opts(dev, MEM_HOST, None, 0, 0, flags)

        def gen():
            h = C.c_void_p()
            check(lib.mlkem_b200_keys_generate(PS, NK, None, C.byref(o), C.byref(h)), "keys_generate")
            lib.mlkem_b200_keys_free(h)

        def from_seeds():
            h = C.c_void_p()
            check(lib.mlkem_b200_keys_from_seeds(PS, NK, P(d), P(z), C.byref(o), C.byref(h)), "keys_from_seeds")
            lib.mlkem_b200_keys_free(h)

        res = race({"keys_from_seeds": from_seeds, "keys_generate": gen}, args.reps)
        for k, (med, mn) in res.items():
            emit({"what": "table", "table": kind, "variant": k, "keys": NK, "reps": args.reps, "median_ms": round(1e3 * med, 3),
                  "min_ms": round(1e3 * mn, 3), "vs_from_seeds": round(res["keys_from_seeds"][0] / med, 4)})

    # ---- share of k_expand_seed in each seeded call's kernel time (profiling pass, one stream)
    lib.mlkem_b200_set_streams(1)
    kem = ck.MLKEM()
    n = 1 << 20
    ek, dk = buf((n, EK), MEM_DEVICE), buf((n, DK), MEM_DEVICE)
    c, K = buf((n, CT), MEM_DEVICE), buf((n, 32), MEM_DEVICE)
    steps = {
        "kem_keygen_seeded": lambda o: lib.mlkem_b200_kem_keygen_seeded_batch(PS, n, None, P(ek), P(dk), C.byref(o)),
        "kem_encaps_seeded": lambda o: lib.mlkem_b200_kem_encaps_seeded_batch(PS, n, P(ek), EK, None, P(c), P(K), C.byref(o)),
        "kem_encaps_keyed_expanded": lambda o: lib.mlkem_b200_kem_encaps_keyed_batch(handle, n, None, None, P(c), P(K), C.byref(o)),
    }
    for name, fn in steps.items():
        o = opts(MEM_DEVICE)
        check(fn(o), name)  # warm
        torch.cuda.synchronize()
        kem.profile_report()
        kem.profile(True)
        check(fn(o), name)
        torch.cuda.synchronize()
        kem.profile(False)
        rep = kem.profile_report()
        total = sum(v["ms"] for v in rep.values())
        mine = rep.get("k_expand_seed", {"ms": 0.0})["ms"]
        emit({"what": "profile", "step": name, "items": n, "kernel_ms_total": round(total, 4), "k_expand_seed_ms": round(mine, 4),
              "k_expand_seed_share": round(mine / total, 5) if total else None,
              "kernels": {k: round(v["ms"], 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}})
    lib.mlkem_b200_set_streams(0)
    lib.mlkem_b200_keys_free(handle)
    if args.out:
        out.close()


if __name__ == "__main__":
    main()
