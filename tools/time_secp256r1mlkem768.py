#!/usr/bin/env python3
"""What P-256 and the SecP256r1MLKEM768 hybrid cost on the device, next to the plain ML-KEM-768 calls and the X25519MLKEM768
hybrid:

  p256       mlkem_b200_p256_public_batch and _p256_ecdh_batch at 2^20 and 2^22 items, device memory;
  hybrid     at 2^22 items, device memory and host memory (pinned buffers): the five SecP256r1MLKEM768 calls (keygen, encaps,
             decaps, seeded keygen, seeded encaps), the plain FIPS ML-KEM-768 calls (_kem_keygen_seeded_batch,
             _kem_encaps_seeded_batch, _decaps_batch) and the seeded X25519MLKEM768 calls, alternating within each repetition;
  profile    the per-kernel split of each SecP256r1MLKEM768 call (mlkem_b200_profile, one stream, a separate pass);
  host       `cryptography`'s P-256 ECDH on one core of this host: exchange() with ready key objects, and key construction +
             exchange, the work the device path replaces;
  ceiling    the SASS of k_p256 (cuobjdump): instructions of the ladder loop body times 256, over the measured issue rates of
             mlkem_b200_int32_peak (IMAD and IMAD.HI for the fma-pipe instructions).

Every call is timed with the host clock around the call and a device synchronise, after one warm-up call of the same size.
One JSON object per line (GPU name, power limit and max SM clock in the first), to --out or stdout.
    python tools/time_secp256r1mlkem768.py --out profiles/secp256r1mlkem768_r04.jsonl
"""
import argparse
import collections
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import crystals_kyber_b200 as ck
from crystals_kyber_b200.lib import MEM_DEVICE, MEM_HOST, Opts
from time_device_rng import Pinned, gpu_info

FIPS = 1
SEED = C.c_char_p(bytes(range(32)))


def P(t):
    return C.c_void_p(t.data_ptr())


def timed(fn, reps):
    fn()  # warm-up of this size
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        rc = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        assert rc == 0, rc
    return ts


def alternate(fns, reps):
    """{name: [seconds]} with the calls of one repetition in turn."""
    for fn in fns.values():
        assert fn() == 0
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            t0 = time.perf_counter()
            assert fn() == 0
            torch.cuda.synchronize()
            out[k].append(time.perf_counter() - t0)
    return out


def buffers(device, n, widths):
    if device:
        return [torch.empty((n, w), dtype=torch.uint8, device="cuda") for w in widths]
    return [Pinned(ck.load(), (n, w)) for w in widths]


def hybrid_fns(lib, n, device):
    """The calls, on buffers of their memory space: client shares / secrets come from a seeded KeyGen, the server shares from a
    seeded Encaps of them; the explicit-randomness calls reuse the scalars of the client secrets."""
    mem = MEM_DEVICE if device else MEM_HOST
    stream = torch.cuda.current_stream().cuda_stream if device else None
    o = Opts(-1, mem, stream, 0, 0, FIPS)
    cs, sec, share, ss, ek, dk, ct, K, xcs, xsec, xshare, rnd = buffers(device, n, [1249, 2432, 1153, 64, 1184, 2400, 1088, 32, 1216, 2432,
                                                                                    1120, 32])
    status = torch.empty(n, dtype=torch.int32, device="cuda") if device else Pinned(lib, (n * 4,))
    if device:
        rnd.copy_(torch.randint(0, 128, (n, 32), dtype=torch.uint8, device="cuda"))  # < 2^255: in-range scalars, also d / z / m
    else:
        rnd.a[:] = np.random.default_rng(4).integers(0, 128, rnd.a.shape, dtype=np.uint8)
    fns = {
        "secp_keygen_seeded": lambda: lib.mlkem_b200_secp256r1mlkem768_keygen_seeded_batch(n, SEED, P(cs), P(sec), C.byref(o)),
        "secp_keygen": lambda: lib.mlkem_b200_secp256r1mlkem768_keygen_batch(n, P(rnd), P(rnd), P(rnd), P(cs), P(sec), P(status), C.byref(o)),
        "x25519_keygen_seeded": lambda: lib.mlkem_b200_x25519mlkem768_keygen_seeded_batch(n, SEED, P(xcs), P(xsec), C.byref(o)),
        "mlkem_keygen_seeded": lambda: lib.mlkem_b200_kem_keygen_seeded_batch(768, n, SEED, P(ek), P(dk), C.byref(o)),
        "secp_encaps_seeded": lambda: lib.mlkem_b200_secp256r1mlkem768_encaps_seeded_batch(n, P(cs), SEED, P(share), P(ss), P(status),
                                                                                           C.byref(o)),
        "secp_encaps": lambda: lib.mlkem_b200_secp256r1mlkem768_encaps_batch(n, P(cs), P(rnd), P(rnd), P(share), P(ss), P(status), C.byref(o)),
        "x25519_encaps_seeded": lambda: lib.mlkem_b200_x25519mlkem768_encaps_seeded_batch(n, P(xcs), SEED, P(xshare), P(ss), P(status),
                                                                                          C.byref(o)),
        "mlkem_encaps_seeded": lambda: lib.mlkem_b200_kem_encaps_seeded_batch(768, n, P(ek), 1184, SEED, P(ct), P(K), C.byref(o)),
        "secp_decaps": lambda: lib.mlkem_b200_secp256r1mlkem768_decaps_batch(n, P(sec), P(share), P(ss), P(status), C.byref(o)),
        "x25519_decaps": lambda: lib.mlkem_b200_x25519mlkem768_decaps_batch(n, P(xsec), P(xshare), P(ss), P(status), C.byref(o)),
        "mlkem_decaps": lambda: lib.mlkem_b200_decaps_batch(768, n, P(dk), P(ct), P(K), C.byref(o)),
    }
    return fns, (cs, sec, share, ss, ek, dk, ct, K, xcs, xsec, xshare, rnd, status)


def host_p256_rate(seconds=2.0):
    try:
        from cryptography.hazmat.primitives import serialization
        from cryptography.hazmat.primitives.asymmetric import ec
    except ImportError:
        return {"what": "host_p256_ecdh", "result": "not measured: cryptography is not installed"}
    enc = serialization.Encoding.X962, serialization.PublicFormat.UncompressedPoint
    curve = ec.SECP256R1()
    sk = [ec.generate_private_key(curve) for _ in range(256)]
    pk = [k.public_key() for k in sk[::-1]]
    raw_sk = [k.private_numbers().private_value for k in sk]
    raw_pk = [p.public_bytes(*enc) for p in pk]
    out = {"what": "host_p256_ecdh", "cryptography": __import__("cryptography").__version__, "threads": 1}
    for name, body in (("exchange_only", lambda i: sk[i].exchange(ec.ECDH(), pk[i])),
                       ("with_key_objects", lambda i: ec.derive_private_key(raw_sk[i], curve).exchange(
                           ec.ECDH(), ec.EllipticCurvePublicKey.from_encoded_point(curve, raw_pk[i])))):
        done, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            for i in range(256):
                body(i)
            done += 256
        out[f"{name}_per_s"] = round(done / (time.perf_counter() - t0))
    return out


def sass_ladder():
    """Opcode counts of k_p256's ladder loop from cuobjdump: the largest innermost loop (the others are the squaring runs of the
    inversion, one squaring each)."""
    so = ck.load()._name
    txt = subprocess.run(f"cuobjdump -sass {so} | c++filt", shell=True, capture_output=True, text=True).stdout
    insts, cur = [], ""
    for line in txt.splitlines():
        f = re.search(r"Function : (.*)", line)
        if f:
            cur = f.group(1)
            continue
        if "k_p256(" not in cur:
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(@!?U?P\d+\s+)?([A-Z0-9_.]+)(.*?);", line)
        if m:
            insts.append((int(m.group(1), 16), m.group(3), m.group(4)))
    spans = []
    for addr, op, rest in insts:
        t = re.search(r"0x([0-9a-f]+)", rest) if op.startswith("BRA") else None
        if t and int(t.group(1), 16) < addr:
            spans.append((int(t.group(1), 16), addr))
    inner = [(lo, hi) for lo, hi in spans if not any(lo <= a < hi for _, a in spans if a != hi)]  # no loop inside (the grid-stride loop has)
    if not inner:
        return None
    lo, hi = max(inner, key=lambda s: s[1] - s[0])
    body = [o for a, o, _ in insts if lo <= a <= hi]
    hist = collections.Counter(o.split(".")[0] if not o.startswith("IMAD") else o for o in body)
    return {"loop_instructions": len(body), "total_instructions": len(insts), "histogram": dict(hist.most_common())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n", type=int, default=1 << 22)
    args = ap.parse_args()
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    lib = ck.load()
    kem = ck.MLKEM()
    emit({"what": "setup", **gpu_info()})
    # the P-256 primitive in device memory
    for n in (1 << 20, args.n):
        g = torch.Generator(device="cuda").manual_seed(n)
        k = torch.randint(0, 128, (n, 32), dtype=torch.uint8, device="cuda", generator=g)  # < 2^255: in range
        pub = torch.empty((n, 65), dtype=torch.uint8, device="cuda")
        ss = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
        status = torch.empty(n, dtype=torch.int32, device="cuda")
        o = Opts(-1, MEM_DEVICE, torch.cuda.current_stream().cuda_stream, 0, 0, 0)
        assert lib.mlkem_b200_p256_public_batch(n, P(k), P(pub), P(status), C.byref(o)) == 0
        peer = pub.roll(1, 0).contiguous()  # item i's key against item i - 1's public key
        for name, fn in (("p256_public", lambda: lib.mlkem_b200_p256_public_batch(n, P(k), P(pub), P(status), C.byref(o))),
                         ("p256_ecdh", lambda: lib.mlkem_b200_p256_ecdh_batch(n, P(k), P(peer), P(ss), P(status), C.byref(o)))):
            ts = timed(fn, args.reps)
            assert int((status != 0).sum()) == 0
            emit({"what": name, "mem": "device", "n": n, "s": [round(t, 5) for t in ts], "M_per_s": round(n / statistics.median(ts) / 1e6, 2)})
        del k, pub, peer, ss, status
    # the hybrid next to the plain calls and the X25519 hybrid
    for device in (True, False):
        try:
            fns, keep = hybrid_fns(lib, args.n, device)
        except MemoryError as e:
            emit({"what": "hybrid", "mem": "device" if device else "host", "n": args.n, "result": f"not measured: {e}"})
            continue
        # inputs: keys of every group, then a server share / ciphertext for each
        for name in ("secp_keygen_seeded", "x25519_keygen_seeded", "mlkem_keygen_seeded", "secp_encaps_seeded", "x25519_encaps_seeded",
                     "mlkem_encaps_seeded"):
            assert fns[name]() == 0
        torch.cuda.synchronize()
        groups = (("secp_keygen_seeded", "secp_keygen", "x25519_keygen_seeded", "mlkem_keygen_seeded"),
                  ("secp_encaps_seeded", "secp_encaps", "x25519_encaps_seeded", "mlkem_encaps_seeded"),
                  ("secp_decaps", "x25519_decaps", "mlkem_decaps"))
        for grp in groups:
            if grp[0] == "secp_decaps":  # the server shares of the seeded keys again (secp_keygen / _encaps overwrote them)
                for name in ("secp_keygen_seeded", "secp_encaps_seeded", "x25519_encaps_seeded"):
                    assert fns[name]() == 0
            r = alternate({k: fns[k] for k in grp}, args.reps)
            for name, ts in r.items():
                emit({"what": name, "mem": "device" if device else "host", "n": args.n, "s": [round(t, 5) for t in ts],
                      "M_per_s": round(args.n / statistics.median(ts) / 1e6, 2)})
        if device:  # per-kernel split, one stream
            kem.set_streams(1)
            for name in ("secp_keygen_seeded", "secp_encaps_seeded", "secp_decaps"):
                kem.profile(True)
                assert fns[name]() == 0
                torch.cuda.synchronize()
                rep = kem.profile_report()
                kem.profile(False)
                total = sum(v["ms"] for v in rep.values())
                split = {k.strip("()"): {"ms": round(v["ms"], 3), "share": round(v["ms"] / total, 4)} for k, v in
                         sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
                emit({"what": "profile", "call": name, "n": args.n, "kernel_ms_total": round(total, 3), "kernels": split})
            kem.set_streams(0)
        del fns, keep
        torch.cuda.empty_cache()
    emit(host_p256_rate())
    peak = kem.int32_peak()
    emit({"what": "int32_peak", **{k: round(v / 1e12, 3) for k, v in peak.items()}, "unit": "T thread-ops/s"})
    s = sass_ladder()
    if s is None:
        emit({"what": "ceiling", "result": "not measured: cuobjdump gave no SASS"})
    else:
        fma = sum(v for k, v in s["histogram"].items() if k.startswith("IMAD"))
        wide = sum(v for k, v in s["histogram"].items() if k.startswith(("IMAD.WIDE", "IMAD.HI")))
        per_sm = 256 * s["loop_instructions"]
        ceil_fma = 1.0 / (256 * ((fma - wide) / peak["imad"] + wide / peak["imad_hi"]))  # IMAD.WIDE issued at the IMAD.HI rate
        ceil_issue = peak["lop3+imad"] / per_sm
        emit({"what": "ceiling", "ladder_loop": s, "ladder_instructions_per_scalarmult": per_sm, "ladder_fma_pipe_per_scalarmult": 256 * fma,
              "ceiling_fma_M_per_s": round(ceil_fma / 1e6, 2), "ceiling_issue_M_per_s": round(ceil_issue / 1e6, 2),
              "note": "ladder only (the inversion adds 255 squarings and 13 products, the point check 4 products); fma pipe: IMAD at the IMAD rate, IMAD.WIDE / IMAD.HI at the IMAD.HI rate"})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
