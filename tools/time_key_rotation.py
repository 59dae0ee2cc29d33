#!/usr/bin/env python3
"""Cost of rotating keys in a resident ML-KEM-768 key table of 2^16 keys, plain and expanded (MLKEM_B200_FLAG_EXPAND_KEYS):

  replace      wall time of mlkem_b200_keys_replace (from dk) / _replace_from_seeds of 1, 256 and 2^16 slots, with host
               (numpy) and device (torch) sources -- a set-up call, so the host clock around it includes the device work;
  export_ek    wall time of mlkem_b200_keys_export_ek of all 2^16 rows to host and to device memory;
  keyed        device-resident keyed Encaps + Decaps of 2^22 items per step, steps alternating between two variants in the same
               run: with a replace of 256 slots (from device seeds) after the step's Decaps, and without.

One JSON object per line (GPU name and power limit in the first), to --out or stdout.
    python tools/time_key_rotation.py --out profiles/key_rotation_r03.jsonl
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

import crystals_kyber_b200 as ck

PS, NK = 768, 1 << 16


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch": torch.__version__, "lib": ck.load()._name}


def wall(fn, reps):
    """Median and minimum host time of fn() in ms; fn returns when its device work is done."""
    fn()  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return {"median_ms": round(statistics.median(ts), 3), "min_ms": round(min(ts), 3), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--items", type=int, default=1 << 22, help="keyed Encaps + Decaps items per step")
    ap.add_argument("--steps", type=int, default=6, help="steps per variant of the keyed measurement")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the library has no CPU fallback")
    out = open(args.out, "w") if args.out else sys.stdout
    emit = lambda rec: (out.write(json.dumps(rec) + "\n"), out.flush())
    emit({"what": "setup", "param_set": PS, "keys": NK, **gpu_info()})

    kem = ck.MLKEM()
    rng = np.random.default_rng(1)
    d, z = (rng.integers(0, 256, (NK, 32), dtype=np.uint8) for _ in range(2))
    nd, nz = (rng.integers(0, 256, (NK, 32), dtype=np.uint8) for _ in range(2))
    _, ndk = kem.keygen(PS, nd, nz)
    dev = {"d": torch.from_numpy(nd).cuda(), "z": torch.from_numpy(nz).cuda(), "dk": torch.from_numpy(ndk).cuda()}
    torch.cuda.synchronize()
    for expand in (False, True):
        table = kem.keys_load(PS, seeds=(d, z), expand=expand)
        kind = "expanded" if expand else "plain"
        for count in (1, 256, NK):
            slots = rng.permutation(NK)[:count].astype(np.uint32)
            for src in ("seeds", "dk"):
                for mem in ("host", "device"):
                    if mem == "host":
                        args_ = {"seeds": (nd[:count], nz[:count])} if src == "seeds" else {"dk": ndk[:count]}
                    else:
                        args_ = {"seeds": (dev["d"][:count], dev["z"][:count])} if src == "seeds" else {"dk": dev["dk"][:count]}
                    r = wall(lambda: table.replace(slots, **args_), 3 if count == NK else 10)
                    emit({"what": "replace", "table": kind, "slots": count, "source": src, "mem": mem, **r})
        r = wall(lambda: table.export_ek(), 5)
        emit({"what": "export_ek", "table": kind, "rows": NK, "mem": "host", **r})

        def export_dev():
            table.export_ek(device=True)
            torch.cuda.synchronize()

        r = wall(export_dev, 10)
        emit({"what": "export_ek", "table": kind, "rows": NK, "mem": "device", **r})

        # keyed throughput with and without a 256-slot rotation per step, alternating
        n = args.items
        g = torch.Generator(device="cuda").manual_seed(2)
        m = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
        slots = rng.permutation(NK)[:256].astype(np.uint32)
        times = {"without": [], "with_replace_256": []}

        def step(rotate):
            c, K = kem.encaps_keyed(table, None, m)
            Kd = kem.decaps_keyed(table, None, c)
            if rotate:
                table.replace(slots, seeds=(dev["d"][:256], dev["z"][:256]))
            torch.cuda.synchronize()
            return K, Kd

        K, Kd = step(False)
        assert bool((K == Kd).all())
        step(True)
        for i in range(2 * args.steps):
            variant = "without" if i % 2 == 0 else "with_replace_256"
            t0 = time.perf_counter()
            step(variant != "without")
            times[variant].append(time.perf_counter() - t0)
        for variant, ts in times.items():
            med = statistics.median(ts)
            emit({"what": "keyed_encaps_decaps", "table": kind, "items_per_step": n, "variant": variant, "steps": len(ts),
                  "median_step_ms": round(1e3 * med, 3), "min_step_ms": round(1e3 * min(ts), 3),
                  "pairs_per_s_median": round(n / med)})
        del m
        table.free()
        torch.cuda.empty_cache()
    if args.out:
        out.close()


if __name__ == "__main__":
    main()
