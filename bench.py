#!/usr/bin/env python3
"""bench.py -- BASELINE.json's headline metric on B200: batched ML-KEM-768 Encaps + Decaps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--log2-items L] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[3]): 2^22 synthetic ML-KEM-768 items PER GPU; one step = Encaps_internal over
all items followed by Decaps_internal over the resulting ciphertexts with 10 % of them tampered (FO
re-encryption + implicit rejection on the device).  Inputs are derived on the device from the global item
index (crystals-kyber_b200/workload.py), keys are generated on the device before the timed region.

  value     encaps+decaps pairs per second, whole job, inputs and outputs resident in HBM
  e2e       the same step through the C ABI with HOST buffers (pinned): H2D of ek, m, dk, c and D2H of
            c, K, K' inside the timed region; e2e.copy_ceiling = the same buffers through the same staging
            pipeline with no kernels (mlkem_b200_copy_probe), measured in the same run on all ranks at once
  e2e_keyed the same step with the keys resident on the GPU (mlkem_b200_keys_*): only m, c and K cross PCIe
  cross_n_digest
            a FIXED global range of 2^20 items split over the ranks; checksum of checksums of c, K, K'
            compared with the oracle-derived fixture tests/golden/config4_digest.json at every rank count
  roofline  the dominant kernel (fused matrix expansion + matrix-vector product) against the INT32
            alu-pipe issue rate measured live on the same GPU (mlkem_b200_int32_peak)
  cpu_baseline / --impl reference
            the reference itself (oracle/_ref, compiled from /root/reference by oracle/Makefile) timed on
            the box's host cores on a bounded sample of the same workload

Multi-GPU: one process per GPU under torchrun; ranks take contiguous shards of the global index range, no
collective on the data path; timing is the max over ranks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PS = 768
METRIC = "ML-KEM-768 Encaps+Decaps ops/s"
UNIT = "encaps+decaps pairs/s"


def emit(obj):
    print(json.dumps(obj), flush=True)


# --dump-outputs: 8192 items x (1088 + 32 + 32) values as float32 = 37.7 MB per dump, whatever the batch size
DUMP_ROWS = 8192


def dump_rows(n: int):
    """Indices (sorted) of the items whose outputs --dump-outputs writes: every item when n <= DUMP_ROWS, else a sample drawn
    with a fixed seed, so that two builds run with the same arguments dump the same items."""
    import numpy as np

    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU code on the host cores
# ----------------------------------------------------------------------------------------------------
def reference_pairs_per_s(threads: int, pairs_per_thread: int, steps: int, warmup: int, detail: bool = False):
    """Times oracle/_ref (the unmodified reference behind ref_shim.c) on `threads` host threads.
    Falls back to the oracle port when the compiled reference did not travel.  Returns a dict.
    detail: also one thread alone (-O2), and the per-call times of NTT / InverseNTT / MultiplyNTTs (SURVEY 8(d))."""
    import numpy as np

    from oracle.oracle import REF_G_SO, REF_SO, Oracle, Reference, build

    build()
    orc = Oracle()
    n = threads * pairs_per_thread
    rng = np.random.default_rng(20261018)
    d, z, m = (rng.integers(0, 256, (n, 32), dtype=np.uint8) for _ in range(3))
    ek, dk = orc.keygen(PS, d, z)  # setup only (not timed, not part of the measured path)
    out = {"cores": threads, "sample": f"{n} ML-KEM-768 encaps+decaps pairs per step on {threads} threads"}
    if os.path.exists(REF_SO):
        ref = Reference(REF_SO)
        for _ in range(warmup):  # a warm-up step is one pair per thread (20 ms per operation: nothing to warm but the caches)
            ref.time_pairs(PS, ek[:threads], dk[:threads], m[:threads], threads)
        out["warmup_steps_run"] = warmup
        ts = [ref.time_pairs(PS, ek, dk, m, threads)[0] for _ in range(steps)]
        t = sum(ts) / len(ts)
        _, c, K = ref.time_pairs(PS, ek[:threads], dk[:threads], m[:threads], threads)
        oc, oK = orc.encaps(PS, ek[:threads], m[:threads])
        assert (c == oc).all() and (K == oK).all(), "reference and oracle disagree"
        out.update(kind="reference", value=n / t, ms_per_step=1e3 * t,
                   build="gcc -O2 of /root/reference/{ml_kem.c,sha3.c} via oracle/ref_shim.c")
        if os.path.exists(REF_G_SO):  # the reference's own makefile flags (-Wall -g => -O0), one thread, for the record
            rg = Reference(REF_G_SO)
            tg, _, _ = rg.time_pairs(PS, ek[:2], dk[:2], m[:2], 1)
            out["makefile_flags_1thread_pairs_per_s"] = 2 / tg
        if detail:
            t1, _, _ = ref.time_pairs(PS, ek[:4], dk[:4], m[:4], 1)
            out["O2_1thread_pairs_per_s"] = 4 / t1
            # SURVEY 8(d): the three operations on their own through the reference's *_internal functions, and KeyGen on all threads
            tk, ek4, dk4 = ref.time_keygen(PS, d[:4], z[:4], 1)
            te, c4, K4 = ref.time_encaps(PS, ek[:4], m[:4], 1)
            td, Kd4 = ref.time_decaps(PS, dk[:4], c4, 1)
            assert (ek4 == ek[:4]).all() and (dk4 == dk[:4]).all() and (Kd4 == K4).all(), "reference and oracle disagree"
            tka, _, _ = ref.time_keygen(PS, d[: 8 * threads], z[: 8 * threads], threads)
            out["O2_1thread_per_operation"] = {"keygen_per_s": 4 / tk, "encaps_per_s": 4 / te, "decaps_per_s": 4 / td,
                                               "sample": "4 calls each of KeyGen_internal / Encaps_internal / Decaps_internal (-O2), one thread"}
            out["keygen_per_s_all_threads"] = 8 * threads / tka
            f = rng.integers(0, 3329, 256, dtype=np.uint16)
            g = rng.integers(0, 3329, 256, dtype=np.uint16)
            tn, ti, tm = ref.time_ring(f, g, 2000)  # ml_kem.c:287, :336, :415 -- 2 000 calls each, one thread
            out["ring_1thread"] = {"ntt_polys_per_s": 1 / tn, "intt_polys_per_s": 1 / ti, "multiply_ntts_polys_per_s": 1 / tm,
                                   "sample": "2000 calls each of NTT / InverseNTT / MultiplyNTTs of the reference (-O2), one thread"}
    else:
        import ctypes

        t0 = time.perf_counter()
        for _ in range(steps):
            c, K = orc.encaps(PS, ek, m)
            orc.decaps(PS, dk, c)
        t = (time.perf_counter() - t0) / steps
        out.update(kind="port", value=n / t, ms_per_step=1e3 * t, build="oracle/mlkem_oracle.c (OpenMP), reference .so absent")
    out["unit"] = UNIT
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # 32 pairs per thread and step: about 1.3 s per step at 20 ms per operation, whatever the core count
    r = reference_pairs_per_s(threads, 32, args.steps, max(0, args.warmup))
    emit({
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16/u64 integer", "data": "synthetic",
        "config": {"workload": f"ML-KEM-768 Encaps_internal + Decaps_internal over 2^{args.log2_items} items per GPU, 10% of the ciphertexts tampered "
                               "(BASELINE configs[3]); 1 op = 1 encaps + 1 decaps",
                   "sample": r["sample"] + " (a bounded sample of that workload; the reference's Decaps_internal always re-encrypts and "
                                           "hashes, so its time does not depend on the tampered fraction)"},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                         "build": r["build"], "makefile_flags_1thread_pairs_per_s": r.get("makefile_flags_1thread_pairs_per_s"),
                         "warmup_steps_run": r.get("warmup_steps_run", 0)},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0, t1):
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power)}


# ----------------------------------------------------------------------------------------------------
# the GPU arm
# ----------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-items", type=int, default=22, help="items per GPU = 2^L (BASELINE config: 22)")
    ap.add_argument("--e2e-log2-items", type=int, default=None, help="items per GPU for the host-buffer leg (default: same)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--wc-inputs", action="store_true",
                    help="e2e input buffers in write-combined pinned memory where the box grants it (default: ordinary pinned memory)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm only (refused with --impl reference): write c, K (Encaps) and K' (Decaps) of the last timed step as "
                         "float32 DIR/<name>.npy, rank 0's items (all of them up to %d, else a fixed seeded sample of that many: "
                         "dump_rows)" % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the GPU arm computed; it does not apply to --impl reference")
        return run_reference_arm(args)

    import numpy as np
    import torch

    import crystals_kyber_b200 as ck
    from crystals_kyber_b200 import workload as wl
    from crystals_kyber_b200.lib import MEM_DEVICE, MEM_HOST, Opts

    FLAG_ASYNC = 2  # MLKEM_B200_FLAG_ASYNC

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Run this rank on the CPUs of its GPU's NUMA node: the pinned host buffers of the e2e leg are then first-touched in
    # the memory next to the GPU's PCIe root, which matters once 8 ranks pull 50 GB/s each out of host memory.
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = None
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        numa_cpus = len(os.sched_getaffinity(0))
    except Exception:  # no NVML / not permitted: keep the inherited affinity
        pass
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    kem = ck.MLKEM()
    lib = kem.lib
    sz = ck.sizes(PS)
    n = 1 << args.log2_items
    begin = rank * n  # weak scaling: every rank owns 2^L consecutive global items
    steps, warmup = args.steps, max(args.warmup, 3)

    # ---- setup (untimed): inputs from the global index, keys, the tampered ciphertexts
    d, z, m = wl.derive_inputs(lambda msg, ln: kem.hash_batch(1, msg, ln), begin, begin + n, dev)
    ek, dk = kem.keygen(PS, d, z)
    c0, K0 = kem.encaps(PS, ek, m)
    c_t = c0.clone()
    tampered = wl.tamper_inplace(c_t, begin)
    del d, z, c0
    c = torch.empty((n, sz["c"]), dtype=torch.uint8, device=dev)
    K = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    Kd = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    o_dev = Opts(local, MEM_DEVICE, stream.cuda_stream, 0, 0, 0)
    P = lambda t: C.c_void_p(t.data_ptr())

    def step_device():
        rc = lib.mlkem_b200_encaps_batch(PS, n, P(ek), P(m), P(c), P(K), C.byref(o_dev))
        rc |= lib.mlkem_b200_decaps_batch(PS, n, P(dk), P(c_t), P(Kd), C.byref(o_dev))
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    for _ in range(warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    launches0 = lib.mlkem_b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record(stream)
    for _ in range(steps):
        step_device()
    e1.record(stream)
    barrier()
    t_wall1 = time.time()
    launches = lib.mlkem_b200_launch_count() - launches0
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.summary(t_wall0, t_wall1)
    value = world * n * steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # here, before the legs below reuse c, K and Kd
        rows = torch.from_numpy(dump_rows(n)).to(dev)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("encaps_c", c), ("encaps_K", K), ("decaps_K", Kd)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.index_select(0, rows).cpu().numpy().astype(np.float32))

    # ---- the two operations on their own (SURVEY 8(d): Encaps/s, Decaps/s and pairs/s = 1 / (1/E + 1/D)), device-resident, per GPU
    def timed_device(fn, reps=3):
        fn()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a0.record(stream)
        for _ in range(reps):
            fn()
        a1.record(stream)
        torch.cuda.synchronize()
        return a0.elapsed_time(a1) / reps * 1e-3

    def only_encaps():
        if lib.mlkem_b200_encaps_batch(PS, n, P(ek), P(m), P(c), P(K), C.byref(o_dev)):
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    def only_decaps():
        if lib.mlkem_b200_decaps_batch(PS, n, P(dk), P(c_t), P(Kd), C.byref(o_dev)):
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    t_enc, t_dec = timed_device(only_encaps), timed_device(only_decaps)
    per_op = {"encaps_per_s_per_gpu": n / t_enc, "decaps_per_s_per_gpu": n / t_dec, "pairs_per_s_per_gpu_from_the_two": n / (t_enc + t_dec)}

    # ---- per-kernel durations: the same steps again with the chunks serialised on one stream (in the timed region
    # above, kernels of different chunks overlap on two streams, so a kernel's own duration cannot be read there)
    kem.set_streams(1)
    kem.profile(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    p0.record(stream)
    for _ in range(steps):
        step_device()
    p1.record(stream)
    barrier()
    kem.profile(False)
    kem.set_streams(0)  # back to the library default
    serial_ms = p0.elapsed_time(p1)
    prof = kem.profile_report()

    # ---- correctness of what was just timed (outside the timed region)
    ok = torch.ones(n, dtype=torch.bool, device=dev)
    ok[tampered] = False
    same = (Kd == K0).all(dim=1)
    assert bool((K == K0).all()) and bool(same[ok].all()) and not bool(same[~ok].any()), "KEM round trip failed"

    # ---- e2e: host buffers through the C ABI (H2D + kernels + D2H per step)
    ne = 1 << (args.e2e_log2_items if args.e2e_log2_items is not None else args.log2_items)
    ne = min(ne, n)

    wc_allocs, wc_bytes = [], [0, 0]  # write-combined / ordinary pinned bytes of the e2e input buffers

    def pinned_copy(t):
        """Host copy of a device tensor in an INPUT buffer of the e2e legs: pinned, and with --wc-inputs write-combined
        (mlkem_b200_host_alloc_wc) where the box grants it.  The CPU only ever fills these buffers; write-combined pages are not
        snooped when the GPU reads them, which is worth nothing on one GPU and 7 % (H2D alone) to 44 % (both directions busy) of
        the box's aggregate copy rate with eight (tools/pcie_bw.py, profiles/pcie_bw_r02_8gpu.json) -- but such mappings are a
        limited resource (8 ranks x 20 GB were refused), so the default is ordinary pinned memory."""
        nbytes = t.numel() * t.element_size()
        ptr = lib.mlkem_b200_host_alloc_wc(nbytes) if args.wc_inputs else None
        if ptr:
            wc_allocs.append(ptr)
            wc_bytes[0] += nbytes
            h = torch.frombuffer((C.c_ubyte * nbytes).from_address(ptr), dtype=torch.uint8).view(t.dtype).view(t.shape)
        else:  # write-combined mappings are a limited resource (8 ranks x 20 GB did not fit on the 8-GPU box): ordinary pinned memory
            wc_bytes[1] += nbytes
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        return h

    def timed_host(step_fn):
        """`steps` synchronous host-memory steps, all ranks at once, max over ranks; one untimed step first."""
        step_fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step_fn()  # synchronous: returns when the results are in host memory
        barrier()
        return max_over_ranks(time.perf_counter() - t0)

    def copy_probe(ins, outs, o=None):
        """mlkem_b200_copy_probe over the given pinned tensors: the copies of a real call, no kernels."""
        o = o_host if o is None else o
        ni, no = len(ins), len(outs)
        ip = (C.c_void_p * ni)(*[t.data_ptr() for t in ins])
        ib = (C.c_size_t * ni)(*[t.shape[1] * t.element_size() for t in ins])
        op = (C.c_void_p * no)(*[t.data_ptr() for t in outs])
        ob = (C.c_size_t * no)(*[t.shape[1] * t.element_size() for t in outs])
        rc = lib.mlkem_b200_copy_probe(ins[0].shape[0], ni, ip, ib, no, op, ob, C.byref(o))
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    def probe_pair(a_ins, a_outs, b_ins, b_outs):
        """The copies of an Encaps call and of a Decaps call issued like the measured step: both asynchronous, one wait."""
        copy_probe(a_ins, a_outs, o_async)
        copy_probe(b_ins, b_outs, o_async)
        if lib.mlkem_b200_synchronize(local, None):
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    hek, hm, hdk, hct = (pinned_copy(t[:ne]) for t in (ek, m, dk, c_t))
    hc = torch.empty((ne, sz["c"]), dtype=torch.uint8, pin_memory=True)
    hK = torch.empty((ne, 32), dtype=torch.uint8, pin_memory=True)
    hKd = torch.empty((ne, 32), dtype=torch.uint8, pin_memory=True)
    o_host = Opts(local, MEM_HOST, None, 0, 0, 0)
    o_async = Opts(local, MEM_HOST, None, 0, 0, FLAG_ASYNC)

    def step_host():
        rc = lib.mlkem_b200_encaps_batch(PS, ne, P(hek), P(hm), P(hc), P(hK), C.byref(o_host))
        rc |= lib.mlkem_b200_decaps_batch(PS, ne, P(hdk), P(hct), P(hKd), C.byref(o_host))
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    def step_host_overlapped():
        # the same two calls issued back to back without waiting in between (MLKEM_B200_FLAG_ASYNC), one wait at the end: the D2H
        # tail of Encaps overlaps the H2D head of Decaps
        rc = lib.mlkem_b200_encaps_batch(PS, ne, P(hek), P(hm), P(hc), P(hK), C.byref(o_async))
        rc |= lib.mlkem_b200_decaps_batch(PS, ne, P(hdk), P(hct), P(hKd), C.byref(o_async))
        rc |= lib.mlkem_b200_synchronize(local, None)
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    e2e_sync_s = timed_host(step_host)
    assert bool((hK == K0[:ne].cpu()).all()) and bool((hKd == Kd[:ne].cpu()).all()), "host-buffer path disagrees with device path"
    hK.zero_(); hKd.zero_()
    e2e_s = timed_host(step_host_overlapped)
    assert bool((hK == K0[:ne].cpu()).all()) and bool((hKd == Kd[:ne].cpu()).all()), "asynchronous host-buffer path disagrees with device path"
    e2e_value = world * ne * steps / e2e_s
    h2d = ne * (sz["ek"] + 32 + sz["dk"] + sz["c"])
    d2h = ne * (sz["c"] + 32 + 32)
    # the copy-only ceiling of exactly these calls, on this box, now, every rank at once
    hscratch = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (hc, hK, hKd)]  # (empty_like would not be pinned)
    ceil_s = timed_host(lambda: probe_pair([hek, hm], hscratch[:2], [hdk, hct], hscratch[2:]))
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "items_per_gpu": ne,
           "ms_per_step": 1e3 * e2e_s / steps, "h2d_GBps_per_gpu": h2d * steps / e2e_s / 1e9,
           "input_buffers": {"write_combined_bytes": wc_bytes[0], "pinned_bytes": wc_bytes[1],
                             "note": "--wc-inputs: write-combined (mlkem_b200_host_alloc_wc) where the box grants it; default ordinary pinned memory"},
           "path": "mlkem_b200_encaps_batch + mlkem_b200_decaps_batch with MLKEM_B200_MEM_HOST (pinned buffers), distinct keys per item; the two "
                   "calls of a step are issued with MLKEM_B200_FLAG_ASYNC and followed by one mlkem_b200_synchronize",
           "blocking_calls": {"value": world * ne * steps / e2e_sync_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_sync_s / steps,
                              "path": "the same two calls, each returning only when its results are in host memory (round 1's e2e)"},
           "copy_ceiling": {"value": world * ne * steps / ceil_s, "unit": UNIT, "ms_per_step": 1e3 * ceil_s / steps,
                            "h2d_GBps_per_gpu": h2d * steps / ceil_s / 1e9,
                            "how": "mlkem_b200_copy_probe: the same buffers through the same chunks / staging slots / streams, issued the same way "
                                   "(two asynchronous calls, one wait), no kernels; all ranks concurrently, same run"},
           "frac_of_copy_ceiling": ceil_s / e2e_s, "cpus_of_gpu_numa_node": numa_cpus}
    del hdk  # (10 GB of pinned memory per rank; the buffers below are reused for the keyed legs)

    # ---- e2e_keyed: the keys live on the GPU (SURVEY 8(d) config 4 allows 2^16 distinct keys reused cyclically); per step only
    # m (32 B) in and c, K (1120 B) out for Encaps, c (1088 B) in and K' (32 B) out for Decaps cross PCIe.  The table is built
    # from the 64-byte seeds once (set-up, like the pinned copies above).
    nk = min(1 << 16, ne)
    d16, z16, _ = wl.derive_inputs(lambda msg, ln: kem.hash_batch(1, msg, ln), begin, begin + nk, dev)
    table = kem.keys_load(PS, seeds=(d16, z16), expand=True)  # MLKEM_B200_FLAG_EXPAND_KEYS: A^ of every key sampled once, here
    hck, hKk, hKdk = hscratch  # outputs of the keyed calls

    def step_keyed_encaps():
        if lib.mlkem_b200_encaps_keyed_batch(table.handle, ne, None, P(hm), P(hck), P(hKk), C.byref(o_host)):
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    step_keyed_encaps()
    hctk = hct  # the ciphertexts Decaps receives: those of the keyed Encaps, 10 % tampered (tampered in cached memory, then copied)
    wl.tamper_inplace(hck.numpy(), begin)
    hctk.copy_(hck)

    def step_keyed(o=o_host):
        rc = lib.mlkem_b200_encaps_keyed_batch(table.handle, ne, None, P(hm), P(hck), P(hKk), C.byref(o))
        rc |= lib.mlkem_b200_decaps_keyed_batch(table.handle, ne, None, P(hctk), P(hKdk), C.byref(o))
        rc |= lib.mlkem_b200_synchronize(local, None)
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    keyed_sync_s = timed_host(step_keyed)
    keyed_s = timed_host(lambda: step_keyed(o_async))
    # parity of the keyed path: identical to the unkeyed device-memory calls with the keys gathered explicitly (a 2^17-item slice,
    # two trips around the table), and the round trip holds on everything
    nv = min(ne, 1 << 17)
    ek16, dk16 = kem.keygen(PS, d16, z16)
    gidx = torch.arange(nv, device=dev) % nk
    cv, Kv = kem.encaps(PS, ek16[gidx], m[:nv])
    Kdv = kem.decaps(PS, dk16[gidx], hctk[:nv].to(dev))
    torch.cuda.synchronize()
    assert bool((hck[:nv] == cv.cpu()).all()) and bool((hKk[:nv] == Kv.cpu()).all()) and bool((hKdk[:nv] == Kdv.cpu()).all()), \
        "keyed calls disagree with the unkeyed calls"
    same_k = (hKdk == hKk).all(dim=1)
    tam_k = torch.zeros(ne, dtype=torch.bool)
    tam_k[tampered[tampered < ne].cpu()] = True
    assert bool(same_k[~tam_k].all()) and not bool(same_k[tam_k].any()), "keyed KEM round trip failed"
    ceil_k_s = timed_host(lambda: probe_pair([hm], [hc, hK], [hctk], [hKd]))
    # the keyed step with everything resident in HBM (CUDA events on the launching stream, like `value`)
    dctk = hctk[:n].to(dev) if ne == n else None
    keyed_dev_ms = None
    if dctk is not None:
        def step_keyed_device():
            rc = lib.mlkem_b200_encaps_keyed_batch(table.handle, n, None, P(m), P(c), P(K), C.byref(o_dev))
            rc |= lib.mlkem_b200_decaps_keyed_batch(table.handle, n, None, P(dctk), P(Kd), C.byref(o_dev))
            if rc:
                raise RuntimeError(lib.mlkem_b200_last_error().decode())

        for _ in range(2):
            step_keyed_device()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        k0.record(stream)
        for _ in range(steps):
            step_keyed_device()
        k1.record(stream)
        barrier()
        keyed_dev_ms = max_over_ranks(k0.elapsed_time(k1))
        assert bool((Kd.cpu() == hKdk).all()) and bool((K.cpu() == hKk).all()), "keyed device path disagrees with keyed host path"
        del dctk
    h2d_k, d2h_k = ne * (32 + sz["c"]), ne * (sz["c"] + 32 + 32)
    e2e_keyed = {"value": world * ne * steps / keyed_s, "unit": UNIT, "h2d_bytes_per_step": h2d_k, "d2h_bytes_per_step": d2h_k,
                 "items_per_gpu": ne, "distinct_keys_per_gpu": nk, "ms_per_step": 1e3 * keyed_s / steps,
                 "path": "mlkem_b200_encaps_keyed_batch + mlkem_b200_decaps_keyed_batch with MLKEM_B200_MEM_HOST; key table built once by "
                         "mlkem_b200_keys_from_seeds, key of item i = i mod 2^16; outputs checked against the unkeyed calls",
                 "blocking_calls": {"value": world * ne * steps / keyed_sync_s, "unit": UNIT, "ms_per_step": 1e3 * keyed_sync_s / steps},
                 "copy_ceiling": {"value": world * ne * steps / ceil_k_s, "unit": UNIT, "ms_per_step": 1e3 * ceil_k_s / steps,
                                  "how": "copy probe of the same buffers, issued the same way (two asynchronous calls, one wait)"},
                 "frac_of_copy_ceiling": ceil_k_s / keyed_s, "vs_unkeyed_e2e": e2e_s / keyed_s,
                 "device_resident": None if keyed_dev_ms is None else {
                     "value": world * n * steps / (keyed_dev_ms * 1e-3), "unit": UNIT, "ms_per_step": keyed_dev_ms / steps,
                     "note": "the same keyed step with m, c and the keys' expanded matrices resident in HBM: 23 instead of 86 Keccak permutations per pair"},
                 "key_table": "MLKEM_B200_FLAG_EXPAND_KEYS: 2400 B dk + 32 B H(ek) + 4608 B expanded matrix per key"}
    # decaps keyed only (a server), encaps with one 1184-byte ek per item (clients with distinct keys)

    def step_keyed_decaps_only():
        rc = lib.mlkem_b200_encaps_batch(PS, ne, P(hek), P(hm), P(hc), P(hK), C.byref(o_async))
        rc |= lib.mlkem_b200_decaps_keyed_batch(table.handle, ne, None, P(hctk), P(hKdk), C.byref(o_async))
        rc |= lib.mlkem_b200_synchronize(local, None)
        if rc:
            raise RuntimeError(lib.mlkem_b200_last_error().decode())

    kd_s = timed_host(step_keyed_decaps_only)
    e2e_keyed["decaps_keyed_only"] = {"value": world * ne * steps / kd_s, "unit": UNIT, "h2d_bytes_per_step": ne * (sz["ek"] + 32 + sz["c"]),
                                      "d2h_bytes_per_step": d2h_k, "ms_per_step": 1e3 * kd_s / steps, "vs_unkeyed_e2e": e2e_s / kd_s}
    table.free()
    del hek, hm, hck, hct, hctk, hc, hscratch, ek16, dk16, cv, Kv, Kdv
    for ptr in wc_allocs:
        lib.mlkem_b200_host_free(ptr)
    os.sched_setaffinity(0, all_cpus)  # the CPU baseline below uses every host core again
    sampler.stop()

    # ---- cross-N byte identity (SURVEY 8(e)): a FIXED global range of 2^20 items, contiguous shards over the ranks; per output a
    # checksum of checksums over 2^14-item blocks, gathered on rank 0 and compared with the oracle-derived fixture
    digest = cross_n_digest(kem, wl, torch, dist, dev, rank, world)

    # ---- roofline of the dominant kernel, INT32 alu pipe
    peaks = kem.int32_peak()
    k_, eta1, _, du, dv = ck.PARAMS[PS]
    ops = wl.op_counts(k_, eta1, du, dv)
    mv = [(name, v) for name, v in prof.items() if "k_sample_matvec" in name]
    mv_ms = sum(v["ms"] for _, v in mv)
    # the fused kernel and its clean-up pass (k_sample_matvec_list, the 2.7 % of rows that need a 4th XOF block) are one
    # unit of work: time of both, launches of the fused kernel
    mv_launches = sum(v["launches"] for name, v in mv if "_list" not in name)
    total_kernel_ms = sum(v["ms"] for v in prof.values())
    items_per_launch = 2.0 * n * steps / max(mv_launches, 1)  # Encrypt runs once in Encaps and once in Decaps
    achieved = ops["matvec_encrypt"] * items_per_launch / (mv_ms / max(mv_launches, 1) * 1e-3) if mv_ms else None
    peak = max(peaks["lop3"], peaks["shf"])
    roofline = {
        "bound": "int32",
        "kernel": "k_sample_matvec + its clean-up pass k_sample_matvec_list (SampleNTT x k^2 + MultiplyNTTs x k^2 + InverseNTT x k, fused)",
        "achieved": achieved / 1e12 if achieved else None, "peak": peak / 1e12, "unit": "Tera int32 op/s",
        "frac": achieved / peak if achieved else None,
        "peak_source": "measured live: mlkem_b200_int32_peak (LOP3/SHF issue rate, alu pipe); MEASURED_PEAKS.json has no integer figure",
        "algorithmic_ops_per_item": ops["matvec_encrypt"], "items_per_launch": items_per_launch,
        "avg_launch_ms": mv_ms / max(mv_launches, 1), "share_of_step_kernel_time": mv_ms / total_kernel_ms if total_kernel_ms else None,
        # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture of this round
        # (profiles/ncu_kem_kernels_r02_summary.csv, 65 536-item launches of tools/prof_kem.py: Encaps' store-mode launch
        # 133.7 + 42.1 MB and its clean-up pass 8.7 MB = 2 815 B/item; Decaps' compare-mode launch 199.7 + 4.2 MB and its clean-up
        # pass 10.8 MB = 3 276 B/item), scaled to this run's launch size -- a figure derived from that capture, not re-measured here
        "traffic": 0.5 * (2815.0 + 3276.0) * items_per_launch, "traffic_bytes_per_item": {"encrypt_store": 2815, "encrypt_compare": 3276},
        "traffic_source": "profiles/ncu_kem_kernels_r02_summary.csv (ncu --set full, tools/prof_kem.py), scaled by items_per_launch",
        "algorithmic_bytes_per_item": 32 + 1536 + 384 + 960,
        "whole_step": {"algorithmic_ops_per_pair": ops["encaps"] + ops["decaps"],
                       "achieved": (ops["encaps"] + ops["decaps"]) * value / world / 1e12, "frac": (ops["encaps"] + ops["decaps"]) * value / world / peak},
        "peaks_tera_ops": {k: v / 1e12 for k, v in peaks.items()},
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16/u64 integer", "data": "synthetic",
        "config": {"workload": f"ML-KEM-768 Encaps_internal + Decaps_internal over 2^{args.log2_items} items per GPU, 10% of the ciphertexts tampered "
                               "(BASELINE configs[3]); 1 op = 1 encaps + 1 decaps",
                   "items_per_gpu": n, "distinct_keys": n, "tamper": "i % 10 == 3", "sharding": f"contiguous index shards x{world}, no collective",
                   "cache": "working set 20 GB per GPU >> 126 MB L2, no flush needed"},
        "per_operation": per_op, "e2e": e2e, "e2e_keyed": e2e_keyed, "cross_n_digest": digest,
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "kernel_ms_per_step": {k: v["ms"] / steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
        "serialized_ms_per_step": serial_ms / steps,
    }

    # ---- extras: the other numbers BASELINE's metric names (NTT polys/s, codec GB/s, KeyGen/s), rank 0 only
    if rank == 0 and not args.no_extras:
        line["extra"] = extras(kem, torch, dev, peaks)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = reference_pairs_per_s(os.cpu_count() or 1, 32, 1, 1, detail=True)
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "build", "makefile_flags_1thread_pairs_per_s",
                                                  "O2_1thread_pairs_per_s", "O2_1thread_per_operation",
                                                  "keygen_per_s_all_threads", "ring_1thread") if k in r}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def cross_n_digest(kem, wl, torch, dist, dev, rank, world):
    """KeyGen -> Encaps -> Decaps(10 % tampered) over global items [0, 2^L) of the workload, rank r taking the contiguous shard
    [r 2^L / W, (r+1) 2^L / W).  Returns {c, K, Kd: sha256 of the per-block sha256s} on rank 0, checked against
    tests/golden/config4_digest.json (made by the ORACLE on the CPU: tests/golden/make_digest.py)."""
    import hashlib

    import crystals_kyber_b200 as ck

    fixture = json.load(open(os.path.join(ROOT, "tests", "golden", "config4_digest.json")))
    L, B = fixture["log2_items"], fixture["log2_block"]
    total, blk = 1 << L, 1 << B
    lo, hi = ck.shard_range(total, rank, world)
    assert lo % blk == 0 and hi % blk == 0, "shard boundaries must be block boundaries"
    d, z, m = wl.derive_inputs(lambda msg, ln: kem.hash_batch(1, msg, ln), lo, hi, dev)
    ek, dk = kem.keygen(PS, d, z)
    c, K = kem.encaps(PS, ek, m)
    ct = c.clone()
    wl.tamper_inplace(ct, lo)
    Kd = kem.decaps(PS, dk, ct)
    torch.cuda.synchronize()
    mine = {name: wl.block_hashes(t.cpu().numpy(), blk) for name, t in (("c", c), ("K", K), ("Kd", Kd))}
    per_rank = {k: hashlib.sha256(v).hexdigest() for k, v in mine.items()}
    if dist is not None:
        parts = [None] * world
        dist.all_gather_object(parts, mine)  # block hashes only (32 B per 2^14 items); not on the measured path
    else:
        parts = [mine]
    if rank != 0:
        return None
    got = {k: wl.combine_block_hashes([p[k] for p in parts]) for k in ("c", "K", "Kd")}
    ok = got == fixture["digest"]
    assert ok, f"cross-N digest mismatch at {world} ranks: {got} != {fixture['digest']}"
    return {"items_total": total, "ranks": world, "block_items": blk, "sha256_of_block_sha256s": got, "rank0_shard_sha256": per_rank,
            "equals_oracle_fixture": ok, "fixture": "tests/golden/config4_digest.json (oracle/mlkem_oracle.c on the CPU, tests/golden/make_digest.py)"}


def extras(kem, torch, dev, peaks):
    """BASELINE config 2 (2^20 polynomials through NTT / InverseNTT / MultiplyNTTs) and the codec kernels,
    device-resident, CUDA-event timed; working sets (0.5-1.5 GB) are far larger than L2."""
    from crystals_kyber_b200 import workload as wl

    out = {}
    n = 1 << 20
    g = torch.Generator(device=dev).manual_seed(20261018)
    f = torch.randint(0, 3329, (n, 256), generator=g, device=dev, dtype=torch.int16).view(torch.uint16)
    h = torch.randint(0, 3329, (n, 256), generator=g, device=dev, dtype=torch.int16).view(torch.uint16)

    def timeit(fn, reps=5):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3

    hbm = None
    try:
        hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    alu = max(peaks["lop3"], peaks["shf"])
    for name, fn, opsn, bytesn in (("ntt", lambda: kem.ntt(f), wl.OPS_NTT, 1024), ("intt", lambda: kem.intt(f), wl.OPS_INTT, 1024),
                                   ("multiply_ntts", lambda: kem.multiply_ntts(f, h), wl.OPS_MULNTT, 1536)):
        t = timeit(fn)
        out[name] = {"polys_per_s": n / t, "int32_frac_of_alu_pipe": opsn * n / t / alu, "gb_per_s": bytesn * n / t / 1e9,
                     "hbm_frac": (bytesn * n / t / 1e9 / hbm) if hbm else None}
    for d in (4, 10, 12):
        t = timeit(lambda: kem.compress_encode(f, d))
        b = (512 + 32 * d) * n
        out[f"compress_encode_{d}"] = {"gb_per_s": b / t / 1e9, "hbm_frac": (b / t / 1e9 / hbm) if hbm else None}
    nk = 1 << 20
    seeds = torch.randint(0, 256, (2, nk, 32), generator=g, device=dev, dtype=torch.uint8)
    for ps in (512, 768, 1024):
        t = timeit(lambda: kem.keygen(ps, seeds[0], seeds[1]), reps=2)
        out[f"keygen_{ps}_per_s"] = nk / t
    out["hbm_peak_gbs"] = hbm
    out.update(caller_view(kem))
    return out


def caller_view(kem):
    """What a caller of the reference gets (VERDICT r01 item 7): the latency of KEM_KeyGen / KEM_Encaps / KEM_Decaps through
    include/ml_kem.h (stride-4 unions, malloc'ed results, a batch of one on the GPU per call), and the throughput of the batched
    host-memory entry points for batches of 2^0 .. 2^14 items in ordinary (pageable) host memory."""
    import statistics

    import numpy as np

    lib = kem.lib

    class PARAMS(C.Structure):
        _fields_ = [("k", C.c_uint), ("n1", C.c_uint), ("n2", C.c_uint), ("du", C.c_uint), ("dv", C.c_uint)]

    class PKE(C.Structure):
        _fields_ = [("ek", C.POINTER(C.c_uint)), ("dk", C.POINTER(C.c_uint)), ("ek_len", C.c_uint), ("dk_len", C.c_uint)]

    class KEM(C.Structure):
        _fields_ = [("K", C.c_uint * 32), ("c", C.POINTER(C.c_uint)), ("c_len", C.c_uint)]

    lib.init.restype, lib.init.argtypes = PARAMS, [C.c_int]
    lib.KEM_KeyGen.restype, lib.KEM_KeyGen.argtypes = PKE, [C.POINTER(PARAMS)]
    lib.KEM_Encaps.restype, lib.KEM_Encaps.argtypes = KEM, [C.POINTER(PARAMS), C.POINTER(C.c_uint), C.c_uint]
    lib.KEM_Decaps.restype = C.POINTER(C.c_uint)
    lib.KEM_Decaps.argtypes = [C.POINTER(PARAMS), C.POINTER(C.c_uint), C.c_uint, C.POINTER(C.c_uint), C.c_uint]
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    p = lib.init(PS)
    lat = {"KEM_KeyGen": [], "KEM_Encaps": [], "KEM_Decaps": []}
    for it in range(23):
        t0 = time.perf_counter()
        keys = lib.KEM_KeyGen(C.byref(p))
        t1 = time.perf_counter()
        enc = lib.KEM_Encaps(C.byref(p), keys.ek, keys.ek_len)
        t2 = time.perf_counter()
        Kd = lib.KEM_Decaps(C.byref(p), keys.dk, keys.dk_len, enc.c, enc.c_len)
        t3 = time.perf_counter()
        assert bool(Kd) and all((Kd[i] & 0xFF) == (enc.K[i] & 0xFF) for i in range(32))
        for ptr in (keys.ek, keys.dk, enc.c, Kd):
            libc.free(ptr)
        if it >= 3:
            for name, dt in zip(lat, (t1 - t0, t2 - t1, t3 - t2)):
                lat[name].append(dt * 1e6)
    out = {"drop_in_api_latency_us": {k: {"median": statistics.median(v), "min": min(v)} for k, v in lat.items()},
           "drop_in_api_note": "include/ml_kem.h entry points, one operation per call: layout conversion + H2D + the kernel chain of one item "
                               "+ D2H + synchronise; the reference takes about 20 ms per operation at -O2 (cpu_baseline.O2_1thread_pairs_per_s)"}
    # is a batch of one launch-bound?  sum of the kernels' own durations (event hooks) against the wall time of the calls
    one = [np.zeros((1, w), np.uint8) for w in (32, 32, 32)]
    ek1, dk1 = kem.keygen(PS, one[0], one[1])
    kem.encaps(PS, ek1, one[2])
    kem.profile(True)
    t0 = time.perf_counter()
    for _ in range(10):
        c1, K1 = kem.encaps(PS, ek1, one[2])
        kem.decaps(PS, dk1, c1)
    wall_us = (time.perf_counter() - t0) / 10 * 1e6
    kem.profile(False)
    rep = kem.profile_report()
    kern_us = sum(v["ms"] for v in rep.values()) / 10 * 1e3
    out["batch_of_one"] = {"wall_us_per_encaps_plus_decaps": wall_us, "kernel_us": kern_us, "launches": sum(v["launches"] for v in rep.values()) // 10,
                           "note": "kernel_us = sum of the kernels' own durations (CUDA events around every launch, which add their own overhead to the "
                                   "wall time here); the rest is launch gaps, the pageable copies and the synchronisation"}
    rng = np.random.default_rng(7)
    nmax = 1 << 14
    d, z, m = (rng.integers(0, 256, (nmax, 32), dtype=np.uint8) for _ in range(3))
    ek, dk = kem.keygen(PS, d, z)
    sweep = {}
    for lg in range(0, 15, 2):
        nb = 1 << lg
        a_ek, a_dk, a_m = (np.ascontiguousarray(x[:nb]) for x in (ek, dk, m))
        reps = 20 if lg <= 8 else 6
        for _ in range(2):
            c, K = kem.encaps(PS, a_ek, a_m)
            kem.decaps(PS, a_dk, c)
        t0 = time.perf_counter()
        for _ in range(reps):
            c, K = kem.encaps(PS, a_ek, a_m)
            Kd = kem.decaps(PS, a_dk, c)
        dt = (time.perf_counter() - t0) / reps
        assert (Kd == K).all()
        sweep[str(nb)] = {"pairs_per_s": nb / dt, "us_per_pair_of_calls": dt * 1e6}
    out["small_batch_host_memory"] = sweep
    return out


if __name__ == "__main__":
    main()
