"""GPU test of bench.py --dump-outputs: the files hold what the timed Encaps + Decaps step returned for the sampled items."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_timed_step_outputs(oracle, tmp_path):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bench import DUMP_ROWS, dump_rows
    from crystals_kyber_b200 import workload as wl

    L = 14  # 2^14 items > DUMP_ROWS: the sampled path

    def bench(steps, *extra):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0", "--log2-items",
                              str(L), "--no-extras", "--no-cpu-baseline", *extra],
                             cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])

    one, two = bench(1), bench(2, "--dump-outputs", str(tmp_path))
    # gpu_launches counts the kernels launched inside the timed region: --steps 2 must launch twice those of --steps 1
    assert one["steps"] == 1 and two["steps"] == 2 and one["gpu_launches"] > 0 and two["gpu_launches"] == 2 * one["gpu_launches"]
    dumped = {name: np.load(tmp_path / f"{name}.npy") for name in ("encaps_c", "encaps_K", "decaps_K")}
    assert sorted(os.listdir(tmp_path)) == sorted(f"{name}.npy" for name in dumped)
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20

    n = 1 << L
    rows = dump_rows(n)
    assert rows.size == DUMP_ROWS and (np.diff(rows) > 0).all()
    d, z, m = wl.derive_inputs(lambda msg, ln: oracle.hash_batch(1, msg, ln), 0, n)
    ek, dk = oracle.keygen(768, d, z)
    c, K = oracle.encaps(768, ek, m)
    ct = c.copy()
    wl.tamper_inplace(ct, 0)  # Decaps of the timed step gets the ciphertexts with bench's 10 % tampered
    Kd = oracle.decaps(768, dk, ct)
    for name, want in (("encaps_c", c), ("encaps_K", K), ("decaps_K", Kd)):
        assert dumped[name].dtype == np.float32 and dumped[name].shape == (DUMP_ROWS, want.shape[1])
        assert (dumped[name] == want[rows].astype(np.float32)).all(), name
    assert (dumped["decaps_K"] != dumped["encaps_K"]).any(axis=1).sum() > 0
