"""CPU: the reference arm of bench.py prints one JSON line with the contract's keys (the GPU arm needs a B200).
GPU: the arrays --dump-outputs writes are the optima of the benchmark batch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args) -> dict:
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), stdout=subprocess.PIPE,
                         text=True, check=True, cwd=ROOT).stdout
    return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])


def test_reference_arm_prints_the_contract_line(tmp_path):
    d = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "lp_relaxations_per_sec" and d["unit"] == "LP/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and "workload" in d["config"]
    out = {k: np.load(tmp_path / f"{k}.npy") for k in ("status", "optF", "x", "basis")}
    assert all(a.dtype == np.float64 for a in out.values())
    count = out["status"].shape[0]
    assert count >= 1 and (out["status"] == 0).all() and out["x"].shape == (count, 128)
    assert out["basis"].shape == (count, 64)


def test_bytes_per_pivot_formula():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.bytes_per_pivot(64, 128) == 131072            # SURVEY.md 8d: C2
    assert bench.bytes_per_pivot(1024, 2048) == 33554432       # C4: 33.55 MB per pivot


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_gpu_arm_dumps_the_last_step(tmp_path):
    """--steps really sets the timed steps, and the dumped arrays are the benchmark batch's optima (oracle parity on
    a slice, 1e-9 relative)."""
    import oracle
    sys.path.insert(0, ROOT)
    import bench
    d = _bench("--steps", "2", "--warmup", "0", "--quick", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    out = {k: np.load(tmp_path / f"{k}.npy") for k in ("status", "optF", "x", "basis", "stats")}
    assert all(a.dtype == np.float64 for a in out.values())
    assert out["x"].shape == (bench.BATCH, bench.N) and out["stats"].shape == (bench.BATCH, 8)
    assert (out["status"] == 0).all()
    c, A, b = bench.make_batch(0)
    sl = slice(0, 64)
    o = oracle.simplex_batch(c[sl], A[sl], b[sl], threads=oracle.num_hw_threads())
    for k in ("optF", "x"):
        assert np.max(np.abs(out[k][sl] - o[k]) / np.maximum(1.0, np.abs(o[k]))) <= 1e-9, k
