"""CPU: the reference arm of bench.py (the CPU restatement timed as the baseline) honours the output contract:
exactly one JSON line on stdout with the agreed keys.  One GPU test runs the B200 arm at C2 and checks what it dumps."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--workload", "c2", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "predicted_queries_per_sec" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and "workload" in d["config"]
    assert d["config"]["test_rows_per_gpu"] == 65536 and d["config"]["n_train"] == 8192   # the B200 arm's config keys
    cb, e2e = d["cpu_baseline"], d["e2e"]
    assert cb["blas_threads"] in (-1, cb["cores"]) and cb["rows_per_step"] == 2048
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    mean, var = np.load(tmp_path / "mean.npy"), np.load(tmp_path / "var.npy")
    assert mean.dtype == var.dtype == np.float64 and mean.shape == var.shape == (2048,)
    assert np.all(np.isfinite(mean)) and np.all(var > 0)


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the timed path returned: the posterior of the seeded C2 test rows, bit for bit what a
    fresh handle predicts for them; --steps sets the number of timed steps."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "c2", "--steps", "2", "--warmup", "1",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and d["config"]["test_rows_per_gpu"] == 65536
    mean, var = np.load(tmp_path / "mean.npy"), np.load(tmp_path / "var.npy")
    assert mean.dtype == var.dtype == np.float64 and mean.shape == var.shape == (65536,)
    from nngp_b200 import _lib, synth
    x = synth.encodings(8192, 128, 1)
    h = _lib.Handle(depth=2, diag_reg=1e-3)
    h.fit(x, synth.labels(x))
    m, v = h.predict(synth.encodings(65536, 128, 2))
    assert np.array_equal(mean, m) and np.array_equal(var, v)


def test_reference_arm_keeps_all_blas_threads_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm must still use every core (VERDICT r1 weak #2)."""
    import os
    env = dict(os.environ, OMP_NUM_THREADS="1", WORLD_SIZE="2", RANK="0", LOCAL_RANK="0")
    code = ("import sys; sys.argv=['bench.py','--impl','reference']; import runpy; m=runpy.run_path(%r, run_name='x'); "
            "print(m['blas_threads'](), m['_CORES'])" % str(ROOT / "bench.py"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(ROOT), env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    threads, cores = map(int, r.stdout.split()[-2:])
    assert threads in (-1, cores), (threads, cores)


def test_b200_arm_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_reference_arm_under_torchrun_only_rank0_works_and_prints():
    """Contract: launched like the B200 arm (torch.distributed.run, N ranks), rank 0 alone runs the CPU arm and prints
    ONE line; the other ranks exit 0 without work."""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(ROOT / "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--workload", "c2"],
                       capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and "x2" in d["config"]["parallelism"]
    cb = d["cpu_baseline"]
    assert cb["blas_threads"] in (-1, cb["cores"]), cb      # torchrun's OMP_NUM_THREADS=1 must not reach OpenBLAS
