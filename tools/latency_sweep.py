"""nngp_predict latency at small and medium batch sizes, default handle vs latency mode (explicit L^-1), plus fit
times with the pieces of the Cholesky (Gram, factorisation, solve).  Host numpy buffers in, mean + variance
out, wall clock around the C-ABI call, averages after warm-up.  Prints one JSON object.
    python tools/latency_sweep.py [N] [D]"""
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "nngp-src_b200"):
    sys.path.insert(0, str(p))
from nngp_b200 import _lib, synth  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
D = int(sys.argv[2]) if len(sys.argv) > 2 else 128
xtr, ytr, xte, _ = synth.make_problem(N, 40000, D)
out = {"what": f"nngp_predict latency (host buffers in, mean+var out) at N={N}, D={D}, depth 2, one B200; wall clock, "
               "average of 10 calls after 3 warm-up calls", "n_train": N, "dim": D}


def sweep(h, sizes, reps=10):
    res = {}
    for t in sizes:
        x = np.ascontiguousarray(xte[:t])
        m, v = np.empty(t), np.empty(t)
        for _ in range(3):
            h.predict(x, mean_out=m, var_out=v)
        t0 = time.perf_counter()
        for _ in range(reps):
            h.predict(x, mean_out=m, var_out=v)
        res[str(t)] = round((time.perf_counter() - t0) / reps * 1e3, 4)
    return res


sizes = [1, 8, 32, 128, 256, 1024, 2048, 4096, 8192, 20000, 40000]
h = _lib.Handle(stats_level=0)
h.fit(xtr, ytr)
out["default_ms"] = sweep(h, sizes)
m_ref, v_ref = h.predict(xte[:4096])
h.close()

hl = _lib.Handle(stats_level=1, latency_mode=True)
hl.fit(xtr, ytr)
hl.stats_reset()
hl.fit(xtr, ytr)
s = hl.stats()
out["latency_mode_fit"] = {"fit_total_ms": s["fit_total_ms"], "inverse_ms": s["inverse_ms"],
                           "inverse_tflops": N**3 / 3 / max(s["inverse_ms"], 1e-9) / 1e9}
hl2 = _lib.Handle(stats_level=0, latency_mode=True)
hl2.fit(xtr, ytr)
os.environ["NNGP_LATENCY_ROWS"] = "1000000"
out["latency_mode_ms"] = sweep(hl2, sizes)
ml, vl = hl2.predict(xte[:4096])
del os.environ["NNGP_LATENCY_ROWS"]
out["latency_vs_default_max_rel_var_diff"] = float(np.max(np.abs(vl - v_ref) / np.abs(v_ref)))
out["latency_vs_default_mean_bitwise"] = bool(np.array_equal(ml, m_ref))
out["flop_floor_ms_1024_rows"] = 1024 * (float(N) * N + 2.0 * N * D) / 37.0e12 * 1e3
hl.close()
hl2.close()

# fit times: N sweep (the key names the panel solve, a DMMA product, as in the earlier sweeps under profiles/)
fits = {}
for n in (2048, 4096, 8192, 16384):
    if n > N and n > 16384:
        continue
    x = synth.encodings(n, D, 1)
    y = synth.labels(x)
    hf = _lib.Handle(stats_level=1)
    hf.fit(x, y)
    hf.stats_reset()
    for _ in range(3):
        hf.fit(x, y)
    s = hf.stats()
    fits[str(n)] = {"fit_total_ms": s["fit_total_ms"] / 3, "chol_ms": s["fit_chol_ms"] / 3, "gram_ms": s["fit_gram_ms"] / 3,
                    "solve_ms": s["fit_solve_ms"] / 3, "chol_tflops": n**3 / 3 / (s["fit_chol_ms"] / 3) / 1e9}
    hf.close()
out["fit_ms_panel_dmma"] = fits
print(json.dumps(out, indent=1))
