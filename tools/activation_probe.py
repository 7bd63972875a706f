"""Cost of the activation in the Gram epilogue: ReLU, LeakyRelu(0.1) and Erf() side by side.

Per activation, on one GPU:
  * the Gram kernel alone (nngp_kernel of N = 32768 rows, D = 256, depth 3, 'nngp': lower tiles + mirror; stats_level 2
    gives the device time of the gemm_nt_kernel<EPI_GRAM, ACT> launches): ms, TFLOP/s of its 2 M N D / 2 flop and the
    share of the DMMA peak measured in the same run (nngp_diag_dmma_peak);
  * the C3 prediction rate: fit N = 32768, D = 256, depth 3, then posterior mean + variance of 131072 test rows (host
    arrays in and out, as bench.py's C3), queries/s over `--reps` calls after one warm-up call.
The card's name and power limit are read in the same run.   python tools/activation_probe.py [--out FILE] [--reps 3]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "nngp-src_b200"):
    sys.path.insert(0, str(p))
from nngp_b200 import _lib, synth  # noqa: E402

N, T, D, DEPTH = 32768, 131072, 256, 3
ACTS = {"relu": _lib.RELU, "leaky_relu_0.1": _lib.Activation("abrelu", 0.1, 1.0),
        "erf": _lib.Activation("erf", 1.0, 1.0, 0.0)}


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        f"--id={torch.cuda.current_device()}"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def gram(act, x_dev, out_dev, reps):
    h = _lib.Handle(depth=DEPTH, stats_level=2, activation=act)
    h.kernel(x_dev, out=out_dev)                      # warm-up
    h.stats_reset()
    for _ in range(reps):
        h.kernel(x_dev, out=out_dev)
    s = h.stats()
    ms = s["gram_ms"] / reps
    return {"gram_ms": ms, "gram_tflops": s["gram_flops"] / reps / ms / 1e9}


def c3(act, xtr, ytr, xte, reps):
    h = _lib.Handle(depth=DEPTH, stats_level=1, activation=act)
    h.fit(xtr, ytr)
    mean, var = np.empty(T), np.empty(T)
    h.predict(xte, mean_out=mean, var_out=var)        # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        h.predict(xte, mean_out=mean, var_out=var)
    sec = (time.perf_counter() - t0) / reps
    assert np.all(np.isfinite(mean)) and np.all(np.isfinite(var))
    return {"c3_predict_s": sec, "c3_queries_per_s": T / sec}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    info = {"card": card(), "workload": {"N": N, "T": T, "D": D, "depth": DEPTH}}
    info["dmma_peak_tflops"] = _lib.Handle().dmma_peak_tflops()
    xtr, ytr, xte, _ = synth.make_problem(N, T, D)
    x_dev = torch.from_numpy(xtr).cuda()
    out_dev = torch.empty((N, N), dtype=torch.float64, device="cuda")
    rows = {}
    for name, act in ACTS.items():
        r = gram(act, x_dev, out_dev, args.reps)
        r["gram_share_of_dmma_peak"] = r["gram_tflops"] / info["dmma_peak_tflops"]
        r.update(c3(act, xtr, ytr, xte, args.reps))
        rows[name] = r
        print(name, json.dumps(r), flush=True)
    for name, r in rows.items():
        r["gram_time_vs_relu"] = r["gram_ms"] / rows["relu"]["gram_ms"]
        r["c3_rate_vs_relu"] = r["c3_queries_per_s"] / rows["relu"]["c3_queries_per_s"]
    info["activations"] = rows
    text = json.dumps(info, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
