"""Cost of the full posterior covariance (nngp_predict_cov) next to the diagonal-only prediction of the same batch.

Workload: N = 32768 training rows, D = 256, depth 3, T in {1024, 4096, 16384} test rows, 'nngp' and 'ntk'.  Inputs and
outputs are device tensors (the wall time is the call, which returns synchronised, without PCIe copies of the T x T
result).  Per case: wall ms per call, the stage split of nngp_stats (stats_level 1) per call, and the rate of the
pred_var stage from the flop model of that stage over its device time, against the DMMA peak measured in the same run:
    'nngp': C -= V V^T on the lower triangle                      T^2 N
    'ntk' : the variance row-dot V M (2 T N^2), P = -V M (2 T N^2), C -= P V^T, U V^T, V U^T (3 T^2 N)
The whole call's flop model: the prediction (T (N^2 + 2 N D); 'ntk': T (4 N^2 + 2 N D), two solves and the row-dot)
+ T^2 D (test x test Gram) + the covariance products above.
The card's name and power limit are read in the same run.   python tools/cov_probe.py [--out FILE] [--t 1024,4096,16384]
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

N, D, DEPTH = 32768, 256, 3


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        f"--id={torch.cuda.current_device()}"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def flops(kind, T):
    """(whole call, pred_var stage, diagonal-only prediction) of nngp_predict_cov; 'ntk' prediction: two solves and
    the variance row-dot V M (2 T N^2), which runs in the pred_var stage."""
    if kind == "nngp":
        pred, extra, var_stage = T * (N * N + 2 * N * D), T * T * N, T * T * N
    else:
        pred, extra, var_stage = T * (4 * N * N + 2 * N * D), 2 * T * N * N + 3 * T * T * N, 4 * T * N * N + 3 * T * T * N
    return pred + T * T * D + extra, var_stage, pred


def timed(fn, reps):
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--t", default="1024,4096,16384")
    args = ap.parse_args()
    import torch
    ts = [int(v) for v in args.t.split(",")]
    xtr, ytr, xte, _ = synth.make_problem(N, max(ts), D)
    xd = torch.from_numpy(np.ascontiguousarray(xte)).cuda()
    rec = {"what": "nngp_predict_cov vs nngp_predict", "N": N, "D": D, "depth": DEPTH, "card": card(), "cases": []}
    for kind in ("nngp", "ntk"):
        h = _lib.Handle(depth=DEPTH, kernel_type=kind, stats_level=1)
        h.fit(xtr, ytr)
        rec.setdefault("dmma_peak_tflops", h.dmma_peak_tflops())
        for T in ts:
            x = xd[:T]
            md = torch.empty(T, dtype=torch.float64, device="cuda")
            vd = torch.empty(T, dtype=torch.float64, device="cuda")
            cd = torch.empty((T, T), dtype=torch.float64, device="cuda")
            reps = 3 if T >= 16384 else 5
            pred_ms = timed(lambda: h.predict(x, mean_out=md, var_out=vd), reps)
            h.predict_cov(x, mean_out=md, cov_out=cd)
            h.stats_reset()
            t0 = time.perf_counter()
            for _ in range(reps):
                h.predict_cov(x, mean_out=md, cov_out=cd)
            cov_ms = (time.perf_counter() - t0) / reps * 1e3
            s = h.stats()
            stages = {k: round(s[k] / reps, 3) for k in ("pred_total_ms", "pred_gram_ms", "pred_trsm_ms", "pred_var_ms",
                                                         "d2h_ms")}
            total_f, var_f, pred_f = flops(kind, T)
            case = {"kind": kind, "T": T, "predict_ms": round(pred_ms, 3), "predict_cov_ms": round(cov_ms, 3),
                    "cov_over_predict_time": round(cov_ms / pred_ms, 3), "cov_over_predict_flop": round(total_f / pred_f, 3),
                    "stages_ms": stages, "flop": total_f, "var_stage_flop": var_f,
                    "var_stage_tflops": round(var_f / (stages["pred_var_ms"] * 1e-3) / 1e12, 2),
                    "call_tflops": round(total_f / (cov_ms * 1e-3) / 1e12, 2)}
            case["var_stage_of_peak"] = round(case["var_stage_tflops"] / rec["dmma_peak_tflops"], 3)
            rec["cases"].append(case)
            print(json.dumps(case), flush=True)
            del cd
        h.close()
        torch.cuda.empty_cache()
    line = json.dumps(rec)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
