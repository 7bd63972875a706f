#!/usr/bin/env python
"""bench.py -- headline benchmark of the NNGP hot path on B200.

Metric (BASELINE.json): predicted queries/s (posterior mean + variance) at 1/2/4/8 B200, plus train-fit
seconds at N = 32k and % of measured FP64 tensor (DMMA) peak.  A "step" is one prediction pass over one batch
of synthetic test queries with the fitted model resident in HBM.  The default workload is C3 (the config
BASELINE.json names for the 1/2/4/8-GPU metric and the N = 32k fit): 32 768 train rows, 256-dim encodings,
depth-3 NNGP, 131 072 test rows per GPU (1M / 8).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c5] [--impl reference] [--dump-outputs DIR]

N>1 is launched by torchrun (one rank per GPU, NCCL): rank 0 fits, the fitted state is broadcast once (packed
lower triangle, nngp_b200.dist.broadcast_fit), each rank predicts its own shard of test rows (weak scaling:
per-GPU rows fixed), no data-path collective.  After that timed region rank 0 also measures the IN-PROCESS
multi-GPU path (one handle with n_gpus = N: peer-to-peer replication + row split behind the same C-ABI call the
reference's single-process callers make) and reports it under "in_process".
Rank 0 prints ONE JSON line.  `--dump-outputs DIR` also writes what the last timed step returned (posterior mean and
variance of every rank's test rows, in rank order) as float64 DIR/mean.npy and DIR/var.npy.  `--impl reference` times
the CPU restatement of the reference path (oracle/nngp_oracle.py: numpy/scipy -> OpenBLAS/LAPACK, the library class
jaxlib calls) on all the box's host cores; jax / neural-tangents are not installable, so no `oracle/_ref` exists
(DESIGN.md).
"""
from __future__ import annotations

import os
import sys

# The CPU legs must use every host core.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which
# would make OpenBLAS single-threaded: fix the BLAS pool size BEFORE numpy is imported.
_CORES = len(os.sched_getaffinity(0))
if "--impl" in sys.argv and "reference" in sys.argv or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_CORES)

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402
from pathlib import Path  # noqa: E402

import numpy as np  # noqa: E402

ROOT = Path(__file__).resolve().parent
for p in (ROOT, ROOT / "nngp-src_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

WORKLOADS = {
    # name: (n_train, n_test_per_gpu, dim, depth, join_dims, description)
    "c2": (8192, 65536, 128, 2, 0, "C2 synthetic single-table: 8k train / 64k test per GPU, 128-dim, depth-2 NNGP"),
    "c3": (32768, 131072, 256, 3, 0, "C3 synthetic: 32k train / 128k test per GPU (1M/8), 256-dim, depth-3 NNGP"),
    "c5": (16384, 524288, 512, 3, 96, "C5 multi-join: 16k train / 512k test per GPU (4M/8), 512-dim, depth-3 NNGP"),
}
METRIC, UNIT = "predicted_queries_per_sec", "queries/s"
CPU_ROWS = {"c2": 2048, "c3": 512, "c5": 1024}     # test rows per CPU step (bounded sample; throughput metric)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--slices", type=int, default=7, help="digit planes of the int8 variance side record (0 = skip it)")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2 side record / fit_n32k / in-process multi-GPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the posterior mean and variance of the last timed step to DIR/mean.npy, DIR/var.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_MAX_ROWS = 1 << 21     # 2 float64 arrays of at most 2M rows: 32 MiB per dump


def dump_outputs(out_dir: str, mean: np.ndarray, var: np.ndarray) -> None:
    """float64 mean.npy / var.npy of one timed step, in test-row order.  The inputs are seeded, so two builds run with
    the same arguments can be compared output for output.  Above DUMP_MAX_ROWS rows the same fixed, seeded sample of
    rows (ascending) is written for every run."""
    if mean.shape[0] > DUMP_MAX_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(mean.shape[0], DUMP_MAX_ROWS, replace=False))
        mean, var = mean[rows], var[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "mean.npy"), np.ascontiguousarray(mean, dtype=np.float64))
    np.save(os.path.join(out_dir, "var.npy"), np.ascontiguousarray(var, dtype=np.float64))


def make_config(workload: str, world: int) -> dict:
    """The `config` object -- identical in both arms (the reference arm states its bounded sample in cpu_baseline)."""
    n, t_rank, d, depth, _jd, desc = WORKLOADS[workload]
    return {"workload": desc, "n_train": n, "test_rows_per_gpu": t_rank, "dim": d, "depth": depth, "diag_reg": 1e-3,
            "parallelism": f"fit on rank 0 + broadcast, test rows sharded x{world}",
            "l2": "inputs larger than L2: per step the factor L (%.0f MB) and the K_* block (%.0f MB) stream "
                  "through a 126 MB L2" % (n * n * 8 / 1e6, t_rank * n * 8 / 1e6)}


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info
        return max([int(i.get("num_threads", 1)) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
    except Exception:  # noqa: BLE001
        return -1


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------- reference arm
def _oracle():
    sys.path.insert(0, str(ROOT / "oracle"))
    import nngp_oracle as oracle
    return oracle


def run_reference(args):
    """The reference's CPU path (restated: oracle) on all host cores.  Per step: posterior mean + variance of a
    bounded sample of test rows against the model fitted at the workload's full N (the fit itself is untimed here,
    its seconds are reported -- `fit_seconds` is the CPU side of "train fit seconds at N = 32k")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    oracle = _oracle()
    from nngp_b200 import synth
    n, _t, d, depth, jd, _desc = WORKLOADS[args.workload]
    rows = CPU_ROWS[args.workload]
    xtr, ytr, xte, _ = synth.make_problem(n, rows, d, join_dims=jd)
    t0 = time.perf_counter()
    fit = oracle.Fit(xtr, ytr, depth)
    t_fit = time.perf_counter() - t0
    for _ in range(args.warmup):
        fit.predict(xte[:256])
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        mean, var = fit.predict(xte)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, mean, var)
    sec = sum(times) / len(times)
    val = rows / sec
    sample = (f"oracle (numpy/scipy -> OpenBLAS, {blas_threads()} BLAS threads, {oracle.THREADS} threads for the "
              f"elementwise recursion): fit at N={n} in {t_fit:.1f}s (untimed), then posterior mean+var of {rows} "
              f"test rows per step ({sec:.2f}s/step); queries/s does not depend on the rows per step")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(args.workload, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": _CORES, "blas_threads": blas_threads(), "kind": "port",
                         "sample": sample, "rows_per_step": rows, "fit_seconds": t_fit},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------- B200 arm
def _traffic(workload: str, world: int):
    """Measured DRAM bytes per launch of the dominant kernel (ncu --set full) for THIS workload, or None.
    profiles/ncu_dominant_kernel.json holds one record per workload; a capture is valid for the per-GPU shape it was
    taken on (rows per GPU are fixed under weak scaling, so it holds at every N)."""
    f = ROOT / "profiles" / "ncu_dominant_kernel.json"
    if not f.exists():
        return None, None
    rec = json.loads(f.read_text()).get(workload)
    if not rec:
        return None, None
    return rec.get("dram_bytes_per_launch"), rec.get("source")


def _guard(fn):
    try:
        return fn()
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def _time_predict(torch, dist, world, h, local, xte_host, steps, warmup, sample_clocks=True, keep=None):
    """(device-resident ms, e2e ms, stats, e2e stats, clocks) of one handle predicting xte_host per step."""
    t = xte_host.shape[0]
    stream = torch.cuda.ExternalStream(h.stream, device=torch.device("cuda", local))
    xte_dev = torch.from_numpy(xte_host).cuda()
    mean_dev = torch.empty(t, dtype=torch.float64, device="cuda")
    var_dev = torch.empty(t, dtype=torch.float64, device="cuda")
    xte_pinned = torch.from_numpy(xte_host).pin_memory()
    mean_pin = torch.empty(t, dtype=torch.float64).pin_memory()
    var_pin = torch.empty(t, dtype=torch.float64).pin_memory()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def step_resident():      # inputs/outputs already in HBM: the C-ABI call on device pointers
        h.predict(xte_dev, want_var=True, mean_out=mean_dev, var_out=var_dev)

    def step_e2e():           # host buffers in, host results out, through the same C-ABI entry point
        h.predict(xte_pinned.numpy(), want_var=True, mean_out=mean_pin.numpy(), var_out=var_pin.numpy())

    for _ in range(warmup):
        step_resident()
    sampler = ClockSampler(local)
    h.stats_reset()
    if sample_clocks:
        sampler.start()
    ms_total = timed(step_resident, steps)
    clocks = sampler.stop() if sample_clocks else {}
    st = h.stats()
    e2e_steps = min(steps, 5)
    for _ in range(2):
        step_e2e()
    h.stats_reset()
    ms_e2e = timed(step_e2e, e2e_steps)
    st_e2e = h.stats()
    if not np.all(np.isfinite(mean_dev[:1024].cpu().numpy())) or not np.array_equal(mean_pin.numpy(), mean_dev.cpu().numpy()):
        raise SystemExit("bench.py: non-finite predictions, or the host-buffer and device-buffer paths disagree")
    if keep is not None:
        keep["mean"], keep["var"] = mean_dev.cpu().numpy(), var_dev.cpu().numpy()
    return ms_total, ms_e2e, e2e_steps, st, st_e2e, clocks


def _sliced_record(torch, dist, world, rank, local, _lib, args, depth, xtr, ytr, xte_host, t_rank, n, kept):
    """The same workload with the variance product on the INT8 tensor cores (cfg.variance_slices: tcgen05.mma kind::i8
    on digit planes of K_* and L^-1, FP64-equivalent to ~2^-7s).  Every rank fits its own handle (same data -> same
    bits) and predicts its shard; timed like the main region (barrier, CUDA events, max over ranks).  A side record:
    `value` stays the all-FP64 path.  Returns the record on rank 0, None elsewhere."""
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    peaks = json.loads(peaks_file.read_text()) if peaks_file.exists() else {}
    hs = _lib.Handle(depth=depth, diag_reg=1e-3, device=local, stats_level=2, variance_slices=args.slices)
    hs.fit(xtr, ytr)
    hs.stats_reset()
    hs.fit(xtr, ytr)
    sfit = hs.stats()
    ks = {}
    k_s = min(args.steps, 5)
    ms_s, ms_se, k_se, st_s, _st_se, clk_s = _time_predict(torch, dist, world, hs, local, xte_host, k_s, 3,
                                                           sample_clocks=(rank == 0), keep=ks if rank == 0 else None)
    hs.close()
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    tops = 2.0 * st_s["sliced_macs"] / max(st_s["sliced_ms"], 1e-9) / 1e9
    pk_s, pk_b = peaks.get("bf16_tflops_sustained"), peaks.get("bf16_tflops")
    tr = _traffic(args.workload + "_sliced", world)
    return {
        "what": "variance_slices=%d: V = K_* L^-T as %d exact int8 plane products on tcgen05 (kind::i8, TMEM "
                "accumulators) against the explicit inverse factor; the mean and the Gram stay FP64; every rank fits "
                "its own handle" % (args.slices, args.slices * (args.slices + 1) // 2 - 1),
        "value": world * k_s * t_rank / (ms_s / 1e3), "unit": UNIT, "n_gpus": world, "ms_per_step": ms_s / k_s, "steps": k_s,
        "e2e_value": world * k_se * t_rank / (ms_se / 1e3),
        "mean_bitwise_equal_fp64_path": bool(np.array_equal(ks["mean"], kept["mean"])),
        "var_max_rel_vs_fp64_path": float(np.max(np.abs(ks["var"] - kept["var"]) / np.abs(kept["var"]))),
        "std_max_rel_vs_fp64_path": float(np.max(np.abs(np.sqrt(ks["var"]) - np.sqrt(kept["var"])) / np.sqrt(kept["var"]))),
        "stage_ms_per_step": {k: st_s[k] / k_s for k in ("pred_gram_ms", "pred_trsm_ms", "sliced_ms", "pred_total_ms")},
        "fit_seconds_device": sfit["fit_total_ms"] / 1e3, "inverse_ms": sfit["inverse_ms"],
        "clocks": clk_s,
        "roofline": {"bound": "tensor", "kernel": "sliced_gemm_kernel (TMA + tcgen05.mma kind::i8 M128 N256 K32, int32 accumulators in TMEM)",
                     "achieved": tops, "unit": "TOP/s (int8, issued; rank 0)",
                     "peak": 2.0 * pk_b if pk_b else None, "frac": tops / (2.0 * pk_b) if pk_b else None,
                     "frac_of_sustained": tops / (2.0 * pk_s) if pk_s else None,
                     "peak_source": "2 x MEASURED_PEAKS.json bf16_tflops (burst; kind::i8 issues twice the MACs of kind::f16 per "
                                    "instruction slot).  The kernel runs for seconds under the 1 kW power cap (see clocks): "
                                    "frac_of_sustained is against 2 x bf16_tflops_sustained, the library's rate in that regime",
                     "traffic": tr[0], "traffic_source": tr[1],
                     "algorithmic_bytes_per_step": float(args.slices) * n * (t_rank + n / 2.0),
                     "fp64_equivalent_tflops": float(t_rank) * n * n * k_s / (st_s["sliced_ms"] / 1e3) / 1e12,
                     "share_of_step": st_s["sliced_ms"] / max(st_s["pred_total_ms"], 1e-9)},
    }


def run_b200(args):
    import torch
    import torch.distributed as dist
    from nngp_b200 import _lib, batch, predict, runtime, stax, synth
    from nngp_b200 import dist as ndist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun (--nproc-per-node {args.gpus}); WORLD_SIZE is 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the nngp_b200 path has no CPU fallback")
    torch.cuda.set_device(local)
    runtime.set_device(local)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gloo = dist.new_group(backend="gloo")       # host-side barrier for the in-process leg (no GPU spinning)

    n, t_rank, d, depth, jd, _desc = WORKLOADS[args.workload]
    warmup = max(args.warmup, 3)
    xtr = synth.encodings(n, d, 1, join_dims=jd)
    ytr = synth.labels(xtr, jd)
    xte_host = synth.encodings(t_rank, d, 2 + rank, join_dims=jd)

    # the reference-facing call chain (train.py:161-172); the engine below is the C-ABI handle behind predict_fn
    _, _, kernel_fn = stax.serial(*([stax.Dense(512)] + [l for _ in range(depth - 1) for l in (stax.Relu(), stax.Dense(1))]))
    kernel_fn = batch.batch(kernel_fn, device_count=0, batch_size=0)
    runtime.set_stats_level(2)
    predict_fn = predict.gradient_descent_mse_ensemble(kernel_fn, xtr, ytr, diag_reg=1e-3)

    fit_info = {}
    if rank == 0:
        h = predict_fn.engine()            # fit #1 (allocations, module load) -- warm-up
        h.stats_reset()
        t0 = time.perf_counter()
        h.fit(xtr, ytr)                    # fit #2, timed
        fit_wall = time.perf_counter() - t0
        s = h.stats()
        fit_info = {"n_train": n, "dim": d, "depth": depth, "seconds_device": s["fit_total_ms"] / 1e3,
                    "seconds_wall_incl_h2d": fit_wall, "gram_ms": s["fit_gram_ms"], "chol_ms": s["fit_chol_ms"],
                    "solve_ms": s["fit_solve_ms"], "chol_tflops": n**3 / 3 / max(s["fit_chol_ms"], 1e-9) / 1e9,
                    "gram_tflops": d * n * (n + 1.0) / max(s["gram_ms"], 1e-9) / 1e9,
                    "gemm_kernel_tflops": s["gemm_flops"] / max(s["gemm_ms"], 1e-9) / 1e9}
    else:
        h = runtime.new_handle(kernel_fn.spec, diag_reg=1e-3)
    bcast = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        ndist.broadcast_fit(h, src=0)
        torch.cuda.synchronize()
        dist.barrier()
        sec = time.perf_counter() - t0
        nbytes = 8 * (n * d + n + n * (n + 1) // 2)
        bcast = {"ms": sec * 1e3, "bytes_per_rank": nbytes, "gb_per_s": nbytes / sec / 1e9,
                 "what": "packed state (X, alpha, lower triangle of L) in 256 MB chunks: pack -> NCCL broadcast -> unpack"}

    kept = {}
    ms_total, ms_e2e, e2e_steps, st, st_e2e, clocks = _time_predict(torch, dist, world, h, local, xte_host, args.steps, warmup,
                                                                    sample_clocks=(rank == 0),
                                                                    keep=kept if rank == 0 or args.dump_outputs else None)
    if args.dump_outputs:
        outs = [kept["mean"], kept["var"]]
        if world > 1:                     # every rank's shard of test rows, in rank order
            for i, a in enumerate(outs):
                parts = [torch.empty(t_rank, dtype=torch.float64, device="cuda") for _ in range(world)]
                dist.all_gather(parts, torch.from_numpy(a).cuda())
                outs[i] = torch.cat(parts).cpu().numpy()
        if rank == 0:
            dump_outputs(args.dump_outputs, *outs)

    sliced = None
    if args.slices > 0 and not args.no_extras:
        try:
            sliced = _sliced_record(torch, dist, world, rank, local, _lib, args, depth, xtr, ytr, xte_host, t_rank, n, kept)
        except Exception as e:  # noqa: BLE001  (a side record must not cost the headline line; all ranks fail alike)
            sliced = {"error": repr(e)}

    in_process = None
    hard_exit = False
    if world > 1 and not args.no_extras:
        # In-process multi-GPU: ONE handle on rank 0 drives all N GPUs through the same nngp_predict call (replicas +
        # row split behind the C ABI).  The other ranks free their state and wait on a host-side (gloo) barrier.
        if rank != 0:
            h.close()
            torch.cuda.empty_cache()
        dist.barrier(group=gloo)
        if rank == 0:
            def leg():
                hm = _lib.Handle(depth=depth, diag_reg=1e-3, stats_level=1, device_ids=list(range(world)))
                xall = np.concatenate([xte_host] + [synth.encodings(t_rank, d, 2 + r, join_dims=jd) for r in range(1, world)])
                hm.fit(xtr, ytr)
                hm.stats_reset()
                hm.fit(xtr, ytr)
                sfit = hm.stats()
                pin = torch.from_numpy(xall).pin_memory()
                mo = torch.empty(xall.shape[0], dtype=torch.float64).pin_memory()
                vo = torch.empty(xall.shape[0], dtype=torch.float64).pin_memory()
                for _ in range(2):
                    hm.predict(pin.numpy(), mean_out=mo.numpy(), var_out=vo.numpy())
                k = min(args.steps, 5)
                t0 = time.perf_counter()
                for _ in range(k):
                    hm.predict(pin.numpy(), mean_out=mo.numpy(), var_out=vo.numpy())
                sec = time.perf_counter() - t0
                rec = {"value": k * xall.shape[0] / sec, "unit": UNIT, "ms_per_step": sec / k * 1e3, "steps": k,
                       "n_gpus": hm.n_gpus, "api": "ONE nngp_handle with n_gpus=N: nngp_fit replicates the packed lower "
                       "triangle peer-to-peer (pipelined chain), nngp_predict splits rows over the GPUs; host buffers in/out, wall clock",
                       "replicate_ms": sfit["replicate_ms"], "replicate_bytes": sfit["replicate_bytes"],
                       "replicate_gb_per_s": sfit["replicate_bytes"] / max(sfit["replicate_ms"], 1e-9) / 1e6,
                       "fit_seconds_device": sfit["fit_total_ms"] / 1e3,
                       "same_bits_as_rank0_shard": bool(np.array_equal(mo.numpy()[:1024], h.predict(xte_host[:1024])[0]))}
                hm.close()
                return rec

            # bounded: a side record must never cost the run its headline line (the worker is a daemon thread)
            box = {}
            th = threading.Thread(target=lambda: box.update(rec=_guard(leg)), daemon=True)
            th.start()
            th.join(timeout=420.0)
            in_process = box.get("rec", {"error": "the in-process multi-GPU leg did not finish within 420 s"})
            hard_exit = th.is_alive()
        dist.barrier(group=gloo)

    if rank != 0:
        if world > 1:
            dist.barrier(group=gloo)      # host-side: rank 0 is busy with its CPU legs / printing
            dist.destroy_process_group()
        return

    queries = world * t_rank * args.steps
    value = queries / (ms_total / 1e3)
    e2e_value = world * t_rank * e2e_steps / (ms_e2e / 1e3)
    peak_dmma = h.dmma_peak_tflops()
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    peaks = json.loads(peaks_file.read_text()) if peaks_file.exists() else {}
    achieved = st["gemm_flops"] / max(st["gemm_ms"], 1e-9) / 1e9
    traffic, traffic_src = _traffic(args.workload, world)
    flops_per_query = float(n) * n + 2.0 * n * d + 4.0 * n
    roofline = {
        "bound": "tensor", "kernel": "trsm_fused_kernel (persistent TMA + DMMA.8x8x4 FP64 triangular solve V = K_* L^-T with fused variance)",
        "achieved": achieved, "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma,
        "traffic": traffic, "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": 8.0 * (2.0 * t_rank * n + n * n / 2.0),
        "peak_source": "FP64 tensor (DMMA) issue-rate microbenchmark measured in this run (burst); MEASURED_PEAKS.json "
                       "has no FP64 entry (bf16 %.0f TF/s, HBM %.0f GB/s are not the bound of an FP64 kernel)" % (
                           peaks.get("bf16_tflops", float("nan")), peaks.get("hbm_gbs", float("nan"))),
        "launches": st["gemm_launches"], "avg_launch_ms": st["gemm_ms"] / max(st["gemm_launches"], 1),
        "algorithmic_flops_per_launch": st["gemm_flops"] / max(st["gemm_launches"], 1),
        "share_of_step": st["gemm_ms"] / max(st["pred_total_ms"], 1e-9),
        "whole_step_tflops_per_gpu": flops_per_query * t_rank * args.steps / (ms_total / 1e3) / 1e12,
        "whole_step_frac_of_peak": flops_per_query * t_rank * args.steps / (ms_total / 1e3) / 1e12 / peak_dmma,
        "gram_kernel": {"tflops": st["gram_flops"] / max(st["gram_ms"], 1e-9) / 1e9,
                        "frac": st["gram_flops"] / max(st["gram_ms"], 1e-9) / 1e9 / peak_dmma,
                        "evals_per_s": st["gram_evals"] / max(st["gram_ms"], 1e-9) * 1e3,
                        "share_of_step": st["gram_ms"] / max(st["pred_total_ms"], 1e-9)},
    }
    if fit_info:
        fit_info["chol_frac_of_fp64_peak"] = fit_info["chol_tflops"] / peak_dmma
        fit_info["gram_frac_of_fp64_peak"] = fit_info["gram_tflops"] / peak_dmma
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": make_config(args.workload, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
                "h2d_bytes_per_step": st_e2e["h2d_bytes"] // e2e_steps, "d2h_bytes_per_step": st_e2e["d2h_bytes"] // e2e_steps,
                "api": "nngp_predict (C ABI) on pinned host buffers == predict_fn(x_test=...) of the neural-tangents mirror"},
        "gpu_launches": st["kernel_launches"],
        "roofline": roofline,
        "stage_ms_per_step": {k: st[k] / args.steps for k in ("pred_gram_ms", "pred_mean_ms", "pred_trsm_ms", "pred_var_ms", "pred_total_ms")},
        "fit": fit_info,
        "build_id": _lib.build_id(),
    }
    if bcast is not None:
        out["fit_broadcast"] = bcast
    if in_process is not None:
        out["in_process"] = in_process
    if sliced is not None:
        if "value" in sliced:
            sliced["speedup_vs_fp64_path"] = sliced["value"] / value
        out["sliced"] = sliced

    if world == 1 and not args.no_extras:
        h.close()
        torch.cuda.empty_cache()
        if args.workload != "c2":          # the round-1 headline config, for continuity
            try:
                n2, t2, d2, dep2, jd2, desc2 = WORKLOADS["c2"]
                x2 = synth.encodings(n2, d2, 1)
                h2 = _lib.Handle(depth=dep2, diag_reg=1e-3, device=local, stats_level=2)
                h2.fit(x2, synth.labels(x2))
                h2.stats_reset()
                h2.fit(x2, synth.labels(x2))
                sf = h2.stats()
                ms2, ms2e, k2e, st2, _st2e, _c = _time_predict(torch, dist, 1, h2, local, synth.encodings(t2, d2, 2), 5, 3)
                out["c2"] = {"workload": desc2, "value": 5 * t2 / (ms2 / 1e3), "e2e_value": k2e * t2 / (ms2e / 1e3),
                             "ms_per_step": ms2 / 5, "trsm_frac": st2["gemm_flops"] / max(st2["gemm_ms"], 1e-9) / 1e9 / peak_dmma,
                             "gram_frac": st2["gram_flops"] / max(st2["gram_ms"], 1e-9) / 1e9 / peak_dmma,
                             "fit_seconds_device": sf["fit_total_ms"] / 1e3, "fit_chol_ms": sf["fit_chol_ms"],
                             "fit_chol_frac": n2**3 / 3 / max(sf["fit_chol_ms"], 1e-9) / 1e9 / peak_dmma}
                h2.close()
            except Exception as e:  # noqa: BLE001
                out["c2"] = {"error": repr(e)}
        if args.workload != "c3":          # "train fit seconds at N = 32k" when the workload itself is not C3
            try:
                n32, d32, depth32 = 32768, 256, 3
                x32 = synth.encodings(n32, d32, 1)
                y32 = synth.labels(x32)
                h32 = _lib.Handle(depth=depth32, diag_reg=1e-3, device=local, stats_level=2)
                h32.fit(x32, y32)
                h32.stats_reset()
                h32.fit(x32, y32)
                s = h32.stats()
                out["fit_n32k"] = {"n_train": n32, "dim": d32, "depth": depth32, "seconds_device": s["fit_total_ms"] / 1e3,
                                   "gram_ms": s["fit_gram_ms"], "chol_ms": s["fit_chol_ms"], "solve_ms": s["fit_solve_ms"],
                                   "chol_tflops": n32**3 / 3 / s["fit_chol_ms"] / 1e9,
                                   "chol_frac_of_fp64_peak": n32**3 / 3 / s["fit_chol_ms"] / 1e9 / peak_dmma,
                                   "gemm_kernel_tflops": s["gemm_flops"] / max(s["gemm_ms"], 1e-9) / 1e9}
                h32.close()
            except Exception as e:  # noqa: BLE001
                out["fit_n32k"] = {"error": repr(e)}

    if world == 1 and not args.no_cpu_baseline:
        # Bounded CPU sample (~20-25 s of host work at C3): the oracle fits the workload's training set itself (all host
        # cores) and predicts `rows` test rows -- the same code `bench.py --impl reference` times over more steps.
        oracle = _oracle()
        rows = CPU_ROWS[args.workload]
        t0 = time.perf_counter()
        cpu_fit = oracle.Fit(xtr, ytr, depth)
        t_fit = time.perf_counter() - t0
        xs = synth.encodings(rows, d, 2, join_dims=jd)
        cpu_fit.predict(xs[:128])
        t1 = time.perf_counter()
        cpu_fit.predict(xs)
        t_pred = time.perf_counter() - t1
        out["cpu_baseline"] = {"value": rows / t_pred, "unit": UNIT, "cores": _CORES, "blas_threads": blas_threads(),
                               "kind": "port", "rows_per_step": rows, "fit_seconds": t_fit,
                               "sample": f"oracle (numpy/scipy, OpenBLAS {blas_threads()} threads + {oracle.THREADS}-thread "
                                         f"elementwise recursion): its own fit at N={n} in {t_fit:.1f}s, then posterior "
                                         f"mean+var of {rows} test rows in {t_pred:.2f}s"}
    print(json.dumps(out))
    if world > 1:
        dist.barrier(group=gloo)
    if hard_exit:            # a stuck side leg still holds CUDA calls: leave without running destructors
        sys.stdout.flush()
        os._exit(0)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    # stdout carries exactly ONE line (rank 0's JSON): library banners (e.g. "NCCL version ...") that are
    # written to fd 1 during the run are diverted to stderr, and fd 1 is restored for the final print.
    sys.stdout.flush()
    _saved_fd = os.dup(1)
    os.dup2(2, 1)
    _real_print = print

    def print(*args, **kw):  # noqa: A001
        sys.stdout.flush()
        os.dup2(_saved_fd, 1)
        _real_print(*args, **kw)
        sys.stdout.flush()
        os.dup2(2, 1)

    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
