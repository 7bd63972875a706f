"""Generates tests/golden/mp_cov.npz: the full posterior covariance of the 50-digit mpmath oracle
(oracle/mp_cov_oracle.py, fit_predict_cov / fit_predict_ntk_cov).

Run from the repo root:  python tests/golden/make_mp_cov_golden.py     (about a minute, CPU only)
Cases: the training sets and configurations of tests/golden/mp_small.npz (make_mp_golden.py: the six 'nngp' cases
and the two 'ntk' cases, same seeds), each with 7 test rows: 4 of mp_small's test rows, a near-duplicate of the
first (relative change 1e-9 in one feature: a pair whose covariance is almost its variance), a scaled copy of the
second, and a copy of a training row (posterior variance about lambda-sized).
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "nngp-src_b200"))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import mp_cov_oracle as mpo  # noqa: E402
from make_mp_golden import CASES  # noqa: E402
from nngp_b200 import synth  # noqa: E402

NTK_CASES = [("ntk_d2", 32, 10, 16, 2, 1.0, 0.0, 1e-3), ("ntk_d3_sigma", 28, 8, 12, 3, 1.5, 0.05, 1e-3)]


def test_rows(xtr, xte):
    x = np.vstack([xte[:4], xte[:1], 1.5 * xte[1:2], xtr[3:4]])
    x[4, 0] *= 1.0 + 1e-9
    return x


def store(out, name, xtr, ytr, xt, cfg, r):
    t = len(xt)
    out[f"{name}/x_train"], out[f"{name}/y_train"], out[f"{name}/x_test"] = xtr, ytr, xt
    out[f"{name}/cfg"] = np.array(cfg)
    out[f"{name}/mean"] = np.array([float(v) for v in r["mean"]])
    out[f"{name}/cov"] = np.array([[float(r["cov"][i][j]) for j in range(t)] for i in range(t)])
    out[f"{name}/K_tt"] = np.array([[float(r["Ktt"][i][j]) for j in range(t)] for i in range(t)])
    print(name, "cov[0,4]", out[f"{name}/cov"][0, 4], "var", np.diag(out[f"{name}/cov"])[:3])


def main():
    out = {}
    for name, n, t, d, depth, sw, sb, reg, absolute in CASES:
        xtr, ytr, xte, _ = synth.make_problem(n, t, d, seed_train=11, seed_test=12)
        if name == "degenerate":       # as in make_mp_golden.py
            xtr[1] = xtr[0]
            xtr[2] = 0.0
            xtr[3] = 2.5 * xtr[0]
            xte[0] = xtr[0]
            xte[1] = 0.0
        xt = test_rows(xtr, xte)
        r = mpo.fit_predict_cov(xtr.tolist(), ytr.tolist(), xt.tolist(), depth, sw, sb, reg, absolute)
        store(out, name, xtr, ytr, xt, [depth, sw, sb, reg, float(absolute), 0.0], r)
    for name, n, t, d, depth, sw, sb, reg in NTK_CASES:
        xtr, ytr, xte, _ = synth.make_problem(n, t, d, seed_train=21, seed_test=22)
        xtr[1] = xtr[0]; xte[0] = xtr[0]; xtr[2] = 0.0
        xt = test_rows(xtr, xte)
        r = mpo.fit_predict_ntk_cov(xtr.tolist(), ytr.tolist(), xt.tolist(), depth, sw, sb, reg)
        store(out, name, xtr, ytr, xt, [depth, sw, sb, reg, 0.0, 1.0], r)
    np.savez_compressed(Path(__file__).with_name("mp_cov.npz"), **out)


if __name__ == "__main__":
    main()
