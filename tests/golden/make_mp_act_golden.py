"""Generates tests/golden/mp_act.npz: 50-digit kernels and posteriors for the ABRelu family and Erf
(oracle/mp_act_oracle.py).

Run from the repo root:  python tests/golden/make_mp_act_golden.py     (a few minutes, CPU only)

Before it writes anything it checks every closed form the oracle uses -- E[phi(u) phi(v)], E[phi'(u) phi'(v)] and
E[phi(u)^2] -- against numerical integration over the bivariate normal at a handful of (q1, q2, k), for each
activation, and stops if one disagrees by more than 1e-12 relative.

Per activation (ACTS):
  <act>/sweep_*   rows at angles 0 .. pi (down to 1e-8 from either end) and lengths 0.5 .. 2 against the first row;
                  K and Theta of the full square at depth 2 (sigma_w 1, sigma_b 0) and depth 3 (1.3, 0.1)
  <act>/mag_*     a zero row, a subnormal row and rows of norm 1e-150 .. the top of the activation's input range
  <act>/post_*    small 'nngp' (depth 2) and 'ntk' (depth 3) posteriors: mean, var, full covariance, lml
  <act>/rag<N>_*  the same posteriors at ragged shapes, N = 1 (D = 1) and N = 65 (D = 7), standard-normal features
                  (every activation but the saturated erf_bigb)
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "nngp-src_b200"))
import mpmath as mp  # noqa: E402

import mp_act_oracle as mpa  # noqa: E402
from nngp_b200 import synth  # noqa: E402

ACTS = {
    "leaky": ("abrelu", 0.1, 1.0, 0.0),       # LeakyRelu(0.1)
    "abs": ("abrelu", -1.0, 1.0, 0.0),        # Abs
    "abrelu": ("abrelu", -0.3, 1.2, 0.0),     # ABRelu(-0.3, 1.2)
    "erf": ("erf", 1.0, 1.0, 0.0),            # Erf()
    "erf_abc": ("erf", 1.5, 0.7, 0.2),        # Erf(1.5, 0.7, 0.2)
    "erf_bigb": ("erf", 1.0, 1.0e3, 0.0),     # Erf(b = 1000): saturated, Q ~ 1e6
}
QUAD_POINTS = [(1.0, 2.0, 0.7), (0.5, 0.3, -0.35), (2.0, 1.5, 1.7), (0.8, 0.8, 1e-3)]
SWEEP_DEPTHS = [(2, 1.0, 0.0), (3, 1.3, 0.1)]
RAGGED = [(1, 1), (65, 7)]           # (N, D); 3 test rows each


def check_closed_forms():
    for name, act in ACTS.items():
        if name == "erf_bigb":
            continue          # (the integrand is a step at this scale; the formulas are those of the other Erf cases)
        for q1, q2, k in QUAD_POINTS:
            e_pp, e_dd, e_p2 = mpa.expectations_by_quadrature(q1, q2, k, act)
            a = mpa._mpf_act(act)
            f_pp, f_dd = mpa.step(mp.mpf(k), mp.mpf(1), mp.mpf(q1), mp.mpf(q2), a)
            f_p2 = mpa.diag_expect(mp.mpf(q1), a)
            for what, x, y in (("E[phi phi]", e_pp, f_pp), ("E[phi' phi']", e_dd, f_dd), ("E[phi^2]", e_p2, f_p2)):
                rel = abs(x - y) / max(abs(y), mp.mpf(1e-30))
                print(f"{name:8s} q=({q1}, {q2}, {k}) {what:13s} closed {mp.nstr(y, 17)}  quad rel diff {mp.nstr(rel, 3)}")
                assert rel < 1e-12, (name, q1, q2, k, what, x, y)


def sweep_rows():
    ang = [0.0, 1e-8, 1e-4, 0.01, 0.3, 1.0, np.pi / 2, 2.0, 3.0, np.pi - 1e-4, np.pi - 1e-8, np.pi]
    rad = [1.0, 0.5, 2.0, 1.0, 1.5, 0.7, 1.0, 1.2, 0.9, 1.0, 1.0, 1.3]
    x = np.zeros((len(ang) + 1, 4))
    x[0, 0] = 1.0
    for i, (t, r) in enumerate(zip(ang, rad)):
        x[i + 1, :2] = r * np.cos(t), r * np.sin(t)
    return x


def mag_rows(act):
    top = 1e70 if act[0] == "erf" else 1e75         # b^2 q < 2^508 (Erf) / q < 2^512
    norms = [0.0, 1e-310, 1e-150, 1e-30, 1.0, 1e30, top]
    rng = np.random.default_rng(5)
    d = rng.standard_normal((len(norms), 4))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return d * np.array(norms)[:, None]


def to_np(m):
    return np.array([[float(v) for v in r] for r in m])


def posteriors(out, pre, act, xtr, ytr, xte):
    for get, depth, sw, sb in (("nngp", 2, 1.0, 0.0), ("ntk", 3, 1.2, 0.1)):
        r = mpa.fit_predict(xtr.tolist(), ytr.tolist(), xte.tolist(), depth, sw, sb, 1e-3, act, ntk=get == "ntk")
        p = f"{pre}_{get}"
        out[p + "_cfg"] = np.array([depth, sw, sb, 1e-3])
        out[p + "_mean"] = np.array([float(v) for v in r["mean"]])
        out[p + "_var"] = np.array([float(v) for v in r["var"]])
        out[p + "_cov"] = to_np(r["cov"])
        out[p + "_lml"] = np.array(float(r["lml"]))


def main():
    check_closed_forms()
    out = {}
    for name, act in ACTS.items():
        for tag, x in (("sweep", sweep_rows()), ("mag", mag_rows(act))):
            out[f"{name}/{tag}_x"] = x
            for depth, sw, sb in SWEEP_DEPTHS:
                for get in ("nngp", "ntk"):
                    out[f"{name}/{tag}_{get}_d{depth}"] = to_np(mpa.kernel(x.tolist(), None, depth, sw, sb, act, get))
        out[f"{name}/act"] = np.array([{"abrelu": 1.0, "erf": 2.0}[act[0]], *act[1:]])
        xtr, ytr, xte, _ = synth.make_problem(10, 4, 4, seed_train=31, seed_test=32)
        out[f"{name}/post_x_train"], out[f"{name}/post_y_train"], out[f"{name}/post_x_test"] = xtr, ytr, xte
        posteriors(out, f"{name}/post", act, xtr, ytr, xte)
        if name != "erf_bigb":
            for n, d in RAGGED:
                rng = np.random.default_rng(100 * n + d)
                xtr, ytr, xte = rng.standard_normal((n, d)), rng.standard_normal(n), rng.standard_normal((3, d))
                out[f"{name}/rag{n}_x_train"], out[f"{name}/rag{n}_y_train"], out[f"{name}/rag{n}_x_test"] = xtr, ytr, xte
                posteriors(out, f"{name}/rag{n}", act, xtr, ytr, xte)
        print(name, "done")
    np.savez_compressed(Path(__file__).with_name("mp_act.npz"), **out)


if __name__ == "__main__":
    main()
