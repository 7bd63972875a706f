"""Generates tests/golden/mp_domain.npz with the 50-digit mpmath oracle: the Gram epilogue's input domain beyond what
the non-negative encodings reach -- signed inputs at prescribed angles in (pi/2, pi), deep and per-layer networks,
and inputs scaled towards the ends of the FP64 range.

  sweep/...      pairs of rows at the angles ANGLES (+ a block of standard-normal pairs), at D = 2, 37 and 130, for
                 every network in CONFIGS: K(x1, x2), K(x1, x1), K(x2, x2) and Theta(x1, x2)
  mag/...        the fixed pair x = (3, 1), y = (2, -0.5) (and the same times 2^20) with x, or x and y, scaled by 2^e;
                 plus a near-parallel pair whose q lies in [2^511, 2^512)
  post/...       a small signed fit / predict (NNGP and NTK posterior)

Run from the repo root:  python tests/golden/make_mp_domain_golden.py     (CPU only, about a minute)
"""
import sys
from pathlib import Path

import mpmath as mp
import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "oracle"))
import mp_oracle as mpo  # noqa: E402

ANGLES = [0.0, 1e-12, 1e-8, 1e-4, np.pi / 4, np.pi / 2 - 1e-12, np.pi / 2, np.pi / 2 + 1e-12, 3 * np.pi / 4,
          np.pi - 1e-4, np.pi - 1e-8, np.pi - 1e-12, np.pi]
N_NORMAL = 8
DIMS = [2, 37, 130]
_SW16 = [float(np.sqrt(2.0) * (1.0 + 0.1 * np.sin(l))) for l in range(16)]
_SB16 = [0.05 * (l % 3) for l in range(16)]
CONFIGS = {   # name: (depth, sigma_w, sigma_b)
    "d2_b0": (2, 1.0, 0.0), "d2_b01": (2, 1.0, 0.1),
    "d3_b0": (3, 1.2, 0.0), "d3_b01": (3, 1.2, 0.1),
    "d5_b0": (5, 1.4, 0.0), "d5_b01": (5, 1.4, 0.1),
    "pl4": (4, [1.1, 0.9, 1.6, 0.7], [0.2, 0.0, 0.3, 0.1]),
    "pl16": (16, _SW16, _SB16),
    "u20": (20, 1.4, 0.1),
}
MAG_EXPS = [-560, -540, -530, -520, -511, -400, -256, 0, 256, 400, 500]
MAG_DEPTH = 3


def pair_rows(d, seed):
    """Row pairs (x1[i], x2[i]) at the angles ANGLES (signed, random directions and lengths), then N_NORMAL pairs of
    independent standard-normal rows."""
    rng = np.random.default_rng(seed)
    x1, x2 = [], []
    for th in ANGLES:
        u = rng.standard_normal(d)
        u /= np.linalg.norm(u)
        v = rng.standard_normal(d)
        v -= (v @ u) * u
        v /= np.linalg.norm(v)
        a = u * rng.uniform(0.5, 2.0) * np.sqrt(d)
        if th == 0.0:
            b = 0.5 * a
        elif th == np.pi:
            b = -0.5 * a
        else:
            b = rng.uniform(0.5, 2.0) * np.sqrt(d) * (np.cos(th) * u + np.sin(th) * v)
        x1.append(a)
        x2.append(b)
    x1 += list(rng.standard_normal((N_NORMAL, d)))
    x2 += list(rng.standard_normal((N_NORMAL, d)))
    return np.array(x1), np.array(x2)


def k1(a, b, depth, sw, sb, get="nngp"):
    return float(mpo.kernel([a.tolist()], [b.tolist()], depth, sw, sb, get)[0][0])


def mag_cases():
    """(x, y) pairs: base pair B in {(3, 1) / (2, -0.5), the same times 2^20}, x scaled by 2^e ('one') or both rows
    scaled by 2^e ('both'); plus 'near_overflow': x = c (1, 0.1), y = c (1, -0.1), q = 1.01 c^2 / 2 in [2^511, 2^512)."""
    xs, ys, names = [], [], []
    for bi, base in enumerate([1.0, 2.0 ** 20]):
        x0, y0 = np.array([3.0, 1.0]) * base, np.array([2.0, -0.5]) * base
        for mode in ("one", "both"):
            for e in MAG_EXPS:
                xs.append(np.ldexp(x0, e))
                ys.append(np.ldexp(y0, e) if mode == "both" else y0)
                names.append(f"b{bi}_{mode}_{e}")
    c = 1.2 * 2.0 ** 256
    xs.append(c * np.array([1.0, 0.1]))
    ys.append(c * np.array([1.0, -0.1]))
    names.append("near_overflow")
    return np.array(xs), np.array(ys), names


def main():
    out = {"angles": np.array(ANGLES)}
    for d in DIMS:
        x1, x2 = pair_rows(d, 100 + d)
        out[f"sweep/x1_D{d}"], out[f"sweep/x2_D{d}"] = x1, x2
        for name, (depth, sw, sb) in CONFIGS.items():
            key = f"sweep/{name}_D{d}"
            out[key + "_K12"] = np.array([k1(a, b, depth, sw, sb) for a, b in zip(x1, x2)])
            out[key + "_K11"] = np.array([k1(a, a, depth, sw, sb) for a in x1])
            out[key + "_K22"] = np.array([k1(b, b, depth, sw, sb) for b in x2])
            out[key + "_T12"] = np.array([k1(a, b, depth, sw, sb, "ntk") for a, b in zip(x1, x2)])
        print("sweep D", d, "done")
    for name, (depth, sw, sb) in CONFIGS.items():
        out[f"cfg/{name}/depth"] = np.array(depth)
        out[f"cfg/{name}/sigma_w"] = np.atleast_1d(np.array(sw, dtype=np.float64))
        out[f"cfg/{name}/sigma_b"] = np.atleast_1d(np.array(sb, dtype=np.float64))

    xs, ys, names = mag_cases()
    out["mag/x"], out["mag/y"], out["mag/names"] = xs, ys, np.array(names)
    out["mag/K_xy"] = np.array([k1(a, b, MAG_DEPTH, 1.0, 0.0) for a, b in zip(xs, ys)])
    out["mag/K_xx"] = np.array([k1(a, a, MAG_DEPTH, 1.0, 0.0) for a in xs])
    out["mag/K_yy"] = np.array([k1(b, b, MAG_DEPTH, 1.0, 0.0) for b in ys])
    # sqrt(K(x,x) K(y,y)) in mpmath: the factors alone can underflow where their geometric mean does not
    out["mag/scale"] = np.array([float(mp.sqrt(mpo.kernel([a.tolist()], None, MAG_DEPTH, 1.0, 0.0)[0][0]
                                               * mpo.kernel([b.tolist()], None, MAG_DEPTH, 1.0, 0.0)[0][0]))
                                 for a, b in zip(xs, ys)])
    print("magnitude cases done")

    rng = np.random.default_rng(7)
    n, t, d, depth, sw, sb, reg = 48, 12, 10, 3, 1.0, 0.05, 1e-3
    x, xt = rng.standard_normal((n, d)), rng.standard_normal((t, d))
    y = np.sin(x[:, 0]) + x[:, 1] * x[:, 2] + 0.1 * rng.standard_normal(n)
    r = mpo.fit_predict(x.tolist(), y.tolist(), xt.tolist(), depth, sw, sb, reg)
    rn = mpo.fit_predict_ntk(x.tolist(), y.tolist(), xt.tolist(), depth, sw, sb, reg)
    out["post/x_train"], out["post/y_train"], out["post/x_test"] = x, y, xt
    out["post/cfg"] = np.array([depth, sw, sb, reg])
    out["post/lam"], out["post/ntk_lam"] = np.array(float(r["lam"])), np.array(float(rn["lam"]))
    out["post/mean"] = np.array([float(v) for v in r["mean"]])
    out["post/var"] = np.array([float(v) for v in r["var"]])
    out["post/ntk_mean"] = np.array([float(v) for v in rn["mean"]])
    out["post/ntk_var"] = np.array([float(v) for v in rn["var"]])
    print("posterior: lam", float(r["lam"]), "mean[0]", out["post/mean"][0], "ntk mean[0]", out["post/ntk_mean"][0])
    np.savez_compressed(Path(__file__).with_name("mp_domain.npz"), **out)


if __name__ == "__main__":
    main()
