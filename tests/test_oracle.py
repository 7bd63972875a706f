"""CPU: pins the numpy/scipy oracle (the parity checker) -- no GPU, no CUDA library involved.

The reference ships no tests or golden vectors for this path (SURVEY.md section 4), so the pins are:
analytic known answers, the 50-digit mpmath restatement (tests/golden/mp_small.npz), a finite-width
Monte-Carlo check of the /D and no-bias conventions, and the forest-workload invariants.
"""
import numpy as np
import pytest

import nngp_oracle as o


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def test_analytic_known_answers():
    rng = np.random.default_rng(0)
    x = rng.uniform(0, 1000, (6, 8))
    d = x.shape[1]
    k = o.kernel_fn(x, None, depth=2)
    # K(x,x) = |x|^2 / (2D)
    assert rel(np.diag(k), np.einsum("ij,ij->i", x, x) / (2 * d)) < 1e-14
    # orthogonal rows: K = sqrt(q q') / (2 pi)
    a = np.zeros((1, 8)); a[0, :4] = rng.uniform(1, 9, 4)
    b = np.zeros((1, 8)); b[0, 4:] = rng.uniform(1, 9, 4)
    qa, qb = a @ a.T / 8, b @ b.T / 8
    assert rel(o.kernel_fn(a, b), np.sqrt(qa * qb) / (2 * np.pi)) < 1e-15
    # x' = -x: K = 0 ; x' = c x: K = c |x|^2 / (2D)
    assert abs(o.kernel_fn(a, -a)[0, 0]) < 1e-15 * qa[0, 0]
    assert rel(o.kernel_fn(a, 3.5 * a), 3.5 * qa / 2) < 1e-15
    # general closed form: sqrt(q q') (sin t + (pi - t) cos t) / (2 pi)
    u, v = x[:1], x[1:2]
    qu, qv = (u @ u.T / d)[0, 0], (v @ v.T / d)[0, 0]
    t = np.arccos((u @ v.T / d)[0, 0] / np.sqrt(qu * qv))
    assert rel(o.kernel_fn(u, v)[0, 0], np.sqrt(qu * qv) * (np.sin(t) + (np.pi - t) * np.cos(t)) / (2 * np.pi)) < 1e-12
    # depth-L diagonal q_L = q_0 / 2^(L-1); zero rows hit the theta = pi/2 branch and give 0
    assert rel(np.diag(o.kernel_fn(x, None, depth=4)), np.einsum("ij,ij->i", x, x) / d / 8) < 1e-14
    z = np.zeros((2, 8))
    assert np.all(o.kernel_fn(z, x) == 0.0) and np.all(np.isfinite(o.kernel_fn(z, z)))


@pytest.mark.parametrize("case", ["ref_d2", "d3", "sigma_variant", "d1_linear", "abs_reg", "degenerate"])
def test_oracle_matches_mpmath_golden(mp_golden, case):
    g = mp_golden[case]
    depth, sw, sb, reg, absolute = g["cfg"]
    depth, absolute = int(depth), bool(absolute)
    kdd = o.kernel_fn(g["x_train"], None, depth, sw, sb)
    ktd = o.kernel_fn(g["x_test"], g["x_train"], depth, sw, sb)
    scale = np.max(np.abs(g["K_dd"]))
    # entries: 1e-14 relative to the kernel scale (near-duplicate rows lose relative accuracy in s, not in K)
    assert np.max(np.abs(kdd - g["K_dd"])) < 1e-14 * scale
    assert np.max(np.abs(ktd - g["K_td"])) < 1e-14 * scale
    fit = o.Fit(g["x_train"], g["y_train"], depth, sw, sb, reg, absolute)
    assert abs(fit.lam - g["lam"]) < 1e-14 * abs(g["lam"])
    mean, var = fit.predict(g["x_test"])
    assert np.max(np.abs(mean - g["mean"])) < 1e-9 * np.max(np.abs(g["mean"]))
    assert np.max(np.abs(var - g["var"])) < 1e-9 * np.max(np.abs(g["var"]))
    m2, cov = fit.predict_full_cov(g["x_test"])
    assert m2.shape == (len(mean), 1) and cov.shape == (len(mean), len(mean))
    assert np.max(np.abs(np.diag(cov) - g["var"])) < 1e-8 * np.max(np.abs(g["var"]))


@pytest.mark.parametrize("case", ["ntk_d2", "ntk_d3_sigma"])
def test_ntk_oracle_matches_mpmath_golden(mp_golden, case):
    g = mp_golden[case]
    depth, sw, sb, reg, _ = g["cfg"]
    depth = int(depth)
    scale = np.max(np.abs(g["Theta_dd"]))
    # Unlike K (dK/dtheta = 0 at theta = 0), Theta is first-order sensitive to theta through kdot = 1/2 - theta/(2 pi):
    # for duplicate rows / the diagonal, s = sqrt(q q' - k^2) is sqrt(rounding noise) ~ 1e-8 sqrt(qq') in ANY FP64
    # evaluation of the nt formula, so entries agree with the 50-digit value to ~1e-9 only there, 1e-14 elsewhere.
    dth = np.abs(o.kernel_fn(g["x_train"], None, depth, sw, sb, get="ntk") - g["Theta_dd"])
    assert np.max(dth) < 1e-8 * scale and np.median(dth) < 1e-14 * scale
    dts = np.abs(o.kernel_fn(g["x_test"], g["x_train"], depth, sw, sb, get="ntk") - g["Theta_td"])
    assert np.max(dts) < 1e-8 * scale and np.median(dts) < 1e-14 * scale
    fit = o.FitNTK(g["x_train"], g["y_train"], depth, sw, sb, reg)
    assert abs(fit.lam - g["lam"]) < 1e-9 * abs(g["lam"])
    mean, var = fit.predict(g["x_test"])
    assert np.max(np.abs(mean - g["mean"])) < 1e-8 * np.max(np.abs(g["mean"]))
    assert np.max(np.abs(var - g["var"])) < 1e-8 * np.max(np.abs(g["var"]))
    # Theta(x,x) closed form: kdot = 1/2 on the diagonal
    q0 = o.layer0_diag(g["x_train"], sw, sb)
    assert np.allclose(np.diag(g["Theta_dd"]), o.final_diag_ntk(q0, depth, sw, sb), rtol=1e-13)   # exact in mpmath


def test_finite_width_monte_carlo_conventions():
    """f(x) = v . relu(W x / sqrt(D)) / sqrt(width): covariance -> K; guards /D, W_std=1, no bias."""
    rng = np.random.default_rng(5)
    d, width, nets = 6, 2048, 200
    x = rng.uniform(0, 3, (4, d))
    acc = np.zeros((4, 4))
    for _ in range(nets):
        w = rng.standard_normal((width, d))
        v = rng.standard_normal(width)
        f = (np.maximum(x @ w.T / np.sqrt(d), 0.0) * v).sum(1) / np.sqrt(width)
        acc += np.outer(f, f)
    emp = acc / nets
    k = o.kernel_fn(x, None, depth=2)
    assert np.max(np.abs(emp - k)) / np.max(k) < 0.2  # 200 draws: ~10% sampling noise
    # a sharper check through the closed-form expectation of relu(u)relu(u') per hidden unit
    w = rng.standard_normal((400000, d))
    h = np.maximum(x @ w.T / np.sqrt(d), 0.0)
    assert np.max(np.abs(h @ h.T / w.shape[0] - k)) / np.max(k) < 1e-2


def test_forest_workload_invariants(forest):
    xtr, ytr, xte, yte = forest["x_train"], forest["y_train"], forest["x_test"], forest["y_test"]
    assert xtr.shape == (10800, 20) and xte.shape == (3600, 20) and xtr.dtype == np.float64
    # lambda = 1e-3 * trace(K)/N = 1e-3 * mean(|x|^2) / (2 D): independent of the solver
    lam = 1e-3 * np.mean(np.einsum("ij,ij->i", xtr, xtr) / 40.0)
    assert abs(lam - 185.5609) < 1e-3     # SURVEY.md section 6 probe value
    sub = slice(0, 1500)
    fit = o.Fit(xtr[sub], ytr[sub])
    mean, var = fit.predict(xte[:300])
    assert np.all(var > 0) and np.all(np.isfinite(mean))
    qe = o.q_error_stats(mean, yte[:300])
    assert qe["median"] < 10.0            # the estimator is doing something sensible


def test_active_selection_rule():
    mean = np.array([[4.0], [8.0], [2.0], [6.0]])
    std = np.array([0.4, 0.1, 0.9, 0.2])
    assert list(o.active_select(mean, std, 2)) == [0, 2]
    assert sorted(o.active_select(mean, std, 10)) == [0, 1, 2, 3]


def test_active_sampling_restatement():
    """Gumbel-top-k restatement of the biased_sample branch (ActiveLearner.py:49-53): splitmix64 known answer, no
    repeats, determinism, zero-probability rows never drawn, inclusion frequencies like numpy's choice(p=...)."""
    u = o.splitmix_uniform(0, 4)
    assert int(u[0] * 2.0 ** 52 - 0.5) == 0xE220A8397B1DCDAF >> 12      # first splitmix64 output for state 0
    assert np.all((u > 0) & (u < 1))
    rng = np.random.default_rng(0)
    s = rng.random(40) + 0.01
    s[7] = 0.0
    a = o.active_sample(np.ones(1), s, 5, seed=3)
    assert len(set(a.tolist())) == 5 and np.array_equal(a, o.active_sample(np.ones(1), s, 5, seed=3))
    cnt, cnt_np = np.zeros(40), np.zeros(40)
    p = s / s.sum()
    for seed in range(3000):
        cnt[o.active_sample(np.ones(1), s, 5, seed)] += 1
        cnt_np[np.random.default_rng(seed).choice(40, 5, replace=False, p=p)] += 1
    assert cnt[7] == 0
    assert np.max(np.abs(cnt - cnt_np)) / 3000 < 0.03 and np.corrcoef(cnt, cnt_np)[0, 1] > 0.98
    assert sorted(o.active_sample(np.ones(1), s[:4], 10, seed=1).tolist()) == [0, 1, 2, 3]
    with pytest.raises(ValueError):
        o.active_sample(np.ones(1), -s, 3)


def test_device_atan2_algorithm_in_numpy():
    """The Gram epilogue's atan2_pos (csrc/gemm_nt.cuh) restated in numpy with the SAME coefficients and range guard
    (parsed from the source) and the flush-to-zero semantics of rcp.approx.ftz.f64: <= 2 ulp of theta against libm and
    40-digit mpmath over the whole double range of s and k, incl. subnormals, the axes and the origin."""
    import re
    from pathlib import Path
    import mpmath as mp
    src = (Path(__file__).resolve().parents[1] / "nngp-src_b200" / "csrc" / "gemm_nt.cuh").read_text()
    body = src[src.index("constexpr double C[21] = {"):]
    body = body[:body.index("};")]
    coef = [float(v) for v in re.findall(r"-?\d+\.\d+(?:e-?\d+)?", body.split("{", 1)[1])]
    assert len(coef) == 21 and coef[0] == 1.0
    # the range guard in front of the reciprocal: biased exponent field of max(s^2, k^2) outside 1..hi, scale 2^+-e
    guard = re.search(r"__double2hiint\(mx2\) >> 20\) - 1u >= (\d+)u\).*?\? 0x1p\+(\d+) : 0x1p-(\d+);", src, re.S)
    assert guard, "atan2_pos: range guard of the reciprocal not found"
    hi, e_up, e_dn = (int(v) for v in guard.groups())
    assert (hi, e_up) == (2044, e_dn)     # [2^-1022, 2^1022): the reciprocal and its result are normal doubles

    tiny = 2.0 ** -1022

    def rcp_newton(x):
        # rcp.approx.ftz.f64: a subnormal input and a subnormal result are flushed to zero (input 0 -> +inf); the seed
        # is correctly rounded here (the MUFU seed is ~20 bits, the two Newton steps make up the difference: <= 1 ulp)
        r = 1.0 / np.where(x < tiny, 0.0, x)
        r = np.where(r < tiny, 0.0, r)
        for _ in range(2):
            r = r * (1.0 - x * r) + r
        return r

    def atan2_pos(s, k, guarded=True):
        # min/max = s |k| / max(s^2, k^2) (reciprocal + product instead of a division),
        # P(u) = Pe(u^2) + u Po(u^2): two Horner chains of 10
        a = np.abs(k)
        s2, a2 = s * s, k * k
        sbig = s2 > a2
        mx2 = np.where(sbig, s2, a2)
        sc = s
        if guarded:
            field = (mx2.view(np.int64) >> 52) & 0x7FF
            rare = (field < 1) | (field > hi)
            f = np.where(field < 1, 2.0 ** e_up, 2.0 ** -e_dn)
            sc = np.where(rare, s * f, s)
            a = np.where(rare, a * f, a)
            sbig = np.where(rare, sc > a, sbig)
            mx2 = np.where(rare, np.where(sbig, sc * sc, a * a), mx2)
        t = (sc * a) * rcp_newton(mx2)
        u = t * t
        w = u * u
        pe = np.full_like(u, coef[20])
        for c in coef[18::-2]:
            pe = pe * w + c
        po = np.full_like(u, coef[19])
        for c in coef[17::-2]:
            po = po * w + c
        at = t * (u * po + pe)
        th0 = np.where(sbig, np.pi / 2 - at, at)
        th = np.where(np.signbit(k), np.pi - th0, th0)
        if not guarded:
            return np.where(mx2 == 0, np.pi / 2, th)
        return np.where((s == 0) & (k == 0), np.pi / 2, th)

    def ref_of(s, k):
        r = np.arctan2(s, k)
        r[(s == 0) & (k == 0)] = np.pi / 2
        return r

    rng = np.random.default_rng(1)
    with np.errstate(all="ignore"):
        # magnitudes of a kernel value in ordinary use
        s = np.abs(rng.standard_normal(200000)) * 10 ** rng.uniform(-12, 9, 200000)
        k = rng.standard_normal(200000) * 10 ** rng.uniform(-12, 9, 200000)
        s[:500] = 0.0; k[500:1000] = 0.0; s[1000] = k[1000] = 0.0; k[1001:1500] = s[1001:1500]
        k[1500:1600] = -0.0
        assert np.max(np.abs(atan2_pos(s, k) - ref_of(s, k))) <= 9e-16            # <= 2 ulp of theta in [0, pi]
        # ... which the guard leaves bitwise alone (mx2 inside [2^-1022, 2^1022) there)
        assert np.array_equal(atan2_pos(s, k), atan2_pos(s, k, guarded=False))
        mp.mp.dps = 40
        hi_ = np.array([float(mp.atan2(mp.mpf(float(a)), mp.mpf(float(b)))) for a, b in zip(s[2000:4000], k[2000:4000])])
        assert np.max(np.abs(atan2_pos(s[2000:4000], k[2000:4000]) - hi_)) <= 9e-16

        # the whole double range: exponents of s and |k| swept independently over [-1074, 1023], subnormals included
        n = 300000
        es, ek = rng.integers(-1074, 1024, n), rng.integers(-1074, 1024, n)
        es[:2000] = ek[:2000] + rng.integers(-3, 4, 2000)               # comparable magnitudes: theta away from the axes
        es[150:250] = ek[150:250] = 511                                  # max(s^2, k^2) in [2^1022, 2^1024)
        s = np.ldexp(rng.uniform(1.0, 2.0, n), es)
        k = np.ldexp(rng.uniform(1.0, 2.0, n), ek) * rng.choice([-1.0, 1.0], n)
        s[:50] = 0.0; k[50:100] = 0.0; k[100:150] = -0.0
        ref = ref_of(s, k)
        got = atan2_pos(s, k)
        assert np.all(np.isfinite(got))
        assert np.max(np.abs(got - ref)) <= 9e-16
        hi_ = np.array([float(mp.atan2(mp.mpf(float(a)), mp.mpf(float(b)))) for a, b in zip(s[:2000], k[:2000])])
        assert np.max(np.abs(got[:2000] - hi_)) <= 9e-16
        # without the guard the flush-to-zero reciprocal breaks exactly there (defects the guard exists for):
        bare = atan2_pos(s, k, guarded=False)
        mx = np.maximum(s, np.abs(k))
        sub = (mx < 2.0 ** -511) & (mx > 0)
        assert np.any(np.isnan(bare[sub]) & (np.maximum(s * s, k * k)[sub] > 0))      # subnormal max(s^2, k^2): NaN
        assert np.any(np.abs(bare[sub] - ref[sub]) == np.pi / 2)                     # k^2 underflows: pi/2, not 0 / pi
        big = (mx >= 2.0 ** 511) & (mx < 2.0 ** 512)                                  # (q < 2^512 keeps |k|, s there)
        assert np.max(np.abs(bare[big] - ref[big])) > 0.1                             # 1/mx2 flushed: t = 0
    # gram_epilogue skips the guard (atan2_pos<false>) when q1 and q2 are normal doubles whose exponents sum to
    # [lo, hi]: then max(s^2, k^2) is inside [2^-1022, 2^1022), even with |k| a little above sqrt(q1 q2) from rounding
    gate = re.search(r"ok &= \(\(unsigned\)\(e2 - 1\) < (\d+)u\) & \(\(unsigned\)\(e1 \+ e2 - \(2046 - (\d+)\)\) <= (\d+)u\)",
                     src)
    assert gate, "gram_epilogue: exponent gate of the unguarded path not found"
    assert re.search(r"bool ok = \(unsigned\)\(e1 - 1\) < %su;" % gate.group(1), src)
    n_normal, lo = int(gate.group(1)), -int(gate.group(2))
    hi_e = lo + int(gate.group(3))
    assert (n_normal, lo, hi_e) == (2046, -1020, 1019)

    def fast(q1, q2):      # the gate, on the biased exponent fields like the device
        f1, f2 = (np.asarray(q1).view(np.int64) >> 52) & 0x7FF, (np.asarray(q2).view(np.int64) >> 52) & 0x7FF
        return (f1 >= 1) & (f1 <= n_normal) & (f2 >= 1) & (f2 <= n_normal) & (f1 + f2 - 2046 >= lo) & (f1 + f2 - 2046 <= hi_e)

    n = 200000
    e1 = rng.integers(-1022, 1023, n)
    e2 = np.where(rng.random(n) < 0.5, lo, hi_e) - e1
    ok = (e2 >= -1022) & (e2 <= 1022)
    q1 = np.ldexp(rng.uniform(1.0, 2.0, n)[ok], e1[ok])
    q2 = np.ldexp(rng.uniform(1.0, 2.0, n)[ok], e2[ok])
    assert np.all(fast(q1, q2))
    kk = np.sqrt(q1) * np.sqrt(q2) * rng.uniform(-1.0 - 8 * 2.0 ** -52, 1.0 + 8 * 2.0 ** -52, q1.size)
    mx2 = np.maximum(np.maximum(q1 * q2 - kk * kk, 0.0), kk * kk)
    assert np.all((mx2 >= 2.0 ** -1022) & (mx2 < 2.0 ** 1022))
    # a row whose q underflowed (to 0 or a subnormal) no longer bounds k: x = (3, 1) 2^-540 against y = (2, -0.5) 2^20
    # has q_x = 0 but k = 2.75 2^-520, k^2 subnormal -- such groups must take the guarded path
    for ex in (-540, -530):
        x, y = np.ldexp(np.array([3.0, 1.0]), ex), np.ldexp(np.array([2.0, -0.5]), 20)
        qx, qy = x @ x / 2, y @ y / 2
        assert not fast(qx, qy) and not fast(qy, qx) and not fast(0.0, 1.0) and not fast(np.inf, 1.0)
    # a pair from the kernel's own domain: x = (3, 1) 2^-530, y = (2, -0.5): k, s ~ 2^-530, k^2 and s^2 subnormal
    x, y = np.ldexp(np.array([3.0, 1.0]), -530), np.array([2.0, -0.5])
    kk, q1, q2 = x @ y / 2, x @ x / 2, y @ y / 2
    ss = np.sqrt(np.array([max(q1 * q2 - kk * kk, 0.0)]))
    with np.errstate(all="ignore"):
        assert np.isnan(atan2_pos(ss, np.array([kk]), guarded=False)[0])
    assert abs(atan2_pos(ss, np.array([kk]))[0] - np.arctan2(ss[0], kk)) < 1e-3


@pytest.mark.parametrize("case", ["layers_d2", "layers_d3"])
def test_per_layer_sigmas_against_mpmath(case, golden_dir):
    """Dense layers with different W_std / b_std (nt allows it): the numpy oracle against 50-digit mpmath vectors
    (tests/golden/make_mp_layers_golden.py), NNGP and NTK, kernels and posteriors."""
    z = np.load(golden_dir / "mp_layers.npz")
    g = {k.split("/")[1]: z[k] for k in z.files if k.startswith(case + "/")}
    sw, sb, reg = tuple(g["sigma_w"]), tuple(g["sigma_b"]), float(g["diag_reg"])
    depth = len(sw)
    x, y, xt = g["x_train"], g["y_train"], g["x_test"]
    k, th = o.kernel_fn(x, None, depth, sw, sb, get="both")
    ks, ths = o.kernel_fn(xt, x, depth, sw, sb, get="both")

    def rel(a, b):
        return np.max(np.abs(a - b)) / np.max(np.abs(b))

    assert rel(k, g["K_dd"]) < 1e-14 and rel(ks, g["K_td"]) < 1e-14
    assert rel(th, g["Theta_dd"]) < 1e-8 and rel(ths, g["Theta_td"]) < 1e-8      # (theta ~ 1e-8 at duplicates)
    f = o.Fit(x, y, depth, sw, sb, diag_reg=reg)
    m, v = f.predict(xt)
    assert abs(f.lam - float(g["lam"])) < 1e-13 * f.lam
    assert rel(m, g["mean"]) < 1e-9 and rel(v, g["var"]) < 1e-8
    fn = o.FitNTK(x, y, depth, sw, sb, diag_reg=reg)
    mn, vn = fn.predict(xt)
    assert rel(mn, g["ntk_mean"]) < 1e-7 and rel(vn, g["ntk_var"]) < 1e-5
