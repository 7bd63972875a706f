"""GPU: the Gram epilogue (csrc/gemm_nt.cuh: gram_epilogue -> arccos_step(_ntk) -> atan2_pos) over its whole input
domain, against the 50-digit mpmath vectors of tests/golden/make_mp_domain_golden.py and the numpy oracle:

  * signed rows at prescribed angles (theta strictly inside (pi/2, pi) included), D = 2 / 37 / 130, depth 2..20,
    per-layer sigmas up to the 16 Dense layers per_layer allows -- NNGP and NTK, symmetric and rectangular launches;
  * power-of-two scaling: bitwise homogeneity while every intermediate is a normal double, finite and close to mpmath
    down into the subnormal range, and the 2^512 bound on the layer-0 diagonal q (q q' must be a finite double);
  * fit / predict on standard-normal features (NNGP and NTK, default / latency_mode / variance_slices handles).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import nngp_oracle as oracle  # noqa: E402

EPS = np.finfo(np.float64).eps
Q_LIMIT = 2.0 ** 512


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


@pytest.fixture(scope="module")
def dom(golden_dir):
    return dict(np.load(golden_dir / "mp_domain.npz"))


def _cfg(dom, name):
    sw, sb = dom[f"cfg/{name}/sigma_w"], dom[f"cfg/{name}/sigma_b"]
    return int(dom[f"cfg/{name}/depth"]), (sw if sw.size > 1 else float(sw[0])), (sb if sb.size > 1 else float(sb[0]))


def relmax(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


CONFIGS = ["d2_b0", "d2_b01", "d3_b0", "d3_b01", "d5_b0", "d5_b01", "pl4", "pl16", "u20"]


@pytest.mark.parametrize("d", [2, 37, 130])
@pytest.mark.parametrize("name", CONFIGS)
def test_angle_sweep_against_mpmath(lib, dom, name, d):
    """|K - K_mp| <= 8 eps sqrt(K_mp(x,x) K_mp(y,y)) at every angle (relative to the natural scale: K -> 0 as
    theta -> pi; past depth 5, 2 eps per arc-cosine step: each adds an ulp or two), through the symmetric launch
    (>= 512 rows: lower tiles + mirror) and the rectangular one, which must agree bit for bit; Theta within 1e-12 of
    the block maximum (1e-7 where theta <= 1e-4 or >= pi - 1e-4: there Theta is first-order sensitive to theta through kdot = 1/2 - theta/(2 pi), and s = sqrt(q q' - k^2) is the square
    root of a rounding residue in any FP64 evaluation)."""
    depth, sw, sb = _cfg(dom, name)
    x1, x2 = dom[f"sweep/x1_D{d}"], dom[f"sweep/x2_D{d}"]
    key = f"sweep/{name}_D{d}"
    k12, k11, k22, t12 = dom[key + "_K12"], dom[key + "_K11"], dom[key + "_K22"], dom[key + "_T12"]
    p = len(x1)
    fill = np.random.default_rng(d).standard_normal((520 - 2 * p, d))
    x = np.concatenate([x1, x2, fill])
    h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb)
    ks = h.kernel(x)
    kr = h.kernel(x, x)
    assert np.array_equal(ks, kr)
    assert np.array_equal(ks, ks.T)
    i = np.arange(p)
    scale = np.sqrt(k11 * k22)
    bar = EPS * max(8, 2 * (depth - 1))
    err = np.abs(ks[i, p + i] - k12) / scale
    assert np.max(err) <= bar, (np.argmax(err), err.max() / EPS)
    assert np.max(np.abs(ks[i, i] - k11) / k11) <= bar
    assert np.max(np.abs(ks[p + i, p + i] - k22) / k22) <= bar
    h.close()

    hn = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, kernel_type="ntk")
    tn = np.diag(hn.kernel(x1, x2))
    hn.close()
    ang = np.concatenate([dom["angles"], np.full(p - len(dom["angles"]), np.pi / 2)])
    loose = (ang <= 1e-4) | (ang >= np.pi - 1e-4)
    terr = np.abs(tn - t12) / np.max(np.abs(t12))
    assert np.max(terr[~loose]) <= 1e-12, (np.argmax(np.where(loose, 0, terr)), terr[~loose].max())
    assert np.max(terr[loose]) <= 1e-7


def test_per_layer_depth_limit(lib):
    """16 Dense layers with their own sigmas is the most per_layer allows: 17 is rejected (the sweep above runs 16)."""
    sw, sb = np.linspace(1.0, 1.6, 17), np.linspace(0.0, 0.2, 17)
    with pytest.raises(ValueError):
        lib.Handle(depth=17, sigma_w=sw, sigma_b=sb)
    h = lib.Handle(depth=16, sigma_w=sw[:16], sigma_b=sb[:16])
    x = np.random.default_rng(0).standard_normal((40, 9))
    assert relmax(h.kernel(x), oracle.kernel_fn(x, None, 16, tuple(sw[:16]), tuple(sb[:16]))) < 1e-13


def _normal_range(x, y, a, b, sw2):
    """True when every intermediate of the first arc-cosine step of kernel(2^a x, 2^b y) -- q, q', q q', k^2, s^2
    -- and the reciprocal of max(s^2, k^2) are normal doubles with room to spare (deeper layers only shrink by sw2/2)."""
    d = x.shape[1]
    q1 = sw2 * np.einsum("ij,ij->i", x, x) / d
    q2 = sw2 * np.einsum("ij,ij->i", y, y) / d
    k = sw2 * (x @ y.T) / d
    qq = np.outer(q1, q2)
    s2 = qq - k * k
    lo = min(q1.min() * 2.0 ** (2 * a), q2.min() * 2.0 ** (2 * b),
             2.0 ** (2 * (a + b)) * min(s2.min(), (k * k).min()))
    hi = 2.0 ** (2 * (a + b)) * qq.max()
    return lo > 2.0 ** -1000 and hi < 2.0 ** 1000 and q1.max() * 2.0 ** (2 * a) < Q_LIMIT and q2.max() * 2.0 ** (2 * b) < Q_LIMIT


def test_homogeneity_bitwise(lib):
    """sigma_b = 0: kernel(2^a X, 2^b Y) == 2^(a+b) kernel(X, Y) bit for bit wherever every intermediate is a normal
    double -- scaling by a power of two commutes with every rounding there, including the reciprocal seed."""
    rng = np.random.default_rng(11)
    x, y = rng.standard_normal((40, 37)), rng.standard_normal((24, 37))
    for depth, sw in [(3, 1.2), (2, 1.0)]:
        h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=0.0)
        k0 = h.kernel(x, y)
        n = 0
        for a in (-250, -160, -64, 0, 64, 160, 250):
            for b in (-250, -160, -64, 0, 64, 160, 250):
                if not _normal_range(x, y, a, b, sw * sw):
                    continue
                n += 1
                kab = h.kernel(np.ldexp(x, a), np.ldexp(y, b))
                assert np.array_equal(kab, np.ldexp(k0, a + b)), (depth, a, b)
        assert n >= 30
        h.close()


def test_magnitude_cases_against_mpmath(lib, dom):
    """The pair x = (3, 1), y = (2, -0.5) (and x 2^20, y 2^20) with x, or x and y, scaled by 2^e, depth 3, sigma_b = 0:
      * q >= 2^512 in a row: rejected (ValueError);
      * every other case: finite, and within sqrt(K_mp(x,x) K_mp(y,y)) of mpmath (|K| <= that bound is all that
        survives once q or k underflows to zero);
      * where q, q', q q' and k^2 keep >= 10 significant bits (>= 2^-1064): within 1e-3 of that scale -- subnormal
        q's carry few bits, nothing tighter is possible.  This is where the reciprocal's flush-to-zero gave NaN (max(s^2,
        k^2) subnormal) or a factor-2 error (k^2 = 0 read as s == k == 0);
      * the near-parallel pair with q in [2^511, 2^512): 8 eps of the scale (1/max(s^2, k^2) below 2^-1022 was flushed
        to 0, which snapped theta to 0)."""
    xs, ys, names = dom["mag/x"], dom["mag/y"], [str(n) for n in dom["mag/names"]]
    kxy, kxx, scales = dom["mag/K_xy"], dom["mag/K_xx"], dom["mag/scale"]
    h = lib.Handle(depth=3, sigma_w=1.0, sigma_b=0.0)
    n_tight = 0
    for x, y, name, r, rx, scale in zip(xs, ys, names, kxy, kxx, scales):
        q1, q2, kk = x @ x / 2, y @ y / 2, x @ y / 2
        if max(q1, q2) >= Q_LIMIT or not np.isfinite(max(q1, q2)):
            with pytest.raises(ValueError, match="2\\^512"):
                h.kernel(x[None], y[None])
            continue
        k = h.kernel(np.stack([x, y]))
        assert np.all(np.isfinite(k)), name
        err = abs(k[0, 1] - r)
        assert err <= scale * (1 + 1e-3) + 2.0 ** -1060, (name, k[0, 1], r)
        if name == "near_overflow":
            assert err <= 8 * EPS * scale, (name, k[0, 1], r)
            assert abs(k[0, 0] - rx) <= 8 * EPS * rx
            n_tight += 1
        elif min(q1, q2, q1 * q2, kk * kk) >= 2.0 ** -1064:
            assert err <= 1e-3 * scale, (name, k[0, 1], r)
            n_tight += 1
    assert n_tight >= 15
    h.close()


def test_homogeneity_below_the_normal_range(lib, dom):
    """kernel(2^a X, 2^b Y) for a + b from -400 down to -560 (q's and products subnormal): finite everywhere, within
    1e-3 of sqrt(K(x,x) K(y,y)) 2^(a+b) wherever q, q' and q q' keep >= 10 significant bits."""
    rng = np.random.default_rng(12)
    x, y = rng.standard_normal((16, 37)) * 2.0 ** 20, rng.standard_normal((12, 37)) * 2.0 ** 20
    h = lib.Handle(depth=3, sigma_w=1.0, sigma_b=0.0)
    k0 = h.kernel(x, y)
    dx = np.diag(h.kernel(x))
    dy = np.diag(h.kernel(y))
    scale = np.sqrt(np.outer(dx, dy))
    q1, q2 = np.einsum("ij,ij->i", x, x) / 37, np.einsum("ij,ij->i", y, y) / 37
    n = 0
    for a, b in [(-200, -200), (-250, -250), (-280, -280), (-300, -260), (-200, -330), (-230, -300), (-265, -265)]:
        kab = h.kernel(np.ldexp(x, a), np.ldexp(y, b))
        assert np.all(np.isfinite(kab)), (a, b)
        f = 2.0 ** (a + b)
        ok = min(q1.min() * 2.0 ** (2 * a), q2.min() * 2.0 ** (2 * b), np.outer(q1, q2).min() * f * f) >= 2.0 ** -1064
        bar = (1e-3 if ok else 1.0 + 1e-3) * scale * f
        assert np.all(np.abs(kab - k0 * f) <= bar), (a, b, np.max(np.abs(kab - k0 * f) / (scale * f)))
        n += ok
    assert n >= 4
    h.close()


def test_subnormal_training_row(lib):
    """A training row scaled to 2^-530 (q subnormal, k^2 and s^2 subnormal against every other row) fits and predicts
    finite values that agree with the oracle."""
    rng = np.random.default_rng(13)
    x, xt = rng.standard_normal((200, 37)), rng.standard_normal((50, 37))
    y = np.sin(x[:, 0]) + x[:, 1]
    x[5] = np.ldexp(x[5], -530)
    h = lib.Handle(depth=3, sigma_w=1.0, sigma_b=0.0)
    h.fit(x, y)
    m, v = h.predict(xt)
    assert np.all(np.isfinite(m)) and np.all(np.isfinite(v)) and np.all(v > 0)
    ref = oracle.Fit(x, y, 3, 1.0, 0.0)
    rm, rv = ref.predict(xt)
    assert relmax(m, rm) < 1e-6 and np.max(np.abs(v - rv) / np.abs(rv)) < 1e-6


def test_q_overflow_rejected(lib):
    """A row whose layer-0 diagonal reaches 2^512 is NNGP_EINVAL (ValueError) in kernel, fit, predict and append_fit,
    instead of NaN entries, a NaN pivot or NaN means with status OK."""
    rng = np.random.default_rng(14)
    x, y, xt = rng.standard_normal((64, 8)), rng.standard_normal(64), rng.standard_normal((10, 8))
    big = x.copy()
    big[3] = 0.0
    big[3, :2] = 2.0 ** 257                          # q = |x|^2 / D = 2^515 / 8 = 2^512 exactly
    just = big.copy()
    just[3, 1] = np.nextafter(2.0 ** 257, 0.0)       # q = 2^512 - 2^460: accepted
    h = lib.Handle(depth=3)
    with pytest.raises(ValueError, match="2\\^512"):
        h.kernel(big)
    with pytest.raises(ValueError, match="2\\^512"):
        h.kernel(x, big)
    assert np.all(np.isfinite(h.kernel(just, x)))
    with pytest.raises(ValueError, match="2\\^512"):
        h.fit(big, y)
    h.fit(x, y)
    with pytest.raises(ValueError, match="2\\^512"):
        h.predict(big[:10])
    m, v = h.predict(xt)
    assert np.all(np.isfinite(m)) and np.all(np.isfinite(v))
    with pytest.raises(ValueError, match="2\\^512"):
        h.append_fit(big[:4], y[:4])
    h.close()
    ha = lib.Handle(depth=3, diag_reg_absolute=True, diag_reg=1e-2)   # the incremental append
    ha.fit(x, y)
    with pytest.raises(ValueError, match="2\\^512"):
        ha.append_fit(big[:4], y[:4])
    ha.close()


def _signed_problem(n, t, d, seed):
    rng = np.random.default_rng(seed)
    x, xt = rng.standard_normal((n, d)), rng.standard_normal((t, d))
    w = rng.standard_normal(d)
    return x, np.sin(x @ w) * 4.0 + x[:, 0] ** 2, xt


def _check_posterior(m, v, rm, rv):
    e_mean = relmax(m, rm)
    e_var = float(np.max(np.abs(v - rv) / np.abs(rv)))
    e_q = float(np.max(np.abs(2.0 ** np.abs(m - rm) - 1.0)))
    assert e_mean < 1e-6 and e_var < 1e-6 and e_q < 1e-3, (e_mean, e_var, e_q)


def test_signed_features_posterior(lib):
    """Standard-normal features (first-layer k < 0 for about half the pairs): NNGP against oracle.Fit, and the same
    problem on latency_mode and variance_slices=7 handles (mean bitwise the default handle's)."""
    x, y, xt = _signed_problem(3000, 2000, 37, 15)
    depth, sw, sb = 3, 1.0, 0.1
    ref = oracle.Fit(x, y, depth, sw, sb)
    rm, rv = ref.predict(xt)
    h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb)
    h.fit(x, y)
    m, v = h.predict(xt)
    _check_posterior(m, v, rm, rv)
    h.close()
    for kw in ({"latency_mode": True}, {"variance_slices": 7}):
        hk = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, **kw)
        hk.fit(x, y)
        mk, vk = hk.predict(xt)
        assert np.array_equal(mk, m), kw
        assert float(np.max(np.abs(vk - rv) / np.abs(rv))) < 1e-6, kw
        hk.close()


def test_signed_features_posterior_ntk(lib):
    x, y, xt = _signed_problem(3000, 2000, 37, 16)
    depth, sw, sb = 3, 1.0, 0.1
    ref = oracle.FitNTK(x, y, depth, sw, sb)
    rm, rv = ref.predict(xt)
    h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, kernel_type="ntk")
    h.fit(x, y)
    m, v = h.predict(xt)
    _check_posterior(m, v, rm, rv)
    h.close()


@pytest.mark.parametrize("kernel_type", ["nngp", "ntk"])
def test_signed_golden_posterior(lib, dom, kernel_type):
    """The small signed fit / predict of the golden file (50-digit mpmath) at 1e-8 (NTK: 1e-7, the bar of
    test_ntk_against_mpmath_golden)."""
    x, y, xt = dom["post/x_train"], dom["post/y_train"], dom["post/x_test"]
    depth, sw, sb, reg = dom["post/cfg"]
    h = lib.Handle(depth=int(depth), sigma_w=sw, sigma_b=sb, diag_reg=reg, kernel_type=kernel_type)
    h.fit(x, y)
    m, v = h.predict(xt)
    pre = "post/" if kernel_type == "nngp" else "post/ntk_"
    # (NTK: Theta's diagonal -- hence lambda -- is first-order sensitive to the rounding residue in s, as in
    #  test_ntk_against_mpmath_golden)
    assert abs(h.dims()[2] - float(dom[pre + "lam"])) < (1e-12 if kernel_type == "nngp" else 1e-8) * float(dom[pre + "lam"])
    tol = 1e-8 if kernel_type == "nngp" else 1e-7
    assert relmax(m, dom[pre + "mean"]) < tol
    assert relmax(v, dom[pre + "var"]) < tol
    h.close()
