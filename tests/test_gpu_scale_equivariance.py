"""GPU: fit and every prediction path against the exact power-of-two symmetries of the posterior.

With sigma_b = 0 and a positively homogeneous activation (ReLU, LeakyRelu, Abs, ABRelu), scaling X and X* by 2^a
scales K, lambda (relative diag_reg) and the variance by 4^a, L by 2^a and alpha by 4^-a, and leaves the mean alone.
Every operation of the paths commutes exactly with that scaling while its operands and results are normal doubles, so
inside a window computed from the unscaled problem (_window) each path must give the scaled result bit for bit: a
hidden absolute constant, a clamp, a flushed subnormal or an exponent computation would all show.  The same holds for
y -> 2^c y (alpha and the mean scale, the variance and covariance do not move), for sigma_w -> 2^t sigma_w, and for
Erf with X -> 2^t X, b -> 2^-t b.  Between the window and the documented range limits (K subnormal, q subnormal) the
calls must return finite results close to the scaled ones, or fail with a message.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

Q_LIMIT_EXP = 512                   # layer-0 q (and, with ABRelu, every layer's diagonal) must stay below 2^512
MARGIN = 2.0 ** 20                  # room for GPU summation order against the normal range's edges


def _window(parts, margin=MARGIN):
    """Integer range [lo, hi] of a for which every part stays a normal double with ``margin`` to spare.

    ``parts``: (array, p) or (array, p, top) -- the array scales as 2^(p a); every nonzero magnitude m must keep
    m 2^(p a) >= 2^-1022 margin and m 2^(p a) < 2^top / margin (top: 1024 unless given; margin a power of two)."""
    lo, hi = -math.inf, math.inf
    for part in parts:
        arr, p = np.abs(np.asarray(part[0], dtype=np.float64)), part[1]
        top = part[2] if len(part) > 2 else 1024
        nz = arr[arr > 0]
        if nz.size == 0:
            continue
        # binary exponents: m in [2^small, 2^(big+1))
        small, big = math.floor(math.log2(float(nz.min()))), math.floor(math.log2(float(nz.max())))
        floor_, ceil_ = -1022 + math.log2(margin), top - 1 - math.log2(margin)
        if p == 0:
            if small < floor_ or big > ceil_:
                return 1, 0
            continue
        # floor_ <= small + p a  and  big + p a <= ceil_
        b1, b2 = (floor_ - small) / p, (ceil_ - big) / p
        lo, hi = (max(lo, b1), min(hi, b2)) if p > 0 else (max(lo, b2), min(hi, b1))
    return math.ceil(lo), math.floor(hi)


def _step_parts(k, top=1024):
    """What one activation step forms from the covariance k (the layer it reads): q, q q', k^2, s^2 = q q' - k^2 and
    the reciprocal of max(s^2, k^2); all scale with X (q as 4^a, the products as 16^a)."""
    q = np.diag(k)
    qq = np.outer(q, q)
    s2 = np.maximum(qq - k * k, 0.0)
    # (qq 2^-53: the rounding residue s^2 of a pair at angle 0, the diagonal of a symmetric Gram, must stay normal)
    return [(q, 2, top), (qq, 4), (k * k, 4), (s2, 4), (qq * 2.0 ** -53, 4), (1.0 / np.maximum(s2, k * k), -4)]


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


def _problem(n, t, d, seed, signed_rows=8):
    """Features with nonzero magnitudes in [0.5, 1) (every partial product of the Gram stays normal wherever the
    result is), about 10 % exact zeros, a few rows with signed entries; labels O(1)."""
    rng = np.random.default_rng(seed)

    def feats(rows):
        x = rng.uniform(0.5, 1.0, size=(rows, d))
        x[rng.random((rows, d)) < 0.1] = 0.0
        sel = rng.choice(rows, signed_rows, replace=False)
        x[sel] *= np.where(rng.random((signed_rows, d)) < 0.5, -1.0, 1.0)
        return x

    x, xt = feats(n), feats(t)
    y = np.sin(3.0 * x[:, 0]) + x[:, 1] - 0.5
    return x, y, xt


ACTS = {
    "relu_d1": dict(depth=1),
    "relu_d2": dict(depth=2),
    "relu_d3": dict(depth=3),
    "leaky_d2": dict(depth=2, act=("abrelu", 0.1, 1.0)),
    "abs_d2": dict(depth=2, act=("abrelu", -1.0, 1.0)),
    "abrelu_d3": dict(depth=3, act=("abrelu", -0.4, 1.6)),
    "per_layer_d3": dict(depth=3, sigma_w=[1.3, 0.75, 1.1]),
}


def _handle(lib, cfg, **kw):
    act = cfg.get("act")
    activation = lib.Activation(*act) if act else None
    return lib.Handle(depth=cfg["depth"], sigma_w=cfg.get("sigma_w", 1.0), sigma_b=0.0, activation=activation, **kw)


def _prefix_cfg(cfg, depth):
    sub = dict(cfg, depth=depth)
    if isinstance(cfg.get("sigma_w"), list):
        sub["sigma_w"] = cfg["sigma_w"][:depth] if depth > 1 else cfg["sigma_w"][0]
    return sub


def _posterior_parts(lib, cfg, x, y, xt, h0, kernel_type="nngp"):
    """Every intermediate the fit and the prediction paths form, from the unscaled problem: each layer's step inputs
    (_step_parts), K, lambda, L, L^2, L^-1, alpha, K_*, K_**, V = L^-1 K_*^T, V^2 and the products K_* alpha."""
    xa = np.vstack([x, xt])
    parts = []
    for layer in range(1, cfg["depth"]):
        hl = _handle(lib, _prefix_cfg(cfg, layer))
        parts += _step_parts(hl.kernel(xa), top=Q_LIMIT_EXP)
        hl.close()
    hk = _handle(lib, cfg)
    ka = hk.kernel(xa)
    hk.close()
    n = x.shape[0]
    st = h0.get_state()
    L, alpha, lam = st["l"], st["alpha"], st["lambda"]
    q0 = np.einsum("ij,ij->i", xa, xa) / xa.shape[1]
    sw = cfg.get("sigma_w", 1.0)
    sw0 = sw[0] if isinstance(sw, list) else sw
    linv = np.linalg.inv(L)
    ks = ka[n:, :n]
    v = linv @ ks.T
    parts += [(q0 * sw0 * sw0, 2, Q_LIMIT_EXP), (ka, 2), (np.array([lam]), 2), (L, 1), (L * L, 2), (linv, -1),
              (alpha, -2), (v, 1), (v * v, 2), (ks * alpha[None, :], 0), (ks @ alpha, 0)]
    if kernel_type == "ntk":
        parts += [(st["m"], 0)]
    return parts


def _scaled(a, x):
    return np.ldexp(x, a)


def _pick(lo, hi, n=4):
    """The window's edges and a few points inside (never 0, which is the unscaled problem itself)."""
    pts = {lo, hi, (lo + hi) // 2 + 1, lo + (hi - lo) // 5, hi - (hi - lo) // 5}
    return sorted(a for a in pts if a != 0 and lo <= a <= hi)[: n + 1]


@pytest.mark.parametrize("name", list(ACTS))
def test_fit_and_every_prediction_path_scale_bitwise(lib, name, monkeypatch):
    """Inside the window: lambda x4^a, L x2^a, alpha x4^-a; the mean bitwise unchanged and the variance x4^a on the
    persistent substitution, the right-looking path, latency_mode and the digit-plane (variance_slices=7) path;
    predict_cov x4^a; active_select TOPK the same rows with scores x2^a; the log marginal likelihood moves by exactly
    the terms the scaling adds."""
    cfg = ACTS[name]
    n, t = (1000, 300) if cfg["depth"] != 2 else (577, 513)
    x, y, xt = _problem(n, t, 21, seed=len(name))
    xc = xt[:96]
    h0 = _handle(lib, cfg)
    h0.fit(x, y)
    st0 = h0.get_state()
    lam0 = h0.dims()[2]
    m0, v0 = h0.predict(xt)
    monkeypatch.setenv("NNGP_SMALL_BATCH_TILES", "1000000")
    mr0, vr0 = h0.predict(xt)
    monkeypatch.delenv("NNGP_SMALL_BATCH_TILES")
    _mc0, c0 = h0.predict_cov(xc)
    idx0, sc0 = h0.active_select(xt, 17, return_scores=True)
    lml0 = h0.log_marginal_likelihood()
    hl0 = _handle(lib, cfg, latency_mode=True)
    hl0.fit(x, y)
    ml0, vl0 = hl0.predict(xt)
    hs0 = _handle(lib, cfg, variance_slices=7)
    hs0.fit(x, y)
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")
    ms0, vs0 = hs0.predict(xt)
    monkeypatch.delenv("NNGP_LATENCY_ROWS")

    lo, hi = _window(_posterior_parts(lib, cfg, x, y, xt, h0))
    assert lo < -100 and hi > 100, (lo, hi)
    ytal0 = float(y @ st0["alpha"])
    slog0 = float(np.sum(np.log(np.diag(st0["l"]))))
    checked = 0
    for a in _pick(lo, hi):
        xs, xts = _scaled(a, x), _scaled(a, xt)
        h = _handle(lib, cfg)
        h.fit(xs, y)
        st = h.get_state()
        assert h.dims()[2] == np.ldexp(lam0, 2 * a), a
        assert np.array_equal(st["x"], xs)
        assert np.array_equal(st["l"], np.ldexp(st0["l"], a)), a
        assert np.array_equal(st["alpha"], np.ldexp(st0["alpha"], -2 * a)), a
        m, v = h.predict(xts)
        assert np.array_equal(m, m0) and np.array_equal(v, np.ldexp(v0, 2 * a)), ("persistent", a)
        monkeypatch.setenv("NNGP_SMALL_BATCH_TILES", "1000000")
        m, v = h.predict(xts)
        monkeypatch.delenv("NNGP_SMALL_BATCH_TILES")
        assert np.array_equal(m, mr0) and np.array_equal(v, np.ldexp(vr0, 2 * a)), ("right-looking", a)
        _mc, c = h.predict_cov(xts[:96])
        assert np.array_equal(c, np.ldexp(c0, 2 * a)), ("predict_cov", a)
        idx, sc = h.active_select(xts, 17, return_scores=True)
        assert np.array_equal(idx, idx0) and np.array_equal(sc, np.ldexp(sc0, a), equal_nan=True), ("active_select", a)
        want = -0.5 * math.ldexp(ytal0, -2 * a) - (slog0 + n * a * math.log(2.0)) - 0.5 * n * math.log(2 * math.pi)
        terms = 0.5 * abs(math.ldexp(ytal0, -2 * a)) + abs(slog0) + n * abs(a) + n
        assert abs(h.log_marginal_likelihood() - want) <= 1e-12 * terms, (a, h.log_marginal_likelihood(), want, lml0)
        h.close()

        hl = _handle(lib, cfg, latency_mode=True)
        hl.fit(xs, y)
        m, v = hl.predict(xts)
        assert np.array_equal(m, ml0) and np.array_equal(v, np.ldexp(vl0, 2 * a)), ("latency_mode", a)
        hl.close()
        hs = _handle(lib, cfg, variance_slices=7)
        hs.fit(xs, y)
        monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")
        m, v = hs.predict(xts)
        monkeypatch.delenv("NNGP_LATENCY_ROWS")
        assert hs.stats()["sliced_macs"] > 0
        assert np.array_equal(m, ms0) and np.array_equal(v, np.ldexp(vs0, 2 * a)), ("variance_slices", a)
        hs.close()
        checked += 1
    assert checked >= 3
    for hh in (h0, hl0, hs0):
        hh.close()


def test_ntk_covariance_and_m_scale_bitwise(lib):
    """'ntk' (ReLU, depth 3): Theta, K and the covariance x4^a, M = L^-1 K_dd L^-T bitwise unchanged."""
    cfg = dict(depth=3)
    x, y, xt = _problem(700, 200, 19, seed=7)
    h0 = _handle(lib, cfg, kernel_type="ntk")
    h0.fit(x, y)
    st0 = h0.get_state()
    m0, v0 = h0.predict(xt)
    _mc0, c0 = h0.predict_cov(xt)
    hn = _handle(lib, cfg, kernel_type="ntk")
    theta = hn.kernel(np.vstack([x, xt]))
    hn.close()
    lo, hi = _window(_posterior_parts(lib, cfg, x, y, xt, h0, "ntk") + [(theta, 2)])
    assert lo < -100 and hi > 100, (lo, hi)
    for a in _pick(lo, hi, 3):
        h = _handle(lib, cfg, kernel_type="ntk")
        h.fit(_scaled(a, x), y)
        st = h.get_state()
        assert np.array_equal(st["m"], st0["m"]), a
        assert np.array_equal(st["l"], np.ldexp(st0["l"], a)), a
        m, v = h.predict(_scaled(a, xt))
        assert np.array_equal(m, m0) and np.array_equal(v, np.ldexp(v0, 2 * a)), a
        _mc, c = h.predict_cov(_scaled(a, xt))
        assert np.array_equal(c, np.ldexp(c0, 2 * a)), a
        h.close()
    h0.close()


def test_append_fit_and_imported_states_scale_bitwise(lib):
    """append_fit (the refit with relative diag_reg, and the incremental path with an absolute lambda scaled by 4^a)
    and states imported through set_state and through pack / unpack predict the scaled posterior bit for bit."""
    cfg = dict(depth=2)
    x, y, xt = _problem(1300, 300, 23, seed=3)
    n1 = 1000
    lam_abs = 0.01
    base = {}
    for mode in ("refit", "incremental"):
        kw = dict(diag_reg=lam_abs, diag_reg_absolute=True) if mode == "incremental" else {}
        h = _handle(lib, cfg, **kw)
        h.fit(x[:n1], y[:n1])
        h.append_fit(x[n1:], y[n1:])
        base[mode] = (h.get_state(), *h.predict(xt))
        h.close()
    h0 = _handle(lib, cfg)
    h0.fit(x, y)
    lo, hi = _window(_posterior_parts(lib, cfg, x, y, xt, h0) + [(np.array([lam_abs]), 2)])
    st0 = h0.get_state()
    m0, v0 = h0.predict(xt)
    size = h0.packed_size()
    assert lo < -100 and hi > 100, (lo, hi)
    for a in _pick(lo, hi, 3):
        xs, xts = _scaled(a, x), _scaled(a, xt)
        for mode in ("refit", "incremental"):
            kw = dict(diag_reg=np.ldexp(lam_abs, 2 * a), diag_reg_absolute=True) if mode == "incremental" else {}
            h = _handle(lib, cfg, **kw)
            h.fit(xs[:n1], y[:n1])
            h.append_fit(xs[n1:], y[n1:])
            stb, mb, vb = base[mode]
            st = h.get_state()
            assert np.array_equal(st["l"], np.ldexp(stb["l"], a)), (mode, a)
            assert np.array_equal(st["alpha"], np.ldexp(stb["alpha"], -2 * a)), (mode, a)
            m, v = h.predict(xts)
            assert np.array_equal(m, mb) and np.array_equal(v, np.ldexp(vb, 2 * a)), (mode, a)
            h.close()
        # imported: the scaled state of the unscaled fit, through set_state and through the packed stream
        himp = _handle(lib, cfg)
        himp.set_state(xs, np.ldexp(st0["l"], a), np.ldexp(st0["alpha"], -2 * a), np.ldexp(st0["lambda"], 2 * a))
        m, v = himp.predict(xts)
        assert np.array_equal(m, m0) and np.array_equal(v, np.ldexp(v0, 2 * a)), ("set_state", a)
        packed = np.empty(size)
        himp.state_pack(0, size, packed)
        hp = _handle(lib, cfg)
        hp.state_import_begin(*xs.shape)
        hp.state_unpack(0, size, packed)
        hp.state_import_end(np.ldexp(st0["lambda"], 2 * a))
        m, v = hp.predict(xts)
        assert np.array_equal(m, m0) and np.array_equal(v, np.ldexp(v0, 2 * a)), ("pack / unpack", a)
        himp.close(); hp.close()
    h0.close()


def test_label_scaling_leaves_variance_and_covariance_bitwise(lib):
    """y -> 2^c y: alpha and the mean x2^c; the variance (every path) and the covariance do not move at all."""
    cfg = dict(depth=3)
    x, y, xt = _problem(900, 250, 17, seed=5)
    out = {}
    for c in (0, -300, -37, 41, 500):
        yc = np.ldexp(y, c)
        h, hl = _handle(lib, cfg), _handle(lib, cfg, latency_mode=True)
        h.fit(x, yc)
        hl.fit(x, yc)
        out[c] = (h.get_state()["alpha"], *h.predict(xt), h.predict_cov(xt[:64])[1], *hl.predict(xt))
        h.close(); hl.close()
    a0, m0, v0, c0, ml0, vl0 = out[0]
    for c, (a, m, v, cv, ml, vl) in out.items():
        assert np.array_equal(a, np.ldexp(a0, c)) and np.array_equal(m, np.ldexp(m0, c)), c
        assert np.array_equal(ml, np.ldexp(ml0, c)), c
        assert np.array_equal(v, v0) and np.array_equal(cv, c0) and np.array_equal(vl, vl0), c


@pytest.mark.parametrize("depth,ts", [(2, (3,)), (3, (-5,)), (3, (2, -3, 4))])
def test_sigma_w_scaling_bitwise(lib, depth, ts):
    """sigma_b = 0: sigma_w -> 2^t sigma_w scales K by 4^(t depth); per-layer sigma_w_l -> 2^(t_l) sigma_w_l by
    4^(sum t_l).  The posterior follows: lambda and the variance by the same factor, the mean unchanged."""
    x, y, xt = _problem(600, 150, 13, seed=depth)
    sw0 = [1.0, 0.9, 1.2][:depth]
    sws = [np.ldexp(s, ts[i] if len(ts) > 1 else ts[0]) for i, s in enumerate(sw0)]
    shift = sum(ts) if len(ts) > 1 else ts[0] * depth
    h0, h = lib.Handle(depth=depth, sigma_w=sw0), lib.Handle(depth=depth, sigma_w=sws)
    assert np.array_equal(h.kernel(x, xt), np.ldexp(h0.kernel(x, xt), 2 * shift))
    h0.fit(x, y); h.fit(x, y)
    assert h.dims()[2] == np.ldexp(h0.dims()[2], 2 * shift)
    m0, v0 = h0.predict(xt)
    m, v = h.predict(xt)
    assert np.array_equal(m, m0) and np.array_equal(v, np.ldexp(v0, 2 * shift))
    h0.close(); h.close()


@pytest.mark.parametrize("depth", [2, 3])
def test_erf_input_and_b_scaling_bitwise(lib, depth):
    """Erf(a, b, c) reads b^2 q and b^2 k only: X -> 2^t X with b -> 2^-t b leaves the first step's input, and so the
    kernel and the whole posterior, bitwise unchanged (Erf has no input homogeneity, so this is its symmetry).  b is
    shared by every step, so at depth 3 the second step's input must scale too: sigma_w of Dense layer 1 -> 2^t."""
    x, y, xt = _problem(640, 160, 11, seed=depth + 40)
    a_, b_, c_ = 1.3, 0.7, 0.2
    sw = [1.0, 0.9, 1.2][:depth] if depth > 2 else 1.0

    def handle(t):
        swt = [sw[0], np.ldexp(sw[1], t), sw[2]] if depth > 2 else sw
        return lib.Handle(depth=depth, sigma_w=swt, activation=lib.Activation("erf", a_, np.ldexp(b_, -t), c_))

    h0 = handle(0)
    k0 = h0.kernel(x, xt)
    h0.fit(x, y)
    m0, v0 = h0.predict(xt)
    _mc0, c0 = h0.predict_cov(xt[:50])
    for t in (-240, -90, 33, 200):          # (b^2 times a later layer's diagonal bound must stay below 2^508)
        h = handle(t)
        xs, xts = np.ldexp(x, t), np.ldexp(xt, t)
        assert np.array_equal(h.kernel(xs, xts), k0), t
        h.fit(xs, y)
        assert h.dims()[2] == h0.dims()[2]
        m, v = h.predict(xts)
        assert np.array_equal(m, m0) and np.array_equal(v, v0), t
        assert np.array_equal(h.predict_cov(xts[:50])[1], c0), t
        h.close()
    h0.close()


# ---- between the window and the range limits ---------------------------------------------------------------------

def _bar(bits):
    """Bar, relative to K_** (variance) or max |mean|, for a problem whose smallest kernel intermediate keeps ``bits``
    significant bits: 1e-9 while it is normal (53 bits), 2^(12 - bits) below, never looser than the scale itself."""
    return 1e-9 if bits >= 53 else max(1e-9, min(1.0 + 1e-3, 2.0 ** (12 - bits)))


def _bits(v):
    """Significant bits a double of magnitude v keeps (53 when normal, fewer in the subnormal range, 0 below)."""
    return 53 if v >= 2.0 ** -1022 else max(0.0, math.log2(v) + 1074) if v > 0 else 0.0


def test_depth1_sliced_variance_with_k_at_the_bottom_of_the_normal_range(lib, monkeypatch):
    """Depth 1 (the linear kernel) with X, X* scaled by 2^-509: K and K_* entries in [2^-1022, 2^-1018), so every
    K_* row has exponent e <= -1018, where the digit-plane scale-up 2^(6-e) is not a double.  Relative diag_reg 0.5
    keeps lambda normal.  Every path must agree with the unscaled posterior: mean within 1e-9, variance within 1e-9
    4^a K_**.  (The digit planes of such rows used to be split with an infinite scale-up: the variance came out wrong
    by O(K_**) with status OK.)"""
    x, y, xt = _problem(700, 400, 16, seed=9, signed_rows=0)
    a = -509
    xs, xts = np.ldexp(x, a), np.ldexp(xt, a)
    h = lib.Handle(depth=1, diag_reg=0.5)
    kss0 = np.einsum("ij,ij->i", xt, xt) / xt.shape[1]
    ks = h.kernel(xts, xs)
    assert ks.max() < 2.0 ** -1018 and np.mean(ks >= 2.0 ** -1022) > 0.999
    h.close()
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")
    for kw in ({}, {"latency_mode": True}, {"variance_slices": 7}):
        h0, h = lib.Handle(depth=1, diag_reg=0.5, **kw), lib.Handle(depth=1, diag_reg=0.5, **kw)
        h0.fit(x, y)
        m0, v0 = h0.predict(xt)
        h.fit(xs, y)
        m, v = h.predict(xts)
        if kw.get("variance_slices"):
            assert h.stats()["sliced_macs"] > 0
        assert np.all(np.isfinite(m)) and np.all(np.isfinite(v)), kw
        assert np.max(np.abs(m - m0)) <= 1e-9 * max(1.0, np.max(np.abs(m0))), kw
        err = np.abs(np.ldexp(v, -2 * a) - v0) / kss0
        assert np.max(err) <= 1e-9, (kw, float(np.max(err)))
        h0.close(); h.close()


@pytest.mark.parametrize("depth,a", [(1, -511), (1, -516), (1, -530), (2, -258), (2, -262), (3, -270)])
def test_below_the_window_finite_or_clear_error(lib, depth, a, monkeypatch):
    """Depth 1 with K at and below the subnormal boundary, depth >= 2 with q q' subnormal.  lambda is absolute:
    0.05 4^a, or 2^-1020 where that would be subnormal (the unscaled reference then uses 2^-1020 4^-a).  Every path
    (substitution, latency_mode, variance_slices) returns finite outputs or fails with a message; the mean and the
    variance follow the unscaled posterior within _bar of the fewest significant bits that K, q and q q' keep --
    1e-9 while they are normal, the scale itself once they are gone (as test_homogeneity_below_the_normal_range)."""
    x, y, xt = _problem(520, 130, 12, seed=depth + 60, signed_rows=0)
    lam = max(np.ldexp(0.05, 2 * a), 2.0 ** -1020)
    lam0 = np.ldexp(lam, -2 * a)
    xs, xts = np.ldexp(x, a), np.ldexp(xt, a)
    xa = np.vstack([x, xt])
    q = np.einsum("ij,ij->i", xa, xa) / xa.shape[1]
    hk = lib.Handle(depth=depth)
    ka = hk.kernel(xa)
    hk.close()
    kss0 = np.diag(ka)[x.shape[0]:]
    small = [ka[ka > 0].min() * 2.0 ** (2 * a)]
    if depth > 1:
        small += [q.min() * 2.0 ** (2 * a), q.min() ** 2 * 2.0 ** (4 * a)]
    bar = _bar(min(_bits(v) for v in small))
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")
    n_ok = 0
    for kw in ({}, {"latency_mode": True}, {"variance_slices": 7}):
        h0 = lib.Handle(depth=depth, diag_reg=lam0, diag_reg_absolute=True, **kw)
        h0.fit(x, y)
        m0, v0 = h0.predict(xt)
        h0.close()
        h = lib.Handle(depth=depth, diag_reg=lam, diag_reg_absolute=True, **kw)
        try:
            h.fit(xs, y)
            m, v = h.predict(xts)
        except (ValueError, np.linalg.LinAlgError) as e:
            assert "nngp_b200" in str(e) and len(str(e)) > 20, e
            continue
        finally:
            h.close()
        assert np.all(np.isfinite(m)) and np.all(np.isfinite(v)), kw
        e_m = np.max(np.abs(m - m0)) / max(1.0, np.max(np.abs(m0)))
        e_v = np.max(np.abs(np.ldexp(v, -2 * a) - v0) / kss0)
        assert e_m <= bar and e_v <= bar, (kw, bar, e_m, e_v)
        n_ok += 1
    assert n_ok >= 1


def test_alpha_overflow_is_an_error(lib):
    """lambda = 2^-1022 (absolute) against K ~ 2^-1018 of rank D = 8 and labels of about 10: alpha = (K + lambda I)^-1
    y reaches 10 2^1022 along the null space of K and overflows.  nngp_fit, and the incremental nngp_append_fit,
    fail with NNGP_EINVAL naming the overflow instead of a model that predicts inf or NaN means."""
    x, _y, _xt = _problem(400, 50, 8, seed=2, signed_rows=0)
    y = 10.0 * np.random.default_rng(3).standard_normal(400)
    xs = np.ldexp(x, -509)
    h = lib.Handle(depth=1, diag_reg=2.0 ** -1022, diag_reg_absolute=True)
    with pytest.raises(ValueError, match="overflow"):
        h.fit(xs, y)
    h.fit(xs[:300], 1e-6 * y[:300])                     # alpha ~ 2^1005: fits
    assert np.all(np.isfinite(h.get_state()["alpha"]))
    with pytest.raises(ValueError, match="overflow"):
        h.append_fit(xs[300:], y[300:])
    h.close()
