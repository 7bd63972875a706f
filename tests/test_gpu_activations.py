"""GPU: the ABRelu family and Erf in the Gram epilogue (gemm_nt_kernel<EPI_GRAM, ACT_ABRELU / ACT_ERF>) and the
diagonal kernel (q_final_kernel), through every layer above them:

  * the angle sweep and magnitude rows of tests/golden/mp_act.npz (50-digit mpmath), symmetric and rectangular
    launches bitwise equal, and the input range of each activation;
  * fit / predict / full covariance / log marginal likelihood against the mpmath posteriors, against the numpy
    oracle at ragged shapes and at N = 8192 under the 1e-6 parity gate;
  * ABRelu(0, 1) through nngp_create_with_activation is bitwise the default (ReLU) handle;
  * Erf on the latency-mode and variance_slices handles, the covariance diagonal, 2 GPUs, the packed state,
    save / load and the incremental append.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import act_oracle  # noqa: E402
import nngp_oracle as oracle  # noqa: E402

EPS = np.finfo(np.float64).eps
ACTS = {"leaky": ("abrelu", 0.1, 1.0, 0.0), "abs": ("abrelu", -1.0, 1.0, 0.0), "abrelu": ("abrelu", -0.3, 1.2, 0.0),
        "erf": ("erf", 1.0, 1.0, 0.0), "erf_abc": ("erf", 1.5, 0.7, 0.2), "erf_bigb": ("erf", 1.0, 1e3, 0.0)}
SWEEP_CFG = {2: (1.0, 0.0), 3: (1.3, 0.1)}


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


@pytest.fixture(scope="module")
def mpa(golden_dir):
    return dict(np.load(golden_dir / "mp_act.npz"))


def _act(lib, name):
    return lib.Activation(*ACTS[name])


def bounds(name, x, depth, sw, sb):
    """(mask, K bound, Theta bound) per pair of rows of x, relative to sqrt(K_mp(x,x) K_mp(y,y)):
      * the ABRelu family: 8 eps (the ReLU sweep's bound: its step is ReLU's with other constants) wherever the
        layer-0 product q q' is a normal double (below, s and k lose their bits, as for ReLU); Theta 1e-12, and 1e-7 on
        pairs parallel in layer 0 (the diagonal, and with sigma_b > 0 the zero and tiny rows, whose q and k are all
        sigma_b^2): theta is a rounding residue there, first-order in Theta through kdot, as for ReLU;
      * Erf: 16 eps (DESIGN.md 5.12) and Theta 1e-12 on every pair, times act_oracle.erf_amplification -- 1 except on
        near-parallel pairs and the diagonal, where saturated Erf amplifies the rounding of k."""
    q = oracle.layer0_diag(x, sw, sb)
    qq = np.outer(q, q)
    if ACTS[name][0] == "abrelu":
        k0 = sw ** 2 * (x @ x.T) / x.shape[1] + sb ** 2
        with np.errstate(invalid="ignore", divide="ignore"):
            parallel = ~(np.abs(k0) / np.sqrt(qq) < 1.0 - 5e-7)          # (layer-0 angle within 1e-3 of 0 or pi)
        ok = (qq >= 2.0 ** -1000) & (qq <= 2.0 ** 1000)
        return ok, np.full(qq.shape, 8 * EPS), np.where(parallel, 1e-7, 1e-12)
    f, g = act_oracle.erf_amplification(x, depth, sw, sb, ACTS[name])
    return qq <= 2.0 ** 1000, 16 * EPS * f, 1e-12 * g


def _check(k, ref, ok, bar):
    d = np.abs(np.diag(ref))
    scale = np.sqrt(np.outer(d, d))
    ok = ok & (scale > 0)
    err = np.abs(k - ref)[ok] / scale[ok]
    assert err.size and np.all(err <= bar[ok]), (np.max(err / bar[ok]), np.argwhere(ok)[np.argmax(err / bar[ok])])


@pytest.mark.parametrize("name", sorted(ACTS))
@pytest.mark.parametrize("depth", [2, 3])
def test_angle_sweep_against_mpmath(lib, mpa, name, depth):
    """K and Theta within bounds() of mpmath at every angle (0 .. pi, down to 1e-8 from either end); symmetric (>= 512
    rows: lower tiles + mirror) and rectangular launches bitwise equal."""
    sw, sb = SWEEP_CFG[depth]
    x = mpa[f"{name}/sweep_x"]
    p = len(x)
    fill = np.random.default_rng(depth).standard_normal((520 - p, x.shape[1]))
    xx = np.concatenate([x, fill])
    h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, activation=_act(lib, name))
    ks, kr = h.kernel(xx), h.kernel(xx, xx)
    assert np.array_equal(ks, kr) and np.array_equal(ks, ks.T)
    ok, kbar, tbar = bounds(name, x, depth, sw, sb)
    _check(ks[:p, :p], mpa[f"{name}/sweep_nngp_d{depth}"], ok, kbar)
    hn = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, kernel_type="ntk", activation=_act(lib, name))
    t = hn.kernel(x)
    assert np.array_equal(t, hn.kernel(x, x))
    _check(t, mpa[f"{name}/sweep_ntk_d{depth}"], ok, tbar)


@pytest.mark.parametrize("name", sorted(ACTS))
@pytest.mark.parametrize("depth", [2, 3])
def test_magnitude_rows_against_mpmath(lib, mpa, name, depth):
    """A zero row, a subnormal row and norms 1e-150 .. the top of the range (1e75; Erf 1e70): every entry finite, and
    K and Theta within bounds() of mpmath."""
    sw, sb = SWEEP_CFG[depth]
    x = mpa[f"{name}/mag_x"]
    ok, kbar, tbar = bounds(name, x, depth, sw, sb)
    for get, bar in (("nngp", kbar), ("ntk", tbar)):
        h = lib.Handle(depth=depth, sigma_w=sw, sigma_b=sb, kernel_type=get, activation=_act(lib, name))
        k = h.kernel(x)
        assert np.all(np.isfinite(k))
        assert np.array_equal(k, h.kernel(x, x))
        _check(k, mpa[f"{name}/mag_{get}_d{depth}"], ok, bar)


def test_input_range(lib):
    """Layer-0 q up to just below 2^512 for the ABRelu family; Erf also needs b^2 q < 2^508 (NNGP_EINVAL otherwise),
    and rejects at creation what its later layers could push past that."""
    d = 4
    row = lambda q: np.full((1, d), np.sqrt(q))             # q = |x|^2 / d
    x_ok = np.vstack([row(2.0 ** 511.9), row(1.0)])
    h = lib.Handle(depth=3, activation=lib.Activation("abrelu", 0.1, 1.0))
    assert np.all(np.isfinite(h.kernel(x_ok)))
    with pytest.raises(ValueError, match="out of range"):
        h.kernel(np.vstack([row(2.0 ** 512.1), row(1.0)]))
    # Abs with sigma_w = 2: each step multiplies q by sigma_w^2 (a^2+b^2)/2 = 4, so two steps need the layer-0
    # q = sigma_w^2 |x|^2 / D = 4 |x|^2 / D below 2^508
    ha = lib.Handle(depth=3, sigma_w=2.0, activation=lib.Activation("abrelu", -1.0, 1.0))
    k = ha.kernel(np.vstack([row(2.0 ** 505.9), row(1.0)]))
    assert np.all(np.isfinite(k))
    with pytest.raises(ValueError, match="must stay below"):
        ha.kernel(np.vstack([row(2.0 ** 506.1), row(1.0)]))
    with pytest.raises(ValueError, match="reaches 2\\^512"):
        lib.Handle(depth=3, sigma_b=2.0 ** 257, activation=lib.Activation("abrelu", -1.0, 1.0))
    b = 1e3
    he = lib.Handle(depth=3, activation=lib.Activation("erf", 1.0, b, 0.0))
    qtop = 2.0 ** 507.9 / b ** 2
    k = he.kernel(np.vstack([row(qtop), row(1.0), -row(qtop)]))
    assert np.all(np.isfinite(k)) and k[0, 2] < 0
    with pytest.raises(ValueError, match="out of range"):
        he.kernel(np.vstack([row(2.0 ** 508.1 / b ** 2), row(1.0)]))
    with pytest.raises(ValueError, match="out of range"):
        he.fit(np.vstack([row(2.0 ** 508.1 / b ** 2), row(1.0)]), np.ones(2))
    for bad in (lib.Activation("erf", 1.0, 0.0, 0.0), lib.Activation("erf", np.inf, 1.0, 0.0),
                lib.Activation("abrelu", np.nan, 1.0), lib.Activation("erf", 1e200, 1.0, 0.0)):
        with pytest.raises(ValueError):
            lib.Handle(depth=2, activation=bad)
    with pytest.raises(ValueError, match="layer"):
        lib.Handle(depth=3, sigma_w=1e150, activation=lib.Activation("erf", 1.0, 1.0, 0.0))
    cfg = lib.NngpConfig()
    lib.load().nngp_default_config(ctypes.byref(cfg))
    out = ctypes.c_void_p()
    bad_kind = lib.NngpActivation(7, 0, 1.0, 1.0, 0.0)
    assert lib.load().nngp_create_with_activation(ctypes.byref(cfg), ctypes.byref(bad_kind), ctypes.byref(out)) == lib.NNGP_EINVAL
    assert b"unknown activation" in lib.load().nngp_last_error(None)
    assert lib.load().nngp_create_with_activation(ctypes.byref(cfg), None, ctypes.byref(out)) == lib.NNGP_OK
    lib.load().nngp_destroy(out)


# (the saturated Erf(b = 1000) is left to the kernel tests: its posterior inherits the kernel's sqrt(b^2 q)
# conditioning per step, times that of K + lambda I)
@pytest.mark.parametrize("name", sorted(set(ACTS) - {"erf_bigb"}))
@pytest.mark.parametrize("get", ["nngp", "ntk"])
@pytest.mark.parametrize("case", ["post", "rag1", "rag65"])     # N x D = 10 x 4, 1 x 1, 65 x 7
def test_posteriors_against_mpmath(lib, mpa, name, get, case):
    p = f"{name}/{case}_{get}"
    depth, sw, sb, reg = mpa[p + "_cfg"]
    h = lib.Handle(depth=int(depth), sigma_w=sw, sigma_b=sb, diag_reg=reg, kernel_type=get, activation=_act(lib, name))
    h.fit(mpa[f"{name}/{case}_x_train"], mpa[f"{name}/{case}_y_train"])
    xt = mpa[f"{name}/{case}_x_test"]
    mean, var = h.predict(xt)
    mc, cov = h.predict_cov(xt)
    tol = 1e-8 if get == "nngp" else 1e-7
    rel = lambda a, b: float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
    assert rel(mean, mpa[p + "_mean"]) <= tol and rel(var, mpa[p + "_var"]) <= tol
    assert rel(cov, mpa[p + "_cov"]) <= tol
    assert np.array_equal(mc, mean) and np.array_equal(np.diag(cov), var) and np.array_equal(cov, cov.T)
    lml = float(mpa[p + "_lml"])
    assert abs(h.log_marginal_likelihood() - lml) <= tol * abs(lml)


def _problem(n, t, d, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, d)), rng.standard_normal(n), rng.standard_normal((t, d))


def _oracle_fit(kind, x, y, depth, act, reg=1e-3, sw=1.0, sb=0.0):
    cls = act_oracle.FitNTK if kind == "ntk" else act_oracle.Fit
    return cls(x, y, depth, sw, sb, reg, activation=act)


# (N = 1 and 65 are held to the mpmath posteriors above)
@pytest.mark.parametrize("name", sorted(set(ACTS) - {"erf_bigb"}))
@pytest.mark.parametrize("n,d", [(257, 1), (257, 33), (1000, 7), (1000, 33)])
def test_ragged_shapes_against_the_oracle(lib, name, n, d):
    x, y, xt = _problem(n, 37, d, n + d)
    for get, depth in (("nngp", 2), ("ntk", 3)):
        if d == 1 and get == "ntk" and ACTS[name][0] == "abrelu":
            # one feature: every pair of rows is parallel or antiparallel, where the ABRelu family's Theta is first-order
            # sensitive to the rounding residue of theta (in any FP64 evaluation, as for ReLU), and the 257-row solve
            # amplifies it past the gate; D = 1 'ntk' is held to the mpmath posterior at N = 1
            continue
        h = lib.Handle(depth=depth, kernel_type=get, activation=_act(lib, name))
        h.fit(x, y)
        mean, cov = h.predict_cov(xt)
        f = _oracle_fit(get, x, y, depth, ACTS[name])
        rm, rc = f.predict_full_cov(xt)
        assert np.max(np.abs(mean - rm[:, 0])) <= 1e-6 * np.max(np.abs(rm)), (get, n, d)
        assert np.max(np.abs(cov - rc)) <= 1e-6 * np.max(np.abs(rc)), (get, n, d)
        assert abs(h.log_marginal_likelihood() - f.log_marginal_likelihood()) <= 1e-6 * abs(f.log_marginal_likelihood())


@pytest.mark.parametrize("name,get", [("leaky", "nngp"), ("erf", "nngp"), ("erf_abc", "ntk")])
def test_parity_gate_at_8192(lib, name, get):
    """The project's 1e-6 parity gate (max relative error of mean and variance against the numpy oracle)."""
    x, y, xt = _problem(8192, 512, 64, 17)
    h = lib.Handle(depth=3, kernel_type=get, activation=_act(lib, name))
    h.fit(x, y)
    mean, var = h.predict(xt)
    rm, rv = _oracle_fit(get, x, y, 3, ACTS[name]).predict(xt)
    assert np.max(np.abs(mean - rm)) / np.max(np.abs(rm)) <= 1e-6
    assert np.max(np.abs(var - rv)) / np.max(np.abs(rv)) <= 1e-6


@pytest.mark.parametrize("get", ["nngp", "ntk"])
@pytest.mark.parametrize("depth", [2, 3])
def test_abrelu_0_1_is_bitwise_the_default_handle(lib, get, depth):
    x, y, xt = _problem(700, 300, 20, depth)
    h0 = lib.Handle(depth=depth, kernel_type=get)
    h1 = lib.Handle(depth=depth, kernel_type=get, activation=lib.Activation("abrelu", 0.0, 1.0))
    assert np.array_equal(h0.kernel(xt, x), h1.kernel(xt, x)) and np.array_equal(h0.kernel(x), h1.kernel(x))
    h0.fit(x, y)
    h1.fit(x, y)
    for a, b in zip(h0.predict(xt) + h0.predict_cov(xt), h1.predict(xt) + h1.predict_cov(xt)):
        assert np.array_equal(a, b)
    assert h0.log_marginal_likelihood() == h1.log_marginal_likelihood()


def test_erf_latency_mode_and_variance_slices(lib, monkeypatch):
    """The same posterior to the tolerances those paths are tested to for ReLU: latency mode 1e-8 relative (rounding),
    7 digit planes 1e-6 of the variance and the mean bitwise."""
    x, y, xt = _problem(1500, 300, 16, 5)
    act = lib.Activation("erf", 1.5, 0.7, 0.2)
    h = lib.Handle(depth=3, activation=act)
    h.fit(x, y)
    mean, var = h.predict(xt)
    hl = lib.Handle(depth=3, activation=act, latency_mode=True)
    hl.fit(x, y)
    ml, vl = hl.predict(xt)
    assert np.max(np.abs(ml - mean)) <= 1e-10 * np.max(np.abs(mean)) and np.max(np.abs(vl - var) / var) <= 1e-8
    hs = lib.Handle(depth=3, activation=act, variance_slices=7)
    hs.fit(x, y)
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")
    ms, vs = hs.predict(xt)
    assert hs.stats()["sliced_macs"] > 0
    assert np.array_equal(ms, mean) and np.max(np.abs(vs - var) / var) <= 1e-6


def test_erf_structure(lib, tmp_path):
    """Covariance diagonal bitwise the variance; packed state, save / load bitwise; incremental append vs refit."""
    x, y, xt = _problem(900, 200, 12, 9)
    act = lib.Activation("erf", 1.5, 0.7, 0.2)
    h = lib.Handle(depth=3, activation=act)
    h.fit(x, y)
    mean, var = h.predict(xt)
    mc, cov = h.predict_cov(xt)
    assert np.array_equal(np.diag(cov), var) and np.array_equal(mc, mean)
    n, d, lam = h.dims()
    flat = np.empty(h.packed_size())
    h.state_pack(0, flat.size, flat)
    h2 = lib.Handle(depth=3, activation=act)
    h2.state_import_begin(n, d)
    h2.state_unpack(0, flat.size, flat)
    h2.state_import_end(lam)
    m2, v2 = h2.predict(xt)
    assert np.array_equal(m2, mean) and np.array_equal(v2, var)
    h.save(tmp_path / "erf_model")
    h3 = lib.Handle.load(tmp_path / "erf_model")
    assert h3.activation == act
    m3, v3 = h3.predict(xt)
    assert np.array_equal(m3, mean) and np.array_equal(v3, var)
    # a model file without an activation is a ReLU model
    z = dict(np.load(tmp_path / "erf_model.npz"))
    for key in ("act_kind", "act_abc"):
        z.pop(key)
    hrelu = lib.Handle(depth=3)
    hrelu.fit(x, y)
    z.update(dict(zip(("x", "l", "alpha"), (lambda s: (s["x"], s["l"], s["alpha"]))(hrelu.get_state()))))
    z["lam"] = hrelu.dims()[2]
    np.savez(tmp_path / "old.npz", **z)
    hold = lib.Handle.load(tmp_path / "old.npz")
    assert hold.activation == lib.RELU and np.array_equal(hold.predict(xt)[0], hrelu.predict(xt)[0])
    # incremental append (fixed lambda) vs a fresh fit of the stacked rows
    xa, ya, _ = _problem(300, 1, 12, 10)
    ha = lib.Handle(depth=3, activation=act, diag_reg_absolute=True)
    ha.fit(x, y)
    ha.append_fit(xa, ya)
    hf = lib.Handle(depth=3, activation=act, diag_reg_absolute=True)
    hf.fit(np.vstack([x, xa]), np.concatenate([y, ya]))
    ma, va = ha.predict(xt)
    mf, vf = hf.predict(xt)
    assert np.max(np.abs(ma - mf)) <= 1e-9 * np.max(np.abs(mf)) and np.max(np.abs(va - vf) / vf) <= 1e-7


def test_erf_two_gpus_bitwise(lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    x, y, xt = _problem(1200, 2000, 24, 11)
    for get in ("nngp", "ntk"):
        act = lib.Activation("erf", 1.0, 1.0, 0.0)
        h1 = lib.Handle(depth=3, kernel_type=get, activation=act)
        hg = lib.Handle(depth=3, kernel_type=get, activation=act, n_gpus=2)
        h1.fit(x, y)
        hg.fit(x, y)
        for a, b in zip(h1.predict(xt), hg.predict(xt)):
            assert np.array_equal(a, b)
