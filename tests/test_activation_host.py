"""CPU: the ABRelu family and Erf on the host side -- the numpy oracle against the 50-digit vectors of
tests/golden/mp_act.npz and against exactly known kernels, the stax layers and the KernelSpec they build, the shapes
predict_fn returns for each activation (through an oracle-backed fake engine), and the C-ABI struct layout."""
import ctypes

import numpy as np
import pytest

import act_oracle
import nngp_oracle as oracle
from nngp_b200 import _lib, predict, runtime, stax, synth

ACTS = {"leaky": stax.LeakyRelu(0.1), "abs": stax.Abs(), "abrelu": stax.ABRelu(-0.3, 1.2), "erf": stax.Erf(),
        "erf_abc": stax.Erf(1.5, 0.7, 0.2), "erf_bigb": stax.Erf(b=1e3)}
SWEEP_CFG = {2: (1.0, 0.0), 3: (1.3, 0.1)}


def _act(layer):
    return layer.params["activation"]


@pytest.fixture(scope="module")
def mpa(golden_dir):
    return dict(np.load(golden_dir / "mp_act.npz"))


@pytest.mark.parametrize("name", sorted(ACTS))
def test_oracle_kernels_against_mpmath(mpa, name):
    """The angle sweep and the magnitude rows: |K - K_mp| <= 1e-13 sqrt(K_mp(x,x) K_mp(y,y)) wherever q q' is a normal
    double, Erf times act_oracle.erf_amplification (1 except on near-parallel pairs and the diagonal of saturated
    rows); Theta the same at 1e-12 for Erf, and 1e-7 for the ABRelu family (first-order sensitive to theta through
    kdot on near-parallel pairs, as for ReLU)."""
    act = _act(ACTS[name])
    for tag in ("sweep", "mag"):
        x = mpa[f"{name}/{tag}_x"]
        for depth, (sw, sb) in SWEEP_CFG.items():
            kmp, tmp = mpa[f"{name}/{tag}_nngp_d{depth}"], mpa[f"{name}/{tag}_ntk_d{depth}"]
            k, t = act_oracle.kernel_fn(x, None, depth, sw, sb, get="both", activation=act)
            assert np.all(np.isfinite(k)) and np.all(np.isfinite(t))
            q = oracle.layer0_diag(x, sw, sb)
            qq = np.outer(q, q)
            f, g = act_oracle.erf_amplification(x, depth, sw, sb, act)
            erf = act.kind == "erf"
            ok = (qq <= 2.0 ** 1000) & ((qq >= 2.0 ** -1000) | erf)
            for got, ref, bar in ((k, kmp, 1e-13 * f), (t, tmp, 1e-12 * g if erf else np.full(qq.shape, 1e-7))):
                d = np.abs(np.diag(ref))
                scale = np.sqrt(np.outer(d, d))
                m = ok & (scale > 0)
                assert np.all(np.abs(got - ref)[m] / scale[m] <= bar[m]), (tag, depth)
            dd = act_oracle.final_diag(q, depth, sw, sb, act)
            d = np.diag(kmp)
            assert np.max(np.abs(dd - d)[d > 0] / d[d > 0]) <= 1e-13


@pytest.mark.parametrize("name", sorted(ACTS))
@pytest.mark.parametrize("get", ["nngp", "ntk"])
@pytest.mark.parametrize("case", ["post", "rag1", "rag65"])
def test_oracle_posteriors_against_mpmath(mpa, name, get, case):
    if case != "post" and name == "erf_bigb":
        pytest.skip("the ragged posteriors cover the activations of the issue list")
    act = _act(ACTS[name])
    p = f"{name}/{case}_{get}"
    depth, sw, sb, reg = mpa[p + "_cfg"]
    cls = act_oracle.FitNTK if get == "ntk" else act_oracle.Fit
    f = cls(mpa[f"{name}/{case}_x_train"], mpa[f"{name}/{case}_y_train"], int(depth), sw, sb, reg, activation=act)
    xt = mpa[f"{name}/{case}_x_test"]
    mean, cov = f.predict_full_cov(xt)
    m2, var = f.predict(xt)
    # ('ntk' with the ABRelu family: Theta(x, x) carries the theta rounding residue of the diagonal through kdot, as for
    # ReLU, whose NTK posteriors the existing tests hold to 1e-7)
    tol = 1e-7 if get == "ntk" and act.kind == "abrelu" else 1e-9
    assert np.max(np.abs(mean[:, 0] - mpa[p + "_mean"])) <= tol * np.max(np.abs(mpa[p + "_mean"]))
    assert np.max(np.abs(cov - mpa[p + "_cov"])) <= tol * np.max(np.abs(mpa[p + "_cov"]))
    assert np.max(np.abs(var - mpa[p + "_var"])) <= tol * np.max(np.abs(mpa[p + "_var"]))
    assert abs(f.log_marginal_likelihood() - float(mpa[p + "_lml"])) <= tol * abs(float(mpa[p + "_lml"]))


def _rows(n=40, d=6, seed=3):
    return np.random.default_rng(seed).standard_normal((n, d))


@pytest.mark.parametrize("a", [0.7, -1.3, 2.0])
@pytest.mark.parametrize("depth", [2, 3])
def test_abrelu_with_a_equal_b_is_the_linear_kernel(a, depth):
    """ABRelu(a, a) is x -> a x: every step multiplies k (and q) by a^2 -- Dense layers compose linearly."""
    x = _rows()
    sw, sb = 1.2, 0.3
    k, t = act_oracle.kernel_fn(x, None, depth, sw, sb, get="both", activation=("abrelu", a, a))
    lin = sw ** 2 * (x @ x.T) / x.shape[1] + sb ** 2
    ntk = lin.copy()
    for _ in range(1, depth):
        lin = sw ** 2 * a * a * lin + sb ** 2
        ntk = lin + sw ** 2 * a * a * ntk
    for got, want in ((k, lin), (t, ntk)):
        d = np.diag(want)
        assert np.max(np.abs(got - want) / np.sqrt(np.outer(d, d))) <= 1e-13
    k1 = act_oracle.kernel_fn(x, None, depth, sw, sb, activation=_act(stax.LeakyRelu(1.0)))   # LeakyRelu(1) = identity
    assert np.allclose(k1, act_oracle.kernel_fn(x, None, depth, sw, sb, activation=("abrelu", 1.0, 1.0)), rtol=1e-13)


def test_abs_kernel_closed_form():
    """Abs: E[|u| |v|] = (2/pi) (s + (pi/2 - theta) k)."""
    x = _rows()
    q = oracle.layer0_diag(x)
    k0 = (x @ x.T) / x.shape[1]
    s = np.sqrt(np.maximum(np.outer(q, q) - k0 * k0, 0.0))
    theta = np.arctan2(s, k0)
    want = 2 / np.pi * (s + (np.pi / 2 - theta) * k0)
    got = act_oracle.kernel_fn(x, None, 2, activation=_act(stax.Abs()))
    assert np.allclose(got, want, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("depth", [2, 3])
def test_abrelu_0_1_is_bitwise_todays_relu(depth):
    x, xt = _rows(50), _rows(9, seed=4)
    for get in ("nngp", "ntk"):
        want = oracle.kernel_fn(xt, x, depth, 1.1, 0.2, get=get)
        got = act_oracle.kernel_fn(xt, x, depth, 1.1, 0.2, get=get, activation=("abrelu", 0.0, 1.0))
        assert np.array_equal(got, want)
    assert np.array_equal(act_oracle.final_diag(oracle.layer0_diag(xt), depth, 1.1, 0.2, ("abrelu", 0.0, 1.0)),
                          oracle.final_diag(oracle.layer0_diag(xt), depth, 1.1, 0.2))


def test_serial_builds_the_kernel_spec():
    _, _, kf = stax.serial(stax.Dense(512), stax.Relu(), stax.Dense(1))
    assert kf.spec == stax.KernelSpec(2, 1.0, 0.0) and kf.spec.activation == _lib.RELU
    _, _, kf = stax.serial(stax.Dense(8, W_std=1.5, b_std=0.1), stax.Erf(), stax.Dense(8, 1.5, 0.1), stax.Erf(),
                           stax.Dense(1, 1.5, 0.1))
    assert kf.spec == stax.KernelSpec(3, 1.5, 0.1, _lib.Activation("erf", 1.0, 1.0, 0.0))
    _, _, kf = stax.serial(stax.Dense(8), stax.LeakyRelu(0.2), stax.Dense(1, W_std=2.0))
    assert kf.spec == stax.KernelSpec(2, (1.0, 2.0), (0.0, 0.0), _lib.Activation("abrelu", 0.2, 1.0))
    assert _act(stax.Abs()) == _lib.Activation("abrelu", -1.0, 1.0)
    assert _act(stax.Erf(1.5, 0.7, 0.2)) == _lib.Activation("erf", 1.5, 0.7, 0.2)


def test_serial_rejects_mixed_activations_and_other_layers():
    with pytest.raises(NotImplementedError, match="one activation"):
        stax.serial(stax.Dense(8), stax.Relu(), stax.Dense(8), stax.Erf(), stax.Dense(1))
    with pytest.raises(NotImplementedError, match="one activation"):
        stax.serial(stax.Dense(8), stax.Relu(), stax.Dense(8), stax.ABRelu(0, 1), stax.Dense(1))
    with pytest.raises(NotImplementedError):
        stax.Gelu()
    with pytest.raises(NotImplementedError):
        stax.serial(stax.Dense(8), stax.Erf(), stax.Erf(), stax.Dense(1))


class ActFakeHandle:
    """Oracle-backed stand-in for the C-ABI handle (runtime.new_handle is replaced by it)."""

    def __init__(self, spec, diag_reg, kernel_type):
        self.spec, self.diag_reg, self.kt = spec, diag_reg, kernel_type

    def fit(self, x, y):
        cls = act_oracle.FitNTK if self.kt == "ntk" else act_oracle.Fit
        s = self.spec
        self.fit_ = cls(x, y, s.depth, s.sigma_w, s.sigma_b, self.diag_reg, activation=s.activation)

    def predict(self, x, want_var=True):
        return self.fit_.predict(x, want_var)

    def predict_cov(self, x):
        mean, cov = self.fit_.predict_full_cov(x)
        return mean[:, 0], cov


@pytest.mark.parametrize("name", sorted(ACTS))
def test_predict_fn_shapes_for_each_activation(monkeypatch, name):
    monkeypatch.setattr(runtime, "new_handle", lambda spec, diag_reg=0.0, diag_reg_absolute=False, kernel_type="nngp":
                        ActFakeHandle(spec, diag_reg, kernel_type))
    x, y, xt, _ = synth.make_problem(30, 7, 6)
    _, _, kf = stax.serial(stax.Dense(64), ACTS[name], stax.Dense(64), ACTS[name], stax.Dense(1))
    pf = predict.gradient_descent_mse_ensemble(kf, x, y[:, None], diag_reg=1e-3)
    for get in ("nngp", "ntk"):
        mean, lazy = pf(x_test=xt, get=get, compute_cov=True)
        m2, cov = pf.full_covariance(xt, get=get)
        assert mean.shape == (7, 1) and m2.shape == (7, 1) and cov.shape == (7, 7)
        assert np.allclose(np.diag(cov), np.diag(lazy), rtol=1e-10) and np.all(np.diag(cov) > 0)


def test_activation_struct_layout():
    """nngp_activation: int32 kind, int32 reserved, double a, b, c (32 bytes)."""
    S = _lib.NngpActivation
    assert ctypes.sizeof(S) == 32
    assert (S.kind.offset, S.reserved.offset, S.a.offset, S.b.offset, S.c.offset) == (0, 4, 8, 16, 24)
    assert _lib.ACT_KINDS == {"relu": 0, "abrelu": 1, "erf": 2}
    s = _lib.Activation("erf", 1.5, 0.7, 0.2).as_struct()
    assert (s.kind, s.a, s.b, s.c) == (2, 1.5, 0.7, 0.2)
    with pytest.raises(ValueError):
        _lib.Activation("gelu").as_struct()
