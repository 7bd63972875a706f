"""CPU: the full posterior covariance on the host side -- the FP64 oracle's full covariances (symmetric, diagonal = the
posterior variance, agreeing with the 50-digit mpmath vectors of tests/golden/mp_cov.npz) and the shapes
predict_fn.full_covariance returns, through an oracle-backed fake engine."""
import numpy as np
import pytest

import cov_oracle
import nngp_oracle as oracle
from nngp_b200 import predict, runtime, stax, synth


@pytest.fixture(scope="module")
def mp_cov(golden_dir):
    z = np.load(golden_dir / "mp_cov.npz")
    cases = {}
    for key in z.files:
        name, field = key.split("/")
        cases.setdefault(name, {})[field] = z[key]
    return cases


def _fit(kind, x, y, depth=2, sw=1.0, sb=0.0, reg=1e-3, absolute=False):
    cls = oracle.FitNTK if kind == "ntk" else oracle.Fit
    return cls(x, y, depth, sw, sb, reg, absolute)


@pytest.mark.parametrize("kind", ["nngp", "ntk"])
@pytest.mark.parametrize("depth", [1, 2, 3])
def test_oracle_full_covariance_is_symmetric_and_its_diagonal_is_the_variance(kind, depth):
    xtr, ytr, xte, _ = synth.make_problem(300, 60, 16)
    xte[1] = xte[0] * (1 + 1e-9)                 # near-duplicate rows
    xte[2] = xtr[5]                              # a training row
    f = _fit(kind, xtr, ytr, depth)
    mean_c, cov = cov_oracle.predict_full_cov(f, xte)
    mean, var = f.predict(xte)
    assert mean_c.shape == (60, 1) and cov.shape == (60, 60)
    assert np.array_equal(mean_c[:, 0], mean) or np.max(np.abs(mean_c[:, 0] - mean)) <= 1e-12 * np.max(np.abs(mean))
    # relative to the prior scale sqrt(K_ii K_jj): the posterior entries are differences of prior-sized terms
    kss = oracle.final_diag(oracle.layer0_diag(xte), depth)
    scale = np.sqrt(np.outer(kss, kss))
    assert np.max(np.abs(cov - cov.T) / scale) <= 1e-12
    assert np.max(np.abs(np.diag(cov) - var) / kss) <= 1e-12


def test_oracle_agrees_with_the_mpmath_covariances(mp_cov):
    assert len(mp_cov) == 8
    for name, g in mp_cov.items():
        depth, sw, sb, reg, absolute, ntk = g["cfg"]
        f = _fit("ntk" if ntk else "nngp", g["x_train"], g["y_train"], int(depth), sw, sb, reg, bool(absolute))
        mean, cov = cov_oracle.predict_full_cov(f, g["x_test"])
        scale = float(np.max(np.abs(g["cov"])))
        assert np.max(np.abs(mean[:, 0] - g["mean"])) <= 1e-9 * np.max(np.abs(g["mean"])), name
        err = float(np.max(np.abs(cov - g["cov"])))
        assert err <= 1e-9 * scale, (name, err / scale)
        assert np.array_equal(g["cov"], g["cov"].T), name


class CovFakeHandle:
    """Oracle-backed stand-in for the C-ABI handle (runtime.new_handle is replaced by it)."""
    fits = 0

    def __init__(self, spec, diag_reg, absolute, kernel_type="nngp"):
        self.spec, self.diag_reg, self.absolute, self.kt = spec, diag_reg, absolute, kernel_type

    def fit(self, x, y):
        CovFakeHandle.fits += 1
        self.fit_ = _fit(self.kt, x, y, self.spec.depth, self.spec.sigma_w, self.spec.sigma_b, self.diag_reg,
                         self.absolute)

    def predict(self, x, want_var=True):
        return self.fit_.predict(x, want_var)

    def predict_cov(self, x):                    # Handle.predict_cov: mean [T], cov [T, T]
        mean, cov = cov_oracle.predict_full_cov(self.fit_, x)
        return mean[:, 0], cov


@pytest.fixture()
def cov_fake_engine(monkeypatch):
    CovFakeHandle.fits = 0
    monkeypatch.setattr(runtime, "new_handle",
                        lambda spec, diag_reg=0.0, diag_reg_absolute=False, kernel_type="nngp": CovFakeHandle(
                            spec, diag_reg, diag_reg_absolute, kernel_type))
    return CovFakeHandle


def test_full_covariance_is_shaped_like_neural_tangents(cov_fake_engine):
    rng = np.random.default_rng(4)
    x, y, xt = rng.uniform(0, 10, (30, 6)), rng.uniform(0, 8, (30, 1)), rng.uniform(0, 10, (7, 6))
    _, _, kernel_fn = stax.serial(stax.Dense(512), stax.Relu(), stax.Dense(1))
    predict_fn = predict.gradient_descent_mse_ensemble(kernel_fn, x, y, diag_reg=1e-3)
    assert cov_fake_engine.fits == 0
    mean, cov = predict_fn.full_covariance(xt, get="nngp")
    assert cov_fake_engine.fits == 1
    assert mean.shape == (7, 1) and cov.shape == (7, 7) and isinstance(cov, np.ndarray)
    m2, lazy = predict_fn(x_test=xt, get="nngp", compute_cov=True)
    assert cov_fake_engine.fits == 1                               # the same cached fit as predict_fn
    assert np.allclose(np.diag(cov), np.diag(lazy), rtol=1e-12) and np.allclose(mean, m2, rtol=1e-12)
    with pytest.raises(NotImplementedError, match="full_covariance"):
        np.asarray(lazy)                                           # the lazy object still refuses, and says where to go
    mt, ct = predict_fn.full_covariance()                          # x_test=None: the training inputs
    assert mt.shape == (30, 1) and ct.shape == (30, 30)
    mn, cn = predict_fn.full_covariance(xt, get="ntk")
    assert cov_fake_engine.fits == 2 and mn.shape == (7, 1) and cn.shape == (7, 7)
    rn = oracle.FitNTK(x, y)
    assert np.allclose(np.diag(cn), rn.predict(xt)[1], rtol=1e-10)
    m1, c1 = predict.gradient_descent_mse_ensemble(kernel_fn, x, y.ravel(), diag_reg=1e-3).full_covariance(xt)
    assert m1.shape == (7,) and c1.shape == (7, 7)
    with pytest.raises(NotImplementedError):
        predict_fn.full_covariance(xt, get=("nngp", "ntk"))
