"""GPU: the full posterior covariance (nngp_predict_cov) against exactly known answers, the 50-digit mpmath vectors of
tests/golden/mp_cov.npz and the FP64 oracle, plus its bitwise properties, positive semi-definiteness and errors.

Exact answers reuse the construction of test_gpu_factor_exact.py: depth 1, lambda = 0, X = [L~ | 0].  For queries
x = [u | w] and x' = [u' | w'],  K(x, x') = (u.u' + w.w') / D  and  V V^T = u.u' / D,  so the posterior covariance is
exactly w.w' / D.  Error model: that file's variance bound with K(x*, x*) replaced by sqrt(K(x,x) K(x',x')),
    |C^ - C| <= 4 N eps kappa sqrt(K(x,x) K(x',x'))       ('ntk': kappa^2; at depth 1 Theta = K and M = I).
"""
import ctypes as C
import math

import numpy as np
import pytest

from test_gpu_factor_exact import EPS, W256_N, W512_N, W1024_N, Exact, cond_bound, lower_band

pytestmark = pytest.mark.gpu

import cov_oracle  # noqa: E402
import nngp_oracle as oracle  # noqa: E402

RAGGED_T = [1, 2, 65, 130, 257]


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


@pytest.fixture(scope="module")
def synth():
    from nngp_b200 import synth as s
    return s


@pytest.fixture(scope="module")
def mp_cov(golden_dir):
    z = np.load(golden_dir / "mp_cov.npz")
    cases = {}
    for key in z.files:
        name, field = key.split("/")
        cases.setdefault(name, {})[field] = z[key]
    return cases


# ---------------------------------------------------------------------------------------------- exact answers
def _check_exact(lib, n):
    L = lower_band(n, seed=n + 100)
    kappa = cond_bound(L)
    ex = Exact(L, seed=n)
    xq = ex.queries(max(RAGGED_T), seed=n + 1)
    X = ex.x_train()
    w = xq[:, n:]
    exact = (w @ w.T) / ex.D                             # integers / 2^k: exact
    kss = np.einsum("ij,ij->i", xq, xq) / ex.D
    scale = np.sqrt(np.outer(kss, kss))
    for kind, kpow in (("nngp", 1), ("ntk", 2)):
        h = lib.Handle(depth=1, sigma_w=1.0, sigma_b=0.0, diag_reg=0.0, kernel_type=kind)
        h.fit(X, ex.y)
        for t in RAGGED_T:
            mean, cov = h.predict_cov(xq[:t])
            tol = 4 * n * EPS * kappa ** kpow * scale[:t, :t]
            err = np.abs(cov - exact[:t, :t])
            assert np.all(err <= tol), (f"N={n} {kind} T={t}: entry {np.unravel_index(np.argmax(err / tol), err.shape)} "
                                        f"off by {float(np.max(err / tol)):.2f} of its bound")
            assert np.array_equal(cov, cov.T)
            m_p, v_p = h.predict(xq[:t])
            assert np.array_equal(mean, m_p) and np.array_equal(np.diag(cov), v_p)


@pytest.mark.parametrize("n", [W256_N[-3], W512_N[1]])
def test_exact_covariance_w256_w512(lib, n):
    """W = 256 (N = 257) and W = 512 (N = 4097), 'nngp' and 'ntk', T = 1, 2, 65, 130, 257."""
    _check_exact(lib, n)


def test_exact_covariance_w1024(lib):
    """W = 1024 (N = 24641, look-ahead on), 'nngp' and 'ntk', T = 1, 2, 65, 130, 257."""
    _check_exact(lib, W1024_N)


# ---------------------------------------------------------------------------------------------- mpmath, oracle
def test_against_mpmath_covariances(lib, mp_cov):
    assert len(mp_cov) == 8
    for name, g in mp_cov.items():
        depth, sw, sb, reg, absolute, ntk = g["cfg"]
        h = lib.Handle(depth=int(depth), sigma_w=sw, sigma_b=sb, diag_reg=reg, diag_reg_absolute=bool(absolute),
                       kernel_type="ntk" if ntk else "nngp")
        h.fit(g["x_train"], g["y_train"])
        mean, cov = h.predict_cov(g["x_test"])
        cscale = float(np.max(np.abs(g["cov"])))
        err = float(np.max(np.abs(cov - g["cov"])))
        print(f"\n{name}: max |C - C_mp| = {err:.3e} = {err / cscale:.2e} of max |C_mp|")
        assert np.max(np.abs(mean - g["mean"])) < 1e-8 * np.max(np.abs(g["mean"])), name
        assert err < 1e-8 * cscale, name


@pytest.mark.parametrize("n,t,d,depth,kind", [(1500, 700, 64, 3, "nngp"), (8192, 1024, 128, 2, "nngp"),
                                              (2500, 600, 32, 2, "ntk"), (8192, 520, 64, 3, "ntk")])
def test_against_the_oracle(lib, synth, n, t, d, depth, kind):
    """|C^_ij - C_ij| <= 1e-6 sqrt(K_ii K_jj) (the project's parity gate); the measured maximum is printed."""
    xtr, ytr, xte, _ = synth.make_problem(n, t, d)
    xte[1] = xte[0] * (1 + 1e-9)
    xte[2] = xtr[7]
    h = lib.Handle(depth=depth, kernel_type=kind)
    h.fit(xtr, ytr)
    mean, cov = h.predict_cov(xte)
    ref = (oracle.FitNTK if kind == "ntk" else oracle.Fit)(xtr, ytr, depth)
    rm, rc = cov_oracle.predict_full_cov(ref, xte)
    kss = oracle.final_diag(oracle.layer0_diag(xte), depth)
    rel = float(np.max(np.abs(cov - rc) / np.sqrt(np.outer(kss, kss))))
    print(f"\n{kind} N={n} T={t} depth={depth}: max |dC_ij| / sqrt(K_ii K_jj) = {rel:.3e}")
    assert rel <= 1e-6
    assert np.max(np.abs(mean - rm[:, 0])) <= 1e-6 * np.max(np.abs(rm))


# ---------------------------------------------------------------------------------------------- bitwise properties
@pytest.fixture(scope="module")
def problem(synth):
    return synth.make_problem(1500, 1000, 32)


def test_bitwise_properties_default_config(lib, problem):
    import torch
    xtr, ytr, xte, _ = problem
    x = xte[:700]                                        # >= 4 row tiles: the lower-triangle Gram
    h = lib.Handle()
    h.fit(xtr, ytr)
    h.stats_reset()
    mean, cov = h.predict_cov(x)
    st = h.stats()
    assert st["queries"] == 700 and st["pred_var_ms"] > 0 and st["pred_gram_ms"] > 0
    assert np.array_equal(cov, cov.T)
    m_p, v_p = h.predict(x)
    assert np.array_equal(mean, m_p) and np.array_equal(np.diag(cov), v_p)
    m2, c2 = h.predict_cov(x)                            # two calls
    assert np.array_equal(mean, m2) and np.array_equal(cov, c2)
    perm = np.random.default_rng(5).permutation(700)     # a permuted batch
    mp_, cp = h.predict_cov(x[perm])
    assert np.array_equal(cp, cov[np.ix_(perm, perm)]) and np.array_equal(mp_, mean[perm])
    for sub in (np.sort(np.random.default_rng(6).choice(700, 300, replace=False)), np.arange(600, 700)):
        ms, cs = h.predict_cov(x[sub])                   # a sub-batch (300 rows: the full-square Gram)
        assert np.array_equal(cs, cov[np.ix_(sub, sub)]) and np.array_equal(ms, mean[sub])
    xd = torch.from_numpy(x).cuda()                      # device pointers
    md = torch.empty(700, dtype=torch.float64, device="cuda")
    cd = torch.empty((700, 700), dtype=torch.float64, device="cuda")
    h.predict_cov(xd, mean_out=md, cov_out=cd)
    assert np.array_equal(md.cpu().numpy(), mean) and np.array_equal(cd.cpu().numpy(), cov)


@pytest.mark.parametrize("cfg,t", [({"latency_mode": True}, 700), ({"variance_slices": 7}, 1000),
                                   ({"kernel_type": "ntk"}, 700), ({"kernel_type": "ntk"}, 130)])
def test_diagonal_is_the_variance_of_every_path(lib, problem, cfg, t):
    """latency mode (explicit inverse, 700 rows), digit planes (1000 rows: past the 767-row switch) and 'ntk': the
    diagonal is nngp_predict's variance and the mean its mean, bit for bit; the matrix is bitwise symmetric."""
    xtr, ytr, xte, _ = problem
    h = lib.Handle(**cfg)
    h.fit(xtr, ytr)
    mean, cov = h.predict_cov(xte[:t])
    m_p, v_p = h.predict(xte[:t])
    assert np.array_equal(cov, cov.T)
    assert np.array_equal(mean, m_p) and np.array_equal(np.diag(cov), v_p)
    if cfg.get("variance_slices"):
        assert h.stats()["sliced_macs"] > 0


def test_two_gpus_give_the_single_gpu_bits(lib, problem):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    xtr, ytr, xte, _ = problem
    h1, h2 = lib.Handle(), lib.Handle(n_gpus=2)
    h1.fit(xtr, ytr)
    h2.fit(xtr, ytr)
    m1, c1 = h1.predict_cov(xte[:700])
    m2, c2 = h2.predict_cov(xte[:700])
    assert np.array_equal(m1, m2) and np.array_equal(c1, c2)
    _, v2 = h2.predict(xte[:700])
    assert np.array_equal(np.diag(c2), v2)


# ---------------------------------------------------------------------------------------------- PSD
PSD_C = 16     # fixed before the first run


def test_positive_semidefinite_at_c2_size(lib, synth):
    """N = 8192, D = 128, depth 2 (config C2), 1024 test rows: lambda_min(C) >= -c N eps max K_ii, c = 16."""
    xtr, ytr, xte, _ = synth.make_problem(8192, 1024, 128)
    h = lib.Handle()
    h.fit(xtr, ytr)
    _, cov = h.predict_cov(xte)
    kmax = float(np.max(oracle.final_diag(oracle.layer0_diag(xte), 2)))
    lmin = float(np.linalg.eigvalsh(cov)[0])
    print(f"\nlambda_min = {lmin:.3e}, bound {-PSD_C * 8192 * EPS * kmax:.3e}")
    assert lmin >= -PSD_C * 8192 * EPS * kmax


# ---------------------------------------------------------------------------------------------- errors
def test_errors(lib, synth):
    from nngp_b200._lib import NngpError
    xtr, ytr, xte, _ = synth.make_problem(200, 300, 16)
    T = 50
    mean, cov = np.empty(T), np.empty((T, T))
    xt = np.ascontiguousarray(xte[:T])
    h = lib.Handle()
    rc = h._lib.nngp_predict_cov(h._h, C.c_void_p(xt.ctypes.data), T, C.c_void_p(mean.ctypes.data),
                                 C.c_void_p(cov.ctypes.data))
    assert rc == lib.NNGP_ESTATE                               # before a fit
    h.fit(xtr, ytr)
    bad = xt.copy()
    bad[3, 2] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        h.predict_cov(bad)
    with pytest.raises(ValueError):
        h.predict_cov(xt, cov_out=np.empty((T, T + 1)))
    # an imported 'ntk' state without M
    hn = lib.Handle(kernel_type="ntk")
    hn.fit(xtr, ytr)
    st = hn.get_state(m=False)
    imp = lib.Handle(kernel_type="ntk")
    imp.set_state(st["x"], st["l"], st["alpha"], st["lambda"])
    with pytest.raises(NngpError) as e:
        imp.predict_cov(xt)
    assert e.value.code == lib.NNGP_ESTATE
    # T beyond one block: 100 rows of V (33 of V, U and V M) fit in 100 rows x 208 columns x 8 bytes
    per_row = 208 * 8
    for kind, cap in (("nngp", 100), ("ntk", 33)):
        hs = lib.Handle(max_block_bytes=100 * per_row, kernel_type=kind)
        hs.fit(xtr, ytr)
        m_ok, c_ok = hs.predict_cov(xte[:cap])
        assert np.array_equal(np.diag(c_ok), hs.predict(xte[:cap])[1])
        with pytest.raises(ValueError, match=rf"T <= {cap}\b"):
            hs.predict_cov(xte[:cap + 1])
