"""Host-only checks of the exact-answer generator of tests/test_gpu_factor_exact.py: every quantity it calls exact is
an integer below 2^53 (or such an integer over a power of two), its closed-form answers agree with dense linear
algebra, its condition bound holds, and its pivot construction fails exactly where LAPACK says.  No GPU needed."""
import math

import numpy as np
import pytest
import scipy.linalg as sla

import test_gpu_factor_exact as fx

LIMIT = 2.0 ** 53


def _int64(L):
    return L.astype(np.int64)


@pytest.mark.parametrize("n", [1, 5, 65, 513, 4097, 8193, fx.W1024_N])
def test_family_a_is_integer_and_exact(n):
    L = fx.lower_band(n, seed=n + 100)
    assert np.array_equal(L.data, np.round(L.data))
    assert (L.tocoo().row >= L.tocoo().col).all()                  # lower triangular
    assert (L.diagonal() == 16.0).all()
    ex = fx.Exact(L, seed=n)
    xq = ex.queries(64, seed=n + 1)
    rep = fx.exactness_report(L, ex, xq)
    assert max(rep.values()) < LIMIT, rep
    Li = _int64(L)
    ai = ex.a.astype(np.int64)
    num = Li @ (Li.T @ ai)                                          # y * D in exact integer arithmetic
    assert np.array_equal(ex.y * ex.D, num.astype(np.float64)) and np.max(np.abs(num)) < LIMIT
    assert ex.D & (ex.D - 1) == 0 and ex.D >= n + fx.PAD
    m, v, kss, _ = ex.answers(xq)
    ui = xq[:, :n].astype(np.int64)
    assert np.array_equal(m * ex.D, (ui @ (Li.T @ ai)).astype(np.float64))
    assert np.array_equal(kss * ex.D, np.einsum("ij,ij->i", xq, xq))
    assert (v[0::2] == 0.0).all() and (v[1::2] > 0.0).all()         # w = 0 rows: variance exactly 0


@pytest.mark.parametrize("n", [3, 64, 129, 300, 600])
def test_closed_forms_match_dense_linear_algebra(n):
    L = fx.lower_band(n, seed=n + 100)
    kappa = fx.cond_bound(L)
    Ld = L.toarray()
    assert np.linalg.cond(Ld) <= kappa * (1 + 1e-12)
    A = fx.gram_dense(L)
    assert np.array_equal(A, (_int64(L) @ _int64(L).T).toarray().astype(np.float64))
    assert np.max(np.abs(np.linalg.cholesky(A) - Ld)) <= 2 * n * fx.EPS * kappa * 16.0
    ex = fx.Exact(L, seed=n)
    X = ex.x_train()
    K = X @ X.T / ex.D
    assert np.array_equal(K, A / ex.D)
    alpha = sla.cho_solve(sla.cho_factor(K, lower=True), ex.y)
    assert np.max(np.abs(alpha - ex.a)) <= 4 * n * fx.EPS * kappa ** 2 * 3
    xq = ex.queries(20, seed=1)
    ks = xq @ X.T / ex.D
    V = sla.solve_triangular(Ld / math.sqrt(ex.D), ks.T, lower=True).T
    m, v, kss, _ = ex.answers(xq)
    assert np.allclose(ks @ ex.a, m, rtol=1e-12, atol=1e-12)
    assert np.allclose(kss - np.einsum("ij,ij->i", V, V), v, rtol=1e-9, atol=1e-9 * kss.max())
    Lc = sla.cholesky(K, lower=True)
    lml = -0.5 * ex.y @ alpha - np.sum(np.log(np.diag(Lc))) - 0.5 * n * math.log(2 * math.pi)
    assert abs(ex.lml()[0] - lml) <= 1e-9 * abs(lml)
    for rows in (1, n // 2 + 1):                                    # the prefix problems of the append test
        Kp = K[:rows, :rows]
        ap = sla.cho_solve(sla.cho_factor(Kp, lower=True), ex.y[:rows])
        mp, vp, _, _ = ex.answers(xq, rows)
        kp = xq @ X[:rows].T / ex.D
        Vp = sla.solve_triangular(Ld[:rows, :rows] / math.sqrt(ex.D), kp.T, lower=True).T
        assert np.allclose(kp @ ap, mp, rtol=1e-10, atol=1e-10)
        assert np.allclose(kss - np.einsum("ij,ij->i", Vp, Vp), vp, rtol=1e-9, atol=1e-9 * kss.max())
        assert abs(ex.lml(rows)[0] - (-0.5 * ex.y[:rows] @ ap - np.sum(np.log(np.diag(Ld[:rows, :rows]) / math.sqrt(ex.D)))
                                      - 0.5 * rows * math.log(2 * math.pi))) <= 1e-9 * max(1.0, abs(ex.lml(rows)[0]))


@pytest.mark.parametrize("where", [np.arange(0, 64), np.arange(1024, fx.ILL_N), "spread"])
def test_chain_families(where):
    n = fx.ILL_N
    idx = np.sort(np.random.default_rng(3).choice(n, 64, replace=False)) if isinstance(where, str) else where
    L = fx.with_chain(fx.lower_band(n, seed=7), idx)
    assert np.array_equal(L.data, np.round(L.data)) and (L.diagonal() > 0).all()
    coo = L.tocoo()
    assert (coo.row >= coo.col).all()
    assert max(fx.exactness_report(L).values()) < LIMIT
    chain = L[idx][:, idx].toarray()
    assert np.array_equal(chain, np.diag(np.full(idx.size, 4.0)) + np.diag(np.full(idx.size - 1, -5.0), -1))
    assert np.linalg.cond(chain) > 1e5


@pytest.mark.parametrize("n", sorted(fx.PIVOTS))
def test_pivot_construction_fails_where_lapack_does(n):
    L = fx.lower_band(n, seed=n + 5)
    A = fx.gram_dense(L)
    for p in fx.PIVOTS[n]:
        a = A.copy()
        a[p, p] -= L[p, p] ** 2 + 1.0
        assert sla.lapack.dpotrf(a, lower=1)[1] == p + 1
    ex = fx.Exact(L, seed=1)
    X = ex.x_train()
    X[fx.PIVOTS[n][3]] = 0.0                                       # zero training row -> pivot exactly 0
    K = X @ X.T / ex.D
    assert sla.lapack.dpotrf(K, lower=1)[1] == fx.PIVOTS[n][3] + 1
