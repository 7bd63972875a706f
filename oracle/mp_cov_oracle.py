"""CPU ORACLE (high precision) -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED AGAINST THE REFERENCE.

The full posterior covariance in 50-digit mpmath, on top of ``mp_oracle.py``'s fits (same algorithm, see its header).
Used once, by ``tests/golden/make_mp_cov_golden.py``, to produce ``tests/golden/mp_cov.npz``.  Small cases only.
"""
from __future__ import annotations

import mpmath as mp

import mp_oracle as mpo


def fit_predict_cov(x, y, xt, depth, sigma_w, sigma_b, diag_reg, absolute=False):
    """mp_oracle.fit_predict with the full posterior covariance: cov[i][j] = K(x_i, x_j) - v_i . v_j, C v_i = k_i."""
    r = mpo.fit_predict(x, y, xt, depth, sigma_w, sigma_b, diag_reg, absolute)
    c = mp.cholesky(r["K"])
    ks = r["Ks"]
    ktt = mpo.kernel(xt, None, depth, sigma_w, sigma_b)
    vs = [mp.lu_solve(c, ks[i, :].T) for i in range(len(xt))]
    r["Ktt"] = ktt
    r["cov"] = [[ktt[i][j] - mp.fsum(a * b for a, b in zip(vs[i], vs[j])) for j in range(len(xt))]
                for i in range(len(xt))]
    return r


def fit_predict_ntk_cov(x, y, xt, depth, sigma_w, sigma_b, diag_reg, absolute=False):
    """mp_oracle.fit_predict_ntk with the full posterior covariance (SURVEY.md Appendix A.5):
    cov[i][j] = K(x_i, x_j) + w_i^T K_dd w_j - w_i . k_j - w_j . k_i,  A w_i = theta_i."""
    r = mpo.fit_predict_ntk(x, y, xt, depth, sigma_w, sigma_b, diag_reg, absolute)
    n = len(x)
    a = r["Theta"].copy()
    for i in range(n):
        a[i, i] += r["lam"]
    kdd = mp.matrix(mpo.kernel(x, None, depth, sigma_w, sigma_b))
    ks = mp.matrix(mpo.kernel(xt, x, depth, sigma_w, sigma_b))
    ths = r["Thetas"]
    ktt = mpo.kernel(xt, None, depth, sigma_w, sigma_b)
    t = len(xt)
    ws = [mp.cholesky_solve(a, ths[i, :].T) for i in range(t)]
    kw = [kdd * w for w in ws]
    r["Ktt"] = ktt
    r["cov"] = [[ktt[i][j] + mp.fsum(ws[i][k] * kw[j][k] for k in range(n))
                 - mp.fsum(ws[i][k] * ks[j, k] for k in range(n)) - mp.fsum(ws[j][k] * ks[i, k] for k in range(n))
                 for j in range(t)] for i in range(t)]
    return r
