"""CPU ORACLE (high precision) -- TEST INFRASTRUCTURE ONLY.

50-digit mpmath restatement of ``act_oracle.py`` (the ABRelu family and Erf; see its header for the step formulas):
the kernels, the 'nngp' and 'ntk' posteriors with their full covariance, and the log marginal likelihood.  It also
holds the independent check of those formulas, ``expectations_by_quadrature``: E[phi(u) phi(v)], E[phi'(u) phi'(v)]
and E[phi(u)^2] as integrals over the bivariate normal, with no closed form.  Used once, by
``tests/golden/make_mp_act_golden.py``, to produce ``tests/golden/mp_act.npz``.  Small cases only.

A module of its own rather than an ``activation=`` keyword on ``mp_oracle.kernel`` / ``fit_predict(_ntk)`` for the
reason ``act_oracle.py`` gives: ``mp_oracle.py`` and the golden vectors made with it stay exactly as they are.
"""
from __future__ import annotations

import mpmath as mp

import mp_oracle as mpo

mp.mp.dps = 50


def _mpf_act(act):
    kind, a, b, c = act
    return kind, mp.mpf(a), mp.mpf(b), mp.mpf(c)


def step(k, ntk, qa, qb, act):
    """(E[phi(u) phi(v)], ntk * kdot) for the pre-activation covariance [[qa, k], [k, qb]]."""
    kind, a, b, c = act
    s2 = qa * qb - k * k
    s = mp.sqrt(s2) if s2 > 0 else mp.mpf(0)
    if kind == "abrelu":
        theta = mp.pi / 2 if (s == 0 and k == 0) else mp.atan2(s, k)
        kdot = (a * a + b * b) / 2 - (a - b) ** 2 * theta / (2 * mp.pi)
        return (a - b) ** 2 * s / (2 * mp.pi) + kdot * k, ntk * kdot
    b2 = b * b
    p = 1 + 2 * b2 * (qa + qb) + 4 * b2 * b2 * s2 if s2 > 0 else 1 + 2 * b2 * (qa + qb)   # (1+2Q1)(1+2Q2) - 4K^2
    e = a * a * 2 / mp.pi * mp.asin(2 * b2 * k / mp.sqrt((1 + 2 * b2 * qa) * (1 + 2 * b2 * qb))) + c * c
    return e, ntk * (a * a * b2 * 4 / mp.pi / mp.sqrt(p))


def diag_expect(q, act):
    """E[phi(u)^2] at variance q."""
    kind, a, b, c = act
    if kind == "abrelu":
        return (a * a + b * b) / 2 * q
    big_q = b * b * q
    return a * a * 2 / mp.pi * mp.asin(2 * big_q / (1 + 2 * big_q)) + c * c


def kernel(x1, x2, depth, sigma_w, sigma_b, act, get="nngp"):
    act = _mpf_act(act)
    x1 = [[mp.mpf(float(v)) for v in r] for r in x1]
    x2 = x1 if x2 is None else [[mp.mpf(float(v)) for v in r] for r in x2]
    lay = mpo._layers(depth, sigma_w, sigma_b)
    d = len(x1[0])
    q1, q2 = mpo._diag0(x1, *lay[0]), mpo._diag0(x2, *lay[0])
    out = []
    for i, u in enumerate(x1):
        row = []
        for j, v in enumerate(x2):
            sw2, sb2 = lay[0]
            k = sw2 * (mp.fsum(p * q for p, q in zip(u, v)) / d) + sb2
            ntk = k
            qa, qb = q1[i], q2[j]
            for layer in range(1, depth):
                sw2, sb2 = lay[layer]
                e, nk = step(k, ntk, qa, qb, act)
                k = sw2 * e + sb2
                ntk = k + sw2 * nk
                qa = sw2 * diag_expect(qa, act) + sb2
                qb = sw2 * diag_expect(qb, act) + sb2
            row.append(ntk if get == "ntk" else k)
        out.append(row)
    return out


def fit_predict(x, y, xt, depth, sigma_w, sigma_b, diag_reg, act, ntk=False):
    """mean, var (diagonal), cov (T x T) and the log marginal likelihood of the 'nngp' (or 'ntk') posterior."""
    n, t = len(x), len(xt)
    kdd = mp.matrix(kernel(x, None, depth, sigma_w, sigma_b, act))
    a = mp.matrix(kernel(x, None, depth, sigma_w, sigma_b, act, "ntk")) if ntk else kdd.copy()
    lam = mp.mpf(diag_reg) * (mp.fsum(a[i, i] for i in range(n)) / n)
    for i in range(n):
        a[i, i] += lam
    yv = mp.matrix([mp.mpf(float(v)) for v in y])
    alpha = mp.cholesky_solve(a, yv)
    c = mp.cholesky(a)
    lml = -yv.T * alpha / 2
    lml = lml[0] - mp.fsum(mp.log(c[i, i]) for i in range(n)) - n * mp.log(2 * mp.pi) / 2
    ks = mp.matrix(kernel(xt, x, depth, sigma_w, sigma_b, act))
    ths = mp.matrix(kernel(xt, x, depth, sigma_w, sigma_b, act, "ntk")) if ntk else ks
    ktt = kernel(xt, None, depth, sigma_w, sigma_b, act)
    mean = ths * alpha
    ws = [mp.cholesky_solve(a, ths[i, :].T) for i in range(t)]
    if ntk:
        kw = [kdd * w for w in ws]
        cov = [[ktt[i][j] + mp.fsum(ws[i][m] * kw[j][m] for m in range(n))
                - mp.fsum(ws[i][m] * ks[j, m] for m in range(n)) - mp.fsum(ws[j][m] * ks[i, m] for m in range(n))
                for j in range(t)] for i in range(t)]
    else:
        cov = [[ktt[i][j] - mp.fsum(ws[i][m] * ks[j, m] for m in range(n)) for j in range(t)] for i in range(t)]
    return {"mean": [mean[i] for i in range(t)], "cov": cov, "var": [cov[i][i] for i in range(t)], "lml": lml,
            "lam": lam}


# ---- the closed forms' independent check ---------------------------------------------------------------------
def _phi(act, x, deriv):
    kind, a, b, c = act
    if kind == "abrelu":
        if deriv:
            return a if x < 0 else b
        return a * x if x < 0 else b * x
    if deriv:
        return a * b * 2 / mp.sqrt(mp.pi) * mp.exp(-(b * x) ** 2)
    return a * mp.erf(b * x) + c


def expectations_by_quadrature(q1, q2, k, act, dps=17):
    """(E[phi(u) phi(v)], E[phi'(u) phi'(v)], E[phi(u)^2]) for (u, v) ~ N(0, [[q1, k], [k, q2]]) by numerical
    integration in polar coordinates of the whitened variables, u = sqrt(q1) z1, v = k/sqrt(q1) z1 + w z2.  ABRelu:
    the integrands are homogeneous in r (degree 2, 0), so the radial integral is exact (int r^3 e^(-r^2/2) = 2,
    int r e^(-r^2/2) = 1) and the angular one is split where u or v changes sign; Erf: 2-D quadrature."""
    with mp.workdps(dps):
        act = _mpf_act(act)
        q1, q2, k = mp.mpf(q1), mp.mpf(q2), mp.mpf(k)
        su, cu = mp.sqrt(q1), k / mp.sqrt(q1)
        w = mp.sqrt(q2 - cu * cu)
        uv = lambda r, t: (su * r * mp.cos(t), r * (cu * mp.cos(t) + w * mp.sin(t)))
        if act[0] == "abrelu":
            tv = mp.atan2(-cu, w)            # v = 0 at t = tv and tv + pi; u = 0 at +-pi/2
            cuts = sorted({float(x) for x in (-mp.pi / 2, mp.pi / 2, tv, tv + mp.pi if tv < 0 else tv - mp.pi)})
            pts = [-mp.pi] + [mp.mpf(x) for x in cuts if -mp.pi < x < mp.pi] + [mp.pi]

            def ang(f):
                return mp.quad(f, pts) / (2 * mp.pi)
            e_pp = 2 * ang(lambda t: _phi(act, uv(1, t)[0], False) * _phi(act, uv(1, t)[1], False))
            e_dd = ang(lambda t: _phi(act, uv(1, t)[0] + mp.mpf(0), True) * _phi(act, uv(1, t)[1], True))
            e_p2 = 2 * ang(lambda t: _phi(act, su * mp.cos(t), False) ** 2)
            return e_pp, e_dd, e_p2

        def polar(f):
            return mp.quad(lambda t, r: f(*uv(r, t)) * r * mp.exp(-r * r / 2), [-mp.pi, 0, mp.pi], [0, 3, 8, mp.inf]) / (2 * mp.pi)
        e_pp = polar(lambda u, v: _phi(act, u, False) * _phi(act, v, False))
        e_dd = polar(lambda u, v: _phi(act, u, True) * _phi(act, v, True))
        e_p2 = polar(lambda u, v: _phi(act, u, False) ** 2)
        return e_pp, e_dd, e_p2
