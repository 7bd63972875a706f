"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.

The NNGP / NTK kernels and GP posteriors of ``nngp_oracle.py`` for a chain Dense (act Dense)* with one activation
throughout [nt 0.6.1 stax.ABRelu / stax.Erf nngp_fn, nngp_fn_diag and ntk]:

  ABRelu(a, b)   phi(x) = a min(x, 0) + b max(x, 0)   (ReLU (0, 1), LeakyRelu(alpha) (alpha, 1), Abs (-1, 1))
      kdot = (a^2 + b^2)/2 - (a - b)^2 theta / (2 pi);  E[phi(u) phi(v)] = (a - b)^2 s / (2 pi) + kdot k
      E[phi(u)^2] = (a^2 + b^2)/2 q
  Erf(a, b, c)   phi(x) = a erf(b x) + c;  Q = b^2 q, K = b^2 k, P = 1 + 2 (Q1 + Q2) + 4 b^4 s^2
      E[phi(u) phi(v)] = a^2 (2/pi) atan2(2K, sqrt P) + c^2;  kdot = a^2 b^2 (4/pi) / sqrt P
      E[phi(u)^2] = a^2 (2/pi) arcsin(2Q / (1 + 2Q)) + c^2

with s = sqrt(max(q1 q2 - k^2, 0)), theta = atan2(s, k) (pi/2 at s = k = 0); each step is followed by the next Dense
layer, k' = sigma_w^2 E[phi phi] + sigma_b^2, ntk' = k' + sigma_w^2 ntk kdot.  ``activation=None`` is ReLU and runs
``nngp_oracle`` itself.  An activation is ``(kind, a, b, c)`` or any object with those attributes
(``nngp_b200._lib.Activation``).  Pinned by ``tests/golden/mp_act.npz`` (``mp_act_oracle.py``), whose generator
first checks the closed forms against 2-D quadrature over the bivariate normal.

Why a module of its own rather than an ``activation=`` keyword on ``nngp_oracle.kernel_fn`` / ``final_diag`` / ``Fit``
/ ``FitNTK``: ``nngp_oracle.py`` is the yardstick every existing ReLU test, ``smoke()`` and ``bench.py`` compare the
CUDA path against, and it is kept byte-for-byte as it is, so that adding activations cannot move what the ReLU path is
measured by.  The entry points here take the same arguments plus ``activation`` (``None`` calls ``nngp_oracle``
itself), and ``tests/test_activation_host.py`` checks that ``ABRelu(0, 1)`` here is bitwise ``nngp_oracle``'s ReLU.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

import nngp_oracle as base

TWO_PI = base.TWO_PI


def normalize(act):
    """(kind, a, b, c) of an activation, or None for ReLU."""
    if act is None:
        return None
    kind, a, b, c = (act.kind, act.a, act.b, act.c) if hasattr(act, "kind") else tuple(act) + (0.0,) * (4 - len(act))
    if kind == "relu":
        return None
    if kind not in ("abrelu", "erf"):
        raise ValueError(f"unknown activation {kind!r}")
    return kind, float(a), float(b), float(c)


def _step(k, ntk, q1, q2, sw2, sb2, act):
    """One activation step + Dense on the block k (rows q1, columns q2), in place."""
    kind, a, b, c = act
    prod = q1[:, None] * q2[None, :]
    s = np.sqrt(np.maximum(prod - k * k, 0.0))
    if kind == "abrelu":
        c0, c1 = (a * a + b * b) / 2, (a - b) ** 2 / TWO_PI
        theta = np.arctan2(s, k)
        theta[(s == 0.0) & (k == 0.0)] = np.pi / 2
        kdot = c0 - c1 * theta
        k[...] = sw2 * (c1 * s + kdot * k) + sb2
    else:
        b2 = b * b
        sp = np.sqrt(1.0 + 2.0 * b2 * (q1[:, None] + q2[None, :]) + 4.0 * (b2 * s) ** 2)
        kdot = a * a * b2 * (4.0 / np.pi) / sp
        k[...] = sw2 * (a * a * (2.0 / np.pi) * np.arctan2(2.0 * b2 * k, sp) + c * c) + sb2
    if ntk is not None:
        ntk[...] = k + sw2 * (ntk * kdot)


def next_diag(q, sw2, sb2, act):
    """sigma_w^2 E[phi(u)^2] + sigma_b^2 at variance q."""
    kind, a, b, c = act
    if kind == "abrelu":
        return sw2 * ((a * a + b * b) / 2 * q) + sb2
    big_q = b * b * q
    return sw2 * (a * a * (2.0 / np.pi) * np.arctan2(2.0 * big_q, np.sqrt(1.0 + 4.0 * big_q)) + c * c) + sb2


def final_diag(q0, depth=2, sigma_w=1.0, sigma_b=0.0, activation=None):
    """K(x,x) after depth-1 steps."""
    act = normalize(activation)
    if act is None:
        return base.final_diag(q0, depth, sigma_w, sigma_b)
    sw2l, sb2l = base._layer_sigmas(depth, sigma_w, sigma_b)
    q = np.array(q0, dtype=np.float64, copy=True)
    for layer in range(1, depth):
        q = next_diag(q, sw2l[layer], sb2l[layer], act)
    return q


def kernel_fn(x1, x2=None, depth=2, sigma_w=1.0, sigma_b=0.0, chunk=2048, get="nngp", activation=None):
    """nngp_oracle.kernel_fn with an activation (get: 'nngp' | 'ntk' | 'both')."""
    act = normalize(activation)
    if act is None:
        return base.kernel_fn(x1, x2, depth, sigma_w, sigma_b, chunk, get)
    x1 = np.asarray(x1, dtype=np.float64)
    x2 = x1 if x2 is None else np.asarray(x2, dtype=np.float64)
    D = x1.shape[1]
    sw2l, sb2l = base._layer_sigmas(depth, sigma_w, sigma_b)
    q1_all, q2_0 = base.layer0_diag(x1, sigma_w, sigma_b), base.layer0_diag(x2, sigma_w, sigma_b)
    out = np.empty((x1.shape[0], x2.shape[0]))
    out_ntk = np.empty_like(out) if get in ("ntk", "both") else None
    for r0 in range(0, x1.shape[0], chunk):
        r1 = min(r0 + chunk, x1.shape[0])
        k = sw2l[0] * ((x1[r0:r1] @ x2.T) / D) + sb2l[0]
        ntk = k.copy() if out_ntk is not None else None
        q1, q2 = q1_all[r0:r1], q2_0
        for layer in range(1, depth):
            _step(k, ntk, q1, q2, sw2l[layer], sb2l[layer], act)
            q1, q2 = next_diag(q1, sw2l[layer], sb2l[layer], act), next_diag(q2, sw2l[layer], sb2l[layer], act)
        out[r0:r1] = k
        if out_ntk is not None:
            out_ntk[r0:r1] = ntk
    if get == "nngp":
        return out
    return out_ntk if get == "ntk" else (out, out_ntk)


def erf_amplification(x, depth=2, sigma_w=1.0, sigma_b=0.0, activation=None):
    """(F, G): per pair of rows of x, how many times its own rounding an FP64 evaluation of the Erf kernel K (F) and of
    its NTK Theta (G) can be moved by the rounding of its inputs, from the conditioning of the steps in k
    (DESIGN.md 5.12).  One step moves E[phi phi] by (4/pi) a^2 b^2 dk / sqrt P when k moves by dk, and
    sqrt P >= max(2 b^2 s, sqrt(2 b^2 (q1 + q2))): a rounding of k (eps sqrt(q q')) moves E by at most
    eps a^2 min(1/sin theta, sqrt(b^2 min(q, q'))), and by at most sqrt(eps) a^2 once the rounding residue of s^2
    dominates P.  kdot = a^2 b^2 (4/pi) / sqrt P moves by eps min(1/sin^2 theta, 2 b^2 min(q, q'), 1/eps) relative.
    Up to 1/sin theta = 4 that is within the bounds' own budget (2.5 eps), so only near-parallel pairs and the
    diagonal get a factor; the steps compound (product over the steps).  All ones for the ABRelu family, whose
    near-parallel error cancels to first order (as ReLU's)."""
    act = normalize(activation)
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    F, G = np.ones((n, n)), np.ones((n, n))
    if act is None or act[0] != "erf":
        return F, G
    b2, eps = act[2] ** 2, np.finfo(np.float64).eps
    q0 = base.layer0_diag(x, sigma_w, sigma_b)
    for layer in range(depth - 1):                      # step `layer` acts on the pre-activations of Dense layer `layer`
        q = final_diag(q0, layer + 1, sigma_w, sigma_b, activation)
        k = kernel_fn(x, None, layer + 1, sigma_w, sigma_b, activation=activation)
        qq = np.outer(q, q)
        with np.errstate(divide="ignore", invalid="ignore"):
            cos2 = np.where(qq > 0, np.minimum(k * k / qq, 1.0), 0.0)
            inv_sin = 1.0 / np.sqrt(1.0 - cos2)
        qmin = np.minimum.outer(q, q)
        near = inv_sin > 4.0
        F *= np.where(near, np.maximum(1.0, np.minimum(np.minimum(inv_sin, np.sqrt(b2 * qmin)), 1.0 / np.sqrt(eps))), 1.0)
        G *= np.where(near, np.maximum(1.0, np.minimum(np.minimum(inv_sin ** 2, 2.0 * b2 * qmin), 1.0 / eps)), 1.0)
    return F, G


class Fit(base.Fit):
    """nngp_oracle.Fit with an activation."""

    def __init__(self, x, y, depth=2, sigma_w=1.0, sigma_b=0.0, diag_reg=1e-3, diag_reg_absolute=False, activation=None):
        self.x = np.asarray(x, dtype=np.float64)
        self.y = np.asarray(y, dtype=np.float64).reshape(-1)
        self.depth, self.sigma_w, self.sigma_b, self.activation = depth, sigma_w, sigma_b, activation
        n = self.x.shape[0]
        k = kernel_fn(self.x, None, depth, sigma_w, sigma_b, activation=activation)
        self.lam = diag_reg if diag_reg_absolute else diag_reg * (np.trace(k) / n)
        k[np.diag_indices(n)] += self.lam
        self.c = sla.cholesky(k, lower=True, check_finite=False)
        self.alpha = sla.cho_solve((self.c, True), self.y, check_finite=False)

    def _k(self, x1, x2=None, get="nngp"):
        return kernel_fn(x1, x2, self.depth, self.sigma_w, self.sigma_b, get=get, activation=self.activation)

    def _kss(self, x):
        return final_diag(base.layer0_diag(x, self.sigma_w, self.sigma_b), self.depth, self.sigma_w, self.sigma_b,
                          self.activation)

    def predict(self, x_test, want_var=True):
        ks = self._k(x_test, self.x)
        mean = ks @ self.alpha
        if not want_var:
            return mean, None
        v = sla.solve_triangular(self.c, ks.T, lower=True, check_finite=False)
        return mean, self._kss(x_test) - np.einsum("ij,ij->j", v, v)

    def predict_full_cov(self, x_test):
        """(mean (T,1), cov (T,T))."""
        ks = self._k(x_test, self.x)
        mean = ks @ self.alpha
        return mean[:, None], self._k(x_test) - ks @ sla.cho_solve((self.c, True), ks.T, check_finite=False)


class FitNTK(Fit):
    """nngp_oracle.FitNTK with an activation (log_marginal_likelihood: of A = Theta_dd + lambda I)."""

    def __init__(self, x, y, depth=2, sigma_w=1.0, sigma_b=0.0, diag_reg=1e-3, diag_reg_absolute=False, activation=None):
        self.x = np.asarray(x, dtype=np.float64)
        self.y = np.asarray(y, dtype=np.float64).reshape(-1)
        self.depth, self.sigma_w, self.sigma_b, self.activation = depth, sigma_w, sigma_b, activation
        n = self.x.shape[0]
        self.k_dd, th = self._k(self.x, None, get="both")
        self.lam = diag_reg if diag_reg_absolute else diag_reg * (np.trace(th) / n)
        th[np.diag_indices(n)] += self.lam
        self.c = sla.cholesky(th, lower=True, check_finite=False)
        self.alpha = sla.cho_solve((self.c, True), self.y, check_finite=False)

    def predict(self, x_test, want_var=True):
        mean, cov = self.predict_full_cov(x_test) if want_var else (None, None)
        if not want_var:
            return self._k(x_test, self.x, get="ntk") @ self.alpha, None
        return mean[:, 0], np.diag(cov).copy()

    def predict_full_cov(self, x_test):
        ks, ths = self._k(x_test, self.x, get="both")
        mean = ths @ self.alpha
        w = sla.cho_solve((self.c, True), ths.T, check_finite=False)
        cross = ks @ w
        return mean[:, None], self._k(x_test) + w.T @ (self.k_dd @ w) - (cross + cross.T)
