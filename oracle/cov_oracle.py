"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED AGAINST THE REFERENCE.

The full posterior covariance of a test batch, in FP64 numpy, on top of the fits of ``nngp_oracle.py`` (see its
header for the reference call sites): what ``predict_fn(x_test=X, get=..., compute_cov=True)`` returns in
neural-tangents before the reference's callers take its diagonal.  'nngp' is ``nngp_oracle.Fit.predict_full_cov``;
this module adds 'ntk'.  Checked against the 50-digit vectors of ``tests/golden/mp_cov.npz``
(``mp_cov_oracle.py``, ``tests/golden/make_mp_cov_golden.py``).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

import nngp_oracle as oracle


def ntk_predict_full_cov(fit: oracle.FitNTK, x_test):
    """(mean (T,1), cov (T,T)) of get='ntk' at t = infinity (SURVEY.md Appendix A.5)  [nt: gp_inference.predict_fn]:
    cov = K_** + Theta_* A^-1 K_dd A^-1 Theta_*^T - (Theta_* A^-1 K_*^T + transpose)."""
    x_test = np.asarray(x_test, dtype=np.float64)
    ks, ths = oracle.kernel_fn(x_test, fit.x, fit.depth, fit.sigma_w, fit.sigma_b, get="both")
    ktt = oracle.kernel_fn(x_test, None, fit.depth, fit.sigma_w, fit.sigma_b)
    mean = ths @ fit.alpha
    w = sla.cho_solve((fit.c, True), ths.T, check_finite=False)               # A^-1 Theta_*^T   (N x T)
    cross = ks @ w                                                            # K_* A^-1 Theta_*^T
    cov = ktt + w.T @ (fit.k_dd @ w) - (cross + cross.T)
    return mean[:, None], cov


def predict_full_cov(fit, x_test):
    """(mean (T,1), cov (T,T)) of an nngp_oracle.Fit or nngp_oracle.FitNTK."""
    if isinstance(fit, oracle.FitNTK):
        return ntk_predict_full_cov(fit, x_test)
    return fit.predict_full_cov(x_test)
