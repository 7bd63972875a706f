"""Mirror of ``neural_tangents.predict.gradient_descent_mse_ensemble`` for ``get='nngp'`` / ``get='ntk'``.

Reference call sites: train.py:171-172 + 157-158, neuroestimator/estimator/estimator.py:34-35 + 66-67,
active/ActiveLearner.py:27-28 + 35-36,44-45.  Semantics kept ([nt 0.6.1] predict.gp_inference):
  * construction is instantaneous; the fit (K_dd, lambda = diag_reg*trace(K_dd)/N, Cholesky, alpha) runs on
    the first ``predict_fn`` call and is cached; a new ``gradient_descent_mse_ensemble`` call is a new fit
    (the active-learning loop relies on this, active/ActiveLearner.py:69,76);
  * ``predict_fn(x_test=X, get='nngp', compute_cov=True)`` returns ``Gaussian(mean[T,1], covariance)``;
  * every caller only takes ``sqrt(diag(covariance))`` (train.py:180, estimator.py:55, ActiveLearner.py:46),
    so ``covariance`` is a lazy (T,T)-shaped object exposing the posterior-variance diagonal -- the T x T
    matrix the reference materialises (and throws away) is never built;
  * code that needs the joint posterior (correlations between queries, the variance of a sum, joint samples)
    asks for it explicitly: ``predict_fn.full_covariance(x_test, get)`` returns ``Gaussian(mean, cov[T,T])``
    from the same cached fit.
All arithmetic: libnngp_b200.so (sm_100a CUDA).  Unsupported options raise NotImplementedError.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np

from . import runtime
from .stax import KernelFn

Gaussian = namedtuple("Gaussian", ["mean", "covariance"])

_DIAG_FUNCS = {}


class LazyCovariance:
    """(T, T)-shaped stand-in for the posterior covariance; only its diagonal exists."""

    def __init__(self, var):
        self._var = np.asarray(var, dtype=np.float64).reshape(-1)
        t = self._var.shape[0]
        self.shape, self.ndim, self.dtype, self.size = (t, t), 2, np.dtype(np.float64), t * t

    def diagonal(self, offset=0, axis1=0, axis2=1):
        if offset != 0:
            raise NotImplementedError("only the main diagonal of the posterior covariance is computed")
        return self._var

    def __array_function__(self, func, types, args, kwargs):
        if func in (np.diag, np.diagonal) and len(args) == 1 and not kwargs:
            return self._var
        if func is np.trace and len(args) == 1 and not kwargs:
            return float(np.sum(self._var))
        if func is np.shape:
            return self.shape
        return NotImplemented

    def __array__(self, *a, **k):
        raise NotImplementedError(
            "nngp_b200 computes the posterior-variance DIAGONAL only (the reference's callers use nothing else: "
            "train.py:180, estimator.py:55, ActiveLearner.py:46); use np.diag(cov) / cov.diagonal(), or "
            "predict_fn.full_covariance(x_test, get) for the T x T matrix")

    def __repr__(self):
        return f"LazyCovariance(shape={self.shape}, diagonal-only)"


def gradient_descent_mse_ensemble(kernel_fn, x_train, y_train, learning_rate=1.0, diag_reg=0.0,
                                  diag_reg_absolute_scale=False, trace_axes=(-1,), _fitted_engines=None, _reserve=None,
                                  **kernel_fn_train_train_kwargs):
    if not isinstance(kernel_fn, KernelFn):
        raise NotImplementedError("gradient_descent_mse_ensemble: kernel_fn must come from nngp_b200.stax.serial")
    if kernel_fn_train_train_kwargs:
        raise NotImplementedError(f"unsupported kernel_fn kwargs {sorted(kernel_fn_train_train_kwargs)}")
    if tuple(trace_axes) != (-1,):
        raise NotImplementedError("only trace_axes=(-1,) is supported")
    x_train = runtime.as_matrix(x_train, "x_train")
    y_arr = y_train if hasattr(y_train, "data_ptr") else np.asarray(y_train, dtype=np.float64)
    y_shape = tuple(y_arr.shape)
    if len(y_shape) == 2 and y_shape[1] != 1:
        raise NotImplementedError("only a single regression output (y_train of shape [N] or [N,1]) is supported")
    if y_shape[0] != x_train.shape[0]:
        raise ValueError(f"x_train has {x_train.shape[0]} rows but y_train has {y_shape[0]}")
    state = dict(_fitted_engines or {})        # one cached fit per `get`, like nt's lru_cache'd predict_inf
                                               # (_fitted_engines: handles already fitted on exactly this data --
                                               #  the device-side append of the active-learning loop, active.py)

    def _fitted(get="nngp"):
        if get not in state:
            h = runtime.new_handle(kernel_fn.spec, diag_reg=diag_reg, diag_reg_absolute=diag_reg_absolute_scale,
                                   kernel_type=get)
            if _reserve is not None and hasattr(h, "reserve"):      # (n_train_max, n_test_max) of an AL loop
                h.reserve(max(int(_reserve[0]), x_train.shape[0]), x_train.shape[1], int(_reserve[1]))
            h.fit(x_train, y_arr)          # raises ValueError / LinAlgError through the C-ABI error codes
            state[get] = h
        return state[get]

    def predict_fn(t=None, x_test=None, get=None, compute_cov=False, **kwargs):
        if t is not None:
            raise NotImplementedError("predict_fn(t=...): only the infinite-time (t=None) posterior is implemented")
        if kwargs:
            raise NotImplementedError(f"predict_fn: unsupported arguments {sorted(kwargs)}")
        if get is None:
            get = "nngp"
        if get not in ("nngp", "ntk"):
            raise NotImplementedError(f"predict_fn(get={get!r}): 'nngp' and 'ntk' are implemented (one at a time)")
        h = _fitted(get)
        xt = x_train if x_test is None else runtime.as_matrix(x_test, "x_test")
        mean, var = h.predict(xt, want_var=bool(compute_cov))
        mean = mean.reshape(-1, 1) if len(y_shape) == 2 else mean
        if not compute_cov:
            return mean
        return Gaussian(mean, LazyCovariance(var))

    def _full_covariance(x_test=None, get="nngp"):
        """``predict_fn(x_test, get=get, compute_cov=True)`` with the covariance as the dense (T, T) posterior
        covariance neural-tangents returns (mean (T, 1) or (T,) like predict_fn).  x_test=None: the training inputs."""
        if get not in ("nngp", "ntk"):
            raise NotImplementedError(f"full_covariance(get={get!r}): 'nngp' and 'ntk' are implemented (one at a time)")
        h = _fitted(get)
        xt = x_train if x_test is None else runtime.as_matrix(x_test, "x_test")
        mean, cov = h.predict_cov(xt)
        return Gaussian(mean.reshape(-1, 1) if len(y_shape) == 2 else mean, cov)

    def _release(get="nngp"):
        """Hand the fitted engine of ``get`` over to the caller and forget it here: this closure then refits from its
        own (x_train, y_train) the next time it is used -- in the reference every ``gradient_descent_mse_ensemble``
        call is an independent fit, so a predict_fn kept from an earlier active-learning round must not start
        answering with a later round's model (``ActiveLearner.retrain`` appends to the engine it takes from here)."""
        return state.pop(get, None)

    predict_fn.engine = _fitted            # bench / tests: access to the underlying C-ABI handle
    predict_fn.release = _release
    predict_fn.full_covariance = _full_covariance
    predict_fn.spec = kernel_fn.spec
    return predict_fn
