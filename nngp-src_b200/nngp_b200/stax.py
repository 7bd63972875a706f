"""Mirror of the ``neural_tangents.stax`` surface the reference uses on its NNGP path.

Reference call sites: ``stax.serial(stax.Dense(512), stax.Relu(), stax.Dense(1))`` at train.py:161-164,
neuroestimator/estimator/estimator.py:27-30, active/active_train.py:40-43 (and the commented
``W_std=1.5, b_std=0.05`` variant at active/active_train.py:44-49).

Only what defines the infinite-width NNGP kernel is kept: a chain Dense (Act Dense)* with one activation
throughout (Relu, LeakyRelu, Abs, ABRelu or Erf) collapses to a ``KernelSpec(depth, W_std, b_std, activation)``
and ``kernel_fn`` evaluates it with the sm_100a Gram kernel (the activation's steps in its epilogue) through the
C ABI.  ``init_fn`` / ``apply_fn`` (finite-width networks) and every other layer type
raise ``NotImplementedError`` -- never a silent CPU fallback.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import _lib, runtime


@dataclass(frozen=True)
class KernelSpec:
    depth: int           # number of Dense layers; depth-1 activation steps
    sigma_w: object      # W_std: a float when every Dense layer has the same, else a tuple with one value per layer
    sigma_b: object      # b_std (None -> 0): likewise
    activation: _lib.Activation = _lib.RELU   # of every step


class _Layer(tuple):
    """(init_fn, apply_fn, kernel_fn) triple, like neural-tangents' layer constructors return."""
    kind: str
    params: dict

    def __new__(cls, kind, **params):
        def _finite_width(*_a, **_k):
            raise NotImplementedError("nngp_b200 implements the infinite-width NNGP kernel only "
                                      "(init_fn/apply_fn of finite networks are outside the hot path)")
        self = super().__new__(cls, (_finite_width, _finite_width, None))
        self.kind, self.params = kind, params
        return self


def Dense(out_dim, W_std=1.0, b_std=None, batch_axis=0, channel_axis=-1, parameterization="ntk", s=(1, 1)):
    if parameterization != "ntk" or batch_axis != 0 or channel_axis not in (-1, 1) or tuple(s) != (1, 1):
        raise NotImplementedError("nngp_b200.stax.Dense: only the default NTK parameterisation / axes are supported")
    return _Layer("dense", out_dim=int(out_dim), W_std=float(W_std), b_std=0.0 if b_std is None else float(b_std))


def _act_layer(act):
    return _Layer("act", activation=act)


def Relu(do_backprop=False, do_stabilize=False):
    return _act_layer(_lib.RELU)


def ABRelu(a, b, do_stabilize=False):
    """a min(x, 0) + b max(x, 0)   [nt 0.6.1 stax.ABRelu]"""
    return _act_layer(_lib.Activation("abrelu", float(a), float(b)))


def LeakyRelu(alpha, do_stabilize=False):
    """ABRelu(alpha, 1)   [nt 0.6.1 stax.LeakyRelu]"""
    return ABRelu(alpha, 1.0)


def Abs(do_stabilize=False):
    """ABRelu(-1, 1)   [nt 0.6.1 stax.Abs]"""
    return ABRelu(-1.0, 1.0)


def Erf(a=1., b=1., c=0.):
    """a erf(b x) + c   [nt 0.6.1 stax.Erf]"""
    return _act_layer(_lib.Activation("erf", float(a), float(b), float(c)))


def _unsupported(name):
    def ctor(*_a, **_k):
        raise NotImplementedError(f"nngp_b200.stax.{name} is not implemented (the kernels exist for Dense and the "
                                  "Relu / LeakyRelu / Abs / ABRelu / Erf activations)")
    ctor.__name__ = name
    return ctor


for _n in ("Conv", "Gelu", "Flatten", "AvgPool", "GlobalAvgPool", "FanOut",
           "FanInSum", "LayerNorm", "Dropout", "Identity", "parallel"):
    globals()[_n] = _unsupported(_n)


class KernelFn:
    """``kernel_fn(x1, x2=None, get='nngp' | 'ntk')`` -> ndarray[M, N]  (reference: train.py:216, via predict_fn)."""

    def __init__(self, spec: KernelSpec):
        self.spec = spec
        self._handles = {}

    def _engine(self, get="nngp"):
        if get not in self._handles:
            self._handles[get] = runtime.new_handle(self.spec, kernel_type=get)
        return self._handles[get]

    def __call__(self, x1, x2=None, get=None, **kwargs):
        if kwargs:
            raise NotImplementedError(f"kernel_fn: unsupported arguments {sorted(kwargs)}")
        if get is None:
            get = "nngp"
        if get not in ("nngp", "ntk"):
            raise NotImplementedError(f"kernel_fn(get={get!r}): 'nngp' and 'ntk' are implemented (one at a time)")
        x1 = runtime.as_matrix(x1, "x1")
        x2 = None if x2 is None else runtime.as_matrix(x2, "x2")
        return self._engine(get).kernel(x1, x2)

    def __repr__(self):
        return f"KernelFn({self.spec})"


def serial(*layers):
    """Collapse Dense (Act Dense)* into one KernelSpec; returns (init_fn, apply_fn, kernel_fn)."""
    if not layers or any(not isinstance(l, _Layer) for l in layers):
        raise NotImplementedError("nngp_b200.stax.serial: expects layers built by nngp_b200.stax.Dense / an activation")
    kinds = [l.kind for l in layers]
    if kinds[0] != "dense" or kinds[-1] != "dense" or any(
            kinds[i] == kinds[i + 1] for i in range(len(kinds) - 1)):
        raise NotImplementedError(f"nngp_b200.stax.serial: only Dense (Act Dense)* chains are supported, got {kinds}")
    acts = {l.params["activation"] for l in layers if l.kind == "act"}
    if len(acts) > 1:
        raise NotImplementedError(f"nngp_b200.stax.serial: one activation for every hidden layer, got {sorted(map(str, acts))}")
    act = acts.pop() if acts else _lib.RELU
    dense = [l for l in layers if l.kind == "dense"]
    w = tuple(l.params["W_std"] for l in dense)
    b = tuple(l.params["b_std"] for l in dense)
    if len(set(w)) == 1 and len(set(b)) == 1:
        spec = KernelSpec(depth=len(dense), sigma_w=w[0], sigma_b=b[0], activation=act)
    else:                                   # layers differ [nt allows it]: per-layer values (nngp_config.per_layer)
        if len(dense) > 16:
            raise NotImplementedError("nngp_b200.stax.serial: per-layer W_std / b_std support at most 16 Dense layers")
        spec = KernelSpec(depth=len(dense), sigma_w=w, sigma_b=b, activation=act)
    init_fn, apply_fn, _ = dense[0]
    return init_fn, apply_fn, KernelFn(spec)
