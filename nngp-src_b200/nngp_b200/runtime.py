"""Process-wide runtime knobs of the host layer: which GPU new handles bind to, input coercion."""
from __future__ import annotations

import os

import numpy as np

from . import _lib

_device = int(os.environ.get("NNGP_B200_DEVICE", os.environ.get("LOCAL_RANK", "-1")))
_stats_level = int(os.environ.get("NNGP_B200_STATS", "1"))
_max_block_bytes = int(os.environ.get("NNGP_B200_MAX_BLOCK_BYTES", "0"))
# GPUs per handle (in-process row-sharded prediction): "NNGP_B200_GPUS=8" or a list of ordinals "0,1,2,3"
_gpus_env = os.environ.get("NNGP_B200_GPUS", "")
_device_ids = [int(v) for v in _gpus_env.split(",")] if "," in _gpus_env else None
_n_gpus = int(_gpus_env) if _gpus_env and _device_ids is None else (len(_device_ids) if _device_ids else 1)
_latency_mode = os.environ.get("NNGP_B200_LATENCY_MODE", "0") not in ("", "0")
_variance_slices = int(os.environ.get("NNGP_B200_VARIANCE_SLICES", "0") or 0)


def set_device(index: int) -> None:
    """GPU ordinal for handles created from now on (-1 = the CUDA current device)."""
    global _device
    _device = int(index)


def set_stats_level(level: int) -> None:
    """0 none, 1 per-stage CUDA events (default), 2 per-kernel-class events (bench roofline accounting)."""
    global _stats_level
    _stats_level = int(level)


def get_device() -> int:
    return _device


def set_gpus(n_or_ids) -> None:
    """Handles created from now on predict on several GPUs of this process: an int G (devices 0..G-1) or a list of
    CUDA ordinals (the first one fits).  The fitted state is replicated peer-to-peer once per fit and test rows are
    split [g*T/G, (g+1)*T/G) -- ``predict_fn`` / ``Estimator.predict`` / the reference's drivers scale unchanged."""
    global _n_gpus, _device_ids
    if isinstance(n_or_ids, int):
        _n_gpus, _device_ids = int(n_or_ids), None
    else:
        _device_ids = [int(v) for v in n_or_ids]
        _n_gpus = len(_device_ids)


def set_latency_mode(on: bool) -> None:
    """Fits from now on also build the explicit inverse factor; small prediction batches use it (serving case)."""
    global _latency_mode
    _latency_mode = bool(on)


def set_variance_slices(s: int) -> None:
    """Fits from now on keep int8 digit planes of the inverse factor (s = 5..9 planes, 0 = off); the variance of
    large prediction batches then runs on the INT8 tensor cores (tcgen05) instead of the FP64 substitution."""
    global _variance_slices
    _variance_slices = int(s)


def new_handle(spec, diag_reg=0.0, diag_reg_absolute=False, kernel_type="nngp") -> "_lib.Handle":
    return _lib.Handle(depth=spec.depth, sigma_w=spec.sigma_w, sigma_b=spec.sigma_b, diag_reg=diag_reg,
                       diag_reg_absolute=diag_reg_absolute, device=_device, max_block_bytes=_max_block_bytes,
                       stats_level=_stats_level, kernel_type=kernel_type, n_gpus=_n_gpus, device_ids=_device_ids,
                       latency_mode=_latency_mode, variance_slices=_variance_slices if kernel_type == "nngp" else 0,
                       activation=spec.activation)


def as_matrix(x, name="x"):
    """numpy float64 C-contiguous 2-D view of x, or x itself if it is a float64 torch tensor."""
    if hasattr(x, "data_ptr") and hasattr(x, "is_contiguous"):   # torch tensor: host or device, zero-copy
        if x.dim() != 2:
            raise ValueError(f"{name} must be 2-D, got shape {tuple(x.shape)}")
        return x
    a = np.ascontiguousarray(np.asarray(x), dtype=np.float64)
    if a.ndim != 2:
        raise ValueError(f"{name} must be 2-D [rows, features], got shape {a.shape}")
    return a
