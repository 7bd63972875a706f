"""ctypes binding of the C ABI in ``include/nngp_b200.h`` (``libnngp_b200.so``).

This module is the ONLY way the Python host layer reaches arithmetic: every kernel /
fit / predict call goes through the shared library's sm_100a CUDA kernels.  There is no
CPU fallback -- if the library is missing, or no B200 is visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

from . import _build

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("NNGP_B200_LIB", _PKG_DIR.parent / "libnngp_b200.so"))

NNGP_OK, NNGP_EINVAL, NNGP_ENOTPD, NNGP_ECUDA, NNGP_ENOMEM, NNGP_ESTATE, NNGP_ENODEV = 0, -1, -2, -3, -4, -5, -6


class NngpConfig(C.Structure):
    _fields_ = [
        ("depth", C.c_int32),
        ("sigma_w", C.c_double),
        ("sigma_b", C.c_double),
        ("diag_reg", C.c_double),
        ("diag_reg_absolute", C.c_int32),
        ("device", C.c_int32),
        ("max_block_bytes", C.c_int64),
        ("stats_level", C.c_int32),
        ("kernel_type", C.c_int32),
        ("n_gpus", C.c_int32),
        ("device_ids", C.c_int32 * 8),
        ("latency_mode", C.c_int32),
        ("per_layer", C.c_int32),
        ("sigma_w_layers", C.c_double * 16),
        ("sigma_b_layers", C.c_double * 16),
        ("variance_slices", C.c_int32),
        ("reserved0", C.c_int32),
    ]


class NngpStats(C.Structure):
    _fields_ = (
        [(n, C.c_double) for n in (
            "fit_gram_ms", "fit_chol_ms", "fit_solve_ms", "fit_total_ms",
            "pred_gram_ms", "pred_mean_ms", "pred_trsm_ms", "pred_var_ms", "pred_total_ms",
            "h2d_ms", "d2h_ms", "gemm_ms", "gemm_flops")]
        + [("gemm_launches", C.c_int64)]
        + [(n, C.c_double) for n in ("gram_ms", "gram_flops", "gram_evals")]
        + [(n, C.c_int64) for n in ("gram_launches", "kernel_launches", "h2d_bytes", "d2h_bytes", "queries")]
        + [("replicate_ms", C.c_double), ("replicate_bytes", C.c_int64), ("inverse_ms", C.c_double),
           ("sliced_ms", C.c_double), ("sliced_macs", C.c_double), ("device_allocs", C.c_int64)]
    )

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


# every symbol include/nngp_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I64 = C.c_int64
_DP = C.POINTER(C.c_double)
EXPORTS = {
    "nngp_abi_version": (C.c_int, []),
    "nngp_build_id": (C.c_char_p, []),
    "nngp_num_gpus": (C.c_int, [_P]),
    "nngp_sliced_product": (C.c_int, [_P, _P, _I64, _I64, _P, _I64, C.c_int32, C.c_int32, _P, _P]),
    "nngp_state_packed_size": (C.c_int, [_P, C.POINTER(_I64)]),
    "nngp_state_pack": (C.c_int, [_P, _I64, _I64, _P]),
    "nngp_state_import_begin": (C.c_int, [_P, _I64, _I64]),
    "nngp_state_unpack": (C.c_int, [_P, _I64, _I64, _P]),
    "nngp_state_import_end": (C.c_int, [_P, C.c_double]),
    "nngp_default_config": (None, [C.POINTER(NngpConfig)]),
    "nngp_create": (C.c_int, [C.POINTER(NngpConfig), C.POINTER(_P)]),
    "nngp_destroy": (None, [_P]),
    "nngp_last_error": (C.c_char_p, [_P]),
    "nngp_get_stream": (_P, [_P]),
    "nngp_kernel": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "nngp_fit": (C.c_int, [_P, _P, _P, _I64, _I64]),
    "nngp_predict": (C.c_int, [_P, _P, _I64, _P, _P]),
    "nngp_get_dims": (C.c_int, [_P, C.POINTER(_I64), C.POINTER(_I64), _DP]),
    "nngp_get_state": (C.c_int, [_P, _P, _P, _P]),
    "nngp_set_state": (C.c_int, [_P, _P, _P, _P, _I64, _I64, C.c_double]),
    "nngp_get_state_ntk_m": (C.c_int, [_P, _P]),
    "nngp_set_state_ntk_m": (C.c_int, [_P, _P]),
    "nngp_log_marginal_likelihood": (C.c_int, [_P, _DP]),
    "nngp_active_select": (C.c_int, [_P, _P, _I64, _I64, C.c_int32, C.c_uint64, _P, C.POINTER(_I64), _P]),
    "nngp_append_fit": (C.c_int, [_P, _P, _P, _I64]),
    "nngp_reserve": (C.c_int, [_P, _I64, _I64, _I64]),
    "nngp_stats": (C.c_int, [_P, C.POINTER(NngpStats)]),
    "nngp_stats_reset": (C.c_int, [_P]),
    "nngp_diag_dmma_peak": (C.c_int, [_P, _DP]),
    "nngp_diag_gemm_probe": (C.c_int, [_P, _I64, _I64, _I64, C.c_int32, _DP]),
    "nngp_diag_potrf": (C.c_int, [_P, _P, _I64]),
    "nngp_encoder_create": (C.c_int, [C.c_char_p, C.POINTER(_P)]),
    "nngp_encoder_destroy": (None, [_P]),
    "nngp_encoder_dim": (C.c_int, [_P]),
    "nngp_encoder_last_error": (C.c_char_p, [_P]),
    "nngp_encode_lines": (C.c_int, [_P, C.c_char_p, _I64, _I64, C.c_int32, _P, _P, C.c_int32]),
}

_lib = None


class NngpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"nngp_b200 error {code}: {msg}")
        self.code = code


def load() -> C.CDLL:
    """Load libnngp_b200.so (built in-tree by ``__graft_entry__.build()``). Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    custom = "NNGP_B200_LIB" in os.environ          # an explicitly chosen build is taken as it is
    if not custom and (not LIB_PATH.exists() or built_id(LIB_PATH) != _build.source_hash()):
        # missing, or compiled from other sources than the tree we run in (the .so is not tracked by git: it travels
        # to the GPU box as a built file) -> rebuild in-tree; without nvcc this raises, there is no CPU fallback
        _build.build()
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} not found (nngp_b200 has no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def built_id(path=None) -> str | None:
    """nngp_build_id() of a library file, read without loading it into this process, or None."""
    return _build.library_id(path or LIB_PATH)


def build_id() -> str:
    return load().nngp_build_id().decode()


def _raise(lib, handle, code: int):
    msg = lib.nngp_last_error(handle)
    msg = msg.decode("utf-8", "replace") if msg else ""
    if code == NNGP_EINVAL:
        raise ValueError(f"nngp_b200: {msg}")
    if code == NNGP_ENOTPD:
        raise np.linalg.LinAlgError(f"nngp_b200: {msg}")
    raise NngpError(code, msg)


def _ptr(a):
    """(pointer, keepalive) for an INPUT: a numpy array (host) or a torch CUDA/CPU tensor (device/host).
    Inputs of another dtype / layout are converted into a temporary (kept alive by the caller)."""
    if a is None:
        return None, None
    if isinstance(a, np.ndarray):
        if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"]:
            a = np.ascontiguousarray(a, dtype=np.float64)
        return C.c_void_p(a.ctypes.data), a
    if hasattr(a, "data_ptr"):  # torch tensor
        import torch
        if a.dtype != torch.float64 or not a.is_contiguous():
            a = a.to(torch.float64).contiguous()
        if a.is_cuda:
            # the library reads on its own non-blocking stream, which is not ordered with torch's streams: whatever
            # produced (or converted) this tensor on torch's current stream must have finished before the C call
            torch.cuda.current_stream(a.device).synchronize()
        return C.c_void_p(a.data_ptr()), a
    a = np.ascontiguousarray(a, dtype=np.float64)
    return C.c_void_p(a.ctypes.data), a


def _out_ptr(a, shape, name):
    """Pointer of an OUTPUT buffer.  The library writes float64 values straight into it, so it must already be
    float64, C-contiguous, writeable and of the right size -- anything else raises (a silent temporary would leave
    the caller's buffer unfilled)."""
    n = int(np.prod(shape))
    if isinstance(a, np.ndarray):
        if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"] or not a.flags["WRITEABLE"]:
            raise ValueError(f"nngp_b200: output buffer {name} must be a writeable C-contiguous float64 array "
                             f"(got dtype {a.dtype}, contiguous={a.flags['C_CONTIGUOUS']})")
        if a.size != n:
            raise ValueError(f"nngp_b200: output buffer {name} has {a.size} elements, {n} are needed {tuple(shape)}")
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        import torch
        if a.dtype != torch.float64 or not a.is_contiguous():
            raise ValueError(f"nngp_b200: output buffer {name} must be a contiguous float64 tensor (got {a.dtype})")
        if a.numel() != n:
            raise ValueError(f"nngp_b200: output buffer {name} has {a.numel()} elements, {n} are needed {tuple(shape)}")
        if a.is_cuda:
            torch.cuda.current_stream(a.device).synchronize()   # earlier users of the buffer on torch's stream
        return C.c_void_p(a.data_ptr())
    raise ValueError(f"nngp_b200: output buffer {name} must be a numpy array or a torch tensor, got {type(a).__name__}")


def _npz_path(path):
    """np.savez appends '.npz' to a name without it; save() and load() agree on the final name."""
    p = os.fspath(path)
    return p if p.endswith(".npz") else p + ".npz"


class Handle:
    """RAII wrapper of ``nngp_handle*`` (one GPU, not re-entrant)."""

    def __init__(self, depth=2, sigma_w=1.0, sigma_b=0.0, diag_reg=1e-3, diag_reg_absolute=False,
                 device=-1, max_block_bytes=0, stats_level=1, kernel_type="nngp", n_gpus=1, device_ids=None,
                 latency_mode=False, variance_slices=0):
        self._lib = load()
        cfg = NngpConfig()
        self._lib.nngp_default_config(C.byref(cfg))
        # sigma_w / sigma_b: one value for every Dense layer, or one per layer (stax.serial chains whose layers differ)
        sw, sb = np.atleast_1d(np.asarray(sigma_w, dtype=np.float64)), np.atleast_1d(np.asarray(sigma_b, dtype=np.float64))
        if sw.size > 1 or sb.size > 1:
            sw = np.broadcast_to(sw, (int(depth),)) if sw.size == 1 else sw
            sb = np.broadcast_to(sb, (int(depth),)) if sb.size == 1 else sb
            if sw.size != int(depth) or sb.size != int(depth) or int(depth) > 16:
                raise ValueError(f"nngp_b200: per-layer sigma_w / sigma_b need one value per Dense layer "
                                 f"(depth={depth} <= 16), got {sw.size} / {sb.size}")
            if np.all(sw == sw[0]) and np.all(sb == sb[0]):
                sw, sb = sw[:1], sb[:1]                      # uniform after all
        cfg.depth, cfg.sigma_w, cfg.sigma_b = int(depth), float(sw[0]), float(sb[0])
        cfg.per_layer = int(sw.size > 1)
        for i in range(16):
            cfg.sigma_w_layers[i] = float(sw[i]) if i < sw.size and sw.size > 1 else 0.0
            cfg.sigma_b_layers[i] = float(sb[i]) if i < sb.size and sb.size > 1 else 0.0
        cfg.diag_reg, cfg.diag_reg_absolute = float(diag_reg), int(bool(diag_reg_absolute))
        cfg.device, cfg.max_block_bytes, cfg.stats_level = int(device), int(max_block_bytes), int(stats_level)
        if kernel_type not in ("nngp", "ntk"):
            raise NotImplementedError(f"kernel_type {kernel_type!r}: only 'nngp' and 'ntk' exist")
        cfg.kernel_type = 1 if kernel_type == "ntk" else 0
        ids = list(device_ids) if device_ids is not None else []
        n_gpus = len(ids) if ids else int(n_gpus)
        if n_gpus > 8 or n_gpus < 0:
            raise ValueError(f"nngp_b200: n_gpus={n_gpus}: 1..8 GPUs per handle")
        cfg.n_gpus = n_gpus
        for i in range(8):
            cfg.device_ids[i] = int(ids[i]) if i < len(ids) else -1
        cfg.latency_mode = int(bool(latency_mode))
        cfg.variance_slices = int(variance_slices)
        self.cfg = cfg
        h = C.c_void_p()
        rc = self._lib.nngp_create(C.byref(cfg), C.byref(h))
        if rc != NNGP_OK:
            _raise(self._lib, None, rc)
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.nngp_destroy(self._h)
            self._h = None

    __del__ = close

    def _ck(self, rc):
        if rc != NNGP_OK:
            _raise(self._lib, self._h, rc)

    @property
    def stream(self) -> int:
        return int(self._lib.nngp_get_stream(self._h) or 0)

    def kernel(self, x1, x2=None, out=None):
        x1p, k1 = _ptr(x1)
        M, D = k1.shape
        x2p, k2 = _ptr(x2)
        N2 = k2.shape[0] if k2 is not None else M
        if k2 is not None and k2.shape[1] != D:
            raise ValueError(f"nngp_b200: x1 has {D} features but x2 has {k2.shape[1]}")
        if out is None:
            out = np.empty((M, N2), dtype=np.float64)
        op = _out_ptr(out, (M, N2), "out")
        self._ck(self._lib.nngp_kernel(self._h, x1p, M, x2p, N2, D, op))
        return out

    def sliced_product(self, a, b, slices=7, lower=False, want_rowsq=False):
        """Diagnostic: ``a @ b.T`` through ``slices`` int8 digit planes per operand on the tcgen05 kind::i8 kernel
        (the product behind ``variance_slices``).  ``lower=True``: b is lower triangular; ``lower=2``: additionally drop
        the plane pair (slices-1, 0) as the variance path does for b = L^-1.  Returns V, or (V, row sums of V**2) with
        ``want_rowsq``."""
        ap, ka = _ptr(a)
        bp, kb = _ptr(b)
        M, K = ka.shape
        N = kb.shape[0]
        if kb.shape[1] != K:
            raise ValueError(f"nngp_b200: a has {K} columns but b has {kb.shape[1]}")
        v = np.empty((M, N), dtype=np.float64)
        rs = np.empty(M, dtype=np.float64) if want_rowsq else None
        self._ck(self._lib.nngp_sliced_product(self._h, ap, M, K, bp, N, 2 if lower == 2 else int(bool(lower)), int(slices),
                                               _out_ptr(v, (M, N), "v"), _out_ptr(rs, (M,), "rowsq") if want_rowsq else None))
        return (v, rs) if want_rowsq else v

    def fit(self, x, y):
        xp, kx = _ptr(x)
        yp, ky = _ptr(y)
        N, D = kx.shape
        if int(np.prod(ky.shape)) != N:
            raise ValueError(f"nngp_b200: y_train has {int(np.prod(ky.shape))} entries for {N} training rows")
        self._ck(self._lib.nngp_fit(self._h, xp, yp, N, D))

    def _check_width(self, kx, what):
        d = self.dims()[1]          # raises NngpError(NNGP_ESTATE) when nothing is fitted
        if kx.ndim != 2 or kx.shape[1] != d:
            raise ValueError(f"nngp_b200: {what} must be [rows, {d}] like the training set, got {tuple(kx.shape)}")

    def predict(self, x, want_var=True, mean_out=None, var_out=None):
        xp, kx = _ptr(x)
        self._check_width(kx, "x_test")
        T = kx.shape[0]
        if mean_out is None:
            mean_out = np.empty(T, dtype=np.float64)
        if want_var and var_out is None:
            var_out = np.empty(T, dtype=np.float64)
        mp = _out_ptr(mean_out, (T,), "mean_out")
        vp = _out_ptr(var_out, (T,), "var_out") if want_var else None
        self._ck(self._lib.nngp_predict(self._h, xp, T, mp, vp))
        return mean_out, (var_out if want_var else None)

    def dims(self):
        n, d, lam = _I64(), _I64(), C.c_double()
        self._ck(self._lib.nngp_get_dims(self._h, C.byref(n), C.byref(d), C.byref(lam)))
        return n.value, d.value, lam.value

    @property
    def n_gpus(self) -> int:
        return int(self._lib.nngp_num_gpus(self._h))

    # ---- packed state streaming (see include/nngp_b200.h; used by nngp_b200.dist.broadcast_fit) ----
    def packed_size(self) -> int:
        n = _I64()
        self._ck(self._lib.nngp_state_packed_size(self._h, C.byref(n)))
        return n.value

    def state_pack(self, offset: int, count: int, dst) -> None:
        self._ck(self._lib.nngp_state_pack(self._h, int(offset), int(count), _out_ptr(dst, (count,), "dst")))

    def state_import_begin(self, n: int, d: int) -> None:
        self._ck(self._lib.nngp_state_import_begin(self._h, int(n), int(d)))

    def state_unpack(self, offset: int, count: int, src) -> None:
        sp, keep = _ptr(src)
        if int(np.prod(keep.shape)) != int(count):
            raise ValueError(f"nngp_b200: src has {int(np.prod(keep.shape))} elements, count is {count}")
        self._ck(self._lib.nngp_state_unpack(self._h, int(offset), int(count), sp))

    def state_import_end(self, lam: float) -> None:
        self._ck(self._lib.nngp_state_import_end(self._h, float(lam)))

    @property
    def is_ntk(self) -> bool:
        return self.cfg.kernel_type == 1

    def get_state(self, x=True, l=True, alpha=True, out=None, m=None):
        """Copy the fitted state out. ``out`` may be a dict of preallocated arrays/tensors (host or device).
        In 'ntk' mode the state also holds ``m`` = L^-1 K_dd L^-T (exported whenever ``l`` is, unless m=False)."""
        n, d, lam = self.dims()
        out = dict(out or {})
        if m is None:
            m = bool(l) and self.is_ntk
        if m:
            if "m" not in out:
                out["m"] = np.empty((n, n))
            mp = _out_ptr(out["m"], (n, n), "m")
            self._ck(self._lib.nngp_get_state_ntk_m(self._h, mp))
        if x and "x" not in out:
            out["x"] = np.empty((n, d))
        if l and "l" not in out:
            out["l"] = np.empty((n, n))
        if alpha and "alpha" not in out:
            out["alpha"] = np.empty(n)
        xp = _out_ptr(out["x"], (n, d), "x") if x else None
        lp = _out_ptr(out["l"], (n, n), "l") if l else None
        ap = _out_ptr(out["alpha"], (n,), "alpha") if alpha else None
        self._ck(self._lib.nngp_get_state(self._h, xp, lp, ap))
        out["lambda"] = lam
        return out

    def set_state(self, x, l, alpha, lam, m=None):
        xp, kx = _ptr(x)
        lp, _kl = _ptr(l)
        ap, _ka = _ptr(alpha)
        N, D = kx.shape
        self._ck(self._lib.nngp_set_state(self._h, xp, lp, ap, N, D, float(lam)))
        if m is not None:                     # 'ntk' mode: the variance also needs M = L^-1 K_dd L^-T
            mp, km = _ptr(m)
            if tuple(km.shape) != (N, N):
                raise ValueError(f"nngp_b200: m must be [{N}, {N}], got {tuple(km.shape)}")
            self._ck(self._lib.nngp_set_state_ntk_m(self._h, mp))

    def active_select(self, x_pool, budget, biased_sample=False, seed=10, return_scores=False):
        """Device-side ``ActiveLearner.active_test`` (active/ActiveLearner.py:43-55): rows of ``x_pool`` to label
        next -- ``argsort(std/max(mean))[-budget:]`` or, with ``biased_sample``, a draw without replacement with
        probability proportional to that score (Gumbel-top-k, splitmix64 stream of ``seed``)."""
        xp, kx = _ptr(x_pool)
        self._check_width(kx, "x_pool")
        T = kx.shape[0]
        k = min(int(budget), T)
        idx = np.empty(k, dtype=np.int64)
        n_sel = _I64()
        scores = np.empty(T) if return_scores else None
        self._ck(self._lib.nngp_active_select(self._h, xp, T, int(budget), 1 if biased_sample else 0, int(seed),
                                              C.c_void_p(idx.ctypes.data), C.byref(n_sel),
                                              C.c_void_p(scores.ctypes.data) if return_scores else None))
        assert n_sel.value == k
        return (idx, scores) if return_scores else idx

    def append_fit(self, x_new, y_new) -> None:
        """``merge_data`` + ``train`` of the active-learning loop (active/ActiveLearner.py:57-65,76): append labelled
        rows to the training set held on the device and refit."""
        xp, kx = _ptr(x_new)
        yp, ky = _ptr(y_new)
        self._check_width(kx, "x_new")
        M = kx.shape[0]
        if int(np.prod(ky.shape)) != M:
            raise ValueError(f"x_new has {M} rows but y_new has shape {tuple(ky.shape)}")
        self._ck(self._lib.nngp_append_fit(self._h, xp, yp, M))

    def reserve(self, n_train_max, dim, n_test_max=0) -> None:
        """Pre-size the device buffers for the largest problem an active-learning loop will reach (before ``fit``)."""
        self._ck(self._lib.nngp_reserve(self._h, int(n_train_max), int(dim), int(n_test_max)))

    def log_marginal_likelihood(self) -> float:
        v = C.c_double()
        self._ck(self._lib.nngp_log_marginal_likelihood(self._h, C.byref(v)))
        return v.value

    def save(self, path) -> None:
        """Fitted state + hyper-parameters -> .npz (the reference has no model file: it refits on every start,
        neuroestimator/README.md:28-29; its ``load_model`` is a warm-up, estimator.py:37-40)."""
        st = self.get_state()
        extra = {"m": st["m"]} if self.is_ntk else {}
        if self.cfg.per_layer:
            sw = np.array(self.cfg.sigma_w_layers[:self.cfg.depth])
            sb = np.array(self.cfg.sigma_b_layers[:self.cfg.depth])
        else:
            sw, sb = self.cfg.sigma_w, self.cfg.sigma_b
        np.savez(_npz_path(path), x=st["x"], l=st["l"], alpha=st["alpha"], lam=st["lambda"], depth=self.cfg.depth,
                 sigma_w=sw, sigma_b=sb, diag_reg=self.cfg.diag_reg,
                 diag_reg_absolute=self.cfg.diag_reg_absolute, kernel_type="ntk" if self.is_ntk else "nngp", **extra)

    @classmethod
    def load(cls, path, **kw) -> "Handle":
        z = np.load(_npz_path(path))
        kt = str(z["kernel_type"]) if "kernel_type" in z.files else "nngp"
        h = cls(depth=int(z["depth"]), sigma_w=z["sigma_w"], sigma_b=z["sigma_b"],
                diag_reg=float(z["diag_reg"]), diag_reg_absolute=bool(z["diag_reg_absolute"]), kernel_type=kt, **kw)
        h.set_state(z["x"], z["l"], z["alpha"], float(z["lam"]), m=z["m"] if kt == "ntk" else None)
        return h

    def stats(self) -> dict:
        s = NngpStats()
        self._ck(self._lib.nngp_stats(self._h, C.byref(s)))
        return s.as_dict()

    def stats_reset(self):
        self._ck(self._lib.nngp_stats_reset(self._h))

    def dmma_peak_tflops(self) -> float:
        v = C.c_double()
        self._ck(self._lib.nngp_diag_dmma_peak(self._h, C.byref(v)))
        return v.value

    def gemm_probe_ms(self, M, N, K, iters=10) -> float:
        v = C.c_double()
        self._ck(self._lib.nngp_diag_gemm_probe(self._h, M, N, K, iters, C.byref(v)))
        return v.value

    def potrf(self, a: np.ndarray) -> np.ndarray:
        a = np.array(a, dtype=np.float64, order="C", copy=True)
        self._ck(self._lib.nngp_diag_potrf(self._h, C.c_void_p(a.ctypes.data), a.shape[0]))
        return np.tril(a)
