"""GPU tests of cfg.variance_slices: the variance product V = K_* L^-T on the INT8 tensor cores (sliced_gemm.cuh:
digit planes + tcgen05.mma kind::i8 with TMEM accumulators).  Everything goes through the C ABI.

Bars: the integer part is bit-exact (the kernel's V equals a numpy restatement of the same digit planes, which are
exact integers); the posterior variance stays within north_star's 1e-6 relative of the oracle (measured: 1e-9 .. 1e-8
at 7 planes, 1e-11 .. 1e-10 at 8), the mean is bitwise the FP64 path's (it never touches the planes).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import nngp_oracle as oracle  # noqa: E402


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


def _split_rows(a, s, tri=False):
    """Digit planes of the rows of ``a`` and their exponents e (|row| < 2^e, 0 for a zero row): the scale-up by 2^(6-e)
    is exact for every finite row, down to the smallest subnormal (np.ldexp does not form 2^(6-e) on its own)."""
    a = np.tril(a) if tri else a
    amax = np.max(np.abs(a), axis=1)
    _, e = np.frexp(amax)
    e = np.where(amax == 0, 0, e)
    t = np.ldexp(a, (6 - e)[:, None])
    planes = []
    for _ in range(s):
        q = np.rint(t)
        planes.append(q)
        t = (t - q) * 128.0
    return planes, e


def _digit_restatement(a, b, s, tri, skip_weak=False):
    """What sliced_gemm_kernel computes, in numpy: exact integer plane products (FP64 matmuls of small integers),
    groups p + q = g folded by Horner in 2^-7, both row exponents applied at once (one rounding, also where the
    product or a row scale 2^(e-6) leaves the normal range).  ``skip_weak``: without the pair (s-1, 0), as the
    variance path runs it."""
    pa, ea = _split_rows(a, s)
    pb, eb = _split_rows(b, s, tri)
    acc = None
    for g in range(s - 1, -1, -1):
        last = g - 1 if (skip_weak and g == s - 1 and g > 0) else g
        c = sum(pa[p] @ pb[g - p].T for p in range(last + 1))
        assert np.max(np.abs(c)) < 2 ** 31
        acc = c if acc is None else acc * 0.0078125 + c
    return np.ldexp(acc, ea[:, None] + eb[None, :] - 12)


# largest magnitudes of the rows placed at the bottom of the range: 2^-1017 is the last exponent whose scale-up 2^(6-e)
# is a double, 2^-1068 the last whose row scale 2^(e-6) is, 2^-1074 the smallest subnormal
TINY_ROWS = (-1017, -1018, -1030, -1068, -1070, -1074)


def _set_tiny_rows(x, rng, first):
    """Rows first.. of x get largest magnitude exactly 2^E for E in TINY_ROWS (signed entries, some exact zeros)."""
    for i, e in enumerate(TINY_ROWS):
        u = rng.uniform(-1.0, 1.0, size=x.shape[1])
        u[rng.random(x.shape[1]) < 0.1] = 0.0
        u[i % x.shape[1]] = -1.0 if i % 2 else 1.0
        x[first + i] = np.ldexp(u, e)


@pytest.mark.parametrize("m,k,n,tri,s,tiny", [
    pytest.param(128, 128, 256, False, 1, False, id="128-128-256-False-1"),
    pytest.param(200, 300, 500, False, 7, False, id="200-300-500-False-7"),
    pytest.param(1, 40, 3, False, 6, False, id="1-40-3-False-6"),
    pytest.param(515, 1280, 1280, True, 7, False, id="515-1280-1280-True-7"),
    pytest.param(2500, 2304, 2304, True, 9, False, id="2500-2304-2304-True-9"),
    pytest.param(300, 4096, 700, False, 5, False, id="300-4096-700-False-5"),
    # rows of A (and of B when it is rectangular) whose largest magnitude is 2^-1017 .. 2^-1074, among normal rows
    pytest.param(200, 300, 500, False, 7, True, id="200-300-500-False-7-subnormal_rows"),
    pytest.param(515, 1280, 1280, True, 7, True, id="515-1280-1280-True-7-subnormal_rows"),
    pytest.param(300, 700, 260, False, 9, True, id="300-700-260-False-9-subnormal_rows"),
])
def test_sliced_product_is_bit_exact_against_the_digit_restatement(lib, m, k, n, tri, s, tiny):
    rng = np.random.default_rng(m + n + s)
    a = rng.normal(size=(m, k)) * np.exp(3 * rng.normal(size=(m, 1)))       # row scales over ~10 decades
    b = rng.normal(size=(n, k)) * np.exp(3 * rng.normal(size=(n, 1)))
    if m > 100:
        a[7] = 0.0                                                            # an all-zero row: exponent 0, digits 0
    if tiny:
        _set_tiny_rows(a, rng, 20)
        if not tri:
            _set_tiny_rows(b, rng, 30)
    if tri:
        b = np.tril(b)
    h = lib.Handle()
    v, rowsq = h.sliced_product(a, b, slices=s, lower=tri, want_rowsq=True)
    ref = _digit_restatement(a, b, s, tri)
    assert np.array_equal(v, ref)
    assert np.allclose(rowsq, np.einsum("ij,ij->i", v, v), rtol=1e-13, atol=0)
    if s >= 7:      # and the digits carry the product: error relative to |row a|max |row b|max K
        # (the exact product of the rows brought to [0.5, 1) by their exponents, where V is a normal double)
        _, ea = np.frexp(np.max(np.abs(a), axis=1))
        _, eb = np.frexp(np.max(np.abs(np.tril(b) if tri else b), axis=1))
        an, bn = np.ldexp(a, -ea[:, None]), np.ldexp(b, -eb[:, None])
        scale = np.max(np.abs(an), axis=1)[:, None] * np.max(np.abs(bn), axis=1)[None, :] * k + 1e-300
        normal = np.abs(v) >= np.finfo(np.float64).tiny
        err = np.abs(np.ldexp(v, -(ea[:, None] + eb[None, :])) - an @ bn.T) / scale
        assert np.max(np.where(normal, err, 0.0)) < 2.0 ** (-7 * s + 8)
    v2 = h.sliced_product(a, b, slices=s, lower=tri)
    assert np.array_equal(v, v2)
    h.close()


def test_variance_path_drops_only_the_weakest_pair(lib):
    """lower=2 is the product exactly as nngp_predict runs it against W = L^-1: all pairs p + q < s except (s-1, 0).
    Bit-exact against the restatement with the same rule; on a diagonally dominated factor (what L^-1 is) the result
    stays at the accuracy of the full set, on a generic triangular matrix it would not -- hence variance path only."""
    rng = np.random.default_rng(21)
    n, m, s = 1536, 300, 7
    a = rng.random((m, n)) + 0.5                                     # flat rows, like kernel values
    w = np.tril(rng.normal(size=(n, n))) * 0.01 + np.diag(1.0 + rng.random(n))     # diagonal ~100x the rest, like L^-1
    h = lib.Handle()
    v_all = h.sliced_product(a, w, slices=s, lower=True)
    v_skip = h.sliced_product(a, w, slices=s, lower=2)
    assert np.array_equal(v_all, _digit_restatement(a, w, s, True))
    assert np.array_equal(v_skip, _digit_restatement(a, w, s, True, skip_weak=True))
    exact = a @ w.T
    scale = np.max(np.abs(exact))
    e_all, e_skip = np.max(np.abs(v_all - exact)) / scale, np.max(np.abs(v_skip - exact)) / scale
    assert e_skip < 4 * e_all + 1e-15, (e_all, e_skip)
    h.close()


def _problem(n, t, d, seed=11):
    rng = np.random.default_rng(seed)
    x = rng.random((n, d))
    y = rng.normal(size=n) * 3 + 8
    xt = np.vstack([rng.random((t - t // 4, d)), x[rng.integers(0, n, t // 4)] + 1e-3 * rng.normal(size=(t // 4, d))])
    return x, y, xt


@pytest.mark.parametrize("s,tol", [(7, 1e-7), (8, 1e-9)])
def test_variance_slices_parity_with_the_oracle(lib, s, tol):
    x, y, xt = _problem(2048, 9000, 64)
    ref = lib.Handle(depth=2)
    ref.fit(x, y)
    m0, v0 = ref.predict(xt)
    h = lib.Handle(depth=2, variance_slices=s)
    h.fit(x, y)
    m1, v1 = h.predict(xt)                       # 9000 rows > NNGP_LATENCY_ROWS: the tcgen05 path
    assert h.stats()["sliced_macs"] > 0
    assert np.array_equal(m0, m1)
    fit = oracle.Fit(x, y, depth=2)
    sel = np.linspace(0, xt.shape[0] - 1, 600).astype(np.int64)
    _mo, vo = fit.predict(xt[sel])
    assert np.max(np.abs(v1[sel] - vo) / np.abs(vo)) < tol          # north_star: 1e-6
    assert np.max(np.abs(v1 - v0) / np.abs(v0)) < tol
    m2, v2 = h.predict(xt)
    assert np.array_equal(v1, v2)                                    # fixed reduction order: repeatable bit for bit
    # rows predicted in a different batch composition give the same bits (per-row exponents, per-row sums)
    _m3, v3 = h.predict(xt[:5000])
    assert np.array_equal(v3, v1[:5000])
    h.close(); ref.close()


def test_variance_slices_on_the_forest_workload(lib, forest, monkeypatch):
    """Reference workload C1 (cond(K + lambda I) ~ 1e7): 7 planes stay 100x inside the 1e-6 bar."""
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "0")       # 3600 test rows: force the large-batch (tcgen05) path
    x, y, xt = forest["x_train"], forest["y_train"], forest["x_test"]
    h = lib.Handle(depth=2, variance_slices=7)
    h.fit(x, y)
    mean, var = h.predict(xt)
    assert h.stats()["sliced_macs"] > 0
    fit = oracle.Fit(x, y, depth=2)
    mo, vo = fit.predict(xt)
    assert np.max(np.abs(mean - mo)) < 1e-6 * np.max(np.abs(mo))
    assert np.max(np.abs(var - vo) / np.abs(vo)) < 1e-6
    assert np.max(np.abs(np.sqrt(var) - np.sqrt(vo)) / np.sqrt(vo)) < 1e-6
    h.close()


def test_variance_slices_survive_state_import_and_append(lib):
    x, y, xt = _problem(1536, 6000, 48, seed=5)
    h = lib.Handle(depth=2, variance_slices=7)
    h.fit(x[:1024], y[:1024])
    h.append_fit(x[1024:], y[1024:])             # the planes are rebuilt with the extended factor
    _m, v_app = h.predict(xt)
    fresh = lib.Handle(depth=2, variance_slices=7)
    fresh.fit(x, y)
    _m, v_fresh = fresh.predict(xt)
    assert np.max(np.abs(v_app - v_fresh) / np.abs(v_fresh)) < 1e-7
    st = fresh.get_state()
    imp = lib.Handle(depth=2, variance_slices=7)
    imp.set_state(st["x"], st["l"], st["alpha"], st["lambda"])
    _m, v_imp = imp.predict(xt)
    assert np.array_equal(v_imp, v_fresh)
    for hh in (h, fresh, imp):
        hh.close()


def test_variance_slices_multi_gpu_is_bitwise_the_single_gpu_result(lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    x, y, xt = _problem(2048, 12000, 64, seed=9)
    one = lib.Handle(depth=2, variance_slices=7)
    one.fit(x, y)
    m1, v1 = one.predict(xt)
    two = lib.Handle(depth=2, variance_slices=7, n_gpus=2)
    two.fit(x, y)
    m2, v2 = two.predict(xt)
    assert np.array_equal(m1, m2) and np.array_equal(v1, v2)
    one.close(); two.close()


def test_variance_slices_rejects_misuse(lib):
    with pytest.raises((ValueError, lib.NngpError)):
        lib.Handle(variance_slices=3)
    with pytest.raises((ValueError, lib.NngpError)):
        lib.Handle(variance_slices=12)
    with pytest.raises((ValueError, lib.NngpError)):
        lib.Handle(variance_slices=7, kernel_type="ntk")
    h = lib.Handle()
    a = np.ones((4, 8))
    with pytest.raises((ValueError, lib.NngpError)):
        h.sliced_product(a, np.ones((5, 8)), slices=7, lower=True)     # a triangular factor must be square
    with pytest.raises((ValueError, lib.NngpError)):
        h.sliced_product(a, np.ones((5, 8)), slices=0)
    with pytest.raises(ValueError):
        h.sliced_product(a, np.ones((5, 9)))
    h.close()
