"""GPU: the blocked Cholesky, the alpha solve, every prediction solve and the incremental append against answers that
are known exactly.

Construction.  L~ is an integer lower-triangular matrix with positive diagonal, small entries and a few non-zeros per
row, so every partial sum of L~ L~^T stays far below 2^53 and A = L~ L~^T is exact in FP64: its Cholesky factor is
exactly L~.  Through the whole pipeline: depth 1 (the Gram is a plain GEMM), sigma_w = 1, sigma_b = 0, lambda = 0,
D a power of two >= N + 8 and X = [L~ | 0].  The Gram's scale 1/D is exact, so K = L~ L~^T / D exactly and

    factor    L = L~ / sqrt(D)
    labels    y = L~ (L~^T a~) / D for integer a~  (exact)   ->   alpha = a~,   z = L^-1 y = L~^T a~ / sqrt(D)
    query     x* = [u | w] (integer u over the N training columns, integer w over the padding columns):
              V = L^-1 k* = u / sqrt(D),   mean = u . (L~^T a~) / D,   var = |w|^2 / D   (all exact)
    LML       -|z|^2 / 2 - sum log L_ii - N/2 log(2 pi)

Rows with w = 0 have variance exactly 0: K(x*, x*) and |V|^2 cancel completely.

Families of L~ (``lower_band``, ``with_chain``):
  (a) diagonal d = 16, band entries +-1 at offsets 1 and 2, two random +-1 entries per row.  With s_r, s_c the largest
      off-diagonal row and column sums of |L~|, ||L~ - dI||_2 <= sqrt(s_r s_c) = s < d, so every singular value of L~
      lies in [d - s, d + s] and cond_2(L~) <= kappa = (d + s)/(d - s) (``cond_bound``; about 2 here).
  (b) (a) graded by powers of two: S A S with S = diag(2^e).  Its factor is S L~, and every operation of the
      factorisation scales exactly, so the GPU factor must be S times the ungraded GPU factor bit for bit.
  (c) a chain of diagonal 4 and subdiagonal -5 over one 64-row diagonal block (cond(L_JJ) ~ 1e6).
  (d) the same chain on 64 rows spread over the whole matrix.

Error model (DESIGN.md section 5.2).  The factorisation and every solve apply explicit inverses W_J = inv(L_JJ) of
the 64 x 64 diagonal blocks instead of substituting.  With cond(L_JJ) <= cond(L~) <= kappa that keeps the usual
first-order bounds of a Cholesky factorisation and triangular solve, which the tolerances below take with constant 2
(factor) or 4 (everything downstream of two triangular solves):

    |L^ - L|            <= 2 N eps kappa max|L|
    |alpha^ - a~|       <= 4 N eps kappa^2 max|a~|                    (cond(K) <= kappa^2)
    |mean^ - mean|      <= 4 N eps kappa^2 max|a~| sum_i |k*_i|       (alpha's error seen through k*)
    |var^ - var|        <= 4 N eps kappa K(x*, x*)                   (|V|^2 <= K(x*, x*); 'ntk': kappa^2, M = I + O(eps kappa^2))
    |LML^ - LML|        <= 4 N eps kappa^2 (|z|^2 / 2 + sum |log L_ii| + N)

The constants were fixed before the first run.  With concentrated ill-conditioning (family c) the backward error of
the explicit-inverse factorisation is eps cond(L_JJ) ||A||, not eps ||A||: ``test_error_model_of_the_explicit_inverses``
checks exactly that against a long-double reference and LAPACK.
"""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
PAD = 8                  # padding columns of X: room for the w part of the queries
CHAIN_DIAG, CHAIN_SUB = 4.0, -5.0

W256_N = [1, 2, 3, 5, 63, 64, 65, 127, 128, 129, 255, 256, 257, 513, 4095]
W512_N = [4096, 4097, 4159, 4160, 8191, 8193]
W1024_N = 24576 + 65


# ---------------------------------------------------------------------------------------------- generator (host)
def lower_band(n, seed, d=16, extra=2):
    """Family (a): integer lower-triangular L~ (CSR, float64 values): diagonal d, +-1 at offsets 1 and 2, and `extra`
    random +-1 entries per row further left (duplicates are summed, so an entry can be 0 or +-2)."""
    rng = np.random.default_rng(seed)
    rows, cols, vals = [np.arange(n)], [np.arange(n)], [np.full(n, float(d))]
    for off in (1, 2):
        i = np.arange(off, n)
        rows.append(i); cols.append(i - off); vals.append(rng.choice([-1.0, 1.0], i.size))
    for _ in range(extra):
        i = np.arange(3, n)
        rows.append(i); cols.append(np.floor(rng.random(i.size) * (i - 2)).astype(np.int64))
        vals.append(rng.choice([-1.0, 1.0], i.size))
    L = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    L.sum_duplicates()
    L.eliminate_zeros()
    return L


def with_chain(L, idx):
    """Families (c) / (d): rows idx (ascending) of L~ replaced by the chain L[i_k, i_k] = 4, L[i_k, i_(k-1)] = -5.
    Still integer and lower triangular; cond of the chain alone is about (5/4)^len(idx)."""
    idx = np.asarray(idx, dtype=np.int64)
    coo = L.tocoo()
    keep = ~np.isin(coo.row, idx)
    rows = [coo.row[keep], idx, idx[1:]]
    cols = [coo.col[keep], idx, idx[:-1]]
    vals = [coo.data[keep], np.full(idx.size, CHAIN_DIAG), np.full(idx.size - 1, CHAIN_SUB)]
    out = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=L.shape)
    out.sum_duplicates()
    return out


def cond_bound(L):
    """kappa = (d + s)/(d - s) >= cond_2(L~) for a constant diagonal d and s = sqrt(s_r s_c) < d (family a)."""
    diag = L.diagonal()
    d = float(diag[0])
    assert np.all(diag == d), "cond_bound needs a constant diagonal"
    off = abs(sp.tril(L, -1)).tocsr()
    s_r = float(off.sum(axis=1).max()) if off.nnz else 0.0
    s_c = float(off.sum(axis=0).max()) if off.nnz else 0.0
    s = math.sqrt(s_r * s_c)
    assert s < d
    return (d + s) / (d - s)


def gram_dense(L):
    """A = L~ L~^T as a dense C-contiguous float64 array (exact: integer entries far below 2^53)."""
    return np.ascontiguousarray((L @ L.T).toarray(), dtype=np.float64)


def feature_dim(n):
    return 1 << int(math.ceil(math.log2(n + PAD)))


class Exact:
    """The depth-1 pipeline problem of L~ and its exact answers (see the module docstring)."""

    def __init__(self, L, seed):
        self.L = L
        self.n = n = L.shape[0]
        self.D = feature_dim(n)
        rng = np.random.default_rng(seed)
        self.a = rng.integers(-3, 4, n).astype(np.float64)
        self.b = L.T @ self.a                        # integer
        self.y = (L @ self.b) / self.D               # integer / 2^k: exact
        self.colsum = np.asarray(abs(L).sum(axis=0)).ravel()   # sum_i |L~_ic|

    def x_train(self, rows=None):
        n = self.n if rows is None else rows
        coo = self.L.tocoo()
        m = coo.row < n
        x = np.zeros((n, self.D))
        x[coo.row[m], coo.col[m]] = coo.data[m]
        return x

    def queries(self, t, seed):
        """t query rows: u in [-3, 3]^N; odd rows also carry four +-512 entries in the padding columns."""
        rng = np.random.default_rng(seed)
        n, D = self.n, self.D
        x = np.zeros((t, D))
        x[:, :n] = rng.integers(-3, 4, (t, n))
        odd = np.arange(1, t, 2)
        for _ in range(4):
            x[odd, rng.integers(n, D, odd.size)] += rng.choice([-512.0, 512.0], odd.size)
        return x

    def answers(self, xq, rows=None):
        """Exact mean, var, K(x*, x*) and the scale sum_i |k*_i| of the queries against the first `rows` rows."""
        n = self.n if rows is None else rows
        u = xq[:, :n]
        mean = (u @ self.b[:n]) / self.D             # L~ lower triangular: b[:n] is the prefix problem's L~11^T alpha
        kss = np.einsum("ij,ij->i", xq, xq) / self.D
        var = kss - np.einsum("ij,ij->i", u, u) / self.D
        ksum = (np.abs(u) @ self.colsum[:n]) / self.D
        return mean, var, kss, ksum

    def lml(self, rows=None):
        n = self.n if rows is None else rows
        logdiag = np.log(self.L.diagonal()[:n]) - 0.5 * math.log(self.D)
        z2 = float(self.b[:n] @ self.b[:n]) / self.D
        return -0.5 * z2 - float(np.sum(logdiag)) - 0.5 * n * math.log(2 * math.pi), z2, float(np.sum(np.abs(logdiag)))


def exactness_report(L, ex=None, xq=None):
    """Largest magnitudes of every integer quantity the construction relies on (all must stay below 2^53)."""
    absL = abs(L)
    row1 = np.asarray(absL.sum(axis=1)).ravel()
    rep = {"gram": float(row1.max() ** 2)}           # any partial sum of a row dot product of L~
    if ex is not None:
        rep["b"] = float(np.max(absL.T @ np.abs(ex.a)))
        rep["y_num"] = float(np.max(absL @ (absL.T @ np.abs(ex.a))))
    if xq is not None:
        rep["query_dot"] = float(np.max(np.abs(xq[:, :ex.n]))) * float(row1.max())   # any partial sum of x* . x_i
        rep["query_sq"] = float(np.max(np.einsum("ij,ij->i", xq, xq)))
        rep["mean_num"] = float(np.max(np.abs(xq[:, :ex.n]) @ np.abs(ex.b)))
    return rep


# ---------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


def potrf_inplace(h, a):
    """nngp_diag_potrf on a (C-contiguous float64, overwritten: lower triangle = factor, upper left as it was)."""
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    h._ck(h._lib.nngp_diag_potrf(h._h, C.c_void_p(a.ctypes.data), a.shape[0]))


def lower_rows(a, r0, r1):
    return np.tril(a[r0:r1], k=r0)


def factor_error(a, L, scale=1.0, chunk=2048):
    """max |tril(a) - scale * L~| over row chunks (no dense N x N temporaries beyond one chunk)."""
    err = 0.0
    for r0 in range(0, L.shape[0], chunk):
        r1 = min(r0 + chunk, L.shape[0])
        err = max(err, float(np.max(np.abs(lower_rows(a, r0, r1) - scale * L[r0:r1].toarray()))))
    return err


def probe_residual(a, L, kappa, seed, chunk=2048):
    """(A - L^ L^^T) Z for 8 random columns against c N eps kappa |L^| |L^^T| |Z| (c = 2) plus the host's own
    rounding of the two products (2 N eps of the same quantity)."""
    n = L.shape[0]
    Z = np.random.default_rng(seed).standard_normal((n, 8))
    LtZ = np.zeros((n, 8)); aLtZ = np.zeros((n, 8))
    for r0 in range(0, n, chunk):
        r1 = min(r0 + chunk, n)
        blk = lower_rows(a, r0, r1)
        LtZ += blk.T @ Z[r0:r1]
        aLtZ += np.abs(blk).T @ np.abs(Z[r0:r1])
    worst = 0.0
    AZ = L @ (L.T @ Z)
    for r0 in range(0, n, chunk):
        r1 = min(r0 + chunk, n)
        blk = lower_rows(a, r0, r1)
        res = np.abs(AZ[r0:r1] - blk @ LtZ)
        bound = (2 * kappa + 2) * n * EPS * (np.abs(blk) @ aLtZ)
        worst = max(worst, float(np.max(res / bound)))
    return worst


# ---------------------------------------------------------------------------------------------- 1. factor
def _check_factor(lib, n, graded):
    L = lower_band(n, seed=n)
    kappa = cond_bound(L)
    a = gram_dense(L)
    h = lib.Handle()
    potrf_inplace(h, a)
    err = factor_error(a, L)
    tol = 2 * n * EPS * kappa * 16.0
    assert err <= tol, f"N={n}: max|L^ - L~| = {err:.3e} > {tol:.3e}"
    if n >= 4096:
        worst = probe_residual(a, L, kappa, seed=n)
        assert worst <= 1.0, f"N={n}: (A - L^ L^^T) Z reaches {worst:.3f} of its bound"
    if graded:
        e = np.random.default_rng(n + 1).integers(-20, 21, n)
        s = np.ldexp(1.0, e)
        ag = gram_dense(L)
        ag *= s[:, None]
        ag *= s[None, :]
        potrf_inplace(h, ag)
        for r0 in range(0, n, 2048):
            r1 = min(r0 + 2048, n)
            assert np.array_equal(lower_rows(ag, r0, r1), s[r0:r1, None] * lower_rows(a, r0, r1)), \
                f"N={n}: the factor of S A S is not S L^ bit for bit (rows {r0}..{r1})"


@pytest.mark.parametrize("n", W256_N + W512_N)
def test_factor_is_the_integer_factor(lib, n):
    """Families (a) and (b), W = 256 and 512: |L^ - L~| <= 2 N eps kappa max|L~|; for N >= 4096 also the backward
    error on 8 random probes; the graded matrix S A S factors to S L^ bit for bit."""
    _check_factor(lib, n, graded=True)


def test_factor_is_the_integer_factor_w1024(lib):
    """W = 1024 (N = 24641, look-ahead on, ragged last panel and last 64-block): family (a), sparse L~."""
    _check_factor(lib, W1024_N, graded=False)


# ---------------------------------------------------------------------------------------------- 2. error model
def _chol_longdouble(K):
    n = K.shape[0]
    L = np.zeros((n, n), dtype=np.longdouble)
    Kl = K.astype(np.longdouble)
    for j in range(n):
        v = Kl[j:, j] - L[j:, :j] @ L[j, :j]
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    return L


def _trsv_longdouble(L, b, lower):
    n = L.shape[0]
    x = np.zeros(n, dtype=np.longdouble)
    rng_ = range(n) if lower else range(n - 1, -1, -1)
    for i in rng_:
        if lower:
            x[i] = (b[i] - L[i, :i] @ x[:i]) / L[i, i]
        else:
            x[i] = (b[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
    return x


ILL_N = 1024 + 63   # W = 256, look-ahead on, last 64-block ragged (63 rows)


@pytest.mark.parametrize("where", ["first_block", "last_ragged_block", "later_panel", "spread"])
def test_error_model_of_the_explicit_inverses(lib, where):
    """Families (c) and (d) on a non-exact K = fl((sigma_w^2 / D) A), sigma_w^2 ~ 1/3, lambda = 0.

    Reference: factor and alpha in long double.  Asserted:
      backward error  ||K - L^ L^^T||_F <= 16 eps (max_J cond_2(L_JJ) + N) ||K||_F  -- the explicit inverses cost
                      eps cond(L_JJ) (DESIGN.md 5.2); N is the classical floor of any Cholesky factorisation;
      alpha           max|alpha^ - alpha| <= 4 (LAPACK's max|alpha - alpha|) + 16 N eps, relative to max|alpha|.
    (A floor of 16 N eps cond(K) would exceed 1 here -- cond(K) ~ 1e12 -- and make the second check vacuous.)"""
    if np.finfo(np.longdouble).eps > 1e-18:
        pytest.skip("long double is not wider than double on this platform")
    n = ILL_N
    base = lower_band(n, seed=7)
    if where == "first_block":
        idx = np.arange(0, 64)
    elif where == "last_ragged_block":
        idx = np.arange(1024, n)
    elif where == "later_panel":
        idx = np.arange(512, 576)            # first block of the third W = 256 panel
    else:
        idx = np.sort(np.random.default_rng(3).choice(n, 64, replace=False))
    L = with_chain(base, idx)
    D = feature_dim(n)
    sw = 3.0 ** -0.5
    scale = (sw * sw) / D                    # the Gram's scale, as the library forms it
    K = scale * gram_dense(L)                # = what the depth-1 Gram produces, entry for entry
    ex = Exact(L, seed=11)
    y = K @ ex.a
    h = lib.Handle(depth=1, sigma_w=sw, sigma_b=0.0, diag_reg=0.0)
    h.fit(ex.x_train(), y)
    st = h.get_state(x=False)
    Lg, ag = st["l"], st["alpha"]
    Lr = _chol_longdouble(K)
    ar = _trsv_longdouble(Lr, _trsv_longdouble(Lr, y.astype(np.longdouble), True), False)
    conds = [np.linalg.cond(np.asarray(Lr[j:j + 64, j:j + 64], dtype=np.float64)) for j in range(0, n, 64)]
    cmax = max(conds)
    Kl = K.astype(np.longdouble)
    Lgl = Lg.astype(np.longdouble)
    bwd = float(np.linalg.norm(np.asarray(Kl - Lgl @ Lgl.T, dtype=np.float64)) / np.linalg.norm(K))
    Ll = sla.cholesky(K, lower=True)
    bwd_lapack = float(np.linalg.norm(np.asarray(Kl - Ll.astype(np.longdouble) @ Ll.astype(np.longdouble).T,
                                                 dtype=np.float64)) / np.linalg.norm(K))
    al = sla.cho_solve((Ll, True), y)
    arf = np.asarray(ar, dtype=np.float64)
    amax = float(np.max(np.abs(arf)))
    fwd = float(np.max(np.abs(np.asarray(ag.astype(np.longdouble) - ar, dtype=np.float64)))) / amax
    fwd_lapack = float(np.max(np.abs(np.asarray(al.astype(np.longdouble) - ar, dtype=np.float64)))) / amax
    print(f"\n[{where}] N={n} max cond(L_JJ)={cmax:.3e} (block {int(np.argmax(conds))}) cond(K)={np.linalg.cond(K):.2e} "
          f"backward GPU {bwd:.2e} LAPACK {bwd_lapack:.2e} | alpha forward GPU {fwd:.2e} LAPACK {fwd_lapack:.2e}")
    assert bwd <= 16 * EPS * (cmax + n), (bwd, cmax)
    assert fwd <= 4 * fwd_lapack + 16 * n * EPS, (fwd, fwd_lapack)


# ---------------------------------------------------------------------------------------------- 3. pivots
PIVOTS = {300: [0, 1, 3, 4, 63, 64, 127, 128, 255, 256, 299],
          4200: [0, 1, 3, 4, 63, 64, 127, 128, 255, 256, 511, 512, 4199]}


@pytest.mark.parametrize("n", sorted(PIVOTS))
def test_non_positive_pivot_is_reported_at_its_index(lib, n):
    """A = L~ L~^T - (L~_pp^2 + 1) e_p e_p^T: leading minors positive up to p, pivot p = -1 in exact arithmetic.
    nngp_diag_potrf must report pivot p (LAPACK's info - 1), and the same handle must then factor a good matrix of
    another size exactly.  The fit path: a zero training row p makes pivot p of K exactly 0 (lambda = 0)."""
    L = lower_band(n, seed=n + 5)
    A = gram_dense(L)
    good = lower_band(n - 37, seed=n + 6)
    good_A = gram_dense(good)
    gtol = 2 * (n - 37) * EPS * cond_bound(good) * 16.0
    h = lib.Handle()
    for p in PIVOTS[n]:
        a = A.copy()
        a[p, p] -= L[p, p] ** 2 + 1.0
        assert sla.lapack.dpotrf(a.copy(), lower=1)[1] == p + 1
        with pytest.raises(np.linalg.LinAlgError, match=rf"pivot {p}\)"):
            potrf_inplace(h, a)
        g = good_A.copy()
        potrf_inplace(h, g)
        assert factor_error(g, good) <= gtol, f"after the failure at pivot {p}"
    ex = Exact(L, seed=1)
    exg = Exact(good, seed=2)
    X = ex.x_train()
    hf = lib.Handle(depth=1, sigma_w=1.0, sigma_b=0.0, diag_reg=0.0)
    for p in PIVOTS[n]:
        row = X[p].copy()
        X[p] = 0.0
        with pytest.raises(np.linalg.LinAlgError, match=rf"pivot {p} of {n}\b"):
            hf.fit(X, ex.y)
        X[p] = row
    hf.fit(exg.x_train(), exg.y)
    kappa = cond_bound(good)
    assert np.max(np.abs(hf.get_state(x=False, l=False)["alpha"] - exg.a)) <= 4 * good.shape[0] * EPS * kappa ** 2 * 3


# ---------------------------------------------------------------------------------------------- 4. fit + predict
def _check_fit(h, ex, kappa, rows=None, what=""):
    n = ex.n if rows is None else rows
    st = h.get_state(x=False)
    assert h.dims()[0] == n
    ltol = 2 * n * EPS * kappa * 16.0 / math.sqrt(ex.D)
    Lsub = ex.L[:n, :n]
    err = factor_error(st["l"], Lsub, scale=1.0 / math.sqrt(ex.D))
    assert err <= ltol, f"{what}: max|L^ - L~/sqrt(D)| = {err:.3e} > {ltol:.3e}"
    if rows is None or rows == ex.n:
        aref = ex.a
    else:  # prefix problem: alpha = L~11^-T b[:n] (host substitution in FP64, kappa-conditioned)
        aref = sla.solve_triangular(Lsub.toarray(), ex.b[:n], lower=True, trans="T")
    atol = 4 * n * EPS * kappa ** 2 * max(3.0, float(np.max(np.abs(aref))))
    aerr = float(np.max(np.abs(st["alpha"] - aref)))
    assert aerr <= atol, f"{what}: max|alpha^ - alpha| = {aerr:.3e} > {atol:.3e}"
    lml, z2, slog = ex.lml(rows)
    lerr = abs(h.log_marginal_likelihood() - lml)
    assert lerr <= 4 * n * EPS * kappa ** 2 * (0.5 * z2 + slog + n), f"{what}: LML off by {lerr:.3e}"


def _check_pred(h, ex, kappa, xq, what, rows=None, var_kappa=1, var_abs=0.0):
    n = ex.n if rows is None else rows
    mean, var = h.predict(xq)
    m_ex, v_ex, kss, ksum = ex.answers(xq, rows)
    mtol = 4 * n * EPS * kappa ** 2 * 3.0 * ksum + 1e-300
    vtol = 4 * n * EPS * kappa ** var_kappa * kss + var_abs * kss
    bad_m = np.abs(mean - m_ex) > mtol
    bad_v = np.abs(var - v_ex) > vtol
    assert not bad_m.any(), f"{what}: mean row {int(np.argmax(bad_m))}: {mean[bad_m][0]!r} vs exact {m_ex[bad_m][0]!r}"
    assert not bad_v.any(), f"{what}: var row {int(np.argmax(bad_v))}: {var[bad_v][0]!r} vs exact {v_ex[bad_v][0]!r}"


def _handle(lib, **kw):
    return lib.Handle(depth=1, sigma_w=1.0, sigma_b=0.0, diag_reg=0.0, **kw)


@pytest.mark.parametrize("n", W256_N + W512_N)
def test_fit_and_every_prediction_path_against_the_exact_answers(lib, n, monkeypatch):
    """Family (a).  L, alpha, LML, mean and var of:
      the persistent solve -- PIPE (1 and 300 rows); at N = 65 and 257 also the static schedule (296 row tiles) and the
        ungated kernel (370 row tiles);
      the right-looking steps (NNGP_SMALL_BATCH_TILES) with 200 rows (OW = 64) and 700 rows (OW = 256);
      latency mode with 1, 2, 3, 4, 5, 8 rows (tri_gemv<1, 2, 4, 8>), 100 rows (split K), 2000 rows (tiled row-dot
        where N >= 2300) and past NNGP_LATENCY_ROWS;
      a state imported with set_state (inverses recomputed by trtri_diag_kernel);
      variance_slices = 7 (1000 rows), within the header's 1e-8 of K(x*, x*) for the int8 variance product;
      'ntk' at depth 1, where Theta = K and M = I: the NNGP posterior."""
    L = lower_band(n, seed=n + 100)
    kappa = cond_bound(L)
    ex = Exact(L, seed=n)
    big = n in (65, 257)
    t_max = 47360 if big else 2000
    xq = ex.queries(t_max, seed=n + 1)
    X = ex.x_train()

    h = _handle(lib)
    h.fit(X, ex.y)
    _check_fit(h, ex, kappa, what="fit")
    for t in (1, 300):
        _check_pred(h, ex, kappa, xq[:t], f"persistent PIPE, {t} rows")
    if big:
        _check_pred(h, ex, kappa, xq[:296 * 128], "persistent, static schedule")
        _check_pred(h, ex, kappa, xq[:370 * 128], "persistent, ungated")
    monkeypatch.setenv("NNGP_SMALL_BATCH_TILES", "1000000")
    for t in (200, 700):
        _check_pred(h, ex, kappa, xq[:t], f"right-looking, {t} rows")
    monkeypatch.delenv("NNGP_SMALL_BATCH_TILES")

    st = h.get_state()
    imp = _handle(lib)
    imp.set_state(st["x"], st["l"], st["alpha"], st["lambda"])
    _check_pred(imp, ex, kappa, xq[:300], "imported state")
    del imp, st

    lat = _handle(lib, latency_mode=True)
    lat.fit(X, ex.y)
    for t in (1, 2, 3, 4, 5, 8, 100, 2000):
        _check_pred(lat, ex, kappa, xq[:t], f"latency mode, {t} rows")
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "4")
    _check_pred(lat, ex, kappa, xq[:5], "latency mode past NNGP_LATENCY_ROWS")
    monkeypatch.delenv("NNGP_LATENCY_ROWS")
    del lat

    sl = _handle(lib, variance_slices=7)
    sl.fit(X, ex.y)
    _check_pred(sl, ex, kappa, xq[:1000], "variance_slices=7", var_abs=1e-8)
    assert sl.stats()["sliced_macs"] > 0
    del sl

    ntk = _handle(lib, kernel_type="ntk")
    ntk.fit(X, ex.y)
    _check_pred(ntk, ex, kappa, xq[:300], "ntk depth 1", var_kappa=2)


def test_fit_and_predict_w1024(lib):
    """N = 24641 (W = 1024, look-ahead on), D = 32768: L, alpha, LML and the persistent solve's mean and var."""
    n = W1024_N
    L = lower_band(n, seed=n + 100)
    kappa = cond_bound(L)
    ex = Exact(L, seed=n)
    h = _handle(lib)
    X = ex.x_train()
    h.fit(X, ex.y)
    del X
    _check_fit(h, ex, kappa, what="fit W=1024")
    _check_pred(h, ex, kappa, ex.queries(300, seed=n + 1), "persistent, 300 rows")


# ---------------------------------------------------------------------------------------------- 5. append
@pytest.mark.parametrize("n0,steps", [(998, [130, 63, 1, 1, 2]), (1000, [4100])])
def test_incremental_append_is_exact(lib, n0, steps):
    """diag_reg = 0 absolute: fit the first n0 rows of L~, append the next ones.  The leading block of L~ L~^T is
    L~11 L~11^T, so after every append the factor is again L~/sqrt(D) over the rows so far, z = b[:N]/sqrt(D), and the
    posterior of a query is exact (mean u[:N] . b[:N] / D, var (|u[N:]|^2 + |w|^2)/D).
    998 + 130: Schur block off the 64-grid; + 63 leaves N odd, so the next one-row append refits; + 1 from an even N
    leaves N odd again; 1000 + 4100: the Schur Cholesky runs at W = 512."""
    n_tot = n0 + sum(steps)
    L = lower_band(n_tot, seed=n_tot)
    kappa = cond_bound(L)
    ex = Exact(L, seed=n0)
    X = ex.x_train()
    xq = ex.queries(300, seed=n0 + 1)
    h = _handle(lib, diag_reg_absolute=True)
    h.fit(X[:n0], ex.y[:n0])
    _check_fit(h, ex, kappa, rows=n0, what=f"fit {n0}")
    n = n0
    for m in steps:
        h.append_fit(X[n:n + m], ex.y[n:n + m])
        n += m
        _check_fit(h, ex, kappa, rows=n, what=f"append to {n}")
        _check_pred(h, ex, kappa, xq, f"after append to {n}", rows=n)
