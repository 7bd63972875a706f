"""GPU: nngp_reserve keeps its promise, and every way of installing a fitted state checks X as a fit does.

After nngp_reserve(N_max, D, T_max) an active-learning loop (fit, predict, select, append up to N_max) makes no device
allocation at all (nngp_stats_t.device_allocs), on every handle configuration, and computes bit for bit what an
unreserved handle computes.  nngp_set_state and the packed import reject a non-finite or out-of-range X with
NNGP_EINVAL and leave the handle usable; an imported state carries no labels."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

D, N0, N_MAX, T_MAX = 24, 3000, 4200, 1500
APPENDS = (1101, 1, 98)   # 3000 -> 4101 (crosses W = 256 -> 512 at 4096) -> 4102 (from odd N: a refit) -> 4200


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


@pytest.fixture(scope="module")
def synth():
    from nngp_b200 import synth as s
    return s


def _n_gpus():
    import torch
    return torch.cuda.device_count()


HANDLES = {
    "default": {},
    "incremental": dict(diag_reg=50.0, diag_reg_absolute=True),
    "latency": dict(latency_mode=True),
    "sliced": dict(variance_slices=7),
    "ntk": dict(kernel_type="ntk"),
    "default_2gpu": dict(n_gpus=2),
    "latency_2gpu": dict(latency_mode=True, n_gpus=2),
}


def _loop(h, xtr, ytr, xpool, ypool):
    """fit at N0, predict / select at up to T_MAX rows, append up to N_MAX, predict again: every output, in order"""
    out = []
    h.fit(xtr, ytr)
    out += h.predict(xpool)                           # above NNGP_LATENCY_ROWS: persistent solve / digit planes
    out.append(h.predict(xpool, want_var=False)[0])
    for rows in (5, 300):                             # latency mode: the explicit inverse (tri_gemv, then GEMM)
        out += h.predict(xpool[:rows])
    out.append(h.active_select(xpool, 40))
    n = N0
    for m in APPENDS:
        h.append_fit(xpool[n - N0:n - N0 + m], ypool[n - N0:n - N0 + m])
        n += m
    assert h.dims()[0] == N_MAX
    out += h.predict(xpool)
    out += h.predict(xpool[:5])
    return out


@pytest.mark.parametrize("name", list(HANDLES))
def test_reserved_loop_allocates_nothing_and_matches_unreserved(lib, synth, name, monkeypatch):
    kw = HANDLES[name]
    if kw.get("n_gpus", 1) > _n_gpus():
        pytest.skip(f"needs >= {kw['n_gpus']} GPUs")
    monkeypatch.setenv("NNGP_LATENCY_ROWS", "600")
    xtr, ytr, xpool, ypool = synth.make_problem(N0, T_MAX, D)
    h = lib.Handle(**kw)
    h.reserve(N_MAX, D, T_MAX)
    h.stats_reset()
    got = _loop(h, xtr, ytr, xpool, ypool)
    assert h.stats()["device_allocs"] == 0

    ref = lib.Handle(**kw)                            # the same loop without nngp_reserve
    ref.stats_reset()
    want = _loop(ref, xtr, ytr, xpool, ypool)
    assert ref.stats()["device_allocs"] > 0
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), i

    if not kw.get("diag_reg_absolute"):               # every append refits: the final model is a fresh fit's
        fresh = lib.Handle(**kw)
        fresh.fit(np.vstack([xtr, xpool[:N_MAX - N0]]), np.concatenate([ytr, ypool[:N_MAX - N0]]))
        m, v = fresh.predict(xpool)
        assert np.array_equal(got[-4], m) and np.array_equal(got[-3], v)


def _bad_inputs(x):
    nan = x.copy()
    nan[7, 3] = np.nan
    big = x.copy()
    big[11] *= 2.0 ** 300                             # layer-0 diagonal ~ 2^600 >= 2^512
    return {"nan": nan, "out_of_range": big}


def _packed(h):
    flat = np.empty(h.packed_size())
    h.state_pack(0, flat.size, flat)
    return flat


def _import_packed(h, flat, n, d, lam):
    h.state_import_begin(n, d)
    h.state_unpack(0, flat.size, flat)
    h.state_import_end(lam)


@pytest.mark.parametrize("how", ["set_state", "packed"])
def test_import_rejects_bad_x_and_leaves_the_handle_usable(lib, synth, how):
    xtr, ytr, xte, _ = synth.make_problem(500, 200, D)
    src = lib.Handle()
    src.fit(xtr, ytr)
    st, flat = src.get_state(), _packed(src)
    n, d, lam = src.dims()
    want = src.predict(xte)
    for kind, xbad in _bad_inputs(st["x"]).items():
        h = lib.Handle()
        with pytest.raises(ValueError, match="non-finite" if kind == "nan" else "out of range"):
            if how == "set_state":
                h.set_state(xbad, st["l"], st["alpha"], lam)
            else:
                bad = flat.copy()
                bad[:n * d] = xbad.ravel()
                _import_packed(h, bad, n, d, lam)
        with pytest.raises(lib.NngpError) as e:       # no fitted model
            h.dims()
        assert e.value.code == lib.NNGP_ESTATE
        h.fit(xtr, ytr)
        m, v = h.predict(xte)
        assert np.array_equal(m, want[0]) and np.array_equal(v, want[1]), kind


@pytest.mark.parametrize("how", ["set_state", "packed"])
def test_imported_state_has_no_labels_and_builds_the_inverse(lib, synth, how):
    xtr, ytr, xte, yte = synth.make_problem(700, 100, D)
    src = lib.Handle(latency_mode=True)
    src.fit(xtr, ytr)
    st, flat = src.get_state(), _packed(src)
    n, d, lam = src.dims()
    h = lib.Handle(latency_mode=True)
    h.stats_reset()
    if how == "set_state":
        h.set_state(st["x"], st["l"], st["alpha"], lam)
    else:
        _import_packed(h, flat, n, d, lam)
    assert h.stats()["inverse_ms"] > 0
    for call in (h.log_marginal_likelihood, lambda: h.append_fit(xte[:3], yte[:3])):
        with pytest.raises(lib.NngpError) as e:
            call()
        assert e.value.code == lib.NNGP_ESTATE
    m, v = h.predict(xte)
    m0, v0 = src.predict(xte)
    assert np.array_equal(m, m0) and np.array_equal(v, v0)
