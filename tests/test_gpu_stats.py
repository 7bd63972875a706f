"""GPU: the nngp_stats_t contract.

One fixed call sequence (fit, predict of a large and a small batch, predict without variance, predict_cov, kernel,
append_fit, set_state) runs at stats_level 0, 1 and 2 on every handle configuration.  The level decides which device
times are recorded (include/nngp_b200.h) and nothing else: every counter comes out the same at all three levels."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, T, D, T_SMALL, T_COV, M_APPEND = 1500, 1300, 24, 5, 600, 37

HANDLES = {
    "default": {},
    "ntk": dict(kernel_type="ntk"),
    "latency": dict(latency_mode=True),
    "sliced": dict(variance_slices=7),
    "absolute_append": dict(diag_reg=50.0, diag_reg_absolute=True),   # even N: the incremental append
    "2gpu": dict(n_gpus=2),
}

# the lowest stats_level at which each device time is recorded
TIME_LEVEL = {**{f: 1 for f in ("fit_gram_ms", "fit_chol_ms", "fit_solve_ms", "fit_total_ms", "pred_gram_ms",
                                "pred_trsm_ms", "pred_var_ms", "pred_total_ms", "h2d_ms", "d2h_ms")},
              "gemm_ms": 2, "gram_ms": 2, "sliced_ms": 0, "inverse_ms": 0, "replicate_ms": 0}
COUNTERS = ("gemm_flops", "gemm_launches", "gram_flops", "gram_evals", "gram_launches", "kernel_launches", "h2d_bytes",
            "d2h_bytes", "queries", "replicate_bytes", "sliced_macs", "device_allocs")


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def _ran(field, kw):
    """Whether the sequence runs the path that fills a time field, on a handle made with `kw`."""
    if field == "sliced_ms":
        return bool(kw.get("variance_slices"))
    if field == "inverse_ms":
        return bool(kw.get("latency_mode") or kw.get("variance_slices"))
    if field == "replicate_ms":
        return kw.get("n_gpus", 1) > 1
    return True


def run_sequence(lib, synth, kw, level):
    """The call sequence on a new handle: [(step, stats after it)], and the stats around a NaN predict and around a
    call rejected before any GPU work."""
    xtr, ytr, xte, yte = synth.make_problem(N, T + M_APPEND, D)
    xa, ya = xte[T:], yte[T:]
    xte = xte[:T]
    h = lib.Handle(stats_level=level, **kw)
    steps = [
        ("fit", lambda: h.fit(xtr, ytr)),
        ("predict", lambda: h.predict(xte)),
        ("predict_small", lambda: h.predict(xte[:T_SMALL])),
        ("predict_mean", lambda: h.predict(xte, want_var=False)),
        ("predict_cov", lambda: h.predict_cov(xte[:T_COV])),
        ("kernel", lambda: h.kernel(xte[:T_COV])),
        ("append_fit", lambda: h.append_fit(xa, ya)),
    ]
    out = []
    for name, call in steps:
        call()
        out.append((name, h.stats()))
    st = h.get_state()
    h.set_state(st["x"], st["l"], st["alpha"], st["lambda"], m=st.get("m"))
    out.append(("set_state", h.stats()))

    bad = xte.copy()
    bad[0, 3] = np.nan
    with pytest.raises(ValueError, match="non-finite value in x_test"):
        h.predict(bad)
    nan = (out[-1][1], h.stats())

    before = h.stats()
    with pytest.raises(lib.NngpError) as e:          # an imported state has no labels to append to
        h.append_fit(xa, ya)
    assert e.value.code == lib.NNGP_ESTATE
    rejected = (before, h.stats())
    h.close()
    return out, nan, rejected


@pytest.fixture(scope="module")
def lib():
    from nngp_b200 import _lib
    _lib.load()
    return _lib


@pytest.fixture(scope="module")
def synth():
    from nngp_b200 import synth as s
    return s


@pytest.mark.parametrize("name", list(HANDLES))
def test_stats_level_changes_only_which_times_are_recorded(lib, synth, name):
    kw = HANDLES[name]
    if kw.get("n_gpus", 1) > _n_gpus():
        pytest.skip(f"needs >= {kw['n_gpus']} GPUs")
    runs = {level: run_sequence(lib, synth, kw, level) for level in (0, 1, 2)}

    for level, (out, nan, rejected) in runs.items():
        assert [s for s, _ in out] == [s for s, _ in runs[0][0]]
        for (step, st), (_, st0) in zip(out, runs[0][0]):
            assert {c: st[c] for c in COUNTERS} == {c: st0[c] for c in COUNTERS}, (level, step)
            assert st["pred_mean_ms"] == 0.0, (level, step)
        final = out[-1][1]
        for field, lowest in TIME_LEVEL.items():
            if level >= lowest and _ran(field, kw):
                assert final[field] > 0, (level, field)
            else:
                assert final[field] == 0, (level, field)

        # a NaN in x_test: ValueError, after the GPU work of the call -- its stage times are added, its rows are not
        # counted as predicted
        pre, post = nan
        assert post["queries"] == pre["queries"] and post["kernel_launches"] > pre["kernel_launches"]
        for field in ("pred_gram_ms", "pred_trsm_ms", "pred_total_ms", "d2h_ms"):
            assert (post[field] > pre[field]) if level >= 1 else (post[field] == 0), (level, field)

        assert rejected[0] == rejected[1], level
    assert {c: runs[0][1][1][c] for c in COUNTERS} == {c: runs[2][1][1][c] for c in COUNTERS}

    if name == "default":    # closed forms of the flop counters on the default path
        out = runs[2][0]
        delta = {step: {c: st[c] - prev[c] for c in ("gemm_flops", "gram_flops")}
                 for (step, st), (_, prev) in zip(out[1:], out)}
        delta["fit"] = {c: out[0][1][c] for c in ("gemm_flops", "gram_flops")}
        assert delta["fit"]["gram_flops"] == N * N * D
        for step, rows, var in (("predict", T, True), ("predict_small", T_SMALL, True), ("predict_mean", T, False)):
            assert delta[step] == {"gemm_flops": rows * N * N if var else 0, "gram_flops": 2 * rows * N * D}, step
