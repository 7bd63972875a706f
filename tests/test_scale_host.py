"""CPU: the references the scale-equivariance and digit-plane GPU tests judge against, checked where they are used --
the window of scales inside which every intermediate stays a normal double, and the digit-plane restatement of rows at
and below the bottom of the normal range (rebuilt exactly with fractions)."""
import math
from fractions import Fraction

import numpy as np
import pytest

from test_gpu_scale_equivariance import _window
from test_gpu_sliced import TINY_ROWS, _set_tiny_rows, _split_rows


def test_window_on_a_hand_built_case():
    # K-like part (x 4^a): 2^-10 .. 4 must stay in [2^(-1022+20), 2^(1024-20)): -10 + 2a >= -1002, 2 + 2a <= 1003
    assert _window([(np.array([2.0 ** -10, 0.0, -4.0]), 2)]) == (-496, 500)
    # an inverse-like part (x 2^-a) bounds the other side: 3 - a <= 1003 -> a >= -1000; -30 - a >= -1002 -> a <= 972
    assert _window([(np.array([2.0 ** -30, 8.0]), -1)]) == (-1000, 972)
    # a q-like part with its own top (2^512) and a product part (x 16^a): the tightest edge of each side wins
    lo, hi = _window([(np.array([0.5, 2.0]), 2, 512), (np.array([0.25, 4.0]), 4)])
    assert (lo, hi) == (-250, 245)        # -2 + 4a >= -1002 (q q'), 1 + 2a <= 491 (q below 2^(512-20))
    assert _window([(np.array([0.5, 2.0]), 2, 512)]) == (-500, 245)
    # a scale-free part outside the range: empty window; zeros and an all-zero part do not constrain
    lo, hi = _window([(np.array([2.0 ** -1010]), 0)])
    assert lo > hi
    assert _window([(np.zeros(3), 2), (np.array([1.0]), 2)]) == (-501, 501)
    # margin 1: the plain normal range, 2^-1022 .. 2^1023 (a value of [1, 2) times 2^1024 overflows)
    assert _window([(np.array([1.0]), 1)], margin=1.0) == (-1022, 1023)
    assert _window([(np.array([1.5]), 1)], margin=1.0) == (-1022, 1023)


@pytest.mark.parametrize("s", [5, 7, 9])
def test_digit_planes_rebuild_tiny_rows_exactly(s):
    """Rows whose largest magnitude is 2^-1017 .. 2^-1074 (and normal rows beside them): every digit is an integer of
    magnitude <= 64, the exponent bounds the row (|a| < 2^e), and sum_p d_p 2^(e-6-7p), summed exactly, is within
    2^(e-7s) of every entry -- the rounding residue of the last plane; exact once the planes hold all the row's bits."""
    rng = np.random.default_rng(s)
    a = rng.normal(size=(10, 24)) * np.exp(3 * rng.normal(size=(10, 1)))
    a[9] = 0.0
    _set_tiny_rows(a, rng, 2)
    planes, e = _split_rows(a, s)
    assert [int(v) for v in e[2:2 + len(TINY_ROWS)]] == [t + 1 for t in TINY_ROWS]   # max = 2^t exactly -> e = t + 1
    assert e[9] == 0
    for p in planes:
        assert np.all(p == np.rint(p)) and np.all(np.abs(p) <= 64)
    for r in range(a.shape[0]):
        if e[r] == 0 and not np.any(a[r]):
            assert all(not np.any(p[r]) for p in planes)
            continue
        assert np.max(np.abs(a[r])) < 2.0 ** float(e[r])
        for c in range(a.shape[1]):
            rebuilt = sum(Fraction(int(planes[p][r, c])) * Fraction(2) ** int(e[r] - 6 - 7 * p) for p in range(s))
            err = abs(rebuilt - Fraction(a[r, c]))
            assert err <= Fraction(2) ** int(e[r] - 7 * s), (r, c)
            if e[r] - 6 - 7 * (s - 1) <= -1074:
                assert err == 0, (r, c)       # the last plane's unit is at or below 2^-1074: every bit is held
