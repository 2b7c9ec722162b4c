"""The numpy oracle's filters against scipy itself, at the configurations the kernel-path tests drive the device with:
zero-phase Butterworth of orders 1-16 (every compiled section count of the kernels) on records from the shortest one
that is filtered (padlen + 1) up, and Savitzky-Golay windows 3-31 including windows longer than the record, even
windows and windows that leave the record unchanged.  The GPU tests rest on the oracle; this pins the oracle.

scipy fits the SG edge polynomial in float32 (the oracle and the kernel in float64), so the edges agree to the suite's
float bar, not bit for bit; that float32 noise grows with the polynomial degree (degree 5 over 25-31 samples leaves the
bar at 8 k-count samples), so the windows here go up to degree 4, as the device tests do."""

import numpy as np
import pytest

from conftest import ATOL, RTOL

scipy_signal = pytest.importorskip("scipy.signal")

BANDS = ((0.01, 0.1, 0.5), (0.02, 0.2, 1.0), (0.05, 0.06, 0.5), (0.001, 0.45, 1.0))


def _rows(rng, n, L):
    """float32 rows like a wave_pool: a 14-bit baseline, noise and one negative pulse per row."""
    t = np.arange(L)
    x = 8000.0 + rng.normal(0, 3, size=(n, L))
    at = rng.integers(0, max(L, 1), size=n)
    x -= rng.uniform(50, 3000, size=(n, 1)) * np.exp(-np.abs(t[None, :] - at[:, None]) / 4.0)
    return np.round(x).astype(np.float32)


@pytest.mark.parametrize("order", list(range(1, 17)))
def test_bw_filter_rows_is_sosfiltfilt(order):
    from oracle import np_oracle as O

    rng = np.random.default_rng(1000 + order)
    lo, hi, fs = BANDS[order % len(BANDS)]
    sos = scipy_signal.butter(order, [lo, hi], btype="band", output="sos", fs=fs)
    pad = O.bw_padlen(sos)
    for L in (pad + 1, pad + 2, pad + 17, 2 * pad + 33, 800):
        X = _rows(rng, 6, L)
        want = scipy_signal.sosfiltfilt(sos, X, axis=-1, padlen=pad).astype(np.float32)
        got = O.bw_filter_rows(X, sos)
        assert got.dtype == np.float32
        assert np.array_equal(got, want), f"order {order} L {L}: {np.count_nonzero(got != want)} samples differ"
    X = _rows(rng, 3, pad)  # not longer than the padding: unfiltered, as the reference does
    assert np.array_equal(O.bw_filter_rows(X, sos), X)


@pytest.mark.parametrize("window,poly", [(3, 1), (5, 2), (7, 3), (9, 2), (11, 2), (15, 4), (21, 3), (25, 4), (31, 3), (10, 2), (4, 3)])
def test_sg_filter_rows_is_savgol_interp(window, poly):
    from oracle import np_oracle as O

    rng = np.random.default_rng(window * 100 + poly)
    for L in (1, 2, 3, 4, 5, 7, 8, 15, 16, 31, 32, 33, 100):
        X = _rows(rng, 5, L)
        got = O.sg_filter_rows(X, window, poly)
        w = O.effective_sg_window(L, window, poly)
        if w is None:  # window <= poly: the record is left unchanged
            assert np.array_equal(got, X), (window, poly, L)
            continue
        want = scipy_signal.savgol_filter(X, w, poly, mode="interp", axis=-1).astype(np.float32)
        h = w // 2
        assert np.array_equal(got[:, h:L - h], want[:, h:L - h]), f"interior differs: window {window} poly {poly} L {L}"
        assert np.allclose(got, want, rtol=RTOL, atol=ATOL), f"edges: window {window} poly {poly} L {L}"
