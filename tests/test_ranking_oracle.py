"""CPU checks of the ranking restatement (tests/ranking_oracle.py): the f64 FFT correlation against the oracle's
time-domain correlators, the f32 selection, and an emulation of one packed ranking transform showing that two planes
of very different power must be scaled to unit power before they share a transform."""
import numpy as np
import pytest

from oracle import oracle
import lag_edges as E
import ranking_oracle as R


def test_fft_statement_equals_the_oracle_correlators():
    """exact_extended / exact_binary (an f64 FFT) against xcorr_two_sided / tdcorr_binary_lags_mt (time domain)."""
    rng = np.random.default_rng(4)
    y = [(rng.standard_normal(30000) + 1j * rng.standard_normal(30000)).astype(np.complex64) for _ in range(2)]
    L = 1500
    assert np.max(np.abs(R.exact_extended(y[0], y[1], L) - oracle.xcorr_two_sided(y[0], y[1], L))) <= 1e-12
    yj = y[1][:27001]   # unequal lengths: W = 27001, signal 0 the template
    assert np.max(np.abs(R.exact_extended(y[0], yj, L) - E.unequal_statement(y[0], yj, L))) <= 1e-12
    want = oracle.tdcorr_binary_lags_mt(y[0], y[1], y[0].size - 2000, 2000)
    # BINARY rounds every product to f32: the f64 plane is within 1e-9, the one-lag statement bit-near
    assert np.max(np.abs(R.exact_binary(y[0], y[1], 2000, 10000) - want)) <= 1e-9
    for lag in (0, 1, 777, 1999):
        assert abs(R.binary_at(y[0], y[1], 2000, 10000, lag) - want[lag]) <= 1e-12


def test_select_is_f32_arithmetic():
    """A lag exactly one f32 ulp under the threshold is out, one on it is in (f64 would round both alike)."""
    m = np.float32(0.75)
    thr = np.float32(m - np.float32(E.TOL))
    a = np.array([m, thr, np.nextafter(thr, np.float32(0)), 0.1], np.float32)
    assert R.select(a).tolist() == [0, 1]
    assert R.select(a, neighbours=True).tolist() == [0, 1, 2]


def test_margin_statement():
    a = np.array([0.1, -0.9, 0.5, 0.45], np.float32)
    assert R.margin(a, 1, -0.9) == np.float32((0.9 - np.float64(np.float32(0.5))) / 0.9)
    assert R.margin(a, 1, 0.0) == 0.0


def packed_errors(ratio, prescale, seed=0, n_seg=40):
    rng = np.random.default_rng(seed)
    n = 6144 * n_seg
    t = rng.standard_normal(n).astype(np.float32)
    s = (rng.standard_normal(n + 8192) * np.sqrt(ratio)).astype(np.float32)
    sc = 1.0 / np.sqrt(np.mean(t.astype(np.float64) ** 2) * np.mean(s.astype(np.float64) ** 2))
    exact = R.correlate(t, s, n, 2048) / n * sc
    return float(np.max(np.abs(R.emulate_packed(t, s, 2048, 6144, prescale=prescale) - exact)))


def test_packed_transform_error_grows_with_the_power_ratio():
    """Raw planes: each split spectrum carries rounding on the scale of the other plane, so the error in
    correlation units grows like sqrt(P_s / P_t) -- above the selection tolerance at a ratio of 1e8."""
    err = {r: packed_errors(r, False) for r in (1.0, 1e4, 1e8)}
    assert err[1.0] < 1e-7
    assert 20 < err[1e4] / err[1.0] < 500                 # sqrt(1e4) = 100
    assert 20 < err[1e8] / err[1e4] < 500
    assert err[1e8] > E.TOL


@pytest.mark.parametrize("ratio", [1.0, 1e4, 1e6, 1e8, 1e12])
def test_packed_transform_bounded_when_planes_are_prescaled(ratio):
    assert packed_errors(ratio, True, seed=1) < 1e-7
