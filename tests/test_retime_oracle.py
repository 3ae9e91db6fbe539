"""CPU checks of the re-timing restatement (tests/retime_oracle.py): the station-rate fit, the index delta(n), and
what re-timing is for -- on drifting captures built as tests/test_gpu_windows.py builds them, re-timing each
station's whole TGT block by its true clock rate puts every pair's correlation peak on its window-centre lag."""
import math

import numpy as np
import pytest

import retime_oracle as RO
from oracle import oracle
from test_gpu_windows import ST4, drift_captures


def test_rates_recover_station_clocks_exactly():
    S = 6
    g = np.random.default_rng(7)
    c = g.uniform(-40e-6, 40e-6, S)
    c -= c.mean()
    pp = RO.pairs(S)
    beta = np.array([c[j] - c[i] for i, j in pp])
    rate, clock = RO.station_rates(beta, np.full(len(pp), 5.0), S)
    assert np.abs(rate - c).max() <= 1e-18
    assert np.array_equal(rate, clock)
    assert abs(rate.sum()) <= 1e-18


def test_rates_per_component_gauge_and_unfitted_station():
    """pairs within {0, 1, 2} and within {3, 4} are fitted, station 5 has no fitted pair; pairs with one REF window
    (no slope) carry a wild beta that must not enter"""
    S = 6
    c = np.array([3e-6, -1e-6, 7e-6, 20e-6, -4e-6, 50e-6])
    pp = RO.pairs(S)
    comp = [0, 0, 0, 1, 1, 2]
    beta = np.array([c[j] - c[i] if comp[i] == comp[j] else 1.0 for i, j in pp])
    nwin = np.array([4.0 if comp[i] == comp[j] and comp[i] < 2 else 1.0 for i, j in pp])
    rate, clock = RO.station_rates(beta, nwin, S)
    for members in ([0, 1, 2], [3, 4]):
        want = c[members] - c[members].mean()
        assert np.abs(rate[members] - want).max() <= 1e-18
        assert abs(rate[members].sum()) <= 1e-18
    assert rate[5] == 0.0 and math.isnan(clock[5])
    assert np.array_equal(clock[:5], rate[:5])


@pytest.mark.parametrize("c", [3.1e-4, -3.1e-4, 1e-3, -1e-3, 2.5e-5])
@pytest.mark.parametrize("length", [40001, 40000])
def test_delta_at_change_points(c, length):
    d = RO.delta(c, length)
    nc = (length - 1) / 2
    # the statement element by element, in scalar doubles
    want = np.array([math.floor(c * (n - nc) + 0.5) for n in range(length)], np.int64)
    assert np.array_equal(d, want)
    steps = np.diff(d)
    assert set(np.unique(steps)) <= {0, 1 if c > 0 else -1}
    # every change point sits where c (n - n_c) + 0.5 crosses an integer, on both sides of it
    for n in np.flatnonzero(steps)[:50] + 1:
        assert math.floor(c * (n - nc) + 0.5) != math.floor(c * (n - 1 - nc) + 0.5)
    assert abs(int(np.count_nonzero(steps)) - abs(c) * (length - 1)) <= 1
    if length % 2:
        assert d[int(nc)] == 0
    x = np.arange(length, dtype=np.float32) + 1
    y = RO.retime(x, c)
    s = np.arange(length) + d
    ok = (s >= 0) & (s < length)
    assert np.array_equal(y[ok], x[s[ok]]) and (y[~ok] == 0).all()
    # a fast clock's plane is stretched: both ends take indices off the plane (a slow clock's never does)
    assert (not ok[0] and not ok[-1]) == (c >= 1e-4)


def test_extended_window_record_without_decimation_is_the_undecimated_chain():
    """window_record in EXTENDED mode with D = 1 (preprocess_binary_dec) gives the bits of the chain without the
    decimator: preprocess_binary, re-time, two-sided correlation, parabolic peak -- on odd and even lengths, both
    signs of drift, with and without a shift"""
    B = 200_000
    eps = np.array([0.0, 40.0, -40.0, 25.0])
    raws, _, _ = drift_captures(ST4, eps, block=B, seed=12)
    tgt = [oracle.extract_target(oracle.unpack_u8(r)) for r in raws]
    oracle.set_seq_dc_limit(0)
    try:
        for (i, j), (a, z), shift in (((0, 1), (0, B), 0), ((1, 2), (137, 100_138), 0), ((2, 3), (3, 150_002), 5)):
            si, sj = tgt[i][a:z], tgt[j][a:z]
            ci, cj = eps[i] * 1e-6, eps[j] * 1e-6
            yi = RO.retime(oracle.preprocess_binary(si)[0], ci)
            yj = RO.retime(oracle.preprocess_binary(sj)[0], cj)
            if shift:
                yj = np.concatenate([yj[shift:], np.zeros(shift, yj.dtype)])
            idx, frac, val = oracle.peak_parabolic(oracle.xcorr_two_sided(yi, yj, 300))
            assert RO.window_record(si, sj, ci, cj, 300, shift=shift) == (idx - 300 + shift, frac, val)
            assert RO.window_record(si, sj, ci, cj, 300, shift=shift, mode="extended", D=1) == (idx - 300 + shift, frac, val)
    finally:
        oracle.set_seq_dc_limit(-1)


def test_retime_forms_far_indices_in_doubles():
    """a rate far beyond any clock's moves every sample off the plane but the centre one (odd lengths)"""
    x = np.arange(1, 10, dtype=np.float32)
    for c in (1e20, -1e20):
        y = RO.retime(x, c)
        assert y[4] == x[4] and (np.delete(y, 4) == 0).all()


def test_retiming_whole_block_with_true_rates_puts_peaks_on_the_centre_lag():
    B = 4_000_000
    eps = np.array([0.0, 40.0, -40.0, 25.0])
    raws, dR, dT = drift_captures(ST4, eps, block=B, seed=11)
    tgt = [oracle.extract_target(oracle.unpack_u8(r)) for r in raws]
    assert all(t.size == B for t in tgt)
    t_c = B + (B - 1) / 2
    oracle.set_seq_dc_limit(0)
    try:
        for i, j in RO.pairs(len(ST4)):
            want = (dT[j] - dT[i]) + (eps[j] - eps[i]) * 1e-6 * t_c
            lag, frac, _ = RO.window_record(tgt[i], tgt[j], eps[i] * 1e-6, eps[j] * 1e-6, 8, shift=int(round(want)))
            assert abs(lag + frac - want) <= 1.0, (i, j, lag + frac, want)
    finally:
        oracle.set_seq_dc_limit(-1)
