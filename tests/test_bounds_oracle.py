"""The restatement of the bounded lag search (tests/bounds_oracle.py) on hand-made correlation arrays, its interval
arithmetic, and the weak-target scenario the GPU tests run, proven here on the CPU oracle."""
import math

import numpy as np
import pytest

import bounds_oracle as B
import lag_edges as E
import window_oracle as W
from oracle import oracle


@pytest.fixture
def extended_oracle():
    oracle.set_seq_dc_limit(0)
    yield
    oracle.set_seq_dc_limit(-1)


def corr(L, peaks):
    c = np.zeros(2 * L + 1)
    c[:] = 0.01 * np.sin(np.arange(2 * L + 1))       # small, distinct background
    for lag, v in peaks.items():
        c[lag + L] = v
    return c


def test_whole_range_is_the_unbounded_peak():
    c = corr(50, {7: 0.9, 6: 0.5, 8: 0.6, -30: -0.8})
    r = B.bounded_peak(c, -50, 50)
    idx, frac, val = oracle.peak_parabolic(c)
    assert r["lag"] == idx - 50 == 7 and r["corr"] == val and abs(float(r["frac"]) - frac) <= 1e-6
    assert r["flags"] == B.BOUNDED
    assert r["margin"] == np.float32((0.9 - 0.8) / 0.9)


def test_ties_go_to_the_lowest_lag_in_the_run():
    c = corr(50, {-20: 0.7, 3: -0.7, 10: 0.7})
    assert B.bounded_peak(c, -50, 50)["lag"] == -20
    r = B.bounded_peak(c, -19, 50)
    assert r["lag"] == 3 and r["corr"] == -0.7 and r["margin"] == 0.0


def test_peak_outside_gives_edge_on_the_boundary():
    c = corr(50, {20: 0.9, 19: 0.6, 18: 0.4})
    r = B.bounded_peak(c, -5, 18)
    assert r["lag"] == 18 and r["flags"] & B.EDGE and r["frac"] == 0.0
    r = B.bounded_peak(c, -5, 19)
    assert r["lag"] == 19 and r["flags"] & B.EDGE
    assert not B.bounded_peak(c, -5, 21)["flags"] & B.EDGE


def test_one_lag_run():
    c = corr(50, {0: 0.9})
    r = B.bounded_peak(c, 4, 4)
    assert r["lag"] == 4 and r["flags"] == B.BOUNDED | B.EDGE and r["margin"] == 1.0


def test_run_clipped_by_the_range_and_empty_runs():
    c = corr(50, {-50: 0.9, 50: 0.95})
    r = B.bounded_peak(c, -200, -40)
    assert r["lag"] == -50 and r["flags"] & B.EDGE
    r = B.bounded_peak(c, 40, 10 ** 6)
    assert r["lag"] == 50 and r["flags"] & B.EDGE
    for lo, hi in ((51, 60), (-60, -51), (B.I32_MIN, -51), (51, B.I32_MAX)):
        r = B.bounded_peak(c, lo, hi)
        assert r["flags"] == B.BOUNDED | B.EMPTY and r["lag"] == 0 and r["corr"] == 0.0, (lo, hi)


def test_decimated_units_ceil_and_floor():
    D = 4
    assert B.run(-9, -1, 10, D) == (10 - 2, 10 - 1)       # ceil(-9/4) = -2, floor(-1/4) = -1
    assert B.run(-8, -4, 10, D) == (8, 9)
    assert B.run(-7, -5, 10, D) == (9, 8)                 # no multiple of 4 in [-7, -5]: empty
    assert B.run(1, 3, 10, D) == (11, 10)
    assert B.run(-3, 3, 10, D) == (10, 10)
    c = corr(10, {-2: 0.9, -1: 0.5, -3: 0.4})
    assert B.bounded_peak(c, -9, 0, D)["flags"] & B.EDGE       # lags -2 .. 0: the peak is the run's first
    r = B.bounded_peak(c, -12, 0, D)
    assert r["first_lag"] == -8 and r["flags"] == B.BOUNDED
    total = 4.0 * (-2.0 + float(np.float32(0.5 * (0.4 - 0.5) / (0.4 - 1.8 + 0.5))))
    assert r["lag"] == round(total) and abs(float(r["frac"]) - (total - round(total))) < 1e-6
    assert B.bounded_peak(c, -7, -5, D)["flags"] & B.EMPTY


def test_interval_operation_order():
    lo, hi = B.interval(12.25, 1e-6, 1000.0, 0.0, 5000.0, 15000.0, False, 5.0)
    y = 12.25 + 1e-6 * (5000.0 - 1000.0)
    half = 2.0 * 15000.0 / 299792458.0 * 2e6 + 5.0
    assert (lo, hi) == (math.ceil(y - half), math.floor(y + half))
    lo, hi = B.interval(0.0, 0.0, 0.0, 3000.0, 0.0, 15000.0, True, 0.0)
    c = -3000.0 / 299792458.0 * 2e6
    assert (lo, hi) == (math.ceil(c - 15000.0 / 299792458.0 * 2e6), math.floor(c + 15000.0 / 299792458.0 * 2e6))
    assert B.interval(1e12, 0.0, 0.0, 0.0, 0.0, 1.0, True, 0.0) == (B.I32_MAX, B.I32_MAX)


def test_int32_extremes_are_empty_runs():
    c = corr(50, {0: 0.9})
    for lo, hi in ((B.I32_MAX, B.I32_MAX), (B.I32_MAX - 10, B.I32_MAX), (B.I32_MIN, B.I32_MIN), (B.I32_MIN, B.I32_MIN + 10)):
        for D in (1, 4):
            r = B.bounded_peak(c, lo, hi, D)
            assert r["flags"] == B.BOUNDED | B.EMPTY and r["lag"] == 0, (lo, hi, D)


def test_weak_target_scenario_on_the_oracle(extended_oracle):
    """The GPU scenario's captures, every TGT window on the oracle chain: a weak target (the weak branch) that repeats
    every SCN_PERIOD samples, in receiver noise.  Without bounds at least 5 of the 10 lags of every window are more than
    5 samples off (another repeat) and the least-squares fix is more than 10 km off; with guard = 5 every lag is within
    1 sample of the planted one and every fix within 100 m.  Without the repeats (period 0) and with the target
    weakened until the unbounded search strays, the weak branch's 200 kHz low-pass leaves the peak about ten samples
    wide and the bounded lags wander over it: no noise level gives both outcomes for such a target (see
    tools/bounds_bench.py's oracle sweep)."""
    raws, d = B.scenario_captures()
    st, L, S = B.SCN_LLH, B.SCN_MAX_LAG, len(B.SCN_LLH)
    x = W.llh_to_ecef(*B.SCN_TARGET)
    for w in range(B.SCN_NT):
        s0 = w * B.SCN_HOP
        ys = [oracle.preprocess_binary(E.split(r)[1][s0:s0 + B.SCN_WIN]) for r in raws]
        assert all(br == 2 for _, br in ys)                   # the weak branch
        off, rd_u, rd_b = 0, [], []
        for i in range(S):
            for j in range(i + 1, S):
                c = oracle.xcorr_two_sided(ys[i][0], ys[j][0], L)
                want = d[j] - d[i]
                lo, hi = B.interval(0.0, 0.0, 0.0, 0.0, 0.0, B.baseline(st[i], st[j]), False, B.SCN_GUARD)
                assert lo <= want <= hi
                u, b = B.bounded_peak(c, -L, L), B.bounded_peak(c, lo, hi)
                off += abs(u["lag"] - want) > 5
                assert abs(b["lag"] + float(b["frac"]) - want) <= 1.0
                usable = not (u["flags"] & B.EDGE)
                rd_u.append((u["lag"] + float(u["frac"])) / 2e6 * W.C_LIGHT if usable else math.nan)
                rd_b.append((b["lag"] + float(b["frac"])) / 2e6 * W.C_LIGHT)
        assert off >= 5, w
        fu = W.solve_ls(st, np.array(rd_u), None, 2, ~np.isnan(rd_u))
        fb = W.solve_ls(st, np.array(rd_b), None, 2, np.ones(len(rd_b), bool))
        assert fu[2] != 0 or W._dist(x, W.llh_to_ecef(*fu[0])) > 10e3, w
        assert fb[2] == 0 and W._dist(x, W.llh_to_ecef(*fb[0])) <= 100.0, w
