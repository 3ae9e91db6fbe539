"""The station check's restatement (tests/exclusion_oracle.py) on exact range differences from random geometries:
which station it excludes, where it stops, ties, unused slots, components, and that the fix without the station
returns to the truth."""
import math

import numpy as np
import pytest

import closure_oracle as CO
import exclusion_oracle as XO
import window_oracle as WO

MAX_RMS = 100.0   # metres


def geometry(S, seed, dims=2):
    """dims 3: stations between 0 and 3000 m, so that the elevation is determined (with 300..400 m it is not, and
    the fix's elevation stays hundreds of metres off with or without the check)"""
    rng = np.random.default_rng(seed)
    h = (300, 400) if dims == 2 else (0, 3000)
    st = np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), rng.uniform(*h)]
                   for _ in range(S)])
    tx = np.array([41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0 if dims == 2 else 1500.0])
    return st, tx, exact_rd(st, tx), rng


def exact_rd(st, tx):
    x = WO.llh_to_ecef(*tx)
    r = [math.dist(x, WO.llh_to_ecef(*s)) for s in st]
    return np.array([r[j] - r[i] for i, j in CO.pairs(len(st))])


def station_offset(rd, S, s, delta):
    """station s's range read delta too long: every pair (i, s) gains delta, every pair (s, j) loses it"""
    out = rd.copy()
    for p, (i, j) in enumerate(CO.pairs(S)):
        out[p] += delta if j == s else (-delta if i == s else 0.0)
    return out


def metres(a, b):
    return math.dist(WO.llh_to_ecef(*a), WO.llh_to_ecef(*b))


def start(tx):
    return tx + [0.02, -0.02, 0.0]


@pytest.mark.parametrize("S,dims", [(5, 2), (6, 2), (8, 2), (16, 2), (6, 3), (9, 3), (16, 3)])
def test_one_bad_station_is_excluded(S, dims):
    P = S * (S - 1) // 2
    for seed in range(3):
        st, tx, rd, rng = geometry(S, 100 * S + 10 * dims + seed, dims)
        bad = int(rng.integers(0, S))
        rd = station_offset(rd, S, bad, rng.choice([-1, 1]) * rng.uniform(1e3, 2e4))
        out, rounds, srms, n, (fix, rms, status, _) = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), dims, MAX_RMS)
        assert n == 1 and np.flatnonzero(rounds).tolist() == [bad] and rounds[bad] == 1, (seed, rounds)
        assert [p for p, (i, j) in enumerate(CO.pairs(S)) if out[p] == 3] == \
            [p for p, (i, j) in enumerate(CO.pairs(S)) if bad in (i, j)]
        assert status == 0 and metres(fix, tx) < 1e-3, (seed, metres(fix, tx))
        # the diagnostic: every station is a candidate here, and the bad one stands far apart
        assert np.isfinite(srms).all() and srms[bad] < 1e-3 * np.delete(srms, bad).min()


def test_two_bad_stations_and_the_stop():
    S, P = 16, 120
    st, tx, rd, rng = geometry(S, 7)
    rd = station_offset(station_offset(rd, S, 3, 4e3), S, 11, -9e3)
    _, rounds, _, n, (fix, _, status, _) = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, MAX_RMS, max_exclude=2)
    assert n == 2 and sorted(np.flatnonzero(rounds).tolist()) == [3, 11] and sorted(rounds[[3, 11]].tolist()) == [1, 2]
    assert status == 0 and metres(fix, tx) < 1e-3
    out, rounds1, _, n1, (fix1, rms1, _, _) = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, MAX_RMS, max_exclude=1)
    assert n1 == 1 and np.flatnonzero(rounds1).tolist() == [int(np.flatnonzero(rounds == 1)[0])]
    assert rms1 > MAX_RMS and (out == 3).sum() == S - 1   # stopped by max_exclude with the rms still above max_rms
    # max_exclude = 0 is no limit: the same two
    _, rounds0, _, n0, _ = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, MAX_RMS, max_exclude=0)
    assert n0 == 2 and rounds0.tolist() == rounds.tolist()


@pytest.mark.parametrize("S,dims", [(4, 2), (5, 3)])
def test_too_few_stations_exclude_nothing(S, dims):
    P = S * (S - 1) // 2
    st, tx, rd, _ = geometry(S, 40 + S, dims)
    rd = station_offset(rd, S, 1, 5e3)
    out, rounds, srms, n, F = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), dims, MAX_RMS)
    assert F[1] > MAX_RMS   # the fix does not fit ...
    assert n == 0 and not rounds.any() and np.isnan(srms).all() and (out == 1).all()   # ... but no station is a candidate
    assert all(XO.redundancy(XO.without([True] * P, S, k), S, dims) == 0 for k in range(S))


def test_error_below_max_rms_is_kept():
    S, P = 8, 28
    st, tx, rd, _ = geometry(S, 3)
    rd = station_offset(rd, S, 5, 30.0)
    plain = WO.solve_ls(st, rd, start(tx), 2, np.ones(P, bool))
    out, rounds, srms, n, F = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, MAX_RMS)
    assert 0 < plain[1] <= MAX_RMS and n == 0 and np.isnan(srms).all() and (out == 1).all()
    assert F[0].tolist() == plain[0].tolist() and F[1:] == plain[1:]
    _, rounds, _, n, _ = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, 1.0)   # a lower bound finds it
    assert n == 1 and rounds[5] == 1


def test_no_improvement_excludes_nothing():
    """5 m of noise on every pair of five stations and no bad station, from the station mean: the fix's rms exceeds
    max_rms, every station is a candidate, but no solve without one fits better (the seeds of 150 that have such a
    set are 4 and 93), so nothing is excluded and the fix is the plain one"""
    S, P = 5, 10
    for seed in (4, 93):
        rng = np.random.default_rng(5000 + seed)
        st = np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), rng.uniform(300, 400)]
                       for _ in range(S)])
        tx = np.array([41.26 + rng.uniform(-0.6, 0.6), -96.02 + rng.uniform(-0.8, 0.8), 350.0])
        rd = exact_rd(st, tx) + rng.normal(0, 5.0, P)
        plain = WO.solve_ls(st, rd, None, 2, np.ones(P, bool))
        out, rounds, srms, n, F = XO.exclude_set(st, rd, np.ones(P, bool), None, 2, 1.0)
        assert plain[2] == 0 and plain[1] > 1.0 and np.isfinite(srms).all() and srms.min() >= plain[1]
        assert n == 0 and not rounds.any() and (out == 1).all()
        assert F[0].tolist() == plain[0].tolist() and F[1:] == plain[1:]


def test_ties_go_to_the_lowest_station():
    """stations 4 and 5 stand at one place and pair (4, 5) is wrong: without 4 the set is, term by term in pair
    order, the set without 5, so the two solves tie bit for bit and the lower station, 4, is excluded"""
    S = 7
    P = S * (S - 1) // 2
    st, tx, _, _ = geometry(S, 11)
    st[5] = st[4]
    rd = exact_rd(st, tx)
    rd[CO.pairs(S).index((4, 5))] += 5e3
    out, rounds, srms, n, (fix, *_) = XO.exclude_set(st, rd, np.ones(P, bool), start(tx), 2, MAX_RMS, max_exclude=0)
    assert srms[4] == srms[5] and srms[4] < 1e-6 * np.delete(srms, [4, 5]).min()
    assert rounds.tolist() == [0, 0, 0, 0, 1, 0, 0] and n == 1 and metres(fix, tx) < 1e-3


def test_unused_slots_are_never_read():
    S, P = 9, 36
    st, tx, rd, rng = geometry(S, 21)
    rd = station_offset(rd, S, 2, 7e3)
    used = rng.uniform(0, 1, P) < 0.8
    a = XO.exclude_set(st, np.where(used, rd, np.nan), used, start(tx), 2, MAX_RMS)
    b = XO.exclude_set(st, np.where(used, rd, 1e9), used, start(tx), 2, MAX_RMS)
    assert a[0].tolist() == b[0].tolist() and a[1].tolist() == b[1].tolist() and a[3] == b[3] == 1 and a[1][2] == 1
    assert np.array_equal(a[2], b[2], equal_nan=True) and a[4][0].tolist() == b[4][0].tolist()
    assert (a[0] == 0).tolist() == (~used).tolist()


def test_disconnected_mask():
    """two groups of three stations with no pair between them, and station 6 with no pair at all: station 6 is no
    candidate, and an exclusion leaves 5 stations in 2 components (redundancy 1)"""
    S = 7
    P = S * (S - 1) // 2
    st, tx, rd, _ = geometry(S, 5)
    used = np.array([(i < 3) == (j < 3) and j != 6 for i, j in CO.pairs(S)])
    rd = station_offset(rd, S, 4, 6e3)
    assert XO.redundancy(used, S, 2) == 2 and not XO.candidate(used, S, 6, 2)
    assert all(XO.candidate(used, S, k, 2) and XO.redundancy(XO.without(used, S, k), S, 2) == 1 for k in range(6))
    out, rounds, srms, n, (fix, rms, status, _) = XO.exclude_set(st, np.where(used, rd, np.nan), used, start(tx), 2,
                                                                 MAX_RMS)
    assert np.isnan(srms[6]) and np.isfinite(srms[:6]).all()
    assert n == 1 and rounds[4] == 1 and status == 0 and metres(fix, tx) < 1e-3


def test_inert_check():
    S, P = 8, 28
    st, tx, rd, _ = geometry(S, 9)
    rd = station_offset(rd, S, 0, 5e3)
    plain = WO.solve_ls(st, rd, None, 2, np.ones(P, bool))
    out, rounds, srms, n, F = XO.exclude_set(st, rd, np.ones(P, bool), None, 2, math.inf)
    assert n == 0 and (out == 1).all() and np.isnan(srms).all() and not rounds.any()
    assert F[0].tolist() == plain[0].tolist() and F[1:] == plain[1:]
