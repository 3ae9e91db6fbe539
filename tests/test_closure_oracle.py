"""The closure check's restatement (tests/closure_oracle.py) on exact range differences from random geometries:
which pairs it drops, where it stops, and that the fix from the kept pairs returns to the truth."""
import math

import numpy as np

import closure_oracle as CO
import window_oracle as WO

MR = 100.0   # max_residual, metres


def geometry(S, seed):
    rng = np.random.default_rng(seed)
    st = np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), rng.uniform(300, 400)]
                   for _ in range(S)])
    tx = np.array([41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0])
    x = WO.llh_to_ecef(*tx)
    r = [math.dist(x, WO.llh_to_ecef(*s)) for s in st]
    rd = np.array([r[j] - r[i] for i, j in CO.pairs(S)])
    return st, tx, rd, rng


def metres(a, b):
    return math.dist(WO.llh_to_ecef(*a), WO.llh_to_ecef(*b))


def test_one_wrong_pair_of_four():
    for seed in range(6):
        _, _, rd, rng = geometry(4, seed)
        q = int(rng.integers(0, 6))
        rd[q] += rng.choice([-1, 1]) * rng.uniform(3, 30) * MR
        out, e, n = CO.check_set(rd, np.ones(6, bool), 4, max_residual=MR)
        assert n == 1 and np.flatnonzero(out == 2).tolist() == [q], seed
        assert abs(e[q]) > MR and np.all(np.abs(np.delete(e, q)) < 1e-6)


def test_sixteen_stations_up_to_eight_wrong_pairs():
    S, P = 16, 120
    for k in range(1, 9):
        st, tx, rd, rng = geometry(S, 100 + k)
        bad = sorted(rng.choice(P, k, replace=False).tolist())
        rd[bad] += rng.choice([-1, 1], k) * rng.uniform(3, 6, k) * MR
        out, e, n = CO.check_set(rd, np.ones(P, bool), S, max_residual=MR)
        assert np.flatnonzero(out == 2).tolist() == bad and n == k, k
        fix, rms, status, _ = WO.solve_ls(st, rd, tx + [0.02, -0.02, 0.0], 2, out == 1)
        assert status == 0 and metres(fix, tx) < 1e-3, (k, metres(fix, tx))
        wrong, *_ = WO.solve_ls(st, rd, tx + [0.02, -0.02, 0.0], 2, np.ones(P, bool))
        assert metres(wrong, tx) > 1.0


def test_station_with_every_pair_wrong():
    S, s = 8, 5
    _, _, rd, _ = geometry(S, 7)
    mine = [p for p, (i, j) in enumerate(CO.pairs(S)) if s in (i, j)]
    rd[mine] += MR * np.array([5.0, -9.0, 13.0, -17.0, 21.0, 25.0, -29.0])   # tau_5 sees 5, -9, ..., 29
    out, e, n = CO.check_set(rd, np.ones(len(rd), bool), S, max_residual=MR)
    assert np.flatnonzero(out == 2).tolist() == mine and n == S - 1
    # the last pair goes with the one before it (degree rule): one step takes both, so max_drop = S - 2 does not
    # stop short of it
    out2, _, n2 = CO.check_set(rd, np.ones(len(rd), bool), S, max_residual=MR, max_drop=S - 2)
    assert n2 == S - 1 and (out2 == out).all()


def test_single_cycle_drops_nothing():
    _, _, rd, _ = geometry(3, 11)
    rd[1] += 20 * MR
    out, e, n = CO.check_set(rd, np.ones(3, bool), 3, max_residual=MR)
    assert n == 0 and (out == 1).all() and np.all(np.abs(e) > MR)
    S = 5
    _, _, rd, _ = geometry(S, 12)
    ring = np.array([j == i + 1 or (i, j) == (0, S - 1) for i, j in CO.pairs(S)])
    rd[0] += 20 * MR
    out, e, n = CO.check_set(rd, ring, S, max_residual=MR)
    assert n == 0 and (out == ring).all()
    assert np.all(np.abs(e[ring]) > MR) and np.isnan(e[~ring]).all()


def two_blocks_and_a_bridge(S=8):
    """K4 on 0..3, K4 on 4..7, the bridge (3, 4)"""
    return np.array([(i < 4) == (j < 4) or (i, j) == (3, 4) for i, j in CO.pairs(S)])


def test_bridge_is_never_dropped():
    S = 8
    _, _, rd, _ = geometry(S, 13)
    u = two_blocks_and_a_bridge(S)
    br = CO.pairs(S).index((3, 4))
    wrong = CO.pairs(S).index((0, 2))
    rd[br] += 50 * MR
    rd[wrong] += 10 * MR
    out, e, n = CO.check_set(rd, u, S, max_residual=MR)
    assert out[br] == 1 and abs(e[br]) < 1e-6
    assert np.flatnonzero(out == 2).tolist() == [wrong] and n == 1


def test_max_drop_and_status_two_stops():
    S, P = 16, 120
    _, _, rd, rng = geometry(S, 21)
    bad = sorted(rng.choice(P, 4, replace=False).tolist())
    rd[bad] += np.array([4.0, -5.0, 6.0, -7.0]) * MR
    _, e_all, n_all = CO.check_set(rd, np.ones(P, bool), S, max_residual=MR)
    assert n_all == 4
    out, e, n = CO.check_set(rd, np.ones(P, bool), S, max_residual=MR, max_drop=2)
    assert n == 2 and set(np.flatnonzero(out == 2).tolist()) <= set(bad)
    # K3 on 0..2 plus (0, 3), (1, 3); a wrong (0, 3): dropping it leaves station 3 one pair, which goes too
    S = 4
    _, _, rd, _ = geometry(S, 22)
    u = np.array([(i, j) != (2, 3) for i, j in CO.pairs(S)])
    rd[CO.pairs(S).index((0, 3))] += 10 * MR
    out2, _, n2 = CO.check_set(rd, u, S, dims=2, max_residual=MR)
    assert n2 == 2 and np.flatnonzero(out2 == 2).tolist() == [CO.pairs(S).index((0, 3)), CO.pairs(S).index((1, 3))]
    out3, e3, n3 = CO.check_set(rd, u, S, dims=3, max_residual=MR)   # three stations left: status 2, keep m
    assert n3 == 0 and (out3 == u).all() and np.nanmax(np.abs(e3)) > MR


def test_ties_go_to_the_lowest_pair():
    # K4 of zero range differences with the same error on the disjoint pairs (0, 1) and (2, 3): equal residuals
    rd = np.zeros(6)
    rd[0] = rd[5] = 1024.0
    _, e, _ = CO.check_set(rd, np.ones(6, bool), 4, max_residual=math.inf)
    assert abs(e[0]) == abs(e[5]) == np.abs(e).max()
    out, _, n = CO.check_set(rd, np.ones(6, bool), 4, max_residual=MR, max_drop=1)
    assert n == 1 and np.flatnonzero(out == 2).tolist() == [0]


def test_unused_slots_are_never_read():
    S, P = 8, 28
    _, _, rd, rng = geometry(S, 31)
    u = rng.uniform(0, 1, P) < 0.7
    rd[3] += 10 * MR
    u[3] = True
    a = CO.check_set(np.where(u, rd, np.nan), u, S, max_residual=MR)
    b = CO.check_set(np.where(u, rd, 1e300), u, S, max_residual=MR)
    assert (a[0] == b[0]).all() and a[2] == b[2]
    assert a[1].tobytes() == b[1].tobytes() and np.isnan(a[1][~u]).all()


def test_components_and_isolated_stations():
    S = 9
    _, _, rd, _ = geometry(S, 41)
    pp = CO.pairs(S)
    u = np.array([j < 8 and (i < 4) == (j < 4) for i, j in pp])    # K4, K4, station 8 alone
    w1, w2 = pp.index((0, 1)), pp.index((5, 7))
    rd[w1] += 8 * MR
    rd[w2] -= 9 * MR
    out, e, n = CO.check_set(rd, u, S, max_residual=MR)
    assert np.flatnonzero(out == 2).tolist() == [w1, w2] and n == 2
    m = out == 1
    tau = CO.station_values(np.where(u, rd, np.nan), m, S)
    assert CO.components(m, S) == [0, 0, 0, 0, 4, 4, 4, 4, 8]
    assert abs(sum(tau[:4])) < 1e-9 and abs(sum(tau[4:8])) < 1e-9 and tau[8] == 0.0


def test_inert_check_returns_u():
    S, P = 16, 120
    _, _, rd, rng = geometry(S, 51)
    u = rng.uniform(0, 1, P) < 0.8
    rd[u] += rng.normal(0, 30, int(u.sum()))
    _, e, _ = CO.check_set(rd, u, S, max_residual=math.inf)
    out, e2, n = CO.check_set(rd, u, S, max_residual=float(np.nanmax(np.abs(e))) * 1.01)
    assert n == 0 and (out == u).all() and e.tobytes() == e2.tobytes()
