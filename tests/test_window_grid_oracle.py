"""CPU: the masked grid statement (tests/window_grid_oracle.py grid_solve) against orc_grid_solve, the seeded windowed fix
stage's statement (window_fixes(grid=...)) on the transmitters that trap a least-squares fix started at the station
mean, and the rounding bound of the masked ranked form (solve.cu, k_grid_rank with a mask).

The engine's tdoa_grid_masked and the _grid windowed calls are checked against these statements on the GPU
(tests/test_gpu_window_grid.py)."""
from __future__ import annotations

import math

import numpy as np

import window_grid_oracle as WG
import window_oracle as WO
from oracle import oracle
from helpers import STATION_LLH
from test_grid_rank_bound import KAPPA, fma

PEAK = np.dtype([("lag", "<i4"), ("flags", "<u4"), ("corr", "<f8"), ("frac", "<f4"), ("margin", "<f4"),
                 ("first_lag", "<i4"), ("n_blocks", "<i4")])
EMPTY = 0x8
FS, C = 2e6, 299792458.0

ST4 = np.vstack([STATION_LLH, [41.20, -96.20, 340.0]])   # the 4-station table of tests/test_gpu_windows.py
# transmitters outside the station hull, 15 km and 30 km out: from the station mean the fix stops in a local minimum
TRAPPED = [np.array([41.3711, -96.0233, 350.0]), np.array([41.5017, -95.9768, 350.0])]
TRAP_GRID = [40.90, -96.45, 0.005, 0.005, 180, 160, 350.0]


def pairs(S):
    return [(i, j) for i in range(S) for j in range(i + 1, S)]


def exact_rd(stations, tx):
    x = np.array(WO.llh_to_ecef(*tx))
    r = [float(np.linalg.norm(x - np.array(WO.llh_to_ecef(*s)))) for s in stations]
    return np.array([r[j] - r[i] for i, j in pairs(len(stations))])


def metres(a, b):
    return float(np.linalg.norm(np.array(WO.llh_to_ecef(*a)) - np.array(WO.llh_to_ecef(*b))))


# ------------------------------------------------------------------ the statement against orc_grid_solve
def test_unmasked_and_all_true_equal_the_oracle_bit_for_bit():
    rng = np.random.default_rng(11)
    for S in (3, 5):
        st = np.array([[41.26 + rng.uniform(-0.2, 0.2), -96.02 + rng.uniform(-0.25, 0.25), rng.uniform(300, 400)]
                       for _ in range(S)])
        desc = [41.20, -96.08, 0.004, 0.004, 30, 32, 350.0]
        for k in range(3):
            tx = np.array([41.26 + rng.uniform(-0.04, 0.04), -96.02 + rng.uniform(-0.05, 0.05), 350.0])
            rd = exact_rd(st, tx) + rng.normal(0, [0.0, 15.0, 150.0][k], S * (S - 1) // 2)
            wi, wc, wl = oracle.grid_solve(st, rd, *desc[:4], int(desc[4]), int(desc[5]), desc[6])
            for used in (None, np.ones(rd.size, bool)):
                gi, gc, gl = WG.grid_solve(st, rd, desc, used)
                assert gi == wi
                assert np.float64(gc).view(np.uint64) == np.float64(wc).view(np.uint64)
                assert np.array_equal(gl, wl)


def test_unused_slots_are_never_read_and_no_used_pair_has_no_argmin():
    rng = np.random.default_rng(12)
    st = ST4
    rd = exact_rd(st, [41.25, -96.05, 350.0]) + rng.normal(0, 20.0, 6)
    desc = [41.15, -96.15, 0.005, 0.005, 40, 40, 350.0]
    used = np.array([1, 0, 1, 1, 0, 1], bool)
    a, b = rd.copy(), rd.copy()
    a[~used], b[~used] = np.nan, 0.0
    ga, gb = WG.grid_solve(st, a, desc, used), WG.grid_solve(st, b, desc, used)
    assert ga[0] == gb[0] and ga[1] == gb[1] and np.array_equal(ga[2], gb[2])
    assert ga[0] != WG.grid_solve(st, rd, desc)[0] or ga[1] != WG.grid_solve(st, rd, desc)[1]   # the mask matters
    gi, gc, gl = WG.grid_solve(st, rd, desc, np.zeros(6, bool))
    assert gi == -1 and math.isnan(gc) and np.isnan(gl).all()


# ------------------------------------------------------------------ the trapped fixes
def trapped_cases():
    """(transmitter, used mask): both transmitters with every pair, the first one with pair (0, 1) unused"""
    full = np.ones(6, bool)
    no01 = full.copy()
    no01[0] = False
    return [(TRAPPED[0], full), (TRAPPED[1], full), (TRAPPED[0], no01)]


def test_grid_seed_frees_the_trapped_fixes():
    """Exact range differences, dims 2: from the station mean the fix ends more than 4 km from the transmitter;
    from the grid arg-min of the same used pairs it ends within 1 mm."""
    for tx, used in trapped_cases():
        rd = exact_rd(ST4, tx)
        mean_fix, _, st_mean, _ = WO.solve_ls(ST4, rd, None, 2, used)
        assert st_mean == 0 and metres(mean_fix, tx) > 4000.0
        gi, _, cell = WG.grid_solve(ST4, rd, TRAP_GRID, used)
        assert gi >= 0 and metres(cell, tx) < 1000.0   # a cell next to the transmitter (0.005 deg: 556 m of latitude)
        fix, rms, status, _ = WO.solve_ls(ST4, rd, cell, 2, used)
        assert status == 0 and metres(fix, tx) < 1e-3 and rms < 1e-3


# ------------------------------------------------------------------ the seed rule in window_fixes
def test_status_two_windows_are_not_searched():
    """Constructed tables (no drift, window times as tests/test_window_fix_oracle.py's), 4 stations, the first
    trapped transmitter: window 0 uses every pair, window 1 all but pair (0, 1), window 2 only pair (0, 1)
    (status 2 at dims 2: fewer than 2 used pairs), window 3 nothing."""
    b, w = 4000, 500
    n_ref, n_tgt = 16, 4
    P = 6
    y_tgt = exact_rd(ST4, TRAPPED[0]) * FS / C
    ref = np.zeros((n_ref, P), PEAK)
    tgt = np.zeros((n_tgt, P), PEAK)
    tgt["lag"] = np.round(y_tgt).astype(np.int32)
    tgt["frac"] = (y_tgt - np.round(y_tgt)).astype(np.float32)
    tgt["flags"][1, 0] = EMPTY
    tgt["flags"][2, 1:] = EMPTY
    tgt["flags"][3, :] = EMPTY
    grid = [41.15, -96.25, 0.02, 0.02, 16, 16, 350.0]   # a coarse grid keeps the pure-Python search short
    kw = dict(fs=FS, dims=2)
    plain = WO.window_fixes(ST4, [3 * b] * 4, 0, 0, w, w, ref, tgt, **kw)
    seeded = WG.window_fixes(ST4, [3 * b] * 4, 0, 0, w, w, ref, tgt, grid=grid, **kw)
    assert plain["status"].tolist() == [0, 0, 2, 2] == seeded["status"].tolist()
    for k in (2, 3):
        assert seeded["seed_index"][k] == -1 and math.isnan(seeded["seed_cost"][k])
        assert np.array_equal(seeded["position"][k], plain["position"][k])
        assert np.array_equal(seeded["seed"][k], plain["position"][k])   # the start it has without a grid
    for k in (0, 1):
        gi, gc, cell = WG.grid_solve(ST4, seeded["range_differences"][k], grid, seeded["pair_used"][k])
        assert seeded["seed_index"][k] == gi and seeded["seed_cost"][k] == gc and np.array_equal(seeded["seed"][k], cell)
        # the window's range differences are the transmitter's to within a float32 frac: the seeded fix finds it
        assert metres(seeded["position"][k], TRAPPED[0]) < 1.0 < 4000.0 < metres(plain["position"][k], TRAPPED[0])


# ------------------------------------------------------------------ the masked ranked form's rounding bound
def ranked_masked(r, rd, used, exact_fma):
    """k_grid_rank's masked f and tol: the row over the used pairs (grid_row_fill), the bracket less the unused
    pairs' (q_j - q_i)^2 chained by FMA in pair order."""
    S = len(r)
    c = [0.0] * S
    b = c1 = 0.0
    unused = []
    p = 0
    for i in range(S):
        for j in range(i + 1, S):
            if used[p]:
                c[j] += rd[p]
                c[i] -= rd[p]
                b += rd[p] * rd[p]
                c1 += 2.0 * abs(rd[p])
            else:
                unused.append((i, j))
            p += 1
    q = [rk - r[0] for rk in r]
    sq = sl = qm = 0.0
    for x in q:
        sq = fma(x, x, sq) if exact_fma else x * x + sq
        sl = sl + x
        qm = max(qm, abs(x))
    a = S * sq - sl * sl
    su = 0.0
    for i, j in unused:
        d = q[j] - q[i]
        su = fma(d, d, su) if exact_fma else d * d + su
    a = a - su
    mid = 0.0
    for x, ck in zip(q, c):
        mid = fma(x, ck, mid) if exact_fma else x * ck + mid
    f = fma(-2.0, mid, a + b) if exact_fma else -2.0 * mid + (a + b)
    tol = KAPPA * (2.0 * S * sq + (fma(2.0 * qm, c1, b) if exact_fma else 2.0 * qm * c1 + b))
    return f, tol


def _masked_sum(r, rd, used):
    """the masked statement, pair by pair in order"""
    cost, p, S = 0.0, 0, len(r)
    for i in range(S):
        for j in range(i + 1, S):
            if used[p]:
                e = (r[j] - r[i]) - rd[p]
                cost = cost + e * e
            p += 1
    return cost


def test_masked_rounding_bound_holds():
    """The unmasked tol still bounds the masked form's error: the subtracted sum is at most the bracket
    (sum over all pairs of (q_j - q_i)^2), so its m + 3 roundings add at most ~124 u S sum q^2 -- under 2 % of the
    t0 term -- and the used-only c_k, sum rd^2 and sum |rd| only shrink the rest."""
    rng = np.random.default_rng(20261020)
    worst = 0.0
    for n in range(6000):
        S = int(rng.integers(3, 17))
        P = S * (S - 1) // 2
        scale = 10.0 ** rng.uniform(0, 6)
        r = scale * rng.uniform(0.05, 1.0, S)
        true_rd = np.array([r[j] - r[i] for i, j in pairs(S)])
        rd = [true_rd, true_rd + rng.normal(0, 15.0, P), true_rd * rng.uniform(0.5, 1.5),
              scale * rng.uniform(-3, 3, P)][n % 4]
        used = rng.uniform(0, 1, P) < rng.uniform(0.05, 1.0)
        if not used.any():
            used[int(rng.integers(0, P))] = True
        f, tol = ranked_masked(list(r), list(rd), used, exact_fma=(n % 10 == 0))
        err = abs(f - _masked_sum(r, rd, used))
        assert err <= tol, (err, tol, S, int(used.sum()))
        worst = max(worst, err / tol)
    assert worst < 0.1
