"""Plain restatement of the masked grid arg-min and the grid-seeded windowed fix stage (tdoa_grid_masked,
tdoa_process_windows_grid / tdoa_window_fixes_grid; test infrastructure only), on top of tests/window_oracle.py:
  - grid_solve:    orc_grid_solve with a per-pair used mask (the masked statement); with no mask, or an all-true one,
                   it is orc_grid_solve bit for bit (checked);
  - window_fixes:  window_oracle.window_fixes, with every window the least-squares step does not refuse (status 2)
                   started from its grid_solve cell.
Python floats are IEEE doubles with no fused multiply-add, so the operation order below is the rounding.  The product
never imports this module."""
from __future__ import annotations

import math

import numpy as np

import window_oracle as WO


def too_few(used, n, dims):
    """The status-2 rule: fewer than dims used pairs, or used pairs touching fewer than dims + 1 stations."""
    n_used, touched, q = 0, set(), 0
    for i in range(n):
        for j in range(i + 1, n):
            if used[q]:
                n_used += 1
                touched.update((i, j))
            q += 1
    return n_used < dims or len(touched) < dims + 1


def _dist(a, b):
    dx, dy, dz = a[0] - b[0], a[1] - b[1], a[2] - b[2]
    return math.sqrt(dx * dx + dy * dy + dz * dz)


def grid_solve(stations_llh, range_diffs, desc, used=None):
    """The grid arg-min in orc_grid_solve's operation order: cost = sum over the used pairs i<j, in order, of
    ((r_j - r_i) - rd_ij)^2; strict < over the cells in linear order.  desc = (lat0, lon0, dlat, dlon, nlat, nlon,
    elev).  A set with no used pair: (-1, NaN, NaN cell).  Returns (index, cost, llh)."""
    st = [tuple(float(v) for v in row) for row in np.asarray(stations_llh, np.float64).reshape(-1, 3)]
    rd = [float(v) for v in np.asarray(range_diffs, np.float64).reshape(-1)]
    n = len(st)
    P = n * (n - 1) // 2
    u = [True] * P if used is None else [bool(v) for v in np.asarray(used).reshape(-1)[:P]]
    if not any(u):
        return -1, math.nan, np.full(3, math.nan)
    lat0, lon0, dlat, dlon = (float(v) for v in desc[:4])
    nlat, nlon, elev = int(desc[4]), int(desc[5]), float(desc[6])
    s = [WO.llh_to_ecef(*row) for row in st]
    pairs = [(i, j, q) for q, (i, j) in enumerate((i, j) for i in range(n) for j in range(i + 1, n)) if u[q]]
    bi, bc = -1, 0.0
    for a in range(nlat):
        for b in range(nlon):
            x = WO.llh_to_ecef(lat0 + a * dlat, lon0 + b * dlon, elev)
            r = [_dist(x, sk) for sk in s]
            cost = 0.0
            for i, j, q in pairs:
                e = (r[j] - r[i]) - rd[q]
                cost += e * e
            if bi < 0 or cost < bc:
                bi, bc = a * nlon + b, cost
    return bi, bc, np.array([lat0 + float(bi // nlon) * dlat, lon0 + float(bi % nlon) * dlon, elev])


def window_fixes(stations_llh, nsamp, guard, win_start, win_len, hop, ref, tgt, grid, fs=2e6, min_margin=0.0,
                 ref_max_residual=0.0, ref_tx_llh=None, dims=2, init_llh=None):
    """window_oracle.window_fixes with a grid (7 numbers, as tdoa_grid): every window the least-squares step does not
    refuse starts at its grid_solve cell; a refused window (status 2) is not searched (index -1, cost NaN) and keeps
    the start it has without a grid (init_llh, or the mean of the stations).  Returns window_oracle.window_fixes'
    dict plus seed, seed_cost, seed_index."""
    out = WO.window_fixes(stations_llh, nsamp, guard, win_start, win_len, hop, ref, tgt, fs=fs, min_margin=min_margin,
                          ref_max_residual=ref_max_residual, ref_tx_llh=ref_tx_llh, dims=dims, init_llh=init_llh)
    st = np.asarray(stations_llh, np.float64).reshape(-1, 3)
    S = st.shape[0]
    rd, used = out["range_differences"], out["pair_used"]
    nt = rd.shape[0]
    if init_llh is not None:
        start = np.asarray(init_llh, np.float64)
    else:   # k_solve_ls's mean: component sums in station order, then one division
        start = np.zeros(3)
        for row in st:
            start = start + row
        start = start / S
    seed, seed_cost, seed_index = np.tile(start, (nt, 1)), np.full(nt, math.nan), np.full(nt, -1, np.int64)
    for w in range(nt):
        if too_few(used[w], S, dims):
            continue   # status 2: window_oracle.window_fixes' result stands
        seed_index[w], seed_cost[w], seed[w] = grid_solve(st, rd[w], grid, used[w])
        out["position"][w], out["rms"][w], out["status"][w], out["iters"][w] = WO.solve_ls(st, rd[w], seed[w], dims, used[w])
    out.update(seed=seed, seed_cost=seed_cost, seed_index=seed_index)
    return out
