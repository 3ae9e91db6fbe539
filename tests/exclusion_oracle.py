"""Plain restatement of the station check of the windowed fixes (tdoa_exclude_stations, the _exclude calls; test
infrastructure only).

LS(mask, x0) is window_oracle.solve_ls (k_solve_ls's statement with a used mask); the status-2 rule and the
components are closure_oracle's.  The grid's second seed is not restated here: the GPU tests check it against
tdoa_grid_masked on the returned mask.  The product never imports this module."""
from __future__ import annotations

import math

import numpy as np

import closure_oracle as CO
import window_oracle as WO


def without(m, S, k):
    """m without every pair that touches station k"""
    return [bool(m[p]) and k not in (i, j) for p, (i, j) in enumerate(CO.pairs(S))]


def redundancy(m, S, dims):
    """(stations m touches) - (components of m's pair graph) - dims"""
    touched = set()
    for p, (i, j) in enumerate(CO.pairs(S)):
        if m[p]:
            touched.update((i, j))
    comp = CO.components(m, S)
    return len(touched) - sum(1 for s in touched if comp[s] == s) - dims


def candidate(m, S, k, dims):
    if not any(m[p] and k in ij for p, ij in enumerate(CO.pairs(S))):
        return False
    mk = without(m, S, k)
    return CO.ls_used_pairs(mk, S, dims) >= 0 and redundancy(mk, S, dims) >= 1


def exclude_set(stations_llh, rd, used, init_llh=None, dims=2, max_rms=math.inf, max_exclude=1):
    """One set: rd[P], used[P] (only the used slots are read), start init_llh (None: the station mean).  Returns
    (out_used[P] in {0, 1, 3}, station_round[S], station_rms[S], n_excluded, (llh, rms, status, iters))."""
    st = np.asarray(stations_llh, np.float64).reshape(-1, 3)
    S = st.shape[0]
    P = S * (S - 1) // 2
    u = [bool(used[p]) for p in range(P)]
    rdv = [float(rd[p]) if u[p] else math.nan for p in range(P)]   # an unused slot is never read
    m = list(u)
    F = WO.solve_ls(st, rdv, init_llh, dims, m)
    rounds, srms, n_ex = [0] * S, [math.nan] * S, 0
    r = 0
    while True:
        if F[2] != 0 or F[1] <= max_rms or (max_exclude > 0 and n_ex == max_exclude):
            break
        r += 1
        best, best_k = None, -1
        for k in range(S):
            if rounds[k] or not candidate(m, S, k, dims):
                continue
            Fk = WO.solve_ls(st, rdv, init_llh, dims, without(m, S, k))
            if r == 1:
                srms[k] = Fk[1]
            if Fk[2] == 0 and (best is None or Fk[1] < best[1]):
                best, best_k = Fk, k
        if best is None or not (best[1] < F[1]):
            break
        m = without(m, S, best_k)
        rounds[best_k] = r
        n_ex += 1
        F = best
    out = np.array([0 if not u[p] else (1 if m[p] else 3) for p in range(P)], np.uint8)
    return out, np.array(rounds, np.uint8), np.array(srms), n_ex, F


def exclude(stations_llh, rd, used, init_llh=None, dims=2, max_rms=math.inf, max_exclude=1):
    """exclude_set over rows rd[n_sets][>= P], used[n_sets][>= P]; init_llh None, one point or one per set.  Returns
    a dict as Engine.exclude_stations."""
    st = np.asarray(stations_llh, np.float64).reshape(-1, 3)
    S = st.shape[0]
    P = S * (S - 1) // 2
    rd = np.asarray(rd, np.float64)
    used = np.asarray(used)
    n = rd.shape[0]
    init = None if init_llh is None else np.broadcast_to(np.asarray(init_llh, np.float64).reshape(-1, 3), (n, 3))
    outs = [exclude_set(st, rd[k, :P], used[k, :P], None if init is None else init[k], dims, max_rms, max_exclude)
            for k in range(n)]
    return {"used": np.array([o[0] for o in outs], np.uint8).reshape(n, P),
            "station_excluded": np.array([o[1] for o in outs], np.uint8).reshape(n, S),
            "station_rms": np.array([o[2] for o in outs]).reshape(n, S),
            "excluded": np.array([o[3] for o in outs], np.int32),
            "position": np.array([o[4][0] for o in outs]).reshape(n, 3),
            "rms": np.array([o[4][1] for o in outs]), "status": np.array([o[4][2] for o in outs], np.int32),
            "iters": np.array([o[4][3] for o in outs], np.int32)}
