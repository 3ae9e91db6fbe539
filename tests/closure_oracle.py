"""Plain restatement of the closure check of the windowed fixes (tdoa_closure, the _closure calls; test
infrastructure only).

Per set: the station values tau from the used range differences are tests/retime_oracle.station_rates' solve with
rd in place of beta (the pairs of the working mask are its fitted pairs), which is k_station_rates' order of
operations; then the residuals, the stop rules, the tentative drop with the degree rule and the status-2 rule of
include/tdoa_b200.h.  Python floats are IEEE doubles rounded to nearest with no fused multiply-add, so the bits are
the kernel's.  The product never imports this module."""
from __future__ import annotations

import math

import numpy as np

import retime_oracle as RO


def pairs(S):
    return RO.pairs(S)


def ls_used_pairs(m, S, dims):
    """the least-squares step's status-2 rule: the number of used pairs, or -1"""
    n_used, touched = 0, set()
    for p, (i, j) in enumerate(pairs(S)):
        if m[p]:
            n_used += 1
            touched.update((i, j))
    return -1 if n_used < dims or len(touched) < dims + 1 else n_used


def components(m, S):
    """label of every station: the smallest station index of its component of the m-pair graph"""
    comp = list(range(S))
    changed = True
    while changed:
        changed = False
        for p, (i, j) in enumerate(pairs(S)):
            if m[p]:
                c = min(comp[i], comp[j])
                if comp[i] != c or comp[j] != c:
                    comp[i] = comp[j] = c
                    changed = True
    return comp


def station_values(rd, m, S):
    """tau[S]: the zero-sum (per component) least-squares station values of the m-pairs' range differences"""
    P = len(pairs(S))
    tau, _ = RO.station_rates(rd, [2.0 if m[p] else 0.0 for p in range(P)], S)
    return [float(v) for v in tau]


def check_set(rd, used, S, dims=2, max_residual=math.inf, max_drop=0):
    """One set: rd[P], used[P] (only the usable slots are read).  Returns (out_used[P] in {0, 1, 2}, resid[P],
    dropped)."""
    pp = pairs(S)
    P = len(pp)
    u = [bool(used[p]) for p in range(P)]
    m = list(u)
    rdv = [float(rd[p]) if u[p] else math.nan for p in range(P)]   # an unusable slot is never read
    drops = 0
    while True:
        tau = station_values(rdv, m, S)
        e = [rdv[p] - (tau[j] - tau[i]) if u[p] else math.nan for p, (i, j) in enumerate(pp)]
        deg = [0] * S
        for p, (i, j) in enumerate(pp):
            if m[p]:
                deg[i] += 1
                deg[j] += 1
        comp = components(m, S)
        touched = [s for s in range(S) if deg[s] > 0]
        redundancy = sum(deg) // 2 - len(touched) + sum(1 for s in touched if comp[s] == s)
        q, best = -1, -1.0
        for p in range(P):
            if m[p] and abs(e[p]) > best:
                q, best = p, abs(e[p])
        if redundancy < 2 or (max_drop > 0 and drops >= max_drop) or q < 0 or not (best > max_residual):
            break
        m2 = list(m)
        lost = set()
        cut = 0
        while q >= 0:
            i, j = pp[q]
            m2[q] = False
            cut += 1
            deg[i] -= 1
            deg[j] -= 1
            lost.update((i, j))
            q = -1
            for s in range(S):
                if s in lost and deg[s] == 1:
                    q = next(p for p, (a, b) in enumerate(pp) if m2[p] and s in (a, b))
                    break
        if ls_used_pairs(m2, S, dims) < 0:
            break
        m = m2
        drops += cut
    out = np.array([0 if not u[p] else (1 if m[p] else 2) for p in range(P)], np.uint8)
    return out, np.array(e, np.float64), drops


def check(rd, used, S, dims=2, max_residual=math.inf, max_drop=0):
    """check_set over rows rd[n_sets][>= P], used[n_sets][>= P]"""
    rd = np.asarray(rd, np.float64)
    used = np.asarray(used)
    P = S * (S - 1) // 2
    outs = [check_set(rd[k, :P], used[k, :P], S, dims, max_residual, max_drop) for k in range(rd.shape[0])]
    if not outs:
        return np.zeros((0, P), np.uint8), np.zeros((0, P)), np.zeros(0, np.int32)
    return (np.stack([o[0] for o in outs]), np.stack([o[1] for o in outs]),
            np.array([o[2] for o in outs], np.int32))
