"""Plain restatement of the windowed fix stage (tdoa_process_windows / tdoa_window_fixes; test infrastructure only).

Python floats are IEEE doubles with no fused multiply-add and `math` is the C library's, so every function here
rounds as oracle/tdoa_oracle.c does when it is written in the same operation order:
  - llh_to_ecef:   orc_llh_to_ecef (processor.go:125-148), checked bit for bit against it;
  - solve_ls:      orc_solve_ls with a per-pair used mask (the statement k_solve_ls follows with a mask); with no
                   mask, or an all-true one, it is orc_solve_ls bit for bit (checked);
  - window_fixes:  the window times, REF line, range differences and used mask of include/tdoa_b200.h, then
                   solve_ls per TGT window.
The product never imports this module."""
from __future__ import annotations

import math

import numpy as np

EDGE, EMPTY = 0x2, 0x8
C_LIGHT = 299792458.0
_A, _F = 6378137.0, 1.0 / 298.257223563


def llh_to_ecef(lat, lon, elev):
    e2 = 2 * _F - _F * _F
    lr, lo = lat * math.pi / 180, lon * math.pi / 180
    sl, cl, so, co = math.sin(lr), math.cos(lr), math.sin(lo), math.cos(lo)
    N = _A / math.sqrt(1 - e2 * sl * sl)
    return ((N + elev) * cl * co, (N + elev) * cl * so, (N * (1 - e2) + elev) * sl)


def _dist(a, b):
    dx, dy, dz = a[0] - b[0], a[1] - b[1], a[2] - b[2]
    return math.sqrt(dx * dx + dy * dy + dz * dz)


def _ls_cost(s, rd, used, lat, lon, h):
    x = llh_to_ecef(lat, lon, h)
    r = [_dist(x, sk) for sk in s]
    c, q, n = 0.0, 0, len(s)
    for i in range(n):
        for j in range(i + 1, n):
            if used is None or used[q]:
                f = (r[j] - r[i]) - rd[q]
                c += f * f
            q += 1
    return c, r


def _ls_step(A, b, lam, n):
    M = [[A[i][j] for j in range(3)] for i in range(3)]
    for i in range(3):
        M[i][i] = A[i][i] + lam * A[i][i]
    if n == 2:
        det = M[0][0] * M[1][1] - M[0][1] * M[1][0]
        if not (abs(det) > 1e-300):
            return None
        return [-(b[0] * M[1][1] - b[1] * M[0][1]) / det, -(M[0][0] * b[1] - M[1][0] * b[0]) / det, 0.0]
    c00 = M[1][1] * M[2][2] - M[1][2] * M[2][1]
    c01 = M[1][2] * M[2][0] - M[1][0] * M[2][2]
    c02 = M[1][0] * M[2][1] - M[1][1] * M[2][0]
    det = M[0][0] * c00 + M[0][1] * c01 + M[0][2] * c02
    if not (abs(det) > 1e-300):
        return None
    c10 = M[0][2] * M[2][1] - M[0][1] * M[2][2]
    c11 = M[0][0] * M[2][2] - M[0][2] * M[2][0]
    c12 = M[0][1] * M[2][0] - M[0][0] * M[2][1]
    c20 = M[0][1] * M[1][2] - M[0][2] * M[1][1]
    c21 = M[0][2] * M[1][0] - M[0][0] * M[1][2]
    c22 = M[0][0] * M[1][1] - M[0][1] * M[1][0]
    return [-(c00 * b[0] + c10 * b[1] + c20 * b[2]) / det, -(c01 * b[0] + c11 * b[1] + c21 * b[2]) / det,
            -(c02 * b[0] + c12 * b[1] + c22 * b[2]) / det]


def solve_ls(stations_llh, range_diffs, init_llh=None, dims=2, used=None):
    """orc_solve_ls's Levenberg-Marquardt fix; used[p] = False leaves pair p out of the cost, the normal equations
    and the rms.  Fewer than dims used pairs, or used pairs touching fewer than dims + 1 stations: status 2 with
    the start point, rms 0 and no iteration.  Returns (llh, rms, status, iters)."""
    st = [tuple(float(v) for v in row) for row in np.asarray(stations_llh, np.float64).reshape(-1, 3)]
    rd = [float(v) for v in np.asarray(range_diffs, np.float64).reshape(-1)]
    u = None if used is None else [bool(v) for v in np.asarray(used).reshape(-1)]
    n = len(st)
    e2 = 2 * _F - _F * _F
    P = n * (n - 1) // 2
    s = [llh_to_ecef(*row) for row in st]
    if init_llh is not None:
        lat, lon, h = (float(v) for v in init_llh)
    else:
        lat = lon = h = 0.0
        for row in st:
            lat += row[0]; lon += row[1]; h += row[2]
        lat /= n; lon /= n; h /= n
    if u is not None:
        n_used, touched, q = 0, set(), 0
        for i in range(n):
            for j in range(i + 1, n):
                if u[q]:
                    n_used += 1
                    touched.update((i, j))
                q += 1
        if n_used < dims or len(touched) < dims + 1:
            return np.array([lat, lon, h]), 0.0, 2, 0
        P = n_used
    lam = 1e-3
    cost, r = _ls_cost(s, rd, u, lat, lon, h)
    it = 0
    while it < 60:
        lr, lo = lat * math.pi / 180, lon * math.pi / 180
        sl, cl, so, co = math.sin(lr), math.cos(lr), math.sin(lo), math.cos(lo)
        w = math.sqrt(1 - e2 * sl * sl)
        Nr, Mr = _A / w, _A * (1 - e2) / (w * w * w)
        x = llh_to_ecef(lat, lon, h)
        g = []
        for k in range(n):
            ux, uy, uz = (x[0] - s[k][0]) / r[k], (x[1] - s[k][1]) / r[k], (x[2] - s[k][2]) / r[k]
            g.append((-so * ux + co * uy, -sl * co * ux - sl * so * uy + cl * uz, cl * co * ux + cl * so * uy + sl * uz))
        A = [[0.0] * 3 for _ in range(3)]
        b = [0.0] * 3
        q = 0
        for i in range(n):
            for j in range(i + 1, n):
                if u is None or u[q]:
                    fq = (r[j] - r[i]) - rd[q]
                    row = (g[j][0] - g[i][0], g[j][1] - g[i][1], g[j][2] - g[i][2])
                    for a in range(3):
                        b[a] += row[a] * fq
                        for c in range(3):
                            A[a][c] += row[a] * row[c]
                q += 1
        moved, d = False, [0.0, 0.0, 0.0]
        for _ in range(8):
            step = _ls_step(A, b, lam, dims)
            if step is None:
                d = [0.0, 0.0, 0.0]
                lam *= 10.0
                continue
            d = step
            clat = lat + d[1] / (Mr + h) * 180.0 / math.pi
            clon = lon + d[0] / ((Nr + h) * cl) * 180.0 / math.pi
            ch = h + d[2] if dims == 3 else h
            cc, rc = _ls_cost(s, rd, u, clat, clon, ch)
            if cc < cost:
                lat, lon, h, cost, r, moved = clat, clon, ch, cc, rc, True
                lam = max(lam / 3.0, 1e-12)
                break
            lam *= 4.0
        if not moved:
            break
        if math.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]) < 1e-6:
            it += 1
            break
        it += 1
    rms = math.sqrt(cost / P) if P > 0 else 0.0
    return np.array([lat, lon, h]), rms, 0 if cost == cost else 1, it


def _usable(rec, min_margin):
    if int(rec["flags"]) & (EMPTY | EDGE):
        return False
    return not (min_margin > 0 and float(rec["margin"]) < min_margin)


def window_time(nsamp, guard, kind, start, length):
    """centre of the window in the capture (kind 0 REF, 1 TGT); NaN for a REF window across blocks 1 and 3"""
    b = nsamp // 3
    g = min(guard, b)
    if kind == 1:
        k0 = b + g + start
    elif start < b:
        if start + length > b:
            return math.nan
        k0 = start
    else:
        k0 = 2 * b + g + (start - b)
    return float(k0) + 0.5 * float(length - 1)


def _line(ys, ts, keep):
    n, st, sy = 0, 0.0, 0.0
    for y, t, k in zip(ys, ts, keep):
        if k:
            n += 1; st += t; sy += y
    if n == 0:
        return 0.0, 0.0, 0.0, 0
    t_mean, a = st / n, sy / n
    stt = sty = 0.0
    for y, t, k in zip(ys, ts, keep):
        if k:
            dt = t - t_mean
            stt += dt * dt
            sty += dt * (y - a)
    beta = sty / stt if n > 1 and stt > 0.0 else 0.0
    return a, beta, t_mean, n


def window_fixes(stations_llh, nsamp, guard, win_start, win_len, hop, ref, tgt, fs=2e6, min_margin=0.0,
                 ref_max_residual=0.0, ref_tx_llh=None, dims=2, init_llh=None):
    """The windowed fix stage on tables ref[n_ref][P], tgt[n_tgt][P] of 32-byte peak records (win_len > 0).
    Returns a dict as Engine.process_windows."""
    st = np.asarray(stations_llh, np.float64).reshape(-1, 3)
    S = st.shape[0]
    P = S * (S - 1) // 2
    ref = np.asarray(ref).reshape(-1, P)
    tgt = np.asarray(tgt).reshape(-1, P)
    n_ref, nt = ref.shape[0], tgt.shape[0]
    min_margin = float(np.float32(min_margin))
    ref_fit = np.zeros((P, 3), np.float64)
    rd = np.full((nt, P), np.nan)
    used = np.zeros((nt, P), bool)
    p = 0
    for i in range(S):
        for j in range(i + 1, S):
            ts = [window_time(int(nsamp[i]), guard, 0, win_start + w * hop, win_len) for w in range(n_ref)]
            ys = [float(ref[w, p]["lag"]) + float(ref[w, p]["frac"]) for w in range(n_ref)]
            keep = [_usable(ref[w, p], min_margin) and not math.isnan(ts[w]) for w in range(n_ref)]
            a, beta, tm, n = _line(ys, ts, keep)
            if ref_max_residual > 0.0 and n > 0:
                keep = [k and not (abs(y - (a + beta * (t - tm))) > ref_max_residual) for y, t, k in zip(ys, ts, keep)]
                a, beta, tm, n = _line(ys, ts, keep)
            geo = 0.0
            if ref_tx_llh is not None:
                x = llh_to_ecef(*(float(v) for v in ref_tx_llh))
                geo = _dist(x, llh_to_ecef(*st[j])) - _dist(x, llh_to_ecef(*st[i]))
            b = int(nsamp[i]) // 3
            ref_fit[p] = (a + beta * ((float(b) + 0.5 * float(b - 1)) - tm) if n > 0 else 0.0, beta, float(n))
            for w in range(nt):
                rec = tgt[w, p]
                if n > 0 and _usable(rec, min_margin):
                    tw = window_time(int(nsamp[i]), guard, 1, win_start + w * hop, win_len)
                    y_ref = a + beta * (tw - tm)
                    rd[w, p] = ((float(rec["lag"]) + float(rec["frac"])) / fs - y_ref / fs) * C_LIGHT + geo
                    used[w, p] = True
            p += 1
    fix, rms = np.zeros((nt, 3)), np.zeros(nt)
    status, iters = np.zeros(nt, np.int32), np.zeros(nt, np.int32)
    for w in range(nt):
        fix[w], rms[w], status[w], iters[w] = solve_ls(st, rd[w], init_llh, dims, used[w])
    return {"ref_fit": ref_fit, "range_differences": rd, "pair_used": used, "position": fix, "rms": rms,
            "status": status, "iters": iters}
