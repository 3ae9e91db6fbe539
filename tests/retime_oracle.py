"""Plain restatement of re-timed target correlation (tdoa_process_windows_retimed; test infrastructure only).

  - station_rates:  the station clock rates from the per-pair REF fits, in k_station_rates' order of operations
                    (Python floats are IEEE doubles rounded to nearest, with no fused multiply-add);
  - delta, retime:  the re-timing index delta(n) = floor(c (n - n_c) + 0.5) and the gather of one plane (numpy
                    evaluates multiply and add as separate roundings, as k_retime does);
  - window_record:  one TGT window of one pair as the engine computes it: in EXTENDED mode (decimated or not)
                    oracle.preprocess_binary_dec, re-time, oracle.xcorr_two_sided, oracle.peak_parabolic; in BINARY
                    mode oracle.preprocess_binary, re-time, oracle.tdcorr_binary.
The range differences and fixes are tests/window_oracle.py's, unchanged.  The product never imports this module."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle


def pairs(S):
    return [(i, j) for i in range(S) for j in range(i + 1, S)]


def station_rates(beta, n_windows, S):
    """beta[p], n_windows[p] per pair p = (i, j), i < j (ref_fit[:, 1] and ref_fit[:, 2]).  Returns (rate, clock_rate):
    rate re-times the planes (0 for a station without a fitted pair), clock_rate is what the call returns (NaN
    there)."""
    pp = pairs(S)
    use = [float(n_windows[p]) >= 2.0 for p in range(len(pp))]
    comp = list(range(S))
    changed = True
    while changed:
        changed = False
        for p, (i, j) in enumerate(pp):
            if use[p]:
                m = min(comp[i], comp[j])
                if comp[i] != m or comp[j] != m:
                    comp[i] = comp[j] = m
                    changed = True
    A = [[1.0 if comp[i] == comp[j] else 0.0 for j in range(S)] for i in range(S)]
    b = [0.0] * S
    fitted = [False] * S
    for p, (i, j) in enumerate(pp):
        if not use[p]:
            continue
        A[i][i] += 1.0; A[j][j] += 1.0; A[i][j] -= 1.0; A[j][i] -= 1.0
        b[i] = b[i] - float(beta[p])
        b[j] = b[j] + float(beta[p])
        fitted[i] = fitted[j] = True
    for k in range(S):
        A[k][k] = math.sqrt(A[k][k])
        for i in range(k + 1, S):
            A[i][k] = A[i][k] / A[k][k]
        for i in range(k + 1, S):
            for j in range(k + 1, i + 1):
                A[i][j] = A[i][j] - A[i][k] * A[j][k]
    for k in range(S):
        b[k] = b[k] / A[k][k]
        for i in range(k + 1, S):
            b[i] = b[i] - A[i][k] * b[k]
    for k in range(S - 1, -1, -1):
        b[k] = b[k] / A[k][k]
        for i in range(k):
            b[i] = b[i] - A[k][i] * b[k]
    rate = np.array(b, np.float64)
    return rate, np.where(fitted, rate, np.nan)


def delta(c, length):
    """delta(n) for n in [0, length): floor(c (n - n_c) + 0.5), n_c = (length - 1) / 2, every step rounded"""
    n = np.arange(length, dtype=np.float64)
    nc = float(length - 1) * 0.5
    return np.floor(np.float64(c) * (n - nc) + 0.5).astype(np.int64)


def retime(x, c):
    """x~[n] = x[n + delta(n)] where that index is on the plane, 0 elsewhere.  The source index is formed in doubles,
    as k_retime forms it, so a rate far beyond any clock's (|delta| past 2^63) still reads 0 rather than a wrapped
    integer."""
    x = np.asarray(x)
    n = np.arange(x.size, dtype=np.float64)
    nc = float(x.size - 1) * 0.5
    s = n + np.floor(np.float64(c) * (n - nc) + 0.5)
    ok = (s >= 0.0) & (s < float(x.size))
    out = np.zeros_like(x)
    out[ok] = x[s[ok].astype(np.int64)]
    return out


def window_record(sig_i, sig_j, c_i, c_j, max_lag, shift=0, mode="extended", D=1, block=10000, sanity=120):
    """(lag, frac, corr) of one TGT window of pair (i, j) on re-timed planes.  sig_*: the two stations' TGT samples
    of the window (complex, as oracle.extract_target gives them).

    mode "extended", decimate D: oracle.preprocess_binary_dec, re-time in the decimated plane's own samples (its
    centre is (n / D - 1) / 2), oracle.xcorr_two_sided over +-(max_lag // D) and oracle.peak_parabolic.  lag and
    frac are in decimated samples (the engine reports D (lag + frac), rounded, in capture samples).  shift: an
    integer the lag is known to be near -- plane j is moved by it before correlating, so that a far lag needs few
    lags (the engine's records always come from the full lag range; this is the same value when the peak lies well
    inside both ranges).
    mode "binary": oracle.preprocess_binary, re-time the complex plane (both parts), oracle.tdcorr_binary with the
    engine's max_lag, block and sanity; frac is 0."""
    if mode == "binary":
        yi = retime(oracle.preprocess_binary(sig_i)[0], c_i)
        yj = retime(oracle.preprocess_binary(sig_j)[0], c_j)
        lag, val, _ = oracle.tdcorr_binary(yi, yj, max_lag, block, sanity)
        return lag, 0.0, val
    assert mode == "extended", mode
    yi = retime(oracle.preprocess_binary_dec(sig_i, D)[0], c_i)
    yj = retime(oracle.preprocess_binary_dec(sig_j, D)[0], c_j)
    max_lag //= D
    if shift:
        z = np.zeros_like(yj)
        if shift > 0:
            z[:-shift] = yj[shift:]
        else:
            z[-shift:] = yj[:shift]
        yj = z
    idx, frac, val = oracle.peak_parabolic(oracle.xcorr_two_sided(yi, yj, max_lag))
    return idx - max_lag + shift, frac, val
