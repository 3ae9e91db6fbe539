"""The FFT search's ranking plane restated (tests/test_ranking_oracle.py, tests/test_gpu_ranking.py).

Every FFT search path ranks the lags on an f32 plane `approx` and evaluates exactly only the lags k_select_candidates
keeps: those within TOL of the maximum |approx|.  Here: the exact plane the ranking approximates (an f64 correlation
of the engine's own normalised planes over every lag the record searches), the selection and the margin stated on
the f32 plane, and a CPU emulation of one packed ranking transform (two real planes in one complex FFT, split with
Z[k] +- conj Z[N - k]) that shows why the planes must share a scale before they share a transform."""
from __future__ import annotations

import numpy as np

import lag_edges as E

TOL = E.TOL


def correlate(t, s, n_t: int, n_lags: int, t_off: int = 0, device=None):
    """c[d] = sum_{m < n_t} t[t_off + m] s[m + d], d in [0, n_lags), in f64 (s is 0 past its end).  An f64 FFT
    (torch on `device` when given, numpy otherwise): exact products and sums up to ~1e-16 of sum |t| |s|."""
    a = np.asarray(t[t_off:t_off + n_t], np.float64)
    b = np.asarray(s[:n_t + n_lags - 1], np.float64)
    N = 1 << int(np.ceil(np.log2(max(2, n_t + n_lags - 1))))
    if device is not None:
        import torch
        A = torch.fft.rfft(torch.from_numpy(a).to(device), n=N)
        B = torch.fft.rfft(torch.from_numpy(b).to(device), n=N)
        c = torch.fft.irfft(torch.conj(A) * B, n=N)[:n_lags].cpu().numpy()
        del A, B
        return c
    return np.fft.irfft(np.conj(np.fft.rfft(a, N)) * np.fft.rfft(b, N), N)[:n_lags]


def exact_extended(yi, yj, L: int, device=None):
    """EXTENDED's plane of pair (i, j) over lags -L..L: signal i the template, W = min(n_i, n_j), t_off = L,
    n_t = W - 2L, corr = sum / n_t (lag_edges.unequal_statement); yi, yj the engine's normalised planes (decimated
    ones included)."""
    W = min(yi.size, yj.size)
    n_t = W - 2 * L
    return correlate(np.real(yi[:W]), np.real(yj[:W]), n_t, 2 * L + 1, t_off=L, device=device) / n_t


def exact_binary(yi, yj, max_lag: int, block: int, device=None):
    """BINARY's first-pass plane: the shorter plane is the template (signal i on a tie), tl_eff = tl - max_lag for
    equal lengths, n_lags = min(max_lag, sl - tl_eff) (at least 1), sum over nb whole blocks of B / (nb B)."""
    t, s = (yj, yi) if yi.size > yj.size else (yi, yj)
    tl, sl = t.size, s.size
    tl_eff = tl - max_lag if sl == tl else tl
    n_lags = max(1, min(max_lag, sl - tl_eff))
    n_t = (tl_eff // block) * block
    return correlate(np.real(t), np.real(s), n_t, n_lags, device=device) / n_t


def binary_at(yi, yj, max_lag: int, block: int, lag: int) -> float:
    """BINARY's correlation at one lag as the reference sums it: each product rounded to f32 (which the f64 plane
    above does not do: it differs from this by ~1e-9), block sums / B, their mean over the nb blocks."""
    t, s = (yj, yi) if yi.size > yj.size else (yi, yj)
    tl_eff = t.size - max_lag if s.size == t.size else t.size
    nb = tl_eff // block
    p = (np.real(t[:nb * block]).astype(np.float32) * np.real(s[lag:lag + nb * block]).astype(np.float32))
    return float(np.mean(p.reshape(nb, block).astype(np.float64).sum(axis=1) / block))


def select(approx, tol: float = TOL, neighbours: bool = False, sanity: int = 0):
    """k_select_candidates on the f32 plane: lag_edges.candidates in f32 arithmetic."""
    return E.candidates(np.asarray(approx, np.float32), neighbours, sanity, tol)


def margin(approx, best: int, corr: float) -> np.float32:
    """k_peak_candidates' margin: f32((|corr| - max_{i != best} |approx_i|) / |corr|), the maximum taken in f32 and
    the rest in f64; best and corr are the first pass's (first_lag's index, and its correlation)."""
    a = np.abs(np.asarray(approx, np.float32))
    ru = np.float32(np.max(np.delete(a, best))) if a.size > 1 else np.float32(0.0)
    if corr == 0.0:
        return np.float32(0.0)
    return np.float32((abs(corr) - np.float64(ru)) / abs(corr))


# ------------------------------------------------------------------ CPU emulation of one packed transform
def emulate_packed(t, s, n_lags: int, seg: int, N: int = 8192, prescale: bool = False):
    """The ranking of c[d] = sum_m t[m] s[m + d] / n as the tile kernels compute it, in f32 (scipy.fft on
    complex64): each segment of `seg` template samples and its N-sample signal span packed as z = t + i s, one
    FFT, T[k] = (Z[k] + conj Z[N-k]) / 2 and S[k] = (Z[k] - conj Z[N-k]) / 2i, conj(T) S summed over the segments
    in complex64, one inverse.  The planes carry their scales sc_t = 1 / rms(t), sc_s = 1 / rms(s): applied after
    the inverse (prescale False), or to every sample before packing (prescale True)."""
    import scipy.fft as F
    t = np.asarray(t, np.float32)
    s = np.asarray(s, np.float32)
    sc_t = np.float32(1.0 / np.sqrt(np.mean(t.astype(np.float64) ** 2)))
    sc_s = np.float32(1.0 / np.sqrt(np.mean(s.astype(np.float64) ** 2)))
    n = t.size
    if prescale:
        t, s = t * sc_t, s * sc_s
    acc = np.zeros(N, np.complex64)
    k = np.arange(N)
    for t0 in range(0, n, seg):
        z = np.zeros(N, np.complex64)
        m = min(seg, n - t0)
        z.real[:m] = t[t0:t0 + m]
        span = s[t0:t0 + N]
        z.imag[:span.size] = span
        Z = F.fft(z)
        Zc = np.conj(Z[(-k) % N])
        T = (Z + Zc) * np.float32(0.5)
        S = (Z - Zc) * np.complex64(-0.5j)
        acc += np.conj(T) * S
    c = F.ifft(acc).real[:n_lags].astype(np.float64)
    return c / n if prescale else c * (np.float64(sc_t) * np.float64(sc_s)) / n
