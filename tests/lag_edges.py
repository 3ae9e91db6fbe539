"""Captures for the lag-search edge tests (tests/test_lag_edges_oracle.py, tests/test_gpu_lag_edges.py): lags
planted on the edges of the lag range and of the search's chunks, exact ties whose count straddles the candidate
cap, a station with its I and Q bytes swapped, stations of unequal length.  The properties the GPU tests rely on
are proven on the CPU oracle by tests/test_lag_edges_oracle.py."""
from __future__ import annotations

import numpy as np

from helpers import fm_capture, fm_signal, quantise
from oracle import oracle

TOL = 2e-5        # k_select_candidates' ranking tolerance (|approx| within TOL of the maximum is a candidate)
MAX_CAND = 64     # kMaxCand: more candidates than this and the pair is redone lag by lag
BINARY_LAGS = 2000
SANITY = 120


def split(raw):
    d = oracle.unpack_u8(raw)
    return oracle.extract_reference(d), oracle.extract_target(d)


def planted(block: int, lag: int, n_stations: int = 2, others=(), seed: int = 0, **kw):
    """fm_capture whose pair (0, 1) has TGT lag d_1 - d_0 = lag (station 0 is delayed for a negative lag);
    `others` are the delays of stations 2.. relative to station 0's."""
    d0 = max(0, -lag)
    d = [d0, d0 + lag] + [d0 + x for x in others]
    assert len(d) == n_stations
    return fm_capture(block, d, d, seed=seed, **kw), d


def swap_iq(raw: np.ndarray) -> np.ndarray:
    """The capture with I and Q exchanged: x -> i conj(x), whose FM discriminator output is the negation."""
    out = np.empty_like(raw)
    out[0::2], out[1::2] = raw[1::2], raw[0::2]
    return out


# EXTENDED cases: (name, stations, max_lag, window, planted lag of pair (0, 1), delays of stations 2.. from station 0)
START = 200   # first TGT sample of the correlated window
EDGE_CASES = [
    ("range_lo", 2, 300, 20000, -300, ()),
    ("range_lo1", 2, 300, 20000, -299, ()),
    ("range_hi1", 2, 300, 20000, 299, ()),
    ("range_hi", 2, 300, 20000, 300, ()),
    ("range_out", 2, 300, 20000, 301, ()),            # just outside: the record is +L with EDGE
    ("range_out_lo", 2, 300, 20000, -301, ()),
    # 6001 lags in 2048-lag chunks: lag indices 2047 | 2048 and 4095 | 4096 (2 x 2 tiles)
    ("chunk1_lo", 2, 3000, 30000, -3000 + 2047, ()),
    ("chunk1_hi", 2, 3000, 30000, -3000 + 2048, ()),
    ("chunk2_lo", 2, 3000, 30000, -3000 + 4095, ()),
    ("chunk2_hi", 2, 3000, 30000, -3000 + 4096, ()),
    # 10 pairs on the parked spectra, 8191 lags in chunks of 4096 and 4095: pair (0, 1) at lag 0 (index 4095),
    # pair (0, 2) at lag 1 (index 4096)
    ("spectra_joint", 5, 4095, 30000, 0, (1, 37, 150)),
    # the 2^21-point transform: 8193 lags put +L alone in row 1
    ("big_lo", 2, 4096, 30000, -4096, ()),
    ("big_lo1", 2, 4096, 30000, -4095, ()),
    ("big_hi1", 2, 4096, 30000, 4095, ()),
    ("big_hi", 2, 4096, 30000, 4096, ()),
    ("big_row_lo", 2, 5000, 40000, -5000 + 8191, ()),   # the row joint of 10001 lags
    ("big_row_hi", 2, 5000, 40000, -5000 + 8192, ()),
]
BINARY_EDGE_LAGS = [0, 1, 119, 120, 121, 1998, 1999]
BINARY_BLOCK = 42000
DEC_L, DEC_D, DEC_W = 320, 4, 24000      # decimate = 4: the lag at +-L, i.e. +-80 at the decimated rate
SWITCH_LAGS = (524287, 524288)           # 2^20 - 1 lags: the big transform; 2^20 + 1: 513 chunks of 2048 lags
SWITCH_LAG, SWITCH_EXTRA = 300000, 60000


def edge_capture(case):
    name, S, L, W, lag, others = case
    raws, d = planted(START + W + 300, lag, S, others, seed=abs(lag) % 97)
    return raws, d


# ------------------------------------------------------------------ exact ties
def periodic(n_samples: int, period: int, delays, seed: int = 7, dev: float = 75e3, taps: int = 8):
    """Captures whose bytes repeat with `period` samples: one period of fm_signal, quantised once and tiled;
    station k is the tile rolled by delays[k] (it lags station 0 by delays[k]), with no noise of its own.  Every
    block of a capture is a window of the same periodic sequence, so REF and TGT are too."""
    one = quantise(fm_signal(period, seed, dev, taps=taps)).reshape(period, 2)
    reps = -(-(n_samples + max(delays) + period) // period)
    tile = np.tile(one, (reps, 1))
    return [np.ascontiguousarray(tile[period - d % period:][:n_samples].reshape(-1)) for d in delays]


# every pair lag is 33, 66, 99 or 132; with these ranges each pair has exactly 21 (22) tied peaks in -L..L, every
# one >= 32 lags inside the range, and the next tie outside it: 63 and 66 candidates with the +-1 neighbours
TIE_PERIOD, TIE_DELAYS, TIE_BLOCK = 165, (0, 33, 66, 99, 132), 165 * 182   # block = whole periods: REF is periodic
TIE_START, TIE_W = 1000, 20000
TIE_L = {21: 1748, 22: 1814}
BTIE_PERIOD, BTIE_DELAYS, BTIE_BLOCK = 31, (0, 20, 10), 31 * 968
BTIE_COUNT = [64, 65, 64]      # pairs (0, 1), (0, 2), (1, 2): ties at 20, 10, 21 (mod 31) in [0, 2000)


def tie_captures(binary: bool = False):
    if binary:
        return periodic(3 * BTIE_BLOCK, BTIE_PERIOD, BTIE_DELAYS)
    return periodic(3 * TIE_BLOCK, TIE_PERIOD, TIE_DELAYS)


def extended_ties(raws, start: int, W: int, L: int, i: int = 0, j: int = 1):
    """Oracle correlation of TGT window [start, start + W) of stations i, j over lags -L..L."""
    yi, _ = oracle.preprocess_binary(split(raws[i])[1][start:start + W])
    yj, _ = oracle.preprocess_binary(split(raws[j])[1][start:start + W])
    return oracle.xcorr_two_sided(yi, yj, L)


def binary_lags(raws, i: int = 0, j: int = 1, max_lag: int = BINARY_LAGS):
    """Every lag of BINARY's first pass over whole TGT signals of equal length (template = signal i shortened
    by max_lag), as the reference computes them."""
    yi, _ = oracle.preprocess_binary(split(raws[i])[1])
    yj, _ = oracle.preprocess_binary(split(raws[j])[1])
    assert yi.size == yj.size
    return oracle.tdcorr_binary_lags_mt(yi, yj, yi.size - max_lag, max_lag)


def candidates(c, neighbours: bool, sanity: int = 0, tol: float = TOL):
    """The lags k_select_candidates keeps, on exact values: within tol of the maximum |c|, within tol of the
    maximum over [0, sanity) when sanity > 0, and (neighbours) the lags either side of a lag of the first set.
    An f32 plane (the FFT ranking) is compared in f32, as the kernel does; anything else in f64."""
    dt = np.float32 if np.asarray(c).dtype == np.float32 else np.float64
    a = np.abs(np.asarray(c, dt))
    tol = dt(tol)
    m1 = a.max()
    take = a >= dt(m1 - tol)
    first = take.copy()
    if sanity > 0:
        m2 = a[:sanity].max()
        take[:sanity] |= a[:sanity] >= dt(m2 - tol)
    if neighbours:
        take[1:] |= first[:-1]
        take[:-1] |= first[1:]
    return np.flatnonzero(take)


def selection_gap(c, sanity: int = 0):
    """How far the candidate set stands from changing: the smallest distance, in |c|, between a lag outside
    the set and the threshold it would need to cross (the maximum, or the [0, sanity) maximum).  A gap over
    5 x TOL means the f32 ranking's error (under 1e-6, tests/test_gpu_ranking.py) cannot change which lags are
    candidates."""
    a = np.abs(np.asarray(c, np.float64))
    m1 = a.max()
    top = a >= m1 - TOL
    gaps = [m1 - a[~top].max()] if (~top).any() else []
    if sanity > 0:
        s = a[:sanity]
        m2 = s.max()
        stop = s >= m2 - TOL
        if (~stop).any():
            gaps.append(m2 - s[~stop].max())
    return min(gaps)


# ------------------------------------------------------------------ unequal lengths
def ragged(blocks, delays, seed: int = 0, noise: float = 0.02, dev_ref: float = 75e3, dev_tgt: float = 60e3,
           amp: float = 0.5):
    """One capture per station with its own block length blocks[k]: all blocks start at the same time (up to
    the station's delay), so the stations differ only at the end.  Block 3 continues the REF signal where block
    1 stopped, so REF (blocks 1 and 3) is one continuous stretch of 2 blocks[k] samples, and every pair of
    REF or TGT signals has the planted lag d_j - d_i over its common length."""
    n = 2 * max(blocks) + max(delays) + 64
    ref = fm_signal(n, 1000 + seed, dev_ref, amp)
    tgt = fm_signal(n, 2000 + seed, dev_tgt, amp)
    pad = max(delays) + 16
    raws = []
    for k, (b, d) in enumerate(zip(blocks, delays)):
        g = np.random.default_rng(3000 + 17 * seed + k)

        def cut(sig, first, m):
            s = sig[pad - d + first:pad - d + first + m]
            return s + noise * (g.standard_normal(m) + 1j * g.standard_normal(m))

        raws.append(quantise(np.concatenate([cut(ref, 0, b), cut(tgt, 0, b), cut(ref, b, b)])))
    return raws


def unequal_statement(yi, yj, L: int):
    """EXTENDED on signals of unequal length: signal i is the template, W = min(n_i, n_j), and the correlation is
    xcorr_two_sided(y_i[:W], y_j[:W], L), each y preprocessed over its own full length."""
    W = min(yi.size, yj.size)
    return oracle.xcorr_two_sided(yi[:W], yj[:W], L)
