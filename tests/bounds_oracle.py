"""Plain restatement of the bounded lag search (tdoa_xcorr_bounded) and of the TGT intervals the windowed calls
compute with tdoa_set_tgt_bounds on (k_tgt_bounds); test infrastructure only, the product never imports it.

Python floats are IEEE doubles with no fused multiply-add, so `tgt_intervals` rounds as k_tgt_bounds does when it
follows the operation order include/tdoa_b200.h states; the REF fit is tests/window_oracle.py's and the baseline is
k_baselines' (llh_to_ecef, then sqrt(dx dx + dy dy + dz dz)).  `bounded_peak` is the statement of one record over the
correlation oracle.xcorr_two_sided gives."""
from __future__ import annotations

import math

import numpy as np

import window_oracle as W
from helpers import fm_signal, quantise

EDGE, EMPTY, BOUNDED = 0x2, 0x8, 0x20
NO_BOUND = (2 ** 31 - 1, -2 ** 31)   # a pair without a REF fit: the search stays unbounded
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


def _ceil_div(a: int, d: int) -> int:
    return -((-a) // d)


def run(lo: int, hi: int, L: int, D: int = 1):
    """The run of lag indices i (lag k = i - L, k in -L..L at the correlation's own rate) with lo <= D k <= hi."""
    i0 = max(0, _ceil_div(lo, D) + L)
    i1 = min(2 * L, hi // D + L)
    return i0, i1


def bounded_peak(c, lo: int, hi: int, D: int = 1):
    """One record of the bounded search over c = xcorr_two_sided(..., L) (index i is lag i - L): dict of lag,
    corr, frac, margin, flags (EDGE / EMPTY / BOUNDED) and first_lag, in capture samples (k_lag_units for D > 1)."""
    c = np.asarray(c, np.float64)
    L = (c.size - 1) // 2
    i0, i1 = run(lo, hi, L, D)
    rec = dict(lag=0, corr=0.0, frac=np.float32(0.0), margin=np.float32(0.0), flags=BOUNDED, first_lag=0)
    if i0 > i1:
        rec["flags"] |= EMPTY
        return rec
    a = np.abs(c[i0:i1 + 1])
    b = int(np.argmax(a))                       # the first maximum: the lowest lag wins ties
    if a[b] == 0.0:
        b = 0
    v = float(c[i0 + b]) if a[b] != 0.0 else 0.0
    second = float(np.max(np.delete(a, b))) if a.size > 1 else 0.0
    idx = i0 + b
    rec["corr"] = v
    rec["margin"] = np.float32((abs(v) - second) / abs(v)) if v != 0.0 else np.float32(0.0)
    if i0 < idx < i1:
        x, m, y = abs(c[idx - 1]), abs(c[idx]), abs(c[idx + 1])
        den = x - 2.0 * m + y
        rec["frac"] = np.float32(0.5 * (x - y) / den) if den != 0.0 else np.float32(0.0)
    else:
        rec["flags"] |= EDGE
    k = idx - L
    if D > 1:                                    # k_lag_units: D (lag + frac), rounded to the nearest lag
        total = float(D) * (float(k) + float(rec["frac"]))
        whole = float(np.rint(total))
        rec["lag"], rec["frac"], rec["first_lag"] = int(whole), np.float32(total - whole), k * D
    else:
        rec["lag"] = rec["first_lag"] = k
    return rec


def baseline(a_llh, b_llh) -> float:
    """k_baselines: sqrt(dx dx + dy dy + dz dz) between the ECEF points."""
    a, b = W.llh_to_ecef(*(float(v) for v in a_llh)), W.llh_to_ecef(*(float(v) for v in b_llh))
    dx, dy, dz = b[0] - a[0], b[1] - a[1], b[2] - a[2]
    return math.sqrt(dx * dx + dy * dy + dz * dz)


def _clamp(v: float) -> int:
    return I32_MIN if v <= -2147483648.0 else (I32_MAX if v >= 2147483647.0 else int(v))


def interval(a, beta, t_mean, geo, t_w, d, has_ref_tx, guard, fs=2e6):
    """The header's operation order for one (TGT window, pair) with a REF fit."""
    y_ref = a + beta * (t_w - t_mean)
    centre = y_ref - geo / W.C_LIGHT * fs
    half = (d if has_ref_tx else 2.0 * d) / W.C_LIGHT * fs + guard
    return _clamp(math.ceil(centre - half)), _clamp(math.floor(centre + half))


def tgt_intervals(stations_llh, nsamp, cfg_guard, ref_geom, tgt_geom, ref, guard, fs=2e6, min_margin=0.0,
                  ref_max_residual=0.0, ref_tx_llh=None):
    """lo, hi [n_tgt][P] (int64 holding int32 values; NO_BOUND where the pair has no REF fit) from the REF table
    ref[n_ref][P], as k_window_ref_fit + k_baselines + k_tgt_bounds compute them.  *_geom = (start, len, n, hop)."""
    st = np.asarray(stations_llh, np.float64).reshape(-1, 3)
    S = st.shape[0]
    P = S * (S - 1) // 2
    ref = np.asarray(ref).reshape(-1, P)
    rs, rl, rn, rh = ref_geom
    ts_, tl, tn, th = tgt_geom
    min_margin = float(np.float32(min_margin))
    lo = np.zeros((tn, P), np.int64)
    hi = np.zeros((tn, P), np.int64)
    p = 0
    for i in range(S):
        for j in range(i + 1, S):
            ts = [W.window_time(int(nsamp[i]), cfg_guard, 0, rs + w * rh, rl) for w in range(rn)]
            ys = [float(ref[w, p]["lag"]) + float(ref[w, p]["frac"]) for w in range(rn)]
            keep = [W._usable(ref[w, p], min_margin) and not math.isnan(ts[w]) for w in range(rn)]
            a, beta, tm, n = W._line(ys, ts, keep)
            if ref_max_residual > 0.0 and n > 0:
                keep = [k and not (abs(y - (a + beta * (t - tm))) > ref_max_residual) for y, t, k in zip(ys, ts, keep)]
                a, beta, tm, n = W._line(ys, ts, keep)
            geo = 0.0
            if ref_tx_llh is not None:
                x = W.llh_to_ecef(*(float(v) for v in ref_tx_llh))
                geo = W._dist(x, W.llh_to_ecef(*st[j])) - W._dist(x, W.llh_to_ecef(*st[i]))
            d = baseline(st[i], st[j])
            for w in range(tn):
                if n > 0:
                    tw = W.window_time(int(nsamp[i]), cfg_guard, 1, ts_ + w * th, tl)
                    lo[w, p], hi[w, p] = interval(a, beta, tm, geo, tw, d, ref_tx_llh is not None, guard, fs)
                else:
                    lo[w, p], hi[w, p] = NO_BOUND
            p += 1
    return lo, hi


# ------------------------------------------------------------------ the weak-target scenario
# Five stations 10-17 km apart around a target; the REF transmitter is equidistant (REF delays 0, no has_ref_tx), so
# every TGT interval is the REF lag +- 2 d fs / c + guard (<= ~170 samples wide on each side) while the search without
# it covers +-SCN_MAX_LAG.  Block 2 is weak (raw power < 0.001: the weak branch, whose band-pass is linear): a faint
# target that repeats its content every SCN_PERIOD samples (a beacon, a looped announcement), in receiver noise of its
# own at each station.  Every repeat of the true lag holds the same target correlation, so outside the interval the
# receiver noise picks one of ~2 SCN_MAX_LAG / SCN_PERIOD equal peaks; inside it there is only the true one.
SCN_LLH = np.array([[39.00, -94.50, 250.0], [39.08, -94.42, 260.0], [38.97, -94.36, 240.0],
                    [39.06, -94.62, 255.0], [38.93, -94.55, 245.0]])
SCN_TARGET = (39.02, -94.49, 250.0)
SCN_MAX_LAG = 20000
SCN_BLOCK = 200000
SCN_WIN, SCN_HOP, SCN_NT = 60000, 65000, 3        # TGT windows [w * hop, + win) of block 2
SCN_REF = (0, 60000, 3, 65000)                    # REF windows in block 1
SCN_GUARD = 5.0
SCN_PERIOD = 1500                                 # > every interval's width: one repeat inside
SCN_AMP, SCN_NOISE = 0.02, 0.01                   # target amplitude and per-component noise of block 2
SCN_SEED = 11


def scenario_delays(fs=2e6):
    """TGT delay of each station (samples, integer, the nearest station 0): round(r_k fs / c) - min."""
    x = W.llh_to_ecef(*SCN_TARGET)
    r = [W._dist(x, W.llh_to_ecef(*s)) for s in SCN_LLH]
    d = [int(round(v * fs / W.C_LIGHT)) for v in r]
    m = min(d)
    return [v - m for v in d]


def scenario_captures(amp: float = SCN_AMP, noise: float = SCN_NOISE, seed: int = SCN_SEED, period: int = SCN_PERIOD):
    """One capture per station: blocks 1 and 3 a strong FM REF programme with no delay (noise 0.02), block 2 a faint
    FM target of amplitude `amp` that repeats every `period` samples (0: never), delayed by scenario_delays(), in
    complex Gaussian noise of `noise` per component, independent per station."""
    d = scenario_delays()
    B = SCN_BLOCK
    pad = max(d) + 16
    ref = fm_signal(2 * B, 100 + seed, 75e3)
    if period:
        one = fm_signal(period, 200 + seed, 60e3, amp, taps=8)
        tgt = np.tile(one, -(-(B + pad) // period))[:B + pad]
    else:
        tgt = fm_signal(B + pad, 200 + seed, 60e3, amp, taps=8)
    raws = []
    for k, dk in enumerate(d):
        g = np.random.default_rng(1000 * seed + k)
        b1 = ref[:B] + 0.02 * (g.standard_normal(B) + 1j * g.standard_normal(B))
        b2 = tgt[pad - dk:pad - dk + B] + noise * (g.standard_normal(B) + 1j * g.standard_normal(B))
        b3 = ref[B:] + 0.02 * (g.standard_normal(B) + 1j * g.standard_normal(B))
        raws.append(quantise(np.concatenate([b1, b2, b3])))
    return raws, d
