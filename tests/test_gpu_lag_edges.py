"""Lag searches where kernels break: planted lags on the edges of the lag range and of every search's chunks,
exact ties whose candidate count straddles the cap of 64 (the lag-by-lag redo in every call that can need it), a
station with its I and Q bytes swapped (corr exactly negated), the margin field on every path, and EXTENDED on
stations of unequal length.  Every case runs on every search path that can serve it (default, use_fft = 2, 3, 4)
against the every-lag path (use_fft = 0) and against the oracle; tests/test_lag_edges_oracle.py proves the
captures' properties on the CPU."""
import numpy as np
import pytest

import tdoa_b200 as T
from oracle import oracle
from helpers import STATION_LLH, fm_capture
import lag_edges as E

pytestmark = pytest.mark.gpu

CORR_TOL = 1e-6
FFT_PATHS = (1, 2, 3, 4)
RESEARCHED, EDGE, BRUTE, EMPTY, OVERFLOW = 0x1, 0x2, 0x4, 0x8, 0x10
# Margin on the FFT paths: the runner-up is the largest |approx| over the other lags, and every approximate value is
# within eps of its exact one (DESIGN §4: ~1e-6 in coefficient units), so |margin_fft - margin_exact| <=
# eps / |corr| plus the f32 rounding of the two margins.  eps is taken as 4 x the stated error.
RANK_EPS = 4e-6
margin_worst = [0.0]   # largest |margin_fft - margin_exact| * |corr| seen (printed with -s)


def ncand(flags):
    return (np.asarray(flags) >> 16) & 0xff


@pytest.fixture
def extended_oracle():
    oracle.set_seq_dc_limit(0)   # EXTENDED mode: exactly rounded DC sum
    yield
    oracle.set_seq_dc_limit(-1)


def load_all(e, raws):
    for k, r in enumerate(raws):
        e.load_u8(k, r)


def run_paths(mode, raws, call, paths=(0,) + FFT_PATHS, **cfg):
    out = {}
    for u in paths:
        with T.Engine(mode, use_fft=u, **cfg) as e:
            load_all(e, raws)
            out[u] = call(e)
    return out


def check_against_every_lag(out, overflow=None):
    """Every FFT path against use_fft = 0.  overflow: mask of the records whose candidates exceed the cap (they
    must come back redone lag by lag, equal to the every-lag record field for field); None: no record overflows."""
    ref = out[0]
    assert np.all(ref["flags"] & BRUTE) and not np.any(ref["flags"] & OVERFLOW)
    over = np.zeros(ref.shape, bool) if overflow is None else np.broadcast_to(overflow, ref.shape)
    for u in out:
        if u == 0:
            continue
        got = out[u]
        for name in ("lag", "first_lag", "n_blocks"):
            assert np.array_equal(got[name], ref[name]), (u, name)
        assert np.array_equal(got["flags"] & (RESEARCHED | EDGE | EMPTY), ref["flags"] & (RESEARCHED | EDGE | EMPTY)), u
        assert np.max(np.abs(got["corr"] - ref["corr"])) <= 1e-12, u
        assert np.max(np.abs(got["frac"] - ref["frac"])) <= 1e-6, u
        assert not np.any(got["flags"] & OVERFLOW), u                         # never left in a returned record
        assert np.all((got["flags"][over] & BRUTE) != 0), u                   # the cap forced the redo
        assert got[over].tobytes() == ref[over].tobytes(), u
        assert np.all(ncand(got["flags"][~over]) > 0) and not np.any(got["flags"][~over] & BRUTE), u   # FFT ran
        fine = ~over & (ref["corr"] != 0)
        dm = np.abs(got["margin"][fine].astype(np.float64) - ref["margin"][fine]) * np.abs(ref["corr"][fine])
        if dm.size:
            margin_worst[0] = max(margin_worst[0], float(dm.max()))
            print(f"margin: path {u} worst |dmargin| * |corr| = {dm.max():.3e} (so far {margin_worst[0]:.3e})")
        assert np.all(dm <= RANK_EPS + 2.0 ** -23 * np.abs(ref["corr"][fine])), (u, dm.max())


def exact_margin(c):
    """margin as k_peak computes it over every lag: f32((|c_max| - max over l != arg-max of |c_l|) / |c_max|)."""
    a = np.abs(c)
    best = int(np.argmax(a))
    second = np.max(np.delete(a, best)) if a.size > 1 else 0.0
    return np.float32((a[best] - second) / a[best]) if c[best] != 0 else np.float32(0.0)


def pairs_of(S):
    return [(i, j) for i in range(S) for j in range(i + 1, S)]


# ------------------------------------------------------------------ 1. planted lags on the edges
@pytest.mark.parametrize("case", E.EDGE_CASES, ids=lambda c: c[0])
def test_planted_edge_lag_on_every_path(case, extended_oracle):
    name, S, L, W, lag, others = case
    raws, _ = E.edge_capture(case)
    out = run_paths(T.MODE_EXTENDED, raws, lambda e: e.xcorr(T.KIND_TGT, E.START, W, 1, 0)[0], n_stations=S, max_lag=L)
    check_against_every_lag(out)
    want_lags = [int(np.clip(lag, -L, L))] + list(others)
    with T.Engine(T.MODE_EXTENDED, n_stations=S, max_lag=L, use_fft=0) as e:
        load_all(e, raws)
        planes = [e.preprocess(k, T.KIND_TGT, E.START, W)[0] for k in range(S)]
    for p, want in enumerate(want_lags):              # pairs (0, 1), (0, 2), ...: the planted ones
        j = p + 1
        yi, _ = oracle.preprocess_binary(E.split(raws[0])[1][E.START:E.START + W])
        yj, _ = oracle.preprocess_binary(E.split(raws[j])[1][E.START:E.START + W])
        idx, frac, val = oracle.peak_parabolic(oracle.xcorr_two_sided(yi, yj, L))
        assert idx - L == want
        for u, rec in out.items():
            r = rec[p]
            assert int(r["lag"]) == want, (u, p)
            assert abs(float(r["frac"]) - frac) <= 1e-3 and abs(float(r["corr"]) - val) <= CORR_TOL, (u, p)
            if abs(want) == L:
                assert r["flags"] & EDGE and r["frac"] == 0.0, (u, p)
            else:
                assert not r["flags"] & EDGE, (u, p)
        # margin of the every-lag path: the statement over every lag of the engine's own planes, bit for bit
        # (one 65536-sample block: the brute sum is the statement's sequential sum)
        c = oracle.xcorr_two_sided(planes[0], planes[j], L)
        assert W - 2 * L <= 65536
        assert out[0][p]["corr"] == c[idx]
        assert out[0][p]["margin"] == exact_margin(c), (out[0][p]["margin"], exact_margin(c))


@pytest.mark.parametrize("sanity", [E.SANITY, 0])
@pytest.mark.parametrize("lag", E.BINARY_EDGE_LAGS)
def test_binary_edge_lag_on_every_path(lag, sanity):
    raws, _ = E.planted(E.BINARY_BLOCK, lag, seed=lag % 53)
    out = run_paths(T.MODE_BINARY, raws, lambda e: e.xcorr(T.KIND_TGT)[0], n_stations=2, sanity_lag=sanity)
    check_against_every_lag(out)
    yi, _ = oracle.preprocess_binary(E.split(raws[0])[1])
    yj, _ = oracle.preprocess_binary(E.split(raws[1])[1])
    d, c, researched = oracle.tdcorr_binary(yi, yj, sanity=sanity)
    for u, rec in out.items():
        r = rec[0]
        assert int(r["lag"]) == d and int(r["first_lag"]) == lag, u
        assert abs(float(r["corr"]) - c) <= CORR_TOL and bool(r["flags"] & RESEARCHED) == researched, u
    assert researched == (sanity > 0 and lag == E.SANITY + 1)


def test_decimated_lag_at_the_range_edge(extended_oracle):
    for lag in (E.DEC_L, -E.DEC_L):
        raws, _ = E.planted(E.START + E.DEC_W + 300, lag, seed=5, dev_tgt=20e3)
        out = run_paths(T.MODE_EXTENDED, raws, lambda e: e.xcorr(T.KIND_TGT, E.START, E.DEC_W, 1, 0)[0], n_stations=2,
                        max_lag=E.DEC_L, decimate=E.DEC_D)
        check_against_every_lag(out)
        for u, rec in out.items():        # k_lag_units: D * (lag + frac), frac 0 on the edge
            assert int(rec[0]["lag"]) == lag and rec[0]["frac"] == 0.0 and rec[0]["flags"] & EDGE, u
            assert int(rec[0]["first_lag"]) == lag, u


@pytest.mark.parametrize("L", E.SWITCH_LAGS)
def test_the_2_20_lag_switch(L, extended_oracle):
    """2^20 - 1 lags... 2^20 + 1 lags: the 2^21-point transform serves up to kBigN / 2 lags; one more and the search
    falls back to 513 chunks of 2048 lags.  Default and use_fft = 3 give the same records at both; the correlation
    at the planted lag and its neighbours is a numpy f64 sum over the oracle's planes."""
    W = 2 * L + E.SWITCH_EXTRA
    raws, _ = E.planted(E.START + W + 300, E.SWITCH_LAG, seed=9)
    out = run_paths(T.MODE_EXTENDED, raws, lambda e: e.xcorr(T.KIND_TGT, E.START, W, 1, 0)[0], paths=(1, 3),
                    n_stations=2, max_lag=L)
    a, b = out[1][0], out[3][0]
    assert a.tobytes() == b.tobytes() or (a["lag"] == b["lag"] and abs(a["corr"] - b["corr"]) <= 1e-12
                                          and abs(a["frac"] - b["frac"]) <= 1e-6)
    assert int(a["lag"]) == E.SWITCH_LAG and ncand(a["flags"]) > 0 and not a["flags"] & BRUTE
    yi, _ = oracle.preprocess_binary(E.split(raws[0])[1][E.START:E.START + W])
    yj, _ = oracle.preprocess_binary(E.split(raws[1])[1][E.START:E.START + W])
    n = W - 2 * L
    t = yi.real[L:L + n].astype(np.float64)
    c = [float(np.dot(t, yj.real[L + l:L + l + n].astype(np.float64)) / n) for l in (E.SWITCH_LAG - 1, E.SWITCH_LAG,
                                                                                        E.SWITCH_LAG + 1)]
    assert abs(float(a["corr"]) - c[1]) <= CORR_TOL
    x, m, y = abs(c[0]), abs(c[1]), abs(c[2])
    assert abs(float(a["frac"]) - 0.5 * (x - y) / (x - 2 * m + y)) <= 1e-3


# ------------------------------------------------------------------ 2. exact ties across the cap
@pytest.mark.parametrize("n_ties", sorted(E.TIE_L))
def test_extended_ties_across_the_cap(n_ties, extended_oracle):
    """21 tied peaks: 63 candidates, the FFT paths settle the ties (lowest lag wins); 22: 66 candidates, the cap
    is exceeded and every pair comes back redone lag by lag (BRUTE), the every-lag record."""
    L = E.TIE_L[n_ties]
    raws = E.tie_captures()
    S = len(E.TIE_DELAYS)
    out = run_paths(T.MODE_EXTENDED, raws, lambda e: e.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 1, 0)[0], n_stations=S,
                    max_lag=L)
    over = n_ties * 3 > E.MAX_CAND
    check_against_every_lag(out, overflow=over)
    for u in FFT_PATHS:
        if not over:
            assert np.all(ncand(out[u]["flags"]) == 3 * n_ties), u
    for p, (i, j) in enumerate(pairs_of(S)):
        c = E.extended_ties(raws, E.TIE_START, E.TIE_W, L, i, j)
        idx, frac, val = oracle.peak_parabolic(c)    # the first of the ties
        for u, rec in out.items():
            assert int(rec[p]["lag"]) == idx - L, (u, p)
            assert abs(float(rec[p]["corr"]) - val) <= CORR_TOL and abs(float(rec[p]["frac"]) - frac) <= 1e-3, (u, p)
        assert out[0][p]["margin"] == 0.0           # the runner-up is another tied lag


def test_binary_ties_across_the_cap():
    """64 candidates (no overflow) on pairs (0, 1) and (1, 2), 65 on pair (0, 2): that pair alone is redone."""
    raws = E.tie_captures(binary=True)
    out = run_paths(T.MODE_BINARY, raws, lambda e: e.xcorr(T.KIND_TGT)[0], n_stations=3)
    over = np.array([c > E.MAX_CAND for c in E.BTIE_COUNT])
    check_against_every_lag(out, overflow=over)
    for u in FFT_PATHS:
        assert ncand(out[u]["flags"])[~over].tolist() == [c for c in E.BTIE_COUNT if c <= E.MAX_CAND], u
    for p, (i, j) in enumerate(pairs_of(3)):
        yi, _ = oracle.preprocess_binary(E.split(raws[i])[1])
        yj, _ = oracle.preprocess_binary(E.split(raws[j])[1])
        d, c, researched = oracle.tdcorr_binary(yi, yj)
        for u, rec in out.items():
            assert int(rec[p]["lag"]) == d and abs(float(rec[p]["corr"]) - c) <= CORR_TOL, (u, p)
            assert bool(rec[p]["flags"] & RESEARCHED) == researched, (u, p)


def test_overflow_redo_in_every_call(extended_oracle):
    """The 66-candidate content through the calls that check the cap after their own synchronisation: tdoa_xcorr
    over 2 windows (the two-stream optimistic pass), tdoa_process (whole signals), tdoa_process_windows (its
    tables are tdoa_xcorr_windows' field for field, margin included), each equal to the every-lag engine's."""
    L = E.TIE_L[22]
    raws = E.tie_captures()[:3]
    with T.Engine(T.MODE_EXTENDED, n_stations=3, max_lag=L) as e, \
            T.Engine(T.MODE_EXTENDED, n_stations=3, max_lag=L, use_fft=0) as b:
        load_all(e, raws)
        load_all(b, raws)
        got, want = e.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 2, 3000), b.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 2, 3000)
        assert np.all(got["flags"] & BRUTE) and got.tobytes() == want.tobytes()
        r, rb = e.process(STATION_LLH), b.process(STATION_LLH)
        for k in ("ref", "tgt"):
            assert np.all(r[k]["flags"] & BRUTE) and r[k].tobytes() == rb[k].tobytes(), k
        for k in ("time_differences", "range_differences", "position"):
            assert np.array_equal(r[k], rb[k]), k
        geo = (E.TIE_START, E.TIE_W, 3, 2, 4000)
        pw, xw, xb = e.process_windows(STATION_LLH, *geo), e.xcorr_windows(*geo), b.xcorr_windows(*geo)
        for k, t in (("ref", 0), ("tgt", 1)):
            assert pw[k].tobytes() == xw[t].tobytes() == xb[t].tobytes(), k
            assert np.all(pw[k]["flags"] & BRUTE), k


def test_overflow_redo_dealt_over_two_gpus(extended_oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = E.TIE_L[22]
    raws = E.tie_captures()[:3]
    with T.Engine(T.MODE_EXTENDED, n_stations=3, max_lag=L, n_devices=2) as e, \
            T.Engine(T.MODE_EXTENDED, n_stations=3, max_lag=L, use_fft=0) as b:
        load_all(e, raws)
        load_all(b, raws)
        got, want = e.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 4, 2000), b.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 4, 2000)
    assert np.all(got["flags"] & BRUTE) and got.tobytes() == want.tobytes()


# ------------------------------------------------------------------ 3. a station with I and Q swapped
@pytest.mark.parametrize("mode", ["BINARY", "EXTENDED"])
def test_swapped_iq_station_negates_its_pairs(mode):
    """i conj(x): the discriminator's products and the arctangent are sign-symmetric, so station 1's planes are
    exactly the negation and every pair with it keeps lag, frac, first_lag and flags, corr exactly negated; margin
    too on the every-lag path.  On the FFT paths margin moves within the ranking bound: every FFT kernel packs two
    real planes into one complex transform (k_fft_tiles: FFT(t0 + i t1); k_fft_segments: t + i s; the parked spectra
    and the 2^21-point transform: two stations per transform), and t + i(-s) is not the negation of t + i s, so
    its f32 rounding -- and the approximate runner-up the margin takes -- differs in the last bits, while the
    candidates' exact values are exactly negated."""
    raws = fm_capture(60000, (0, 5, 12), (0, 9, 31), seed=3)
    sw = [raws[0], E.swap_iq(raws[1]), raws[2]]
    kw = dict(max_lag=300) if mode == "EXTENDED" else {}
    for u in (0,) + FFT_PATHS:
        with T.Engine(getattr(T, "MODE_" + mode), use_fft=u, **kw) as e:
            res = []
            for caps in (raws, sw):
                load_all(e, caps)
                res.append(np.concatenate([e.xcorr(T.KIND_REF)[0], e.xcorr(T.KIND_TGT)[0]]))
        a, b = res
        with_1 = np.array([True, False, True] * 2)          # pairs (0, 1), (0, 2), (1, 2) of REF, then TGT
        for name in ("lag", "frac", "first_lag", "flags", "n_blocks"):
            assert np.array_equal(a[name], b[name]), (u, name)
        if u == 0:
            assert np.array_equal(a["margin"], b["margin"])
        else:
            dm = np.abs(a["margin"].astype(np.float64) - b["margin"]) * np.abs(a["corr"])
            assert np.all(dm <= RANK_EPS + 2.0 ** -23 * np.abs(a["corr"])), (u, dm.max())
        assert np.array_equal(b["corr"][with_1], -a["corr"][with_1]), u
        assert np.array_equal(b["corr"][~with_1], a["corr"][~with_1]), u


# ------------------------------------------------------------------ 5. unequal lengths in EXTENDED
@pytest.mark.parametrize("extra", [1, 7, 3001])
def test_extended_unequal_lengths_keep_signal_1_as_template(extra, extended_oracle):
    """Station i is the template whatever the lengths: with W = min(n_i, n_j) the correlation is
    xcorr_two_sided(y_i[:W], y_j[:W], L), each y preprocessed over its own full length, and the lag d_j - d_i."""
    L, D = 300, 4
    d = (0, 17, 40)
    pairs = pairs_of(3)
    for longer in range(3):
        blocks = [30000 + (extra if k == longer else 0) for k in range(3)]
        raws = E.ragged(blocks, d, seed=extra)
        out = run_paths(T.MODE_EXTENDED, raws, lambda e: np.concatenate([e.xcorr(T.KIND_REF, 0, 0)[0],
                                                                         e.xcorr(T.KIND_TGT, 0, 0)[0]]), max_lag=L)
        check_against_every_lag(out)
        for kind in (0, 1):
            ys = [oracle.preprocess_binary(E.split(r)[kind])[0] for r in raws]
            for p, (i, j) in enumerate(pairs):
                idx, frac, val = oracle.peak_parabolic(E.unequal_statement(ys[i], ys[j], L))
                assert idx - L == d[j] - d[i]
                for u, rec in out.items():
                    r = rec[3 * kind + p]
                    assert int(r["lag"]) == d[j] - d[i], (longer, kind, p, u)
                    assert abs(float(r["frac"]) - frac) <= 1e-3 and abs(float(r["corr"]) - val) <= CORR_TOL, (longer, kind, p, u)
        with T.Engine(T.MODE_EXTENDED, max_lag=L) as e:
            load_all(e, raws)
            r = e.process(STATION_LLH)
        for k, kind in (("ref", 0), ("tgt", 1)):
            assert r[k].tobytes() == out[1][3 * kind:3 * kind + 3].tobytes(), (longer, k)
        with T.Engine(T.MODE_EXTENDED, max_lag=L, decimate=D) as e:
            load_all(e, raws)
            rec = e.xcorr(T.KIND_TGT, 0, 0)[0]
        ys = [oracle.preprocess_binary_dec(E.split(r)[1], D)[0] for r in raws]
        for p, (i, j) in enumerate(pairs):
            idx, frac, _ = oracle.peak_parabolic(E.unequal_statement(ys[i], ys[j], L // D))
            want = D * (idx - L // D + frac)
            got = int(rec[p]["lag"]) + float(rec[p]["frac"])
            assert abs(got - want) <= 1e-3 * D, (longer, p)
            assert abs(got - (d[j] - d[i])) <= 0.75, (longer, p)
