"""Bounded lag search (tdoa_xcorr_bounded) against its restatement (tests/bounds_oracle.py) on every search path, the
TGT intervals of tdoa_set_tgt_bounds in the windowed calls (k_tgt_bounds pinned through the restated intervals), the
weak-target scenario, multi-GPU engines and the refusals."""
import ctypes as C

import numpy as np
import pytest

import tdoa_b200 as T
import bounds_oracle as B
import lag_edges as E
from oracle import oracle

pytestmark = pytest.mark.gpu

EDGE, BRUTE, EMPTY, OVERFLOW, BOUNDED = 0x2, 0x4, 0x8, 0x10, 0x20
STATE = EDGE | EMPTY | BOUNDED
RANK_EPS = 4e-6     # the FFT ranking's error bound, as tests/test_gpu_lag_edges.py takes it


@pytest.fixture
def extended_oracle():
    oracle.set_seq_dc_limit(0)
    yield
    oracle.set_seq_dc_limit(-1)


def load_all(e, raws):
    for k, r in enumerate(raws):
        e.load_u8(k, r)


def ncand(flags):
    return (np.asarray(flags) >> 16) & 0xff


# (name, stations, max_lag, window, planted lag of pair (0, 1), others, decimate): the 2 x 2 tiles over several
# 2048-lag chunks, the parked spectra (10 pairs), the 2^21-point transform, a decimated engine
CASES = [
    ("tiles_chunks", 2, 3000, 30000, -3000 + 2048, (), 1),
    ("spectra", 5, 4095, 30000, 0, (1, 37, 150), 1),
    ("big", 2, 5000, 40000, -5000 + 8192, (), 1),
    ("decimated", 2, 320, 24000, 200, (), 4),
]


def intervals(L, lag, D):
    """(lo, hi) cases in capture samples: the whole range, one lag, the 2048 and 4096 chunk joints, partly and wholly
    outside +-L (up to the int32 limits), and a true peak just outside the interval (EDGE at its boundary)."""
    R = L                                      # +-max_lag in capture samples
    out = [(-R, R), (lag, lag), (lag - 3 * D, lag + 3 * D), (R - 10 * D, R + 100), (R + D, R + 50 * D),
           (-R - 50 * D, -R - D), (lag + D, lag + 200 * D), (lag - 200 * D, lag - D), (-2 ** 31, 2 ** 31 - 1),
           # far beyond the range on either side, up to the int32 limits: empty runs
           (2 ** 31 - 1, 2 ** 31 - 1), (2 ** 31 - 11, 2 ** 31 - 1), (-2 ** 31, -2 ** 31), (-2 ** 31, -2 ** 31 + 10)]
    for j in (2047, 2048, 4095, 4096):
        k = -L // D + j
        if k <= L // D:
            out.append((D * (k - 2), D * (k + 2)))
    return out


def check_record(got, want, exact):
    assert int(got["lag"]) == want["lag"] and int(got["first_lag"]) == want["first_lag"], (got, want)
    assert int(got["flags"]) & STATE == want["flags"], (got, want)
    if exact:
        assert float(got["corr"]) == want["corr"] and got["frac"] == want["frac"] and got["margin"] == want["margin"]
    else:
        assert abs(float(got["corr"]) - want["corr"]) <= 1e-12 and abs(float(got["frac"]) - float(want["frac"])) <= 1e-6
        c = abs(want["corr"])
        assert abs(float(got["margin"]) - float(want["margin"])) * c <= RANK_EPS + 2.0 ** -23 * c


@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_statement_on_every_path(case, extended_oracle):
    name, S, L, W, lag, others, D = case
    raws, _ = E.planted(E.START + W + 300, lag, S, others, seed=abs(lag) % 97)
    cfg = dict(n_stations=S, max_lag=L, decimate=D)
    with T.Engine(T.MODE_EXTENDED, use_fft=0, **cfg) as e:
        load_all(e, raws)
        planes = [e.preprocess(k, T.KIND_TGT, E.START, W)[0] for k in range(S)]
    P = S * (S - 1) // 2
    pairs = [(i, j) for i in range(S) for j in range(i + 1, S)]
    corr = [oracle.xcorr_two_sided(planes[i], planes[j], L // D) for i, j in pairs]
    assert W // D - 2 * (L // D) <= 65536          # one block: the every-lag sum is the statement's sequential sum
    for u in (0, 1, 2, 3, 4):
        with T.Engine(T.MODE_EXTENDED, use_fft=u, **cfg) as e:
            load_all(e, raws)
            plain = e.xcorr(T.KIND_TGT, E.START, W, 1, 0)[0]
            for lo, hi in intervals(L, lag, D):
                got = e.xcorr_bounded(T.KIND_TGT, lo, hi, E.START, W, 1, 0)[0]
                for p in range(P):
                    check_record(got[p], B.bounded_peak(corr[p], lo, hi, D), exact=(u == 0))
                    assert got[p]["n_blocks"] == plain[p]["n_blocks"]
                    assert not got[p]["flags"] & OVERFLOW
                    assert bool(got[p]["flags"] & BRUTE) == (u == 0), (u, lo, hi)
                if lo <= -L and hi >= L:   # the whole range: tdoa_xcorr's record apart from the flag
                    g = got.copy()
                    g["flags"] &= ~np.uint32(BOUNDED)
                    assert g.tobytes() == plain.tobytes(), (u, lo, hi)


@pytest.mark.parametrize("n_ties", sorted(E.TIE_L))
def test_ties_across_the_cap(n_ties, extended_oracle):
    """63 / 66 tied candidates inside a whole-range run (the latter redone lag by lag, with its interval), and the 66
    ties of the unbounded search cut to one inside a run of 80 lags: no overflow, no redo."""
    L = E.TIE_L[n_ties]
    raws = E.tie_captures()
    S = len(E.TIE_DELAYS)
    P = S * (S - 1) // 2
    with T.Engine(T.MODE_EXTENDED, n_stations=S, max_lag=L) as e:
        load_all(e, raws)
        plain = e.xcorr(T.KIND_TGT, E.TIE_START, E.TIE_W, 1, 0)[0]
        whole = e.xcorr_bounded(T.KIND_TGT, -L, L, E.TIE_START, E.TIE_W, 1, 0)[0]
        assert np.all(whole["flags"] & BOUNDED)
        whole["flags"] &= ~np.uint32(BOUNDED)
        assert whole.tobytes() == plain.tobytes()
        assert np.all((plain["flags"] & BRUTE) != 0) == (3 * n_ties > E.MAX_CAND)
        lo = plain["lag"].astype(np.int64) - 40      # the first tie alone: the next ones are 165 lags away
        got = e.xcorr_bounded(T.KIND_TGT, lo, lo + 80, E.TIE_START, E.TIE_W, 1, 0)[0]
    assert not np.any(got["flags"] & (BRUTE | OVERFLOW)) and np.all(ncand(got["flags"]) <= 3)
    for p, (i, j) in enumerate([(i, j) for i in range(S) for j in range(i + 1, S)]):
        c = E.extended_ties(raws, E.TIE_START, E.TIE_W, L, i, j)
        want = B.bounded_peak(c, int(lo[p]), int(lo[p]) + 80)
        assert int(got[p]["lag"]) == want["lag"] and abs(float(got[p]["corr"]) - want["corr"]) <= 1e-6


# ------------------------------------------------------------------ the setting in the windowed calls
SCN_GEOM = (0, B.SCN_WIN, B.SCN_NT, B.SCN_HOP)
GRID = (38.90, -94.65, 0.005, 0.005, 40, 70, 250.0)


def scenario_engine(**kw):
    e = T.Engine(T.MODE_EXTENDED, n_stations=len(B.SCN_LLH), max_lag=B.SCN_MAX_LAG, **kw)
    return e


REF_TX = (39.20, -94.30, 300.0)
# the REF transmitter's geometric term (half = d, centre moved by -geo fs / c) with the refit
REF_OPTS = dict(ref_tx_llh=REF_TX, ref_max_residual=2.0)
# a margin test no REF record passes: no pair has a REF fit, so every TGT search stays unbounded
NO_FIT = dict(min_margin=0.99)


def windowed_calls():
    """name -> (call, the same options for window_fixes, the options of the REF fit for the restated intervals)"""
    s, w, n, h = SCN_GEOM
    llh = B.SCN_LLH
    clo = dict(closure=dict(max_residual=300.0, max_drop=0))
    exc = dict(exclusion=dict(max_rms=300.0, max_exclude=1))
    return {
        "plain": (lambda e: e.process_windows(llh, s, w, n, n, h), {}, {}),
        "ref_tx": (lambda e: e.process_windows(llh, s, w, n, n, h, **REF_OPTS), REF_OPTS, REF_OPTS),
        "no_fit": (lambda e: e.process_windows(llh, s, w, n, n, h, **NO_FIT), NO_FIT, NO_FIT),
        "grid": (lambda e: e.process_windows(llh, s, w, n, n, h, grid=GRID), dict(grid=GRID), {}),
        "retimed": (lambda e: e.process_windows_retimed(llh, SCN_GEOM, SCN_GEOM), {}, {}),
        "closure": (lambda e: e.process_windows(llh, s, w, n, n, h, **clo), clo, {}),
        "exclude": (lambda e: e.process_windows(llh, s, w, n, n, h, **exc), exc, {}),
    }


@pytest.fixture(scope="module")
def scenario():
    return B.scenario_captures()


@pytest.mark.parametrize("name", list(windowed_calls()))
def test_setting_in_the_windowed_calls(name, scenario):
    raws, _ = scenario
    call, fix_kw, fit_kw = windowed_calls()[name]
    s, w, n, h = SCN_GEOM
    nsamp = [r.size // 2 for r in raws]
    with scenario_engine() as e, scenario_engine() as fresh:
        load_all(e, raws)
        load_all(fresh, raws)
        base = call(fresh)
        t0 = fresh.stats()["launches_total"]
        base2 = call(fresh)
        fresh_launches = fresh.stats()["launches_total"] - t0
        e.set_tgt_bounds(B.SCN_GUARD)
        got = call(e)
        assert got["ref"].tobytes() == base["ref"].tobytes()              # the REF table is the unbounded call's
        lo, hi = B.tgt_intervals(B.SCN_LLH, nsamp, 0, SCN_GEOM, SCN_GEOM, got["ref"], B.SCN_GUARD, **fit_kw)
        if name == "no_fit":      # k_tgt_bounds' pair without a REF fit: the unbounded record, no BOUNDED flag
            assert np.all(lo == B.NO_BOUND[0]) and np.all(hi == B.NO_BOUND[1])
            assert got["tgt"].tobytes() == base["tgt"].tobytes()
            lo, hi = np.full_like(lo, -B.SCN_MAX_LAG), np.full_like(hi, B.SCN_MAX_LAG)
        else:
            assert not np.any(lo > hi)
            assert np.all(got["tgt"]["flags"] & BOUNDED)
        if name not in ("retimed", "no_fit"):     # the re-timed planes are not tdoa_xcorr's: their lags are checked against the intervals
            want = e.xcorr_bounded(T.KIND_TGT, lo, hi, s, w, n, h)
            assert got["tgt"].tobytes() == want.tobytes()                 # pins k_tgt_bounds bit for bit
        assert np.all((got["tgt"]["lag"] >= lo) & (got["tgt"]["lag"] <= hi))
        fx = e.window_fixes(B.SCN_LLH, s, w, got["ref"], got["tgt"], h, **fix_kw)
        for k in ("range_differences", "pair_used", "position", "rms", "status"):
            assert np.array_equal(fx[k], got[k], equal_nan=True) if fx[k].dtype.kind == "f" else np.array_equal(fx[k], got[k]), k
        e.set_tgt_bounds(None)
        t0 = e.stats()["launches_total"]
        off = call(e)
        assert e.stats()["launches_total"] - t0 == fresh_launches
        for k in ("ref", "tgt"):
            assert off[k].tobytes() == base2[k].tobytes() == base[k].tobytes(), k
        assert np.array_equal(off["position"], base2["position"])


def test_weak_target_scenario(scenario):
    """A weak target that repeats every 1500 samples (tests/bounds_oracle.py; the outcome established on the CPU
    oracle by tests/test_bounds_oracle.py).  Without bounds the receiver noise picks one of the target's repeats in
    +-20 000 lags: in every TGT window at least 5 of the 10 lags are more than 5 samples off and the fix is more than
    10 km off.  With guard = 5 the interval holds the true repeat alone: every TGT lag is within 1 sample and every
    fix within 100 m (the oracle's: 11, 34 and 44 m; measured on a B200: 12, 41 and 50 m)."""
    raws, d = scenario
    S = len(B.SCN_LLH)
    s, w, n, h = SCN_GEOM
    want = np.array([d[j] - d[i] for i in range(S) for j in range(i + 1, S)])
    x = B.W.llh_to_ecef(*B.SCN_TARGET)
    with scenario_engine() as e:
        load_all(e, raws)
        free = e.process_windows(B.SCN_LLH, s, w, n, n, h)
        e.set_tgt_bounds(B.SCN_GUARD)
        bnd = e.process_windows(B.SCN_LLH, s, w, n, n, h)
    err_free = np.abs(free["tgt"]["lag"] - want)
    err_bnd = np.abs(bnd["tgt"]["lag"] + bnd["tgt"]["frac"] - want)
    dist = lambda r: np.array([B.W._dist(x, B.W.llh_to_ecef(*p)) for p in r["position"]])
    print("unbounded lag errors", err_free.tolist(), "fix errors (m)", np.round(dist(free)).tolist(), free["status"].tolist())
    print("bounded lag errors", np.round(err_bnd, 3).tolist(), "fix errors (m)", np.round(dist(bnd), 1).tolist())
    assert np.all(np.count_nonzero(err_free > 5, axis=1) >= 5)
    assert np.all((dist(free) > 10e3) | (free["status"] != 0))
    assert np.all(err_bnd <= 1.0)
    assert np.all(bnd["status"] == 0) and np.all(dist(bnd) <= 100.0)


# ------------------------------------------------------------------ more than one GPU
def test_one_rank_communicator_and_two_devices(scenario):
    import torch
    raws, _ = scenario
    s, w, n, h = SCN_GEOM
    P = 10
    rng = np.random.default_rng(3)
    lo = rng.integers(-300, 0, (n, P)).astype(np.int32)
    hi = lo + rng.integers(0, 400, (n, P)).astype(np.int32)
    with scenario_engine() as one:
        load_all(one, raws)
        want_x = one.xcorr_bounded(T.KIND_TGT, lo, hi, s, w, n, h)
        one.set_tgt_bounds(B.SCN_GUARD)
        want_w = one.process_windows(B.SCN_LLH, s, w, n, n, h)
    engines = [("comm", {})]
    if torch.cuda.device_count() >= 2:
        engines.append(("n_devices", dict(n_devices=2)))
    for name, kw in engines:
        with scenario_engine(**kw) as e:
            if name == "comm":
                e.comm_init(T.comm_unique_id(), 0, 1)
            load_all(e, raws)
            got_x = e.xcorr_bounded(T.KIND_TGT, lo, hi, s, w, n, h)
            e.set_tgt_bounds(B.SCN_GUARD)
            got_w = e.process_windows(B.SCN_LLH, s, w, n, n, h)
        assert got_x.tobytes() == want_x.tobytes(), name
        for k in ("ref", "tgt"):
            assert got_w[k].tobytes() == want_w[k].tobytes(), (name, k)
        assert np.array_equal(got_w["position"], want_w["position"]), name


# ------------------------------------------------------------------ refusals
def test_refusals():
    raws, _ = E.planted(30000, 10, seed=1)
    with T.Engine(T.MODE_BINARY, n_stations=2) as b:
        load_all(b, raws)
        with pytest.raises(T.TdoaError):
            b.xcorr_bounded(T.KIND_TGT, -5, 5)
        with pytest.raises(T.TdoaError):
            b.set_tgt_bounds(5.0)
    with T.Engine(T.MODE_EXTENDED, n_stations=2, max_lag=300) as e:
        load_all(e, raws)
        with pytest.raises(T.TdoaError):
            e.xcorr_bounded(T.KIND_TGT, 5, 4, 0, 20000, 1, 0)
        out = np.zeros(1, T.PEAK_DTYPE)
        lo = np.zeros(1, np.int32)
        ptr = C.c_void_p(out.ctypes.data)
        lp = C.c_void_p(lo.ctypes.data)
        assert e._lib.tdoa_xcorr_bounded(e._h, T.KIND_TGT, 0, 20000, 1, 0, None, lp, ptr) == -1
        assert e._lib.tdoa_xcorr_bounded(e._h, T.KIND_TGT, 0, 20000, 1, 0, lp, None, ptr) == -1
        for on, g in ((2, 5.0), (-1, 5.0), (1, float("nan")), (1, float("inf")), (1, -1.0)):
            assert e._lib.tdoa_set_tgt_bounds(e._h, on, g) == -1, (on, g)
        e.set_tgt_bounds(0.0)
        e.set_tgt_bounds(None)
