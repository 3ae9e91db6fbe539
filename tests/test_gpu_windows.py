"""Windowed ProcessTDOA (tdoa_process_windows / tdoa_window_fixes; window_fix.cu): one fix per TGT window with
the REF clock drift fitted across blocks 1 and 3.

The captures here drift: station k's sample n is src[n - d_k - round(eps_k n)] over the WHOLE capture (the clock
runs on through the retunes), d_k from the REF transmitter in blocks 1 and 3 and from the TX in block 2.  So the
lag of pair (i, j) at capture sample t is (d_j - d_i) + (eps_j - eps_i) t: the REF windows see a line of slope
eps_j - eps_i, and the time difference a TGT window should report is (dT_j - dT_i) - (dR_j - dR_i) whatever
its time."""
import numpy as np
import pytest
import torch

import tdoa_b200 as T
from helpers import STATION_LLH, fm_capture, fm_signal, quantise
import window_oracle as WO
from oracle import oracle

FS, C = 2e6, 299792458.0
B, W = 4_000_000, 500_000            # test-sized block; windows of W at hop W
N_REF, N_TGT = 2 * B // W, B // W    # 16 REF windows (8 per REF block), 8 TGT windows
L = 300                              # lags: delays up to ~100 samples + drift up to 60 samples
ST4 = np.vstack([STATION_LLH, [41.20, -96.20, 340.0]])
TX = np.array([41.25, -96.05, 350.0])
REF_TX = np.array([41.10, -95.80, 400.0])
EPS_PPM = np.array([0.0, 4.0, -5.0, 2.0])


def pairs(S):
    return [(i, j) for i in range(S) for j in range(i + 1, S)]


def delays(stations, x_llh):
    x = oracle.llh_to_ecef(*x_llh)
    r = np.array([np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in stations])
    d = np.round(r / C * FS).astype(np.int64)
    return d - d.min()


def drift_captures(stations=ST4, eps_ppm=EPS_PPM, block=B, seed=5, noise=0.02):
    dR, dT = delays(stations, REF_TX), delays(stations, TX)
    n = 3 * block
    pad = int(max(dR.max(), dT.max()) + np.abs(eps_ppm).max() * 1e-6 * n) + 16
    ref = fm_signal(n + 2 * pad, 1000 + seed, 75e3)
    tgt = fm_signal(n + 2 * pad, 2000 + seed, 60e3)
    t = np.arange(n)
    in_tgt = (t >= block) & (t < 2 * block)
    raws = []
    for k in range(len(stations)):
        d = np.where(in_tgt, dT[k], dR[k]) + np.round(eps_ppm[k] * 1e-6 * t).astype(np.int64)
        idx = pad + t - d
        x = np.where(in_tgt, tgt[idx], ref[idx])
        g = np.random.default_rng(3000 + 17 * seed + k)
        x = x + noise * (g.standard_normal(n) + 1j * g.standard_normal(n))
        raws.append(quantise(x))
    return raws, dR, dT


@pytest.fixture(scope="module")
def drift():
    return drift_captures()


def window_lag(raws, i, j, kind, w):
    """the oracle pipeline (the binary's preprocessing, two-sided correlation, parabolic peak) on one window"""
    out = []
    for k in (i, j):
        d = oracle.unpack_u8(raws[k])
        sig = oracle.extract_reference(d) if kind == T.KIND_REF else oracle.extract_target(d)
        y, _ = oracle.preprocess_binary(sig[w * W:(w + 1) * W])
        out.append(y)
    idx, frac, _ = oracle.peak_parabolic(oracle.xcorr_two_sided(out[0], out[1], L))
    return idx - L + frac


def test_drift_captures_give_the_lags_the_tests_assert(drift):
    """CPU: the captures carry lag (d_j - d_i) + (eps_j - eps_i) t, t the window centre (checked on a REF window
    of block 1, one of block 3 and a TGT window, on the pair with the largest drift)."""
    raws, dR, dT = drift
    i, j = 1, 2
    deps = (EPS_PPM[j] - EPS_PPM[i]) * 1e-6
    oracle.set_seq_dc_limit(0)
    try:
        for kind, w, d, t0 in ((T.KIND_REF, 0, dR, 0), (T.KIND_REF, N_REF - 1, dR, B), (T.KIND_TGT, 3, dT, B)):
            t = t0 + w * W + (W - 1) / 2
            assert abs(window_lag(raws, i, j, kind, w) - ((d[j] - d[i]) + deps * t)) < 1.0
    finally:
        oracle.set_seq_dc_limit(-1)


def load_all(e, raws):
    for k, r in enumerate(raws):
        e.load_u8(k, r)


def y_of(tab):
    return tab["lag"].astype(np.float64) + tab["frac"].astype(np.float64)


# ------------------------------------------------------------------ drift, end to end
@pytest.mark.gpu
def test_drift_end_to_end(drift):
    raws, dR, dT = drift
    S = len(ST4)
    pp = pairs(S)
    truth = np.array([(dT[j] - dT[i]) - (dR[j] - dR[i]) for i, j in pp], np.float64)
    deps = np.array([(EPS_PPM[j] - EPS_PPM[i]) * 1e-6 for i, j in pp])
    init = [ST4[:, 0].mean(), ST4[:, 1].mean(), TX[2]]
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=S) as e:
        load_all(e, raws)
        out = e.process_windows(ST4, 0, W, N_REF, N_TGT, W)
        geo = e.process_windows(ST4, 0, W, N_REF, N_TGT, W, ref_tx_llh=REF_TX, init_llh=init)
    assert out["pair_used"].all()
    td = out["range_differences"] * FS / C
    assert np.abs(td - truth).max() <= 1.0
    assert np.abs(out["ref_fit"][:, 1] - deps).max() <= 0.05e-6
    assert np.array_equal(out["ref_fit"][:, 2], [N_REF] * len(pp))
    # the naive corrections, from the returned tables, miss by far more than 1 sample
    ref_y, tgt_y = y_of(out["ref"]), y_of(out["tgt"])
    same_index = tgt_y - ref_y[:N_TGT]
    whole_signal = tgt_y - ref_y.mean(axis=0)
    assert np.abs(same_index - truth).max() > 10.0
    assert np.abs(whole_signal - truth).max() > 5.0
    # with the REF transmitter's position the range differences are TDOAs and the fixes find the TX.
    # Bound: each range difference is off by at most 1 sample (above) + 1 sample of rounding in the REF
    # delays (the captures hold round(r / c * fs) per station, the geometric term the exact distances) + 1 of
    # rounding in the TX delays: delta <= 3 c / fs = 450 m per pair.  Linearised at the TX, the horizontal error
    # is pinv(J) delta, J the P x 2 matrix of d rd_p / d(east, north): |error| <= ||pinv(J)||_2 sqrt(P) 450 m.
    x0 = oracle.llh_to_ecef(*TX)

    def rds(lat, lon):
        x = oracle.llh_to_ecef(lat, lon, TX[2])
        r = [np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in ST4]
        return np.array([r[j] - r[i] for i, j in pp])
    h = 1e-5
    m_lat = np.linalg.norm(oracle.llh_to_ecef(TX[0] + h, TX[1], TX[2]) - x0)
    m_lon = np.linalg.norm(oracle.llh_to_ecef(TX[0], TX[1] + h, TX[2]) - x0)
    J = np.column_stack([(rds(TX[0], TX[1] + h) - rds(*TX[:2])) / m_lon, (rds(TX[0] + h, TX[1]) - rds(*TX[:2])) / m_lat])
    bound = np.linalg.norm(np.linalg.pinv(J), 2) * np.sqrt(len(pp)) * 3 * C / FS
    assert (geo["status"] == 0).all()
    for w in range(N_TGT):
        assert np.linalg.norm(oracle.llh_to_ecef(*geo["position"][w]) - x0) <= bound


# ------------------------------------------------------------------ tables
@pytest.mark.gpu
def test_tables_are_xcorr_windows_tables(drift):
    raws = drift[0]
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=len(ST4)) as e:
        load_all(e, raws)
        ref, tgt = e.xcorr_windows(0, W, N_REF, N_TGT, W)
        out = e.process_windows(ST4, 0, W, N_REF, N_TGT, W)
    assert out["ref"].tobytes() == ref.tobytes()
    assert out["tgt"].tobytes() == tgt.tobytes()


# ------------------------------------------------------------------ fix stage vs the oracle
def injected(S, seed, n_ref=16, n_tgt=8, b=4000, w=500):
    """tables whose TGT lags are a TX's range differences on top of a per-pair REF drift line, with some
    EMPTY / EDGE / low-margin records and one outlier; stations scattered around the three collectors"""
    g = np.random.default_rng(seed)
    st = np.vstack([STATION_LLH, STATION_LLH.mean(0) + g.uniform([-0.15, -0.2, -30], [0.15, 0.2, 30], (S - 3, 3))])[:S]
    P = S * (S - 1) // 2
    x = oracle.llh_to_ecef(*TX)
    r = np.array([np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in st])
    xr = oracle.llh_to_ecef(*REF_TX)
    q = np.array([np.linalg.norm(xr - oracle.llh_to_ecef(*s)) for s in st])
    rd = np.array([(r[j] - r[i]) - (q[j] - q[i]) for i, j in pairs(S)])   # what the REF term adds back
    a0, beta = g.uniform(-50, 50, P), g.uniform(-5e-6, 5e-6, P)
    tc = b + (b - 1) / 2
    t_ref = np.array([(k * w if k * w < b else 2 * b + (k * w - b)) + (w - 1) / 2 for k in range(n_ref)])
    t_tgt = np.array([b + k * w + (w - 1) / 2 for k in range(n_tgt)])
    ref_y = a0 + beta * (t_ref[:, None] - tc) + g.normal(0, 0.05, (n_ref, P))
    tgt_y = a0 + beta * (t_tgt[:, None] - tc) + rd * FS / C + g.normal(0, 0.05, (n_tgt, P))
    tabs = []
    for y in (ref_y, tgt_y):
        t = np.zeros(y.shape, T.PEAK_DTYPE)
        t["lag"] = np.round(y).astype(np.int32)
        t["frac"] = (y - np.round(y)).astype(np.float32)
        t["margin"] = g.uniform(0.05, 0.9, y.shape).astype(np.float32)
        tabs.append(t)
    ref, tgt = tabs
    ref["flags"][2, 0] = T.PEAK_EMPTY
    ref["flags"][5, P - 1] = T.PEAK_EDGE
    ref["lag"][7, 1] += 200                                  # an outlier for the refit
    ref["flags"][:, 2] |= T.PEAK_EMPTY                       # pair 2: no REF fit
    tgt["flags"][1, P - 1] = T.PEAK_EMPTY
    tgt["flags"][n_tgt - 1, :] = T.PEAK_EMPTY                # status 2: nothing left
    tgt["flags"][n_tgt - 1, 0] = 0
    caps = [np.random.default_rng(seed + k).integers(0, 256, 6 * b, dtype=np.uint8) for k in range(S)]
    return st, ref, tgt, caps, b, w


@pytest.mark.gpu
@pytest.mark.parametrize("S,dims,mode", [(3, 2, T.MODE_BINARY), (3, 2, T.MODE_EXTENDED), (16, 2, T.MODE_EXTENDED),
                                         (16, 3, T.MODE_EXTENDED)])
def test_fix_stage_matches_oracle(S, dims, mode):
    st, ref, tgt, caps, b, w = injected(S, 40 + S + dims)
    P = S * (S - 1) // 2
    # dims 3 starts 1.4 km from the TX: from the station mean (2 km) the nearly flat station layout leaves the
    # elevation column so weak that no damped step lowers the cost and the solver stops where it started
    init = [STATION_LLH[:, 0].mean(), STATION_LLH[:, 1].mean(), TX[2]] if dims == 2 else [TX[0] + 0.01, TX[1] - 0.01, TX[2]]
    kw = dict(min_margin=0.1, ref_max_residual=20.0, ref_tx_llh=REF_TX, init_llh=init)
    with T.Engine(mode, n_stations=S) as e:
        load_all(e, caps)
        got = e.window_fixes(st, 0, w, ref, tgt, w, dims=dims, **kw)
    want = WO.window_fixes(st, [3 * b] * S, 0, 0, w, w, ref, tgt, fs=FS, dims=dims, **kw)
    assert np.abs(got["ref_fit"] - want["ref_fit"]).max() <= 1e-9
    assert np.array_equal(got["pair_used"], want["pair_used"])
    u = want["pair_used"]
    assert np.abs(got["range_differences"][u] - want["range_differences"][u]).max() <= 1e-6
    assert np.isnan(got["range_differences"][~u]).all()
    assert np.array_equal(got["status"], want["status"])
    assert want["status"][-1] == 2 and got["iters"][-1] == 0
    assert (want["status"][:-1] == 0).all()
    # fixes within 1e-4 m of the statement's -- plus what the statement itself does with range differences one
    # rounding apart: the device's sin / cos / sqrt are not the C library's in the last bit, and on a flat valley
    # (the elevation of a ground transmitter, dims 3) that moves the stopping point (0.36 mm measured on one window)
    g = np.random.default_rng(1)
    for k in range(len(got["status"])):
        sens = 0.0
        if want["status"][k] == 0:
            x0 = np.array(WO.llh_to_ecef(*want["position"][k]))
            for _ in range(3):
                rd1 = want["range_differences"][k] * (1 + g.uniform(-1, 1, P) * 2.0 ** -52)
                p1 = WO.solve_ls(st, rd1, init, dims, want["pair_used"][k])[0]
                sens = max(sens, float(np.linalg.norm(np.array(WO.llh_to_ecef(*p1)) - x0)))
        d = oracle.llh_to_ecef(*got["position"][k]) - oracle.llh_to_ecef(*want["position"][k])
        assert np.linalg.norm(d) <= 1e-4 + 10 * sens
    assert np.abs(got["rms"] - want["rms"]).max() <= 1e-6
    assert (got["iters"][:-1] > 0).all()
    # the fixes are where the TX is (noise 0.05 samples = 7.5 m per pair; dims 3 also solves the poorly observed
    # elevation of a ground transmitter seen by ground stations)
    for k in range(len(got["status"]) - 1):
        assert np.linalg.norm(oracle.llh_to_ecef(*got["position"][k]) - oracle.llh_to_ecef(*TX)) < (100 if dims == 2 else 500)


# ------------------------------------------------------------------ the reference's own correction
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [T.MODE_BINARY, T.MODE_EXTENDED])
def test_whole_blocks_are_tdoa_process(mode):
    """win_len = hop = b, guard 0, no drift, no REF position: REF windows = blocks 1 and 3, the TGT window =
    block 2, the line through two points evaluated at their midpoint = their mean."""
    b = 300000
    raws = fm_capture(b, (0, 3, 8), (0, 20, 41), seed=3)
    with T.Engine(mode, chunk_samples=0) as e:
        load_all(e, raws)
        whole = e.process(STATION_LLH)
        got = e.process_windows(STATION_LLH, 0, b, 2, 1, b)
    want = whole["range_differences"]
    assert got["pair_used"].all()
    assert got["tgt"].tobytes() == whole["tgt"].tobytes()   # the TGT window is the whole TGT signal
    if mode == T.MODE_BINARY:
        assert np.array_equal(got["range_differences"][0], want)
    else:
        # the one difference is the REF value: mean of the two block records instead of the whole-signal record
        ref_mean = y_of(got["ref"]).mean(axis=0)
        assert np.abs(got["range_differences"][0] - (want + (y_of(whole["ref"]) - ref_mean) * C / FS)).max() <= 1e-6
        # and the two REF values agree to 0.01 samples here (measured on a B200: 0.0075; the preprocessing and the
        # lag-range edges of one 2b-sample signal are not those of two b-sample blocks)
        assert np.abs(y_of(whole["ref"]) - ref_mean).max() <= 0.01


# ------------------------------------------------------------------ more than one GPU
def multi_case():
    return fm_capture(220000, (0, 3, 8), (0, 20, 41), seed=17)


@pytest.mark.gpu
def test_one_rank_communicator_gives_the_one_gpu_results():
    raws = multi_case()
    args = (STATION_LLH, 1000, 30000, 7, 4, 25000)
    with T.Engine(T.MODE_EXTENDED, max_lag=300) as e:
        load_all(e, raws)
        want = e.process_windows(*args)
    with T.Engine(T.MODE_EXTENDED, max_lag=300) as e:
        e.comm_init(T.comm_unique_id(), 0, 1)
        load_all(e, raws)
        got = e.process_windows(*args)
    for k in want:
        assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), k


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_one_gpu_results():
    raws = multi_case()
    args = (STATION_LLH, 1000, 30000, 7, 4, 25000)
    with T.Engine(T.MODE_EXTENDED, max_lag=300) as e:
        load_all(e, raws)
        want = e.process_windows(*args)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_devices=2) as e:
        load_all(e, raws)
        got = e.process_windows(*args)
    for k in want:
        assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), k


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_argument_errors():
    raws = fm_capture(60000, (0, 3, 8), (0, 20, 41), seed=2)
    with T.Engine(T.MODE_SOURCE) as e:
        load_all(e, raws)
        with pytest.raises(T.TdoaError, match="SOURCE"):
            e.process_windows(STATION_LLH, 0, 10000, 2, 1, 10000)
    with T.Engine(T.MODE_BINARY, n_stations=2) as e:
        load_all(e, raws[:2])
        with pytest.raises(T.TdoaError, match="stations"):
            e.process_windows(STATION_LLH[:2], 0, 10000, 2, 1, 10000)
    with pytest.raises(T.TdoaError, match="n_stations"):   # more than 64 stations: no engine holds them
        T.Engine(T.MODE_BINARY, n_stations=65)
    with T.Engine(T.MODE_BINARY) as e:
        load_all(e, raws)
        for kw, msg in ((dict(dims=4), "dims"), (dict(dims=3), "4 stations")):
            with pytest.raises(T.TdoaError, match=msg):
                e.process_windows(STATION_LLH, 0, 10000, 2, 1, 10000, **kw)
            with pytest.raises(T.TdoaError, match=msg):
                e.window_fixes(STATION_LLH, 0, 10000, np.zeros((2, 3), T.PEAK_DTYPE), np.zeros((1, 3), T.PEAK_DTYPE),
                               10000, **kw)
        for nr, nt in ((0, 1), (1, 0)):
            with pytest.raises(T.TdoaError, match="window"):
                e.process_windows(STATION_LLH, 0, 10000, nr, nt, 10000)
        with pytest.raises(T.TdoaError, match="windows end"):
            e.process_windows(STATION_LLH, 0, 10000, 2, 7, 10000)   # TGT: 60000 samples
        with pytest.raises(T.TdoaError, match="bad window"):
            e.process_windows(STATION_LLH, 0, 10000, 2, 2, 0)
