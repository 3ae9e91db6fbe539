"""Re-timed target correlation (tdoa_process_windows_retimed; retime.cu): station clock rates fitted from the REF
windows re-time every TGT plane, so one TGT window may span the whole block.

The captures drift as in tests/test_gpu_windows.py: station k's sample n is src[n - d_k - round(eps_k n)]."""
import ctypes
import sys

import numpy as np
import pytest
import torch

import retime_oracle as RO
import tdoa_b200 as T
from helpers import STATION_LLH, fm_signal, quantise
from oracle import oracle
from test_gpu_windows import C, FS, REF_TX, ST4, TX, delays, drift_captures

CORR_TOL = 1e-6


def load_all(e, raws):
    for k, r in enumerate(raws):
        e.load_u8(k, r)


def y_of(tab):
    return tab["lag"].astype(np.float64) + tab["frac"].astype(np.float64)


def tgt_planes(raws):
    return [oracle.extract_target(oracle.unpack_u8(r)) for r in raws]


def check_clock(out, S):
    """clock_rate is the restatement's fit of the returned REF fits, bit for bit (NaN at the same stations)"""
    _, clock = RO.station_rates(out["ref_fit"][:, 1], out["ref_fit"][:, 2], S)
    got = np.asarray(out["clock_rate"], np.float64)
    assert got.view(np.uint64).tolist() == clock.view(np.uint64).tolist(), (got, clock)


def check_parity(out, raws, L, pair_ids):
    """TGT window 0 (the whole block) of the given pairs against the restatement re-timed by the returned rates"""
    S = len(raws)
    check_clock(out, S)
    tg = tgt_planes(raws)
    pp = RO.pairs(S)
    oracle.set_seq_dc_limit(0)
    try:
        for p in pair_ids:
            i, j = pp[p]
            lag, frac, val = RO.window_record(tg[i], tg[j], out["clock_rate"][i], out["clock_rate"][j], L)
            got = out["tgt"][0][p]
            assert int(got["lag"]) == lag, (p, int(got["lag"]), lag)
            assert abs(float(got["frac"]) - frac) <= 1e-3, p
            assert abs(float(got["corr"]) - val) <= CORR_TOL, p
    finally:
        oracle.set_seq_dc_limit(-1)


# ------------------------------------------------------------------ restatement parity, per correlator path
@pytest.mark.gpu
def test_parity_three_stations_tile_fft():
    B, W, L = 400_000, 100_000, 300
    st = ST4[:3]
    raws, _, _ = drift_captures(st, np.array([0.0, 40.0, -40.0]), block=B, seed=21)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=3) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=(0, W, 2 * B // W, W), tgt=(0, B, 1, B))
    assert out["pair_used"].all()
    check_parity(out, raws, L, range(3))


@pytest.mark.gpu
def test_parity_sixteen_stations_parked_spectra():
    B, W, L, S = 200_000, 50_000, 400, 16
    g = np.random.default_rng(3)
    st = np.vstack([ST4, ST4.mean(0) + g.uniform([-0.06, -0.08, -20], [0.06, 0.08, 20], (S - 4, 3))])
    raws, _, _ = drift_captures(st, g.uniform(-20.0, 20.0, S), block=B, seed=22)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=S) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=(0, W, 2 * B // W, W), tgt=(0, B, 1, B))
    assert out["pair_used"].all()
    check_parity(out, raws, L, range(0, S * (S - 1) // 2, 11))


@pytest.mark.gpu
def test_parity_wide_lags_big_transform():
    B, W, L = 200_000, 50_000, 4100   # 8201 lags: the 2^21-point transform
    st = ST4[:3]
    raws, _, _ = drift_captures(st, np.array([0.0, -30.0, 35.0]), block=B, seed=23)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=3) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=(0, W, 2 * B // W, W), tgt=(0, B, 1, B))
    check_parity(out, raws, L, range(3))


# ------------------------------------------------------------------ identity
@pytest.mark.gpu
def test_without_drift_it_is_process_windows():
    B, W, L = 400_000, 100_000, 300
    raws, _, _ = drift_captures(ST4, np.zeros(4), block=B, seed=24)
    nr, nt = 2 * B // W, B // W
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=4) as e:
        load_all(e, raws)
        ref_alone = e.xcorr(T.KIND_REF, 0, W, nr, W)
        want = e.process_windows(ST4, 0, W, nr, nt, W)
        got = e.process_windows_retimed(ST4, ref=(0, W, nr, W), tgt=(0, W, nt, W))
    assert got["ref"].tobytes() == ref_alone.tobytes()
    check_clock(got, 4)
    # rates this small shift no sample of a W-sample plane: delta is 0 everywhere
    assert (np.abs(got["clock_rate"]) * W / 2 < 0.5).all()
    for k in want:
        assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), k


# ------------------------------------------------------------------ what it is for
B4, W4, L4 = 4_000_000, 500_000, 1100
EPS40 = np.array([0.0, 40.0, -40.0, 25.0])
# Per component, TGT block only, on top of the 0.02 of every block.  At this level the 0.5 M-sample windows are
# noise-limited (on a B200: worst 2.83 samples off) while the whole block stays within 1 sample (worst 0.93).  The
# lag error of a window falls as 1 / sqrt(its length), so the whole block's is sqrt(8) = 2.8x smaller: a level at which
# a 0.5 M window misses by 5 samples leaves the whole block ~2 samples off (1.93 measured at 0.28) -- more integration
# than 8x is what such a target needs.  The margin is no test of a weak window in EXTENDED mode: the runner-up of an
# exactly evaluated peak is its neighbour lag, so margins are ~1e-3 for short and long windows alike.
WEAK_NOISE = 0.21


def fix_bound(pp):
    """test_drift_end_to_end's bound: 3 samples of range difference per pair through pinv of the geometry"""
    x0 = oracle.llh_to_ecef(*TX)

    def rds(lat, lon):
        x = oracle.llh_to_ecef(lat, lon, TX[2])
        r = [np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in ST4]
        return np.array([r[j] - r[i] for i, j in pp])
    h = 1e-5
    m_lat = np.linalg.norm(oracle.llh_to_ecef(TX[0] + h, TX[1], TX[2]) - x0)
    m_lon = np.linalg.norm(oracle.llh_to_ecef(TX[0], TX[1] + h, TX[2]) - x0)
    J = np.column_stack([(rds(TX[0], TX[1] + h) - rds(*TX[:2])) / m_lon, (rds(TX[0] + h, TX[1]) - rds(*TX[:2])) / m_lat])
    return np.linalg.norm(np.linalg.pinv(J), 2) * np.sqrt(len(pp)) * 3 * C / FS


def weak_target_captures(tgt_noise, seed=5):
    """drift_captures with extra noise in the TGT block only (the REF transmitter stays strong)"""
    dR, dT = delays(ST4, REF_TX), delays(ST4, TX)
    n = 3 * B4
    pad = int(max(dR.max(), dT.max()) + np.abs(EPS40).max() * 1e-6 * n) + 16
    ref = fm_signal(n + 2 * pad, 1000 + seed, 75e3)
    tgt = fm_signal(n + 2 * pad, 2000 + seed, 60e3)
    t = np.arange(n)
    in_tgt = (t >= B4) & (t < 2 * B4)
    raws = []
    for k in range(len(ST4)):
        d = np.where(in_tgt, dT[k], dR[k]) + np.round(EPS40[k] * 1e-6 * t).astype(np.int64)
        idx = pad + t - d
        x = np.where(in_tgt, tgt[idx], ref[idx])
        g = np.random.default_rng(3000 + 17 * seed + k)
        x = x + 0.02 * (g.standard_normal(n) + 1j * g.standard_normal(n))
        x = x + np.where(in_tgt, tgt_noise, 0.0) * (g.standard_normal(n) + 1j * g.standard_normal(n))
        raws.append(quantise(x))
    return raws, dR, dT


@pytest.mark.gpu
def test_whole_block_tgt_window_with_drift():
    raws, dR, dT = drift_captures(ST4, EPS40, block=B4, seed=25)
    pp = RO.pairs(4)
    truth = np.array([(dT[j] - dT[i]) - (dR[j] - dR[i]) for i, j in pp], np.float64)
    ref_geo = (0, W4, 2 * B4 // W4, W4)
    with T.Engine(T.MODE_EXTENDED, max_lag=L4, n_stations=4) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(ST4, ref=ref_geo, tgt=(0, B4, 1, B4))
        geo = e.process_windows_retimed(ST4, ref=ref_geo, tgt=(0, B4, 1, B4), ref_tx_llh=REF_TX,
                                        init_llh=[ST4[:, 0].mean(), ST4[:, 1].mean(), TX[2]])
        plain = e.process_windows(ST4, 0, B4, 2, 1, B4)
    assert out["pair_used"].all()
    check_clock(out, 4)
    check_clock(geo, 4)
    td = out["range_differences"][0] * FS / C
    assert np.abs(td - truth).max() <= 1.0, td - truth
    c = out["clock_rate"] - out["clock_rate"].mean()
    assert np.abs(c - (EPS40 - EPS40.mean()) * 1e-6).max() <= 0.05e-6
    assert geo["status"][0] == 0
    assert np.linalg.norm(oracle.llh_to_ecef(*geo["position"][0]) - oracle.llh_to_ecef(*TX)) <= fix_bound(pp)
    # the same whole-block TGT window without re-timing: the drift inside it smears the peaks
    assert np.abs(plain["range_differences"][0] * FS / C - truth).max() > 5.0


@pytest.mark.gpu
def test_weak_target_needs_the_long_window():
    raws, dR, dT = weak_target_captures(WEAK_NOISE)
    pp = RO.pairs(4)
    truth = np.array([(dT[j] - dT[i]) - (dR[j] - dR[i]) for i, j in pp], np.float64)
    ref_geo = (0, W4, 2 * B4 // W4, W4)
    with T.Engine(T.MODE_EXTENDED, max_lag=L4, n_stations=4) as e:
        load_all(e, raws)
        short = e.process_windows_retimed(ST4, ref=ref_geo, tgt=(0, W4, B4 // W4, W4))
        whole = e.process_windows_retimed(ST4, ref=ref_geo, tgt=(0, B4, 1, B4))
    check_clock(short, 4)
    check_clock(whole, 4)
    es = short["range_differences"] * FS / C - truth        # 8 windows x 6 pairs
    ew = whole["range_differences"][0] * FS / C - truth
    # every pair from the whole block within 1 sample
    assert np.abs(ew).max() <= 1.0, (ew, es)
    # the 0.5 M-sample windows (drift-free after re-timing, but noise-limited) miss by more than twice that
    assert np.abs(es).max() > 2.0, (ew, es)
    # 8x the integration: the rms lag error falls by sqrt(8) in expectation, by at least 2 here
    assert np.sqrt(np.mean(ew ** 2)) <= np.sqrt(np.mean(es ** 2)) / 2.0, (ew, es)


# ------------------------------------------------------------------ more than one GPU
def multi_args():
    raws, _, _ = drift_captures(ST4, EPS40, block=400_000, seed=26)
    return raws, dict(ref=(0, 100_000, 8, 100_000), tgt=(0, 200_000, 2, 200_000))


def same_results(want, got):
    """Everything bit for bit, but the tables' margin, which a dealt call may move by ~1e-7 (the runner-up lags are
    evaluated in other batches; see tests/test_gpu_window_grid.py)"""
    check_clock(want, 4)
    for k in want:
        if k in ("ref", "tgt"):
            for f in want[k].dtype.names:
                if f == "margin":
                    assert np.abs(got[k][f] - want[k][f]).max() <= 1e-6, (k, f)
                else:
                    assert got[k][f].tobytes() == want[k][f].tobytes(), (k, f)
        else:
            assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), k


@pytest.mark.gpu
def test_one_rank_communicator_gives_the_one_gpu_results():
    raws, kw = multi_args()
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        load_all(e, raws)
        want = e.process_windows_retimed(ST4, **kw)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        e.comm_init(T.comm_unique_id(), 0, 1)
        load_all(e, raws)
        got = e.process_windows_retimed(ST4, **kw)
    same_results(want, got)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_one_gpu_results():
    raws, kw = multi_args()
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        load_all(e, raws)
        want = e.process_windows_retimed(ST4, **kw)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4, n_devices=2) as e:
        load_all(e, raws)
        got = e.process_windows_retimed(ST4, **kw)
    same_results(want, got)


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_refusals():
    from helpers import fm_capture
    raws = fm_capture(60000, (0, 3, 8), (0, 20, 41), seed=2)
    ref = (0, 10000, 2, 10000)
    with T.Engine(T.MODE_SOURCE) as e:
        load_all(e, raws)
        with pytest.raises(T.TdoaError, match="SOURCE"):
            e.process_windows_retimed(STATION_LLH, ref=ref, tgt=(0, 10000, 1, 10000))
    with T.Engine(T.MODE_BINARY, n_stations=2) as e:
        load_all(e, raws[:2])
        with pytest.raises(T.TdoaError, match="stations"):
            e.process_windows_retimed(STATION_LLH[:2], ref=ref, tgt=(0, 10000, 1, 10000))
    with T.Engine(T.MODE_EXTENDED) as e:
        load_all(e, raws)
        for tgt, msg in (((0, 10000, 0, 10000), "window"), ((0, 30000, 3, 30000), "windows end"),
                         ((0, 10000, 2, 0), "bad window"), ((-1, 10000, 1, 10000), "bad window")):
            with pytest.raises(T.TdoaError, match=msg):
                e.process_windows_retimed(STATION_LLH, ref=ref, tgt=tgt)
        # fix_llh NULL (the one C-level refusal the binding cannot produce)
        native = sys.modules[type(e).__module__]
        o = native.WindowOpts(dims=2)
        st = np.ascontiguousarray(STATION_LLH, np.float64)
        status = np.zeros(1, np.int32)
        with pytest.raises(T.TdoaError, match="NULL"):
            e._check(e._lib.tdoa_process_windows_retimed(e._h, native._ptr(st), ctypes.byref(o), 0, 10000, 2, 10000, 0, 10000,
                                                         1, 10000, None, None, None, None, None, None, None,
                                                         native._ptr(status), None, None))
