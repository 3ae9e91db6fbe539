"""Configurations of tdoa_process_windows_retimed beyond EXTENDED mode with whole-block TGT windows: BINARY mode,
the decimating box-car, TGT windows that start off zero, overlap and have odd lengths, and guard samples -- each
against the restatement (tests/retime_oracle.py) re-timed by the returned rates, and against the injected delays.

The captures drift as in tests/test_gpu_windows.py: station k's sample n is src[n - d_k - round(eps_k n)]."""
import numpy as np
import pytest

import retime_oracle as RO
import tdoa_b200 as T
from oracle import oracle
from test_gpu_retimed import CORR_TOL, check_clock, fix_bound, load_all, tgt_planes
from test_gpu_windows import C, FS, REF_TX, ST4, TX, drift_captures

B, W = 400_000, 100_000
REF = (0, W, 2 * B // W, W)


def truth_of(dR, dT, S):
    """range differences in samples: the TGT delay difference less the REF one (the REF position is not given)"""
    return np.array([(dT[j] - dT[i]) - (dR[j] - dR[i]) for i, j in RO.pairs(S)], np.float64)


@pytest.mark.gpu
def test_binary_mode_with_drift():
    """BINARY mode re-times the preprocessed planes too; the restatement re-times both parts of each plane, so a
    BINARY correlator that read an imaginary part would differ (the engine drops the imaginary plane)"""
    st = ST4[[1, 2, 3]]                    # every pair's lag positive: the BINARY correlator's lags are one-sided
    eps = np.array([-20.0, 0.0, 20.0])
    raws, dR, dT = drift_captures(st, eps, block=B, seed=31)
    with T.Engine(T.MODE_BINARY, n_stations=3) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=REF, tgt=(0, B, 1, B))
        ml, blk, san = e.cfg.max_lag, e.cfg.block_size, e.cfg.sanity_lag
    assert out["pair_used"].all()
    check_clock(out, 3)
    tg = tgt_planes(raws)
    t_c = B + (B - 1) / 2
    for p, (i, j) in enumerate(RO.pairs(3)):
        lag, _, val = RO.window_record(tg[i], tg[j], out["clock_rate"][i], out["clock_rate"][j], ml, mode="binary",
                                       block=blk, sanity=san)
        got = out["tgt"][0][p]
        assert int(got["lag"]) == lag, (p, int(got["lag"]), lag)
        assert abs(float(got["corr"]) - val) <= CORR_TOL, p
        # the window-centre lag of the injected delays and drift
        assert abs(lag - ((dT[j] - dT[i]) + (eps[j] - eps[i]) * 1e-6 * t_c)) <= 1.0, p
    assert np.abs(out["range_differences"][0] * FS / C - truth_of(dR, dT, 3)).max() <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("D", [2, 4])
def test_extended_decimated_with_drift(D):
    """decimate = D: each plane is re-timed in its own n / D samples, about (n / D - 1) / 2"""
    L = 300
    st = ST4[:3]
    eps = np.array([0.0, 40.0, -40.0])
    raws, dR, dT = drift_captures(st, eps, block=B, seed=32 + D)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=3, decimate=D) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=REF, tgt=(0, B, 1, B))
    assert out["pair_used"].all()
    check_clock(out, 3)
    tg = tgt_planes(raws)
    oracle.set_seq_dc_limit(0)
    try:
        for p, (i, j) in enumerate(RO.pairs(3)):
            lag, frac, val = RO.window_record(tg[i], tg[j], out["clock_rate"][i], out["clock_rate"][j], L, D=D)
            got = out["tgt"][0][p]
            got_total = int(got["lag"]) + float(got["frac"])
            assert abs(got_total - D * (lag + frac)) <= 1e-3 * D, (p, got_total, D * (lag + frac))
            assert abs(float(got["corr"]) - val) <= CORR_TOL, p
    finally:
        oracle.set_seq_dc_limit(-1)
    td = out["range_differences"][0] * FS / C
    assert np.abs(td - truth_of(dR, dT, 3)).max() <= D / 2 + 1, td - truth_of(dR, dT, 3)


@pytest.mark.gpu
def test_offset_overlapping_odd_windows():
    """TGT windows from sample 137, of odd length 100 001, 99 000 apart (overlapping): each is re-timed about its
    own centre, (len - 1) / 2"""
    L = 300
    q0, n, nw, hop = 137, 100_001, 3, 99_000
    st = ST4[:3]
    eps = np.array([0.0, 40.0, -40.0])
    raws, dR, dT = drift_captures(st, eps, block=B, seed=33)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=3) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(st, ref=REF, tgt=(q0, n, nw, hop))
    assert out["pair_used"].all()
    check_clock(out, 3)
    tg = tgt_planes(raws)
    oracle.set_seq_dc_limit(0)
    try:
        for w in range(nw):
            a = q0 + w * hop
            for p, (i, j) in enumerate(RO.pairs(3)):
                lag, frac, val = RO.window_record(tg[i][a:a + n], tg[j][a:a + n], out["clock_rate"][i],
                                                  out["clock_rate"][j], L)
                got = out["tgt"][w][p]
                assert int(got["lag"]) == lag, (w, p, int(got["lag"]), lag)
                assert abs(float(got["frac"]) - frac) <= 1e-3, (w, p)
                assert abs(float(got["corr"]) - val) <= CORR_TOL, (w, p)
    finally:
        oracle.set_seq_dc_limit(-1)
    err = out["range_differences"] * FS / C - truth_of(dR, dT, 3)
    assert np.abs(err).max() <= 1.0, err


@pytest.mark.gpu
def test_guard_samples_with_drift():
    """guard_samples = G: TGT = block 2[G:], REF = block 1 ++ block 3[G:] (seven REF windows, none across the
    joint); the whole guarded TGT block as one window, re-timed, and the fix"""
    G, L = 5000, 300
    eps = np.array([0.0, 40.0, -40.0, 25.0])
    raws, dR, dT = drift_captures(ST4, eps, block=B, seed=34)
    with T.Engine(T.MODE_EXTENDED, max_lag=L, n_stations=4, guard_samples=G) as e:
        load_all(e, raws)
        out = e.process_windows_retimed(ST4, ref=(0, W, 7, W), tgt=(0, B - G, 1, B - G), ref_tx_llh=REF_TX,
                                        init_llh=[ST4[:, 0].mean(), ST4[:, 1].mean(), TX[2]])
    assert out["pair_used"].all()
    check_clock(out, 4)
    tg = [t[G:] for t in tgt_planes(raws)]
    oracle.set_seq_dc_limit(0)
    try:
        for p, (i, j) in enumerate(RO.pairs(4)):
            lag, frac, val = RO.window_record(tg[i], tg[j], out["clock_rate"][i], out["clock_rate"][j], L)
            got = out["tgt"][0][p]
            assert int(got["lag"]) == lag, (p, int(got["lag"]), lag)
            assert abs(float(got["frac"]) - frac) <= 1e-3, p
            assert abs(float(got["corr"]) - val) <= CORR_TOL, p
    finally:
        oracle.set_seq_dc_limit(-1)
    assert out["status"][0] == 0
    assert np.linalg.norm(oracle.llh_to_ecef(*out["position"][0]) - oracle.llh_to_ecef(*TX)) <= fix_bound(RO.pairs(4))
