"""CPU: the windowed fix stage's statement (tests/window_oracle.py) against constructed tables, and its
least-squares fix and geodesy against the C oracle's (orc_solve_ls, orc_llh_to_ecef) bit for bit.

The engine's k_window_ref_fit / k_window_rd / masked k_solve_ls are checked against this statement on the GPU
(tests/test_gpu_windows.py); here the statement itself is checked against what it is meant to recover."""
from __future__ import annotations

import numpy as np

import window_oracle as WO
from oracle import oracle
from helpers import STATION_LLH

PEAK = np.dtype([("lag", "<i4"), ("flags", "<u4"), ("corr", "<f8"), ("frac", "<f4"), ("margin", "<f4"),
                 ("first_lag", "<i4"), ("n_blocks", "<i4")])
EDGE, EMPTY = 0x2, 0x8
FS, C = 2e6, 299792458.0
B = 4_000_000            # block: capture of 3 B samples
W = 500_000              # window length = hop
N_REF, N_TGT = 16, 8     # REF signal 2 B, TGT signal B


def ref_time(w):         # centre of REF window w in the capture (guard 0)
    k0 = w * W if w * W < B else 2 * B + (w * W - B)
    return k0 + (W - 1) / 2


def tgt_time(w):
    return B + w * W + (W - 1) / 2


def tables(P, ref_y, tgt_y):
    """records whose lag + frac = the given values (frac in [-0.5, 0.5], exactly representable)"""
    ref = np.zeros((N_REF, P), PEAK)
    tgt = np.zeros((N_TGT, P), PEAK)
    for tab, y in ((ref, ref_y), (tgt, tgt_y)):
        lag = np.round(y)
        tab["lag"] = lag.astype(np.int32)
        tab["frac"] = (y - lag).astype(np.float32)
        tab["margin"] = 0.5
    return ref, tgt


def run(ref, tgt, **kw):
    return WO.window_fixes(STATION_LLH, [3 * B] * 3, 0, 0, W, W, ref, tgt, fs=FS, **kw)


def test_linear_drift_and_offset_recovered_exactly():
    # lag = a0 + beta (t - block-2 centre); values chosen as dyadic rationals so every sum is exact
    beta = np.array([2.0 ** -20, -3 * 2.0 ** -21, 2.0 ** -19])      # ~1, -1.4, 1.9 ppm
    a0 = np.array([12.25, -40.5, 7.0])
    tc = B + (B - 1) / 2
    ref_y = np.array([[a0[p] + beta[p] * (ref_time(w) - tc) for p in range(3)] for w in range(N_REF)])
    tgt_lag = np.array([30.0, -10.0, 5.5])
    tgt_y = np.array([[a0[p] + beta[p] * (tgt_time(w) - tc) + tgt_lag[p] for p in range(3)] for w in range(N_TGT)])
    ref, tgt = tables(3, ref_y, tgt_y)
    # what the records hold is what the statement sees: y = lag + f32(frac)
    assert np.array_equal(ref["lag"] + ref["frac"].astype(np.float64), ref_y)
    out = run(ref, tgt)
    assert np.array_equal(out["ref_fit"][:, 1], beta)
    assert np.array_equal(out["ref_fit"][:, 0], a0)
    assert np.array_equal(out["ref_fit"][:, 2], [N_REF] * 3)
    assert out["pair_used"].all()
    np.testing.assert_allclose(out["range_differences"], np.broadcast_to(tgt_lag * C / FS, (N_TGT, 3)), rtol=0, atol=1e-6)


def test_exclusions_straddle_empty_edge_margin():
    ref_y = np.full((N_REF, 3), 10.0)
    tgt_y = np.full((N_TGT, 3), 12.0)
    ref, tgt = tables(3, ref_y, tgt_y)
    ref["lag"][3, 0] = 900; ref["flags"][3, 0] = EMPTY          # pair 0: one EMPTY window of 16
    ref["lag"][5, 1] = 900; ref["flags"][5, 1] = EDGE           # pair 1: one EDGE window
    ref["lag"][7, 2] = 900; ref["margin"][7, 2] = 0.01          # pair 2: one low-margin window
    tgt["flags"][2, 1] = EMPTY
    tgt["margin"][4, 2] = 0.01
    out = run(ref, tgt, min_margin=0.1)
    assert np.array_equal(out["ref_fit"][:, 2], [N_REF - 1] * 3)
    assert np.array_equal(out["ref_fit"][:, 0], [10.0] * 3) and np.array_equal(out["ref_fit"][:, 1], [0.0] * 3)
    used = np.ones((N_TGT, 3), bool)
    used[2, 1] = used[4, 2] = False
    assert np.array_equal(out["pair_used"], used)
    assert np.isnan(out["range_differences"][~used]).all()
    # min_margin = 0: the margin test is off
    assert run(ref, tgt)["ref_fit"][2, 2] == N_REF
    # at a hop of 0.75e6, REF window 5 is [3.75e6, 4.25e6): samples in blocks 1 and 3, no single time
    hop = 750_000
    ref2 = np.zeros((10, 3), PEAK); ref2["margin"] = 0.5; ref2["lag"] = 10
    ref2["lag"][5] = 900                                        # [3.75e6, 4.25e6): blocks 1 and 3
    out = WO.window_fixes(STATION_LLH, [3 * B] * 3, 0, 0, W, hop, ref2, tgt[:1], fs=FS)
    assert np.array_equal(out["ref_fit"][:, 2], [9] * 3)
    assert np.array_equal(out["ref_fit"][:, 0], [10.0] * 3)


def test_outlier_refit_drops_a_200_sample_outlier():
    beta = 2.0 ** -20
    tc = B + (B - 1) / 2
    ref_y = np.array([[beta * (ref_time(w) - tc)] * 3 for w in range(N_REF)])
    ref_y[6, 1] += 200.0
    ref, tgt = tables(3, ref_y, np.zeros((N_TGT, 3)))
    bad = run(ref, tgt)
    assert bad["ref_fit"][1, 2] == N_REF and abs(bad["ref_fit"][1, 0]) > 1.0
    out = run(ref, tgt, ref_max_residual=50.0)
    assert np.array_equal(out["ref_fit"][:, 2], [N_REF, N_REF - 1, N_REF])
    np.testing.assert_allclose(out["ref_fit"][:, 1], [beta] * 3, rtol=1e-12, atol=0)
    np.testing.assert_allclose(out["ref_fit"][:, 0], [0.0] * 3, rtol=0, atol=1e-9)


def test_no_usable_ref_window_leaves_the_pair_unused():
    ref, tgt = tables(3, np.full((N_REF, 3), 1.0), np.full((N_TGT, 3), 2.0))
    ref["flags"][:, 2] = EMPTY
    out = run(ref, tgt)
    assert np.array_equal(out["ref_fit"][2], [0.0, 0.0, 0.0])
    assert not out["pair_used"][:, 2].any() and out["pair_used"][:, :2].all()
    # with 3 stations and one pair gone, the two left touch 3 stations: dims 2 still solves
    assert (out["status"] != 2).all()
    ref["flags"][:, 1] = EMPTY
    out = run(ref, tgt)
    assert (out["status"] == 2).all() and (out["iters"] == 0).all()


def test_geometric_term_is_the_baseline_style_distance():
    tx = np.array([41.30, -96.20, 300.0])
    ref, tgt = tables(3, np.zeros((N_REF, 3)), np.zeros((N_TGT, 3)))
    out = run(ref, tgt, ref_tx_llh=tx)
    p = 0
    for i in range(3):
        for j in range(i + 1, 3):
            geo = oracle.baseline(tx, STATION_LLH[j]) - oracle.baseline(tx, STATION_LLH[i])
            x = oracle.llh_to_ecef(*tx)
            di = np.linalg.norm(x - oracle.llh_to_ecef(*STATION_LLH[i]))
            dj = np.linalg.norm(x - oracle.llh_to_ecef(*STATION_LLH[j]))
            assert abs(out["range_differences"][0, p] - geo) < 1e-6
            assert abs(out["range_differences"][0, p] - (dj - di)) < 1e-6
            p += 1


def test_masked_ls_ignores_garbage_pairs():
    st = np.vstack([STATION_LLH, [41.22, -96.15, 340.0], [41.30, -95.95, 360.0]])
    tx = np.array([41.26, -96.05, 345.0])
    x = oracle.llh_to_ecef(*tx)
    r = [np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in st]
    rd = np.array([r[j] - r[i] for i in range(5) for j in range(i + 1, 5)])
    used = np.ones(rd.size, bool)
    rd[2] += 7000.0; used[2] = False
    rd[7] = np.nan; used[7] = False
    out, rms, status, _ = WO.solve_ls(st, rd, init_llh=[41.25, -96.0, tx[2]], dims=2, used=used)
    assert status == 0
    assert np.linalg.norm(oracle.llh_to_ecef(*out) - x) < 1e-3
    assert rms < 1e-3
    # without the mask the NaN poisons the fit
    assert WO.solve_ls(st, rd, init_llh=[41.25, -96.0, tx[2]], dims=2)[2] == 1


def test_restatement_is_the_c_oracle_bit_for_bit():
    """no mask and an all-true mask are orc_solve_ls itself (dims 2 and 3, noisy sets, default and given starts)"""
    rng = np.random.default_rng(11)
    st = np.vstack([STATION_LLH, [41.22, -96.15, 340.0], [41.30, -95.95, 360.0]])
    for k in range(6):
        tx = [41.26 + 0.05 * rng.uniform(-1, 1), -96.05 + 0.05 * rng.uniform(-1, 1), 345.0]
        x = oracle.llh_to_ecef(*tx)
        assert WO.llh_to_ecef(*tx) == tuple(x)
        r = [np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in st]
        rd = np.array([r[j] - r[i] for i in range(5) for j in range(i + 1, 5)]) + rng.normal(0, 20, 10)
        init = None if k % 2 else [41.25, -96.0, 345.0]
        for dims in (2, 3):
            want = oracle.solve_ls(st, rd, init_llh=init, dims=dims)
            for used in (None, np.ones(rd.size, bool)):
                got = WO.solve_ls(st, rd, init_llh=init, dims=dims, used=used)
                assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]
