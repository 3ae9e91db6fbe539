"""The closure check of the windowed fixes on the GPU: k_window_closure (tdoa_closure) against its restatement
(tests/closure_oracle.py) bit for bit, the inert check against the calls without it, corrupted tables, a station
that hears another programme (a station offset the check cannot see), the re-timed call with a grid seed, more than one GPU, and the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import tdoa_b200 as T
from helpers import fm_signal, quantise
import closure_oracle as CO
import window_oracle as WO
from oracle import oracle
from test_gpu_window_grid import (ST4, TRAP_GRID, TRAPPED, REF_TX, W, N_REF, WD, trapped_tables, drift_captures,
                                  same_results, exact_rd, metres)

FS, CL = 2e6, 299792458.0
MR = 100.0
INERT = {"max_residual": math.inf}


def stations(S, seed):
    rng = np.random.default_rng(seed)
    return np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), rng.uniform(300, 400)]
                     for _ in range(S)])


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64).tolist()


# ------------------------------------------------------------------ kernel parity
def parity_sets(S, n_sets, seed, n_bad):
    rng = np.random.default_rng(seed)
    st = stations(S, seed)
    P = S * (S - 1) // 2
    rds, used = np.zeros((n_sets, P + 3)), np.zeros((n_sets, P + 3), np.uint8)
    for k in range(n_sets):
        tx = [41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0]
        rd = exact_rd(st, tx) + rng.normal(0, 20, P)
        bad = rng.choice(P, min(n_bad, P), replace=False)
        rd[bad] += rng.choice([-1, 1], bad.size) * rng.uniform(2, 40, bad.size) * MR
        kind = k % 4
        u = np.ones(P, bool) if kind == 0 else rng.uniform(0, 1, P) < (0.7, 0.35, 1.0)[kind - 1]
        if kind == 3:   # two components and an isolated station
            half = S // 2
            u = np.array([(i < half) == (j < half) and j != S - 1 for i, j in CO.pairs(S)])
        rds[k, :P] = np.where(u, rd, np.nan)
        rds[k, P:] = np.nan
        used[k, :P] = u
    return rds, used


@pytest.mark.gpu
@pytest.mark.parametrize("S,n_sets,n_bad,max_drop,dims", [(3, 40, 1, 0, 2), (4, 1000, 1, 0, 2), (8, 300, 3, 0, 2),
                                                          (16, 60, 12, 0, 3), (16, 40, 30, 5, 2), (64, 3, 40, 0, 2)])
def test_kernel_equals_restatement(S, n_sets, n_bad, max_drop, dims):
    rds, used = parity_sets(S, n_sets, 1000 * S + n_sets, n_bad)
    P = S * (S - 1) // 2
    with T.Engine(T.MODE_BINARY) as e:
        out, resid, dropped = e.closure(S, rds, used, dims, max_residual=MR, max_drop=max_drop)
    w_out, w_resid, w_dropped = CO.check(rds, used, S, dims, MR, max_drop)
    assert out[:, :P].tolist() == w_out.tolist()
    assert bits(resid[:, :P]) == bits(w_resid)
    assert dropped.tolist() == w_dropped.tolist()
    assert np.isnan(resid[:, P:]).all() and (out[:, P:] == 0).all()   # past P: left as the caller's arrays were
    assert dropped.max() >= (1 if S > 3 else 0)


# ------------------------------------------------------------------ the inert check equals the calls without it
@pytest.fixture(scope="module")
def trapped_drift():
    return drift_captures(TRAPPED[0])


def same(a, b, keys):
    for k in keys:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


FIX_KEYS = ("ref_fit", "range_differences", "pair_used", "position", "rms", "status", "iters")


@pytest.mark.gpu
def test_inert_check_equals_the_calls_without_it(trapped_drift):
    raws = trapped_drift
    args = (ST4, 0, WD, 6, 3, WD)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        for grid in (None, TRAP_GRID):
            plain = e.process_windows(*args, ref_tx_llh=REF_TX, grid=grid)
            got = e.process_windows(*args, ref_tx_llh=REF_TX, grid=grid, closure=INERT)
            same(plain, got, FIX_KEYS + ("ref", "tgt") + (("seed", "seed_cost", "seed_index") if grid else ()))
            assert not got["pair_dropped"].any() and (got["dropped"] == 0).all()
            fx = e.window_fixes(ST4, 0, WD, plain["ref"], plain["tgt"], WD, ref_tx_llh=REF_TX, grid=grid)
            fx_c = e.window_fixes(ST4, 0, WD, plain["ref"], plain["tgt"], WD, ref_tx_llh=REF_TX, grid=grid, closure=INERT)
            same(fx, fx_c, FIX_KEYS)
        geo = ((0, WD, 6, WD), (0, 0, 1, WD))
        plain = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX)
        got = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX, closure=INERT)
        same(plain, got, FIX_KEYS + ("ref", "tgt", "clock_rate"))
        assert np.isfinite(got["closure_residual"][got["pair_used"]]).all()


# ------------------------------------------------------------------ corrupted tables
B = 4000


def exact_tables(st, txs, n_ref=N_REF):
    S = st.shape[0]
    P = S * (S - 1) // 2
    y = np.stack([exact_rd(st, tx) for tx in txs]) * FS / CL
    ref = np.zeros((n_ref, P), T.PEAK_DTYPE)
    tgt = np.zeros((len(txs), P), T.PEAK_DTYPE)
    tgt["lag"] = np.round(y).astype(np.int32)
    tgt["frac"] = (y - np.round(y)).astype(np.float32)
    caps = [np.random.default_rng(70 + k).integers(0, 256, 6 * B, dtype=np.uint8) for k in range(S)]
    return ref, tgt, caps


@pytest.mark.gpu
@pytest.mark.parametrize("S,k", [(8, 1), (8, 3), (12, 2), (16, 5)])
def test_corrupted_tables(S, k):
    rng = np.random.default_rng(S * 10 + k)
    st = stations(S, 500 + S)
    txs = [np.array([41.26 + rng.uniform(-0.08, 0.08), -96.02 + rng.uniform(-0.1, 0.1), 350.0]) for _ in range(6)]
    ref, tgt, caps = exact_tables(st, txs)
    P = S * (S - 1) // 2
    bad = np.zeros(tgt.shape, bool)
    for w in range(tgt.shape[0]):
        bad[w, rng.choice(P, k, replace=False)] = True
    worse = tgt.copy()
    worse["lag"][bad] += (rng.choice([-1, 1], bad.sum()) * rng.integers(40, 501, bad.sum())).astype(np.int32)
    c = {"max_residual": MR}
    with T.Engine(T.MODE_EXTENDED, n_stations=S) as e:
        for s, cap in enumerate(caps):
            e.load_u8(s, cap)
        clean = e.window_fixes(st, 0, W, ref, tgt, W)
        plain = e.window_fixes(st, 0, W, ref, worse, W)
        got = e.window_fixes(st, 0, W, ref, worse, W, closure=c)
    assert got["pair_dropped"].tolist() == bad.tolist()
    assert (got["pair_used"] == ~bad).all() and got["dropped"].tolist() == [k] * tgt.shape[0]
    off = [metres(plain["position"][w], clean["position"][w]) for w in range(tgt.shape[0])]
    assert min(off) > 100.0 and max(off) > 1000.0
    for w in range(tgt.shape[0]):
        assert metres(got["position"][w], clean["position"][w]) <= 1.0
    # the fix stage against the restatement: range differences, the check bit for bit, the fixes
    want = WO.window_fixes(st, [3 * B] * S, 0, 0, W, W, ref, worse, fs=FS)
    assert want["range_differences"].tobytes() == got["range_differences"].tobytes()
    w_out, w_resid, w_drop = CO.check(want["range_differences"], want["pair_used"], S, 2, MR)
    assert (w_out == 1).tolist() == got["pair_used"].tolist() and w_drop.tolist() == got["dropped"].tolist()
    assert bits(w_resid) == bits(got["closure_residual"])
    for w in range(tgt.shape[0]):
        pos, rms, status, _ = WO.solve_ls(st, want["range_differences"][w], None, 2, w_out[w] == 1)
        assert status == got["status"][w] and metres(pos, got["position"][w]) <= 1e-4


# ------------------------------------------------------------------ a station that hears another programme
ST6 = np.vstack([ST4, [[41.42, -95.80, 330.0], [41.10, -96.30, 360.0]]])
TX6 = np.array([41.28, -96.05, 350.0])
BE = 1_000_000


def interfered_captures(bad=4, block=BE, seed=9, noise=0.02):
    """six stations without drift; station `bad` hears another FM programme than the others in block 2"""
    dR = np.round([np.linalg.norm(oracle.llh_to_ecef(*REF_TX) - oracle.llh_to_ecef(*s)) / CL * FS for s in ST6]).astype(np.int64)
    dT = np.round([np.linalg.norm(oracle.llh_to_ecef(*TX6) - oracle.llh_to_ecef(*s)) / CL * FS for s in ST6]).astype(np.int64)
    dR, dT = dR - dR.min(), dT - dT.min()
    n = 3 * block
    pad = int(max(dR.max(), dT.max())) + 16
    ref = fm_signal(n + 2 * pad, 1000 + seed, 75e3)
    tgt = fm_signal(n + 2 * pad, 2000 + seed, 60e3)
    other = fm_signal(n + 2 * pad, 4000 + seed, 60e3)
    t = np.arange(n)
    in_tgt = (t >= block) & (t < 2 * block)
    raws = []
    for k in range(len(ST6)):
        idx = pad + t - np.where(in_tgt, dT[k], dR[k])
        x = np.where(in_tgt, (other if k == bad else tgt)[idx], ref[idx])
        g = np.random.default_rng(5000 + 17 * seed + k)
        raws.append(quantise(x + noise * (g.standard_normal(n) + 1j * g.standard_normal(n))))
    return raws


@pytest.mark.gpu
def test_station_hearing_another_programme_is_a_station_offset():
    """Station 4 hears another FM programme in block 2.  Its pairs' peaks are wrong, but the peak of pair (i, 4) is
    the other programme's cross-correlation peak moved by station i's own delay, so every one of its pairs is off by
    the same range: a wrong station value, which the station values tau absorb.  The check cannot see it (nothing is
    dropped, every residual stays within max_residual) and the fixes are those of the call without the check."""
    raws = interfered_captures(4)
    args = (ST6, 0, BE // 2, 4, 2, BE // 2)
    with T.Engine(T.MODE_EXTENDED, max_lag=600, n_stations=6) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        plain = e.process_windows(*args, ref_tx_llh=REF_TX, init_llh=TX6 + [0.03, 0.03, 0.0])
        got = e.process_windows(*args, ref_tx_llh=REF_TX, init_llh=TX6 + [0.03, 0.03, 0.0], closure={"max_residual": 300.0})
    same(plain, got, FIX_KEYS)
    assert got["dropped"].tolist() == [0, 0] and got["pair_used"].all()
    assert np.abs(got["closure_residual"]).max() <= 300.0
    assert min(metres(got["position"][w], TX6) for w in range(2)) > 1000.0


# ------------------------------------------------------------------ the re-timed call with a grid seed
@pytest.mark.gpu
def test_retimed_call_with_grid_and_closure(trapped_drift):
    raws = trapped_drift
    geo = ((0, WD, 16, WD), (0, 0, 1, WD))
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        plain = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX)
        got = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX, grid=TRAP_GRID, closure={"max_residual": 300.0})
    same(plain, got, ("ref", "tgt", "ref_fit", "range_differences", "clock_rate"))
    assert got["status"].tolist() == [0] and got["seed_index"][0] >= 0 and got["dropped"].tolist() == [0]
    # the restatement's fix from the returned range differences, started at the returned seed
    want, *_ = WO.solve_ls(ST4, got["range_differences"][0], got["seed"][0], 2, got["pair_used"][0])
    assert metres(got["position"][0], want) <= 1.0
    # the station mean's local minimum holds the plain call kilometres away; the seeded fix is not trapped (outside
    # the 4-station hull a sample of range error moves it by a few hundred metres)
    assert metres(plain["position"][0], TRAPPED[0]) > 4000.0
    assert metres(got["position"][0], TRAPPED[0]) <= 1000.0


# ------------------------------------------------------------------ more than one GPU
def closure_run(raws, **kw):
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4, **kw.pop("engine", {})) as e:
        if kw.pop("comm", False):
            e.comm_init(T.comm_unique_id(), 0, 1)
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        return e.process_windows(ST4, 0, WD, 4, 2, WD, ref_tx_llh=REF_TX, grid=TRAP_GRID, closure={"max_residual": 50.0})


@pytest.mark.gpu
def test_one_rank_communicator_gives_the_one_gpu_results(trapped_drift):
    same_results(closure_run(trapped_drift), closure_run(trapped_drift, comm=True))


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_one_gpu_results(trapped_drift):
    same_results(closure_run(trapped_drift), closure_run(trapped_drift, engine={"n_devices": 2}))


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_argument_errors():
    ref, tgt, caps = trapped_tables()
    rd, u = np.zeros((2, 6)), np.ones((2, 6), np.uint8)
    with T.Engine(T.MODE_EXTENDED, n_stations=4) as e:
        for k, cap in enumerate(caps):
            e.load_u8(k, cap)
        for bad in ({"max_residual": 0.0}, {"max_residual": -1.0}, {"max_residual": math.nan},
                    {"max_residual": 10.0, "max_drop": -1}):
            with pytest.raises(T.TdoaError, match="max_"):
                e.window_fixes(ST4, 0, W, ref, tgt, W, closure=bad)
            with pytest.raises(T.TdoaError, match="max_"):
                e.process_windows(ST4, 0, W, N_REF, 3, W, closure=bad)
            with pytest.raises(T.TdoaError, match="max_"):
                e.closure(4, rd, u, **bad)
        with pytest.raises(T.TdoaError, match="dims"):   # what the base call refuses
            e.window_fixes(ST4, 0, W, ref, tgt, W, dims=4, closure=INERT)
        for S, dims, rds, msg in ((2, 2, rd, "stations"), (65, 2, np.zeros((1, 65 * 32)), "stations"),
                                  (4, 4, rd, "dims"), (4, 2, np.zeros((2, 5)), "rd_stride")):
            with pytest.raises(T.TdoaError, match=msg):
                e.closure(S, rds, np.ones(rds.shape, np.uint8), dims, max_residual=10.0)
        # NULL options, retimed not 0 / 1, n_sets < 0
        o = T._native.WindowOpts(dims=2)
        c = T._native.ClosureOpts(max_residual=10.0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        st = np.ascontiguousarray(ST4)
        fix, status = np.zeros((3, 3)), np.zeros(3, np.int32)
        out = np.zeros((2, 6), np.uint8)
        L = e._lib
        assert L.tdoa_closure(e._h, 4, p(rd), p(u), 2, 6, 2, None, p(out), None, None) == -1
        assert L.tdoa_closure(e._h, 4, p(rd), p(u), -1, 6, 2, C.byref(c), p(out), None, None) == -1
        assert L.tdoa_window_fixes_closure(e._h, p(st), C.byref(o), None, 0, W, N_REF, 3, W, None, p(ref), p(tgt), None,
                                           None, None, None, None, p(fix), None, p(status), None, None, None, None) == -1
        assert "closure options" in e.last_error()
        for retimed in (2, -1):
            rc = L.tdoa_process_windows_closure(e._h, p(st), C.byref(o), C.byref(c), 0, W, N_REF, W, 0, W, 3, W, retimed,
                                                None, None, None, None, None, None, None, None, p(fix), None, p(status),
                                                None, None, None, None, None)
            assert rc == -1 and "retimed" in e.last_error()
