"""Masked grid arg-min (tdoa_grid_masked) and grid-seeded windowed fixes (tdoa_process_windows_grid /
tdoa_window_fixes_grid) on the GPU, against the unmasked grid, the exhaustive (use_fft = 0) engine and the plain
restatements of tests/window_oracle.py and tests/window_grid_oracle.py."""
import ctypes as C

import numpy as np
import pytest
import torch

import tdoa_b200 as T
from helpers import STATION_LLH, fm_signal, quantise
import window_grid_oracle as WG
import window_oracle as WO
from oracle import oracle

FS, CL = 2e6, 299792458.0
ST4 = np.vstack([STATION_LLH, [41.20, -96.20, 340.0]])
TRAPPED = [np.array([41.3711, -96.0233, 350.0]), np.array([41.5017, -95.9768, 350.0])]
TRAP_GRID = [40.90, -96.45, 0.005, 0.005, 180, 160, 350.0]
REF_TX = np.array([41.10, -95.80, 400.0])


def pairs(S):
    return [(i, j) for i in range(S) for j in range(i + 1, S)]


def exact_rd(stations, tx):
    x = oracle.llh_to_ecef(*tx)
    r = [np.linalg.norm(x - oracle.llh_to_ecef(*s)) for s in stations]
    return np.array([r[j] - r[i] for i, j in pairs(len(stations))])


def metres(a, b):
    return float(np.linalg.norm(oracle.llh_to_ecef(*a) - oracle.llh_to_ecef(*b)))


def launches(e):
    return e.stats()["launches_total"]


def grid_masked_null(e, st, desc, rds):
    """tdoa_grid_masked with used = NULL (Engine.grid(used=None) calls tdoa_grid)"""
    st = np.ascontiguousarray(st, np.float64)
    gd = np.ascontiguousarray(desc, np.float64)
    rd = np.ascontiguousarray(rds, np.float64)
    n, stride = rd.shape
    out, cost, idx = np.zeros((n, 3)), np.zeros(n), np.zeros(n, np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    e._check(e._lib.tdoa_grid_masked(e._h, p(st), st.shape[0], p(gd), p(rd), None, n, stride, p(out), p(cost), p(idx)))
    return out, cost, idx


def grid_case(n_st, n_sets, nlat, nlon, dlat, seed):
    """test_grid_ranked_equals_exhaustive's stations, grid and sets"""
    rng = np.random.default_rng(seed)
    st = np.array([[41.26 + rng.uniform(-0.2, 0.2), -96.02 + rng.uniform(-0.25, 0.25), rng.uniform(300, 400)] for _ in range(n_st)])
    desc = [41.26 - 0.5 * nlat * dlat, -96.02 - 0.5 * nlon * 0.002, dlat, 0.002, nlat, nlon, 350.0]
    rds = []
    for k in range(n_sets):
        tx = np.array([41.26 + rng.uniform(-0.05, 0.05), -96.02 + rng.uniform(-0.08, 0.08), 350.0])
        rds.append(exact_rd(st, tx) + rng.normal(0, [0.0, 15.0, 150.0][k % 3], n_st * (n_st - 1) // 2))
    return st, desc, np.stack(rds), rng


SHAPES = [(3, 4, 90, 110, 0.002), (5, 7, 257, 129, 0.001), (16, 9, 300, 300, 0.0015), (16, 3, 64, 500, 0.0),
          (9, 700, 40, 37, 0.003), (2, 2, 50, 50, 0.002)]


# ------------------------------------------------------------------ tdoa_grid_masked
@pytest.mark.gpu
@pytest.mark.parametrize("n_st,n_sets,nlat,nlon,dlat", SHAPES)
def test_masked_without_mask_is_tdoa_grid(n_st, n_sets, nlat, nlon, dlat):
    st, desc, rds, _ = grid_case(n_st, n_sets, nlat, nlon, dlat, 100 * n_st + n_sets)
    with T.Engine(T.MODE_BINARY) as e:
        l0 = launches(e)
        out, cost, idx = e.grid(st, desc, rds)
        l1 = launches(e)
        out_m, cost_m, idx_m = grid_masked_null(e, st, desc, rds)
        l2 = launches(e)
    assert l1 - l0 == l2 - l1
    assert idx.tolist() == idx_m.tolist()
    assert cost.view(np.uint64).tolist() == cost_m.view(np.uint64).tolist()
    assert out.tobytes() == out_m.tobytes()


def masks_for(n_st, n_sets, rng):
    """per set: one unused pair, random subsets, down to a spanning path (station k with k + 1); some sets with no
    used pair"""
    P = n_st * (n_st - 1) // 2
    used = np.ones((n_sets, P), bool)
    path = np.array([j == i + 1 for i, j in pairs(n_st)])
    for k in range(n_sets):
        kind = k % 5
        if kind == 1:
            used[k, int(rng.integers(0, P))] = False
        elif kind == 2:
            used[k] = rng.uniform(0, 1, P) < 0.6
            used[k, 0] = True
        elif kind == 3:
            used[k] = path
        elif kind == 4 and k % 10 == 4:
            used[k] = False
    return used


CASES = [(3, 20, 90, 110, 0.002), (4, 30, 120, 100, 0.0015), (5, 25, 150, 129, 0.001), (16, 15, 300, 300, 0.0015),
         (4, 600, 40, 37, 0.003), (5, 3, 64, 300, 0.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_st,n_sets,nlat,nlon,dlat", CASES)
def test_masked_ranked_equals_exhaustive(n_st, n_sets, nlat, nlon, dlat):
    """One unused pair down to a spanning path, NaN in every unused slot, sets with no used pair, dlat = 0 (every
    cell ties with nlat - 1 others: the lowest index wins), more than 512 sets; ranked vs every cell, bit for bit;
    one set against the restatement (index equal, cost within 1e-9)."""
    st, desc, rds, rng = grid_case(n_st, n_sets, nlat, nlon, dlat, 7 * n_st + n_sets)
    used = masks_for(n_st, n_sets, rng)
    rds = np.where(used, rds, np.nan)
    with T.Engine(T.MODE_BINARY) as e, T.Engine(T.MODE_BINARY, use_fft=0) as ex:
        l0, l1 = launches(e), launches(ex)
        out, cost, idx = e.grid(st, desc, rds, used=used)
        out0, cost0, idx0 = ex.grid(st, desc, rds, used=used)
        n_l = launches(e) - l0, launches(ex) - l1
    assert n_l == (5 * ((n_sets + 511) // 512), 2)   # no fall-back: sets without a used pair are not searched
    assert idx.tolist() == idx0.tolist()
    assert cost.view(np.uint64).tolist() == cost0.view(np.uint64).tolist()
    assert out.tobytes() == out0.tobytes()
    none = ~used.any(axis=1)
    assert none.any() or n_sets < 5
    assert (idx[none] == -1).all() and np.isnan(cost[none]).all() and np.isnan(out[none]).all()
    assert (idx[~none] >= 0).all()
    if dlat == 0.0:
        assert all(int(i) < nlon for i in idx[~none])
    for k in range(1, min(4, n_sets)):
        wi, wc, wl = WG.grid_solve(st, rds[k], desc, used[k])
        assert idx[k] == wi and cost[k] == pytest.approx(wc, rel=1e-9)


@pytest.mark.gpu
def test_masked_tie_plateau_falls_back():
    """dlat = dlon = 0: every cell of the grid ties, more than the candidate table holds (64 per set + 1024); the
    ranked pass overflows and every cell is evaluated (five launches, then two)."""
    st, _, rds, rng = grid_case(5, 3, 2, 2, 0.0, 77)
    used = masks_for(5, 3, rng)
    desc = [41.26, -96.02, 0.0, 0.0, 50, 50, 350.0]
    with T.Engine(T.MODE_BINARY) as e, T.Engine(T.MODE_BINARY, use_fft=0) as ex:
        l0 = launches(e)
        out, cost, idx = e.grid(st, desc, rds, used=used)
        assert launches(e) - l0 == 5 + 2
        out0, cost0, idx0 = ex.grid(st, desc, rds, used=used)
    assert idx.tolist() == idx0.tolist() == [0, 0, 0]
    assert cost.view(np.uint64).tolist() == cost0.view(np.uint64).tolist()


# ------------------------------------------------------------------ the windowed seed on constructed tables
B, W = 4000, 500
N_REF = 16


def trapped_tables():
    """TGT windows: TRAPPED[0] with every pair, TRAPPED[1] with every pair, TRAPPED[0] without pair (0, 1), then a
    window with pair (0, 1) only (status 2); REF windows at lag 0 (no drift)"""
    P = 6
    ys = [exact_rd(ST4, TRAPPED[0]), exact_rd(ST4, TRAPPED[1]), exact_rd(ST4, TRAPPED[0]), exact_rd(ST4, TRAPPED[0])]
    y = np.stack(ys) * FS / CL
    ref = np.zeros((N_REF, P), T.PEAK_DTYPE)
    tgt = np.zeros((len(ys), P), T.PEAK_DTYPE)
    tgt["lag"] = np.round(y).astype(np.int32)
    tgt["frac"] = (y - np.round(y)).astype(np.float32)
    tgt["flags"][2, 0] = T.PEAK_EMPTY
    tgt["flags"][3, 1:] = T.PEAK_EMPTY
    caps = [np.random.default_rng(60 + k).integers(0, 256, 6 * B, dtype=np.uint8) for k in range(4)]
    return ref, tgt, caps


def verdict(got, want, k):
    """tools/windows_bench.py's fix verdict: within 1e-4 m of the statement's fix, or the same rms to 1e-9"""
    dpos = metres(got["position"][k], want["position"][k])
    return dpos <= 1e-4 or abs(got["rms"][k] - want["rms"][k]) <= 1e-9 * max(want["rms"][k], 1.0)


@pytest.mark.gpu
def test_window_fixes_grid_frees_the_trapped_fixes():
    ref, tgt, caps = trapped_tables()
    with T.Engine(T.MODE_EXTENDED, n_stations=4) as e:
        for k, c in enumerate(caps):
            e.load_u8(k, c)
        got = e.window_fixes(ST4, 0, W, ref, tgt, W, grid=TRAP_GRID)
        plain = e.window_fixes(ST4, 0, W, ref, tgt, W)
    want = WG.window_fixes(ST4, [3 * B] * 4, 0, 0, W, W, ref, tgt, fs=FS, dims=2, grid=TRAP_GRID)
    for key in ("ref_fit", "range_differences", "pair_used", "status"):
        assert np.asarray(got[key]).tobytes() == np.asarray(plain[key]).tobytes(), key
    assert got["status"].tolist() == [0, 0, 0, 2]
    assert got["seed_index"].tolist() == want["seed_index"].tolist()
    assert got["seed_index"][3] == -1 and np.isnan(got["seed_cost"][3])
    assert np.array_equal(got["seed"][3], plain["position"][3])     # status 2 keeps its start
    assert np.array_equal(got["position"][3], plain["position"][3])
    for k, tx in enumerate([TRAPPED[0], TRAPPED[1], TRAPPED[0]]):
        assert metres(got["position"][k], tx) <= 1.0            # the north_star bound
        assert metres(plain["position"][k], tx) > 4000.0        # the station mean's local minimum
        assert got["seed_cost"][k] == pytest.approx(want["seed_cost"][k], rel=1e-9)
        assert verdict(got, want, k)


@pytest.mark.gpu
def test_windowed_fallback_equals_every_cell():
    """A tie plateau (dlat = dlon = 0, more tied cells than the candidate table holds): the optimistic ranked pass
    overflows and the call reruns the grid on every cell and the fixes; seeds and fixes equal a use_fft = 0
    engine's bit for bit."""
    ref, tgt, caps = trapped_tables()
    plateau = [41.30, -96.10, 0.0, 0.0, 40, 40, 350.0]
    res = []
    for use_fft in (None, 0):
        kw = {} if use_fft is None else {"use_fft": use_fft}
        with T.Engine(T.MODE_EXTENDED, n_stations=4, **kw) as e:
            for k, c in enumerate(caps):
                e.load_u8(k, c)
            l0 = launches(e)
            res.append(e.window_fixes(ST4, 0, W, ref, tgt, W, grid=plateau))
            res[-1]["launches"] = launches(e) - l0
    ranked, every = res
    assert ranked["launches"] == 3 + 5 + 1 + 2 + 1     # fit, rd, rows; ranked; fix; then every cell and the fix again
    assert every["launches"] == 3 + 2 + 1
    for key in ("seed", "seed_cost", "seed_index", "position", "rms", "status", "iters"):
        assert np.asarray(ranked[key]).tobytes() == np.asarray(every[key]).tobytes(), key
    assert ranked["seed_index"].tolist() == [0, 0, 0, -1]


# ------------------------------------------------------------------ process_windows_grid on drifting captures
BD, WD = 4_000_000, 500_000
N_REF_D, N_TGT_D = 2 * BD // WD, BD // WD
EPS_PPM = np.array([0.0, 4.0, -5.0, 2.0])


def delays(stations, x_llh):
    d = np.round(np.array([np.linalg.norm(oracle.llh_to_ecef(*x_llh) - oracle.llh_to_ecef(*s)) for s in stations]) / CL * FS)
    d = d.astype(np.int64)
    return d - d.min()


def drift_captures(tx, stations=ST4, block=BD, seed=5, noise=0.02):
    """tests/test_gpu_windows.py's drifting captures with the transmitter at tx"""
    dR, dT = delays(stations, REF_TX), delays(stations, tx)
    n = 3 * block
    pad = int(max(dR.max(), dT.max()) + np.abs(EPS_PPM).max() * 1e-6 * n) + 16
    ref = fm_signal(n + 2 * pad, 1000 + seed, 75e3)
    tgt = fm_signal(n + 2 * pad, 2000 + seed, 60e3)
    t = np.arange(n)
    in_tgt = (t >= block) & (t < 2 * block)
    raws = []
    for k in range(len(stations)):
        d = np.where(in_tgt, dT[k], dR[k]) + np.round(EPS_PPM[k] * 1e-6 * t).astype(np.int64)
        idx = pad + t - d
        x = np.where(in_tgt, tgt[idx], ref[idx])
        g = np.random.default_rng(3000 + 17 * seed + k)
        x = x + noise * (g.standard_normal(n) + 1j * g.standard_normal(n))
        raws.append(quantise(x))
    return raws


@pytest.fixture(scope="module")
def trapped_drift():
    return drift_captures(TRAPPED[0])


@pytest.mark.gpu
def test_process_windows_grid_on_drifting_captures(trapped_drift):
    """Tables, REF fit, range differences and used pairs equal process_windows' bit for bit; every window's fix
    passes the verdict against the restatement on the returned tables and lies nearer the transmitter than the
    station-mean start's fix (which the station mean's local minimum holds kilometres away)."""
    raws = trapped_drift
    args = (ST4, 0, WD, N_REF_D, N_TGT_D, WD)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        plain = e.process_windows(*args, ref_tx_llh=REF_TX)
        got = e.process_windows(*args, ref_tx_llh=REF_TX, grid=TRAP_GRID)
    for key in ("ref", "tgt", "ref_fit", "range_differences", "pair_used"):
        assert np.asarray(got[key]).tobytes() == np.asarray(plain[key]).tobytes(), key
    want = WG.window_fixes(ST4, [r.size // 2 for r in raws], 0, 0, WD, WD, got["ref"], got["tgt"], fs=FS, dims=2,
                           ref_tx_llh=REF_TX, grid=TRAP_GRID)
    assert (got["status"] == 0).all()
    assert got["seed_index"].tolist() == want["seed_index"].tolist()
    for k in range(N_TGT_D):
        assert verdict(got, want, k)
        assert metres(got["position"][k], TRAPPED[0]) < metres(plain["position"][k], TRAPPED[0])


# ------------------------------------------------------------------ more than one GPU
def same_results(want, got):
    """Everything bit for bit, but the tables' margin: the pair loops evaluate the runner-up lags of a dealt call in
    other batches than those of the one-GPU call, which moves a REF margin of these captures by up to 1.2e-7 (the
    same with or without a grid, and in the windowed calls before the grid seed existed).  The fix stage reads
    margins only through min_margin (0 here)."""
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
def test_one_rank_communicator_gives_the_one_gpu_results(trapped_drift):
    raws = trapped_drift
    args = (ST4, 0, WD, 4, 2, WD)
    res = []
    for comm in (False, True):
        with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
            if comm:
                e.comm_init(T.comm_unique_id(), 0, 1)
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            res.append(e.process_windows(*args, ref_tx_llh=REF_TX, grid=TRAP_GRID))
    same_results(*res)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_one_gpu_results(trapped_drift):
    raws = trapped_drift
    args = (ST4, 0, WD, 4, 2, WD)
    res = []
    for n_dev in (1, 2):
        with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4, n_devices=n_dev) as e:
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            res.append(e.process_windows(*args, ref_tx_llh=REF_TX, grid=TRAP_GRID))
    same_results(*res)


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_argument_errors():
    ref, tgt, caps = trapped_tables()
    with T.Engine(T.MODE_EXTENDED, n_stations=4) as e:
        for k, c in enumerate(caps):
            e.load_u8(k, c)
        for desc, msg in (([41.0, -96.0, 0.01, 0.01, 0, 10, 350.0], "empty grid"),
                          ([41.0, -96.0, 0.01, 0.01, 3e9, 10, 350.0], "too large"),
                          ([41.0, -96.0, 0.01, 0.01, 1e6, 1e6, 350.0], "too large")):
            with pytest.raises(T.TdoaError, match=msg):
                e.window_fixes(ST4, 0, W, ref, tgt, W, grid=desc)
            with pytest.raises(T.TdoaError, match=msg):
                e.process_windows(ST4, 0, W, N_REF, 3, W, grid=desc)
            with pytest.raises(T.TdoaError, match=msg):
                e.grid(ST4, desc, np.zeros((1, 6)), used=np.ones((1, 6), bool))
        with pytest.raises(T.TdoaError, match="dims"):   # what the base call refuses
            e.window_fixes(ST4, 0, W, ref, tgt, W, dims=4, grid=TRAP_GRID)
        # a NULL grid_desc
        o = T._native.WindowOpts(dims=2)
        P = 6
        bufs = [np.zeros(n) for n in (3 * P, tgt.shape[0] * P, 3 * tgt.shape[0], tgt.shape[0])]
        status = np.zeros(tgt.shape[0], np.int32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        st = np.ascontiguousarray(ST4)
        for fn, tabs in ((e._lib.tdoa_window_fixes_grid, (p(ref), p(tgt))), (e._lib.tdoa_process_windows_grid, (None, None))):
            rc = fn(e._h, p(st), C.byref(o), 0, W, N_REF, tgt.shape[0], W, None, *tabs, p(bufs[0]), p(bufs[1]), None,
                    p(bufs[2]), p(bufs[3]), p(status), None, None, None, None)
            assert rc == -1 and "grid_desc" in e.last_error()
    # more than 16 stations
    S = 17
    st17 = np.vstack([ST4, ST4[0] + np.arange(1, 14)[:, None] * [0.01, 0.01, 0.0]])
    caps17 = [np.random.default_rng(k).integers(0, 256, 6 * B, dtype=np.uint8) for k in range(S)]
    P17 = S * (S - 1) // 2
    with T.Engine(T.MODE_EXTENDED, n_stations=S) as e:
        for k, c in enumerate(caps17):
            e.load_u8(k, c)
        with pytest.raises(T.TdoaError, match="16 stations"):
            e.window_fixes(st17, 0, W, np.zeros((N_REF, P17), T.PEAK_DTYPE), np.zeros((2, P17), T.PEAK_DTYPE), W, grid=TRAP_GRID)
        with pytest.raises(T.TdoaError, match="16 stations"):
            e.process_windows(st17, 0, W, N_REF, 2, W, grid=TRAP_GRID)
        with pytest.raises(T.TdoaError, match="16 stations"):
            e.grid(st17, TRAP_GRID, np.zeros((1, P17)), used=np.ones((1, P17), bool))
