"""The station check of the windowed fixes on the GPU: k_window_exclude (tdoa_exclude_stations) against its
restatement (tests/exclusion_oracle.py), every candidate against tdoa_solve_ls on the stations without it, the inert
check against the calls without it, a station that hears another programme, corrupted tables, the closure check and
the station check together, the grid's second seed, more than one GPU, and the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import tdoa_b200 as T
import closure_oracle as CO
import exclusion_oracle as XO
from test_gpu_window_grid import ST4, TRAP_GRID, TRAPPED, REF_TX, W, N_REF, WD, drift_captures, same_results, exact_rd, metres
from test_gpu_closure import ST6, TX6, BE, interfered_captures

FS, CL = 2e6, 299792458.0
INERT = {"max_rms": math.inf}
B = 4000


def stations(S, seed, dims=2):
    """dims 3: stations between 0 and 3000 m, where the elevation is determined"""
    rng = np.random.default_rng(seed)
    h = (300, 400) if dims == 2 else (0, 3000)
    return np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), rng.uniform(*h)] for _ in range(S)])


def station_offset(rd, S, s, delta):
    out = np.array(rd, np.float64)
    for p, (i, j) in enumerate(CO.pairs(S)):
        out[..., p] += delta if j == s else (-delta if i == s else 0.0)
    return out


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64).tolist()


def same(a, b, keys):
    for k in keys:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


# ------------------------------------------------------------------ kernel against the restatement
def parity_sets(S, n_distinct, seed, dims):
    """exact range differences + 2 m of noise; per set none, one or two bad stations (2..20 km; at least one in the
    first set) and a full or random mask.  A set is kept only when its first-round candidate rms keep the best and the
    second best apart by 4x (the decision then does not rest on rounding)"""
    rng = np.random.default_rng(seed)
    st = stations(S, seed, dims)
    P = S * (S - 1) // 2
    rds, used, init = [], [], []
    while len(rds) < n_distinct:
        tx = np.array([41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0 if dims == 2 else 1500.0])
        rd = exact_rd(st, tx) + rng.normal(0, 2.0, P)
        n_bad = int(rng.integers(0, 3)) or (0 if rds else 1)   # the first set has a bad station
        for s in rng.choice(S, n_bad, replace=False):
            rd = station_offset(rd, S, int(s), rng.choice([-1, 1]) * rng.uniform(2e3, 2e4))
        u = np.ones(P, bool) if len(rds) % 2 == 0 else rng.uniform(0, 1, P) < 0.85
        x0 = tx + [0.02, -0.02, 0.0]
        _, _, srms, _, _ = XO.exclude_set(st, np.where(u, rd, np.nan), u, x0, dims, 50.0, 0)
        f = np.sort(srms[np.isfinite(srms)])
        if f.size >= 2 and not f[1] > 4 * f[0]:
            continue
        rds.append(np.concatenate([np.where(u, rd, np.nan), [np.nan] * 2]))
        used.append(np.concatenate([u, [0, 0]]).astype(np.uint8))
        init.append(x0)
    return st, np.array(rds), np.array(used), np.array(init)


@pytest.mark.gpu
@pytest.mark.parametrize("S,dims,n_distinct,repeat", [(5, 2, 60, 100), (8, 2, 40, 100), (8, 3, 30, 10), (16, 2, 12, 10),
                                                      (16, 3, 8, 10), (64, 2, 2, 4), (64, 3, 1, 4)])
def test_kernel_equals_restatement(S, dims, n_distinct, repeat):
    """more sets than one wave: the distinct sets repeated"""
    st, rds, used, init = parity_sets(S, n_distinct, 100 * S + dims, dims)
    P = S * (S - 1) // 2
    want = XO.exclude(st, rds, used, init, dims, 50.0, 0)
    with T.Engine(T.MODE_BINARY) as e:
        got = e.exclude_stations(st, np.tile(rds, (repeat, 1)), np.tile(used, (repeat, 1)), np.tile(init, (repeat, 1)),
                                 dims, max_rms=50.0, max_exclude=0)
    n = n_distinct
    for r in range(repeat):
        g = {k: v[r * n:(r + 1) * n] for k, v in got.items()}
        assert g["used"][:, :P].tolist() == want["used"].tolist()
        assert g["station_excluded"].tolist() == want["station_excluded"].tolist()
        assert g["excluded"].tolist() == want["excluded"].tolist() and g["status"].tolist() == want["status"].tolist()
        for k in range(n):
            assert metres(g["position"][k], want["position"][k]) <= 1e-4, (r, k)
        # the same candidates, and the same first-round winner with its rms.  The losing candidates' solves keep a
        # wrong station; at dims 3 they are ill-conditioned, and where the device's sin / cos and the C library's
        # differ in the last bit their Levenberg-Marquardt runs may stop elsewhere, so their rms is not compared
        # here (test_candidates_equal_solve_ls_without_the_station pins every one to tdoa_solve_ls bit for bit)
        fin = np.isfinite(want["station_rms"])
        assert (np.isfinite(g["station_rms"]) == fin).all()
        for k in np.flatnonzero(fin.any(axis=1)):
            best = int(np.nanargmin(want["station_rms"][k]))
            assert int(np.nanargmin(g["station_rms"][k])) == best, (r, k)
            assert abs(g["station_rms"][k, best] - want["station_rms"][k, best]) <= 1e-6 * max(want["station_rms"][k, best], 1.0)
    assert (got["used"][:, P:] == 0).all()   # past P: left as the caller's arrays were
    assert want["excluded"].max() >= 1


@pytest.mark.gpu
def test_candidates_equal_solve_ls_without_the_station():
    """every finite station_rms[k] is, bit for bit, tdoa_solve_ls's rms on the stations without k (their pairs in
    order) from the same start; without a grid the final fix is the winning candidate's solve, bit for bit"""
    S = 8
    P = S * (S - 1) // 2
    rng = np.random.default_rng(3)
    st = stations(S, 77)
    txs = [np.array([41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0]) for _ in range(6)]
    rds = np.stack([station_offset(exact_rd(st, tx) + rng.normal(0, 2.0, P), S, int(rng.integers(0, S)), 5e3) for tx in txs])
    used = np.ones((len(txs), P), np.uint8)   # every pair used: the reduced problem is unmasked
    init = np.stack([tx + [0.02, -0.02, 0.0] for tx in txs])
    with T.Engine(T.MODE_BINARY) as e:
        got = e.exclude_stations(st, rds, used, init, 2, max_rms=50.0, max_exclude=1)
        for w in range(rds.shape[0]):
            assert np.isfinite(got["station_rms"][w]).all() and got["excluded"][w] == 1
            for k in range(S):
                keep = [p for p, (i, j) in enumerate(CO.pairs(S)) if k not in (i, j)]
                pos, rms, status, it = e.solve_ls(np.delete(st, k, 0), rds[w, keep], init[w], 2)
                assert bits([rms]) == bits([got["station_rms"][w, k]]), (w, k)
                if got["station_excluded"][w, k]:
                    assert bits(pos) == bits(got["position"][w]) and bits([rms]) == bits([got["rms"][w]])
                    assert (status, it) == (got["status"][w], got["iters"][w])


# ------------------------------------------------------------------ the inert check equals the calls without it
FIX_KEYS = ("ref_fit", "range_differences", "pair_used", "position", "rms", "status", "iters")


@pytest.fixture(scope="module")
def trapped_drift():
    return drift_captures(TRAPPED[0])


@pytest.mark.gpu
def test_inert_check_equals_the_calls_without_it(trapped_drift):
    args = (ST4, 0, WD, 6, 3, WD)
    with T.Engine(T.MODE_EXTENDED, max_lag=300, n_stations=4) as e:
        for k, r in enumerate(trapped_drift):
            e.load_u8(k, r)
        for grid in (None, TRAP_GRID):
            seeds = ("seed", "seed_cost", "seed_index") if grid else ()
            for closure in (None, {"max_residual": 50.0}):
                plain = e.process_windows(*args, ref_tx_llh=REF_TX, grid=grid, closure=closure)
                got = e.process_windows(*args, ref_tx_llh=REF_TX, grid=grid, closure=closure, exclusion=INERT)
                same(plain, got, FIX_KEYS + ("ref", "tgt") + seeds + (("pair_dropped", "dropped") if closure else ()))
                assert not got["pair_excluded"].any() and (got["excluded"] == 0).all()
                assert np.isnan(got["station_rms"]).all() and not got["station_excluded"].any()
                fx = e.window_fixes(ST4, 0, WD, plain["ref"], plain["tgt"], WD, ref_tx_llh=REF_TX, grid=grid, closure=closure)
                fx_x = e.window_fixes(ST4, 0, WD, plain["ref"], plain["tgt"], WD, ref_tx_llh=REF_TX, grid=grid,
                                      closure=closure, exclusion=INERT)
                same(fx, fx_x, FIX_KEYS + seeds)
        geo = ((0, WD, 6, WD), (0, 0, 1, WD))
        plain = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX)
        got = e.process_windows_retimed(ST4, *geo, ref_tx_llh=REF_TX, exclusion=INERT)
        same(plain, got, FIX_KEYS + ("ref", "tgt", "clock_rate"))


# ------------------------------------------------------------------ a station that hears another programme
@pytest.mark.gpu
def test_station_hearing_another_programme_is_excluded():
    """Station 4 hears another FM programme in block 2 (tests/test_gpu_closure.py: the closure check cannot see it).
    The fix does not fit one position; without station 4 it does, and the check excludes 4 and only 4"""
    raws = interfered_captures(4)
    args = (ST6, 0, BE // 2, 4, 2, BE // 2)
    init = TX6 + [0.03, 0.03, 0.0]
    with T.Engine(T.MODE_EXTENDED, max_lag=600, n_stations=6) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        plain = e.process_windows(*args, ref_tx_llh=REF_TX, init_llh=init)
        got = e.process_windows(*args, ref_tx_llh=REF_TX, init_llh=init, exclusion={"max_rms": MAX_RMS_FM})
        inert = e.process_windows(*args, ref_tx_llh=REF_TX, init_llh=init, exclusion=INERT)
        tgt = plain["tgt"].copy()
        for p, (i, j) in enumerate(CO.pairs(6)):
            if 4 in (i, j):
                tgt["flags"][:, p] |= T.PEAK_EMPTY
        five = e.window_fixes(ST6, 0, BE // 2, plain["ref"], tgt, BE // 2, ref_tx_llh=REF_TX, init_llh=init)
    same(plain, inert, FIX_KEYS + ("ref", "tgt"))
    same(plain, got, ("ref", "tgt", "ref_fit", "range_differences"))
    assert got["station_excluded"].tolist() == [[0, 0, 0, 0, 1, 0]] * 2 and got["excluded"].tolist() == [1, 1]
    assert (got["pair_excluded"] == ~five["pair_used"]).all() and (got["pair_used"] == five["pair_used"]).all()
    same(five, got, ("position", "rms", "status", "iters"))
    assert (plain["rms"] > MAX_RMS_FM).all() and (got["rms"] <= MAX_RMS_FM).all()
    for w in range(2):
        assert metres(plain["position"][w], TX6) > 1000.0
        assert metres(got["position"][w], TX6) <= FM_BOUND


# Measured on these captures (one B200): the plain fixes' rms 7385 / 21816 m, without station 4 42.3 / 42.6 m (the
# next candidate 4635 / 21915 m); the plain fixes 3944 / 164181 m from TX6, the five-station fixes 115.7 / 115.4 m.
# max_rms sits 7x above the leave-4-out rms and 25x below the plain rms; the bound is twice the five-station error.
MAX_RMS_FM = 300.0
FM_BOUND = 250.0


# ------------------------------------------------------------------ corrupted tables
def tables(st, rds, n_ref=N_REF):
    """REF windows at lag 0, TGT windows from the range differences rds[n][P] (lag + float32 frac)"""
    S = st.shape[0]
    y = np.asarray(rds) * FS / CL
    ref = np.zeros((n_ref, y.shape[1]), T.PEAK_DTYPE)
    tgt = np.zeros(y.shape, T.PEAK_DTYPE)
    tgt["lag"] = np.round(y).astype(np.int32)
    tgt["frac"] = (y - np.round(y)).astype(np.float32)
    caps = [np.random.default_rng(70 + k).integers(0, 256, 6 * B, dtype=np.uint8) for k in range(S)]
    return ref, tgt, caps


@pytest.mark.gpu
@pytest.mark.parametrize("S,bad", [(8, (2,)), (8, (0, 5)), (16, (11,)), (16, (3, 9))])
def test_corrupted_tables(S, bad):
    rng = np.random.default_rng(S * 10 + len(bad))
    st = stations(S, 600 + S)
    txs = [np.array([41.26 + rng.uniform(-0.08, 0.08), -96.02 + rng.uniform(-0.1, 0.1), 350.0]) for _ in range(6)]
    clean_rd = np.stack([exact_rd(st, tx) for tx in txs])
    worse = clean_rd
    for s in bad:
        worse = station_offset(worse, S, s, rng.choice([-1, 1]) * rng.uniform(2e3, 2e4))
    ref, tgt, caps = tables(st, clean_rd)
    _, tgt_w, _ = tables(st, worse)
    with T.Engine(T.MODE_EXTENDED, n_stations=S) as e:
        for s, cap in enumerate(caps):
            e.load_u8(s, cap)
        clean = e.window_fixes(st, 0, W, ref, tgt, W)
        plain = e.window_fixes(st, 0, W, ref, tgt_w, W)
        got = e.window_fixes(st, 0, W, ref, tgt_w, W, exclusion={"max_rms": 50.0, "max_exclude": len(bad)})
    want = np.zeros(S, bool)
    want[list(bad)] = True
    assert ((got["station_excluded"] > 0) == want).all() and got["excluded"].tolist() == [len(bad)] * 6
    assert (got["pair_excluded"] == np.array([bool(set(bad) & {i, j}) for i, j in CO.pairs(S)])).all()
    assert max(metres(plain["position"][w], clean["position"][w]) for w in range(6)) > 1000.0
    for w in range(6):
        assert metres(got["position"][w], clean["position"][w]) <= 1.0


@pytest.mark.gpu
def test_closure_and_exclusion_together():
    """one wrong pair and one wrong station in the same window: the closure check drops the pair (2), then the
    station check takes the station (3)"""
    S = 8
    st = stations(S, 31)
    tx = np.array([41.27, -96.03, 350.0])
    rd = station_offset(exact_rd(st, tx), S, 2, 4.5e3)
    q = CO.pairs(S).index((5, 7))
    rd[q] += 30e3
    ref, tgt, caps = tables(st, rd[None])
    _, tgt_c, _ = tables(st, exact_rd(st, tx)[None])
    with T.Engine(T.MODE_EXTENDED, n_stations=S) as e:
        for s, cap in enumerate(caps):
            e.load_u8(s, cap)
        clean = e.window_fixes(st, 0, W, ref, tgt_c, W)
        got = e.window_fixes(st, 0, W, ref, tgt, W, closure={"max_residual": 100.0}, exclusion={"max_rms": 50.0})
    assert got["pair_dropped"][0].tolist() == [p == q for p in range(len(CO.pairs(S)))]
    assert got["pair_excluded"][0].tolist() == [2 in (i, j) for i, j in CO.pairs(S)]
    assert got["dropped"].tolist() == [1] and got["excluded"].tolist() == [1] and got["station_excluded"][0, 2] == 1
    assert metres(got["position"][0], clean["position"][0]) <= 1.0


# ------------------------------------------------------------------ the grid's second seed
ST5 = ST6[:5]


@pytest.mark.gpu
def test_grid_seeds_again_on_the_final_mask():
    """five stations, the transmitter outside their hull, station 4's range 8 km long: the first arg-min (over every
    pair) starts the check's solves where the solve without station 4 is trapped 4.9 km away (the restatement);
    seeded again over the final mask, the fix is not trapped.  The seed outputs are tdoa_grid_masked's arg-min over
    the returned mask, and evaluating every cell (use_fft = 0) gives the same results"""
    S = 5
    rd = station_offset(exact_rd(ST5, TRAPPED[0]), S, 4, 8e3)
    ref, tgt, caps = tables(ST5, rd[None])
    _, tgt_c, _ = tables(ST5, exact_rd(ST5, TRAPPED[0])[None])
    res = []
    for use_fft in (1, 0):
        with T.Engine(T.MODE_EXTENDED, n_stations=S, use_fft=use_fft) as e:
            for s, cap in enumerate(caps):
                e.load_u8(s, cap)
            got = e.window_fixes(ST5, 0, W, ref, tgt, W, grid=TRAP_GRID, exclusion={"max_rms": 50.0})
            clean = e.window_fixes(ST5, 0, W, ref, tgt_c, W, grid=TRAP_GRID)
            first = e.grid(ST5, TRAP_GRID, got["range_differences"], used=np.ones_like(got["pair_used"]))
            seed = e.grid(ST5, TRAP_GRID, got["range_differences"], used=got["pair_used"])
            x0 = e.exclude_stations(ST5, got["range_differences"], np.ones_like(got["pair_used"]), first[0], 2, max_rms=50.0)
        assert got["station_excluded"].tolist() == [[0, 0, 0, 0, 1]]
        assert got["seed_index"].tolist() == seed[2].tolist() != first[2].tolist()
        assert bits(got["seed_cost"]) == bits(seed[1]) and bits(got["seed"]) == bits(seed[0])
        assert metres(x0["position"][0], TRAPPED[0]) > 1000.0       # the check's solve from the first arg-min
        assert metres(got["position"][0], TRAPPED[0]) <= 1.0        # the fix from the second
        assert metres(got["position"][0], clean["position"][0]) <= 1.0
        res.append(got)
    same_results(res[0], res[1])


# ------------------------------------------------------------------ more than one GPU
def interfered_run(raws, **kw):
    with T.Engine(T.MODE_EXTENDED, max_lag=600, n_stations=6, **kw.pop("engine", {})) as e:
        if kw.pop("comm", False):
            e.comm_init(T.comm_unique_id(), 0, 1)
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        return e.process_windows(ST6, 0, BE // 2, 4, 2, BE // 2, ref_tx_llh=REF_TX, grid=TRAP_GRID,
                                 closure={"max_residual": 300.0}, exclusion={"max_rms": 100.0})


@pytest.fixture(scope="module")
def interfered():
    return interfered_captures(4)


@pytest.mark.gpu
def test_one_rank_communicator_gives_the_one_gpu_results(interfered):
    one = interfered_run(interfered)
    assert one["excluded"].tolist() == [1, 1]
    same_results(one, interfered_run(interfered, comm=True))


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_give_the_one_gpu_results(interfered):
    same_results(interfered_run(interfered), interfered_run(interfered, engine={"n_devices": 2}))


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_argument_errors():
    st = stations(6, 1)
    ref, tgt, caps = tables(st, np.zeros((3, 15)))
    rd, u = np.zeros((2, 15)), np.ones((2, 15), np.uint8)
    with T.Engine(T.MODE_EXTENDED, n_stations=6) as e:
        for k, cap in enumerate(caps):
            e.load_u8(k, cap)
        for bad in ({"max_rms": 0.0}, {"max_rms": -1.0}, {"max_rms": math.nan}, {"max_rms": 10.0, "max_exclude": -1}):
            with pytest.raises(T.TdoaError, match="max_"):
                e.window_fixes(st, 0, W, ref, tgt, W, exclusion=bad)
            with pytest.raises(T.TdoaError, match="max_"):
                e.process_windows(st, 0, W, N_REF, 3, W, exclusion=bad)
            with pytest.raises(T.TdoaError, match="max_"):
                e.exclude_stations(st, rd, u, **bad)
        with pytest.raises(T.TdoaError, match="dims"):   # what the base call refuses
            e.window_fixes(st, 0, W, ref, tgt, W, dims=4, exclusion=INERT)
        with pytest.raises(T.TdoaError, match="max_residual"):   # and the closure options
            e.window_fixes(st, 0, W, ref, tgt, W, closure={"max_residual": 0.0}, exclusion=INERT)
        for sts, dims, rds, msg in ((st[:2], 2, np.zeros((2, 1)), "stations"), (stations(65, 2), 2, np.zeros((1, 65 * 32)), "stations"),
                                    (st, 4, rd, "dims"), (st, 2, np.zeros((2, 14)), "rd_stride")):
            with pytest.raises(T.TdoaError, match=msg):
                e.exclude_stations(sts, rds, np.ones(rds.shape, np.uint8), None, dims, max_rms=10.0)
        # NULL options, retimed not 0 / 1, n_sets < 0
        o = T._native.WindowOpts(dims=2)
        x = T._native.ExclusionOpts(max_rms=10.0, max_exclude=1)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        sa = np.ascontiguousarray(st)
        fix, status = np.zeros((3, 3)), np.zeros(3, np.int32)
        out = np.zeros((2, 15), np.uint8)
        L = e._lib
        assert L.tdoa_exclude_stations(e._h, p(sa), 6, p(rd), p(u), 2, 15, None, 2, None, p(out), None, None, None,
                                       p(fix), None, p(status), None) == -1
        assert "exclusion options" in e.last_error()
        assert L.tdoa_exclude_stations(e._h, p(sa), 6, p(rd), p(u), -1, 15, None, 2, C.byref(x), p(out), None, None, None,
                                       p(fix), None, p(status), None) == -1
        assert "n_sets" in e.last_error()
        assert L.tdoa_window_fixes_exclude(e._h, p(sa), C.byref(o), None, None, 0, W, N_REF, 3, W, None, p(ref), p(tgt),
                                           *[None] * 8, p(fix), None, p(status), None, None, None, None) == -1
        assert "exclusion options" in e.last_error()
        for retimed in (2, -1):
            rc = L.tdoa_process_windows_exclude(e._h, p(sa), C.byref(o), None, C.byref(x), 0, W, N_REF, W, 0, W, 3, W,
                                                retimed, *[None] * 11, p(fix), None, p(status), None, None, None, None, None)
            assert rc == -1 and "retimed" in e.last_error()
