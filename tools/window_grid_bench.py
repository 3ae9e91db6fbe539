#!/usr/bin/env python
"""Times grid-seeded windowed fixes (tdoa_process_windows_grid) against tdoa_process_windows on the two windowed
workloads of tools/windows_bench.py (same run, alternating), with the fix stage's device time of both and an oracle
verdict on one window.  With --parent-lib it also times BASELINE config 5 (tdoa_grid, 1000 x 1000 cells, 16 stations,
64 sets) and tdoa_process_windows_grid on both workloads with this tree's library and with a second library (e.g. built
from the parent commit), alternating in one process, and checks that both give the same bits.

    python tools/window_grid_bench.py [--reps K] [--parent-lib PATH] [--out profiles/r4_window_grid.jsonl]

  cfg3      3 stations, 66 REF + 33 TGT windows of 2e6 samples, +-50 000 lags, EXTENDED; grid 400 x 400 cells of
            0.0005 deg around the stations
  configs3  16 stations (120 pairs), weak_signal_simulator.go content, 66 + 33 windows, +-2000 lags, EXTENDED; grid
            1000 x 1000 cells of 0.0005 deg around the ring (config 5's grid)

Verdict: the restatements (tests/window_oracle.py, tests/window_grid_oracle.py) on the returned tables for one TGT window, its grid search over the
11 x 11 cells around the engine's seed cell (as tools/configs_bench.py checks config 5) and windows_bench.py's fix
verdict.  One JSON line per case (stdout and --out) with the card name and power limit read in the same run."""
import argparse
import ctypes
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))

import torch  # noqa: E402

import bench  # noqa: E402
import configs_bench  # noqa: E402
import simulators as S  # noqa: E402
import tdoa_b200 as T  # noqa: E402
import window_grid_oracle as WG  # noqa: E402  (the checker; never on the measured path)
import window_oracle as WO  # noqa: E402
from oracle import oracle  # noqa: E402
from windows_bench import BLOCK, W, card  # noqa: E402

_N = sys.modules[T.Engine.__module__]


def around(stations, n, step=0.0005, elev=350.0):
    st = np.asarray(stations)
    return [float(st[:, 0].mean()) - 0.5 * n * step, float(st[:, 1].mean()) - 0.5 * n * step, step, step, n, n, elev]


def verdict(stations, res, grid, w):
    """the seeded fix stage's statement on the engine's tables, TGT window w: range differences and mask as
    windows_bench.py checks them, the seed cell by the masked grid statement over the 11 x 11 cells around it, the
    fix from that cell by the restatement's least-squares step"""
    want = WO.window_fixes(stations, res["nsamp"], 0, 0, W, W, res["ref"], res["tgt"], fs=2e6, dims=2)
    u = want["pair_used"][w]
    rd = want["range_differences"][w]
    ok = bool(np.array_equal(u, res["pair_used"][w]))
    drd = float(np.abs(rd[u] - res["range_differences"][w][u]).max()) if u.any() else 0.0
    nlat, nlon = int(grid[4]), int(grid[5])
    idx = int(res["seed_index"][w])
    out = {"tgt_window": w, "pairs_used": int(u.sum()), "max_abs_rd_diff_m": drd, "seed_index": idx}
    if idx < 0:
        ok = ok and WG.too_few(u, len(stations), 2) and int(res["status"][w]) == 2
        return {**out, "ok": "ok" if ok else "MISMATCH"}
    a, b = divmod(idx, nlon)
    a0, b0 = min(max(a - 5, 0), max(nlat - 11, 0)), min(max(b - 5, 0), max(nlon - 11, 0))
    sub = [grid[0] + a0 * grid[2], grid[1] + b0 * grid[3], grid[2], grid[3], min(11, nlat), min(11, nlon), grid[6]]
    wi, wc, cell = WG.grid_solve(stations, rd, sub, u)
    same_cell = (a0 + wi // sub[5], b0 + wi % sub[5]) == (a, b)
    dcost = abs(float(res["seed_cost"][w]) - wc) / max(abs(wc), 1e-300)
    fix, rms, status, _ = WO.solve_ls(stations, rd, res["seed"][w], 2, u)
    dpos = float(np.linalg.norm(oracle.llh_to_ecef(*fix) - oracle.llh_to_ecef(*res["position"][w])))
    same_fix = dpos <= 1e-4 or abs(float(res["rms"][w]) - rms) <= 1e-9 * max(rms, 1.0)
    ok = ok and drd <= 1e-6 and same_cell and dcost <= 1e-9 and same_fix and status == int(res["status"][w])
    return {**out, "seed_cost_rel_diff": dcost, "seed_cell_is_local_argmin": bool(same_cell), "fix_diff_m": dpos,
            "rms_m": float(res["rms"][w]), "oracle_rms_m": float(rms), "status": int(res["status"][w]),
            "ok": "ok" if ok else "MISMATCH"}


def run_case(name, e, stations, caps, grid, reps, tx):
    nw_t, nw_r = BLOCK // W, 2 * BLOCK // W

    def pw(g=None):
        return e.process_windows(stations, 0, W, nw_r, nw_t, W, grid=g)

    for _ in range(2):   # warm every shape
        pw(); pw(grid)
    t_pw, t_pg, fix_pw, fix_pg = [], [], [], []
    for _ in range(reps):   # alternating
        torch.cuda.synchronize(); t0 = time.perf_counter(); plain = pw(); t_pw.append(time.perf_counter() - t0)
        fix_pw.append(e.stats()["ms_fix"])
        torch.cuda.synchronize(); t0 = time.perf_counter(); res = pw(grid); t_pg.append(time.perf_counter() - t0)
        fix_pg.append(e.stats()["ms_fix"])
    res["nsamp"] = [c.numel() // 2 for c in caps]
    same = all(np.asarray(res[k]).tobytes() == np.asarray(plain[k]).tobytes()
               for k in ("ref", "tgt", "ref_fit", "range_differences", "pair_used"))
    med = lambda v: 1e3 * float(np.median(v))   # noqa: E731
    err = lambda p: float(np.median([np.linalg.norm(oracle.llh_to_ecef(*x) - oracle.llh_to_ecef(*tx)) for x in p]))  # noqa: E731
    return {"case": name, "windows": {"ref": nw_r, "tgt": nw_t, "samples": W}, "pairs": e.n_pairs, "grid": grid,
            "reps": reps, "process_windows_ms": med(t_pw), "process_windows_grid_ms": med(t_pg),
            "process_windows_ms_all": [1e3 * t for t in t_pw], "process_windows_grid_ms_all": [1e3 * t for t in t_pg],
            "ms_fix": float(np.median(fix_pw)), "ms_fix_grid": float(np.median(fix_pg)),
            "ms_fix_all": fix_pw, "ms_fix_grid_all": fix_pg,
            "tables_rd_used_equal_process_windows": bool(same),
            "status_counts": np.bincount(res["status"], minlength=3).tolist(),
            "unsearched_windows": int((res["seed_index"] < 0).sum()),
            "median_fix_err_m": err(plain["position"]), "median_fix_err_grid_m": err(res["position"]),
            "note": "fix errors are against the simulated transmitter, without the REF transmitter's geometric term",
            "oracle": verdict(stations, res, grid, nw_t // 2)}


def engine_on(lib_path, *args, **kw):
    """an Engine bound to another build of the library (which may lack this build's newer symbols)"""
    other, cur = ctypes.CDLL(str(lib_path)), _N.load_library()
    for name in ("tdoa_default_config", "tdoa_create", "tdoa_destroy", "tdoa_last_error", "tdoa_grid", "tdoa_get_stats",
                 "tdoa_load_u8_device", "tdoa_process_windows_grid"):
        getattr(other, name).argtypes = getattr(cur, name).argtypes
        getattr(other, name).restype = getattr(cur, name).restype
    saved = _N._lib
    try:
        _N._lib = other
        return T.Engine(*args, **kw)
    finally:
        _N._lib = saved


def cfg5_ab(parent_lib, reps):
    """config 5 (tools/configs_bench.py cfg5's sets and grid) on this tree's library and the other, alternating"""
    st16 = configs_bench.ring_stations(16)
    _, dist = configs_bench.delays_for(st16)
    rd = np.array([dist[j] - dist[i] for i in range(16) for j in range(i + 1, 16)])
    rds = rd[None, :] + np.random.default_rng(5).normal(0, 50e-9 * configs_bench.C, (64, rd.size))
    desc = [41.26 - 0.25, -96.02 - 0.25, 0.0005, 0.0005, 1000, 1000, 400.0]
    engines = {"branch": T.Engine(T.MODE_BINARY), "parent": engine_on(parent_lib, T.MODE_BINARY)}
    times = {k: [] for k in engines}
    outs = {}
    for e in engines.values():
        e.grid(st16, desc, rds)
    for _ in range(reps):
        for k, e in engines.items():
            torch.cuda.synchronize(); t0 = time.perf_counter(); outs[k] = e.grid(st16, desc, rds)
            times[k].append(time.perf_counter() - t0)
    for e in engines.values():
        e.close()
    same = (outs["branch"][2].tolist() == outs["parent"][2].tolist() and
            outs["branch"][1].view(np.uint64).tolist() == outs["parent"][1].view(np.uint64).tolist())
    return {"case": "config 5: tdoa_grid 1000 x 1000 cells, 16 stations, 64 sets, branch vs parent build", "reps": reps,
            "branch_ms": 1e3 * float(np.median(times["branch"])), "parent_ms": 1e3 * float(np.median(times["parent"])),
            "branch_ms_all": [1e3 * t for t in times["branch"]], "parent_ms_all": [1e3 * t for t in times["parent"]],
            "same_index_and_cost": bool(same)}


def windows_ab(name, engines, stations, grid, reps):
    """tdoa_process_windows_grid with this tree's library and the other (engines: {"branch", "parent"}, both loaded
    with the same captures), alternating; every returned array must be the same bits"""
    nw_t, nw_r = BLOCK // W, 2 * BLOCK // W
    times = {k: [] for k in engines}
    fix = {k: [] for k in engines}
    outs = {}
    for _ in range(2):   # warm every shape
        for e in engines.values():
            e.process_windows(stations, 0, W, nw_r, nw_t, W, grid=grid)
    for _ in range(reps):
        for k, e in engines.items():
            torch.cuda.synchronize(); t0 = time.perf_counter()
            outs[k] = e.process_windows(stations, 0, W, nw_r, nw_t, W, grid=grid)
            times[k].append(time.perf_counter() - t0)
            fix[k].append(e.stats()["ms_fix"])
    same = all(np.asarray(outs["branch"][k]).tobytes() == np.asarray(outs["parent"][k]).tobytes() for k in outs["branch"])
    med = lambda v: 1e3 * float(np.median(v))   # noqa: E731
    return {"case": name + ": tdoa_process_windows_grid, branch vs parent build", "grid": grid, "reps": reps,
            "branch_ms": med(times["branch"]), "parent_ms": med(times["parent"]),
            "branch_ms_all": [1e3 * t for t in times["branch"]], "parent_ms_all": [1e3 * t for t in times["parent"]],
            "branch_ms_fix": float(np.median(fix["branch"])), "parent_ms_fix": float(np.median(fix["parent"])),
            "branch_ms_fix_all": fix["branch"], "parent_ms_fix_all": fix["parent"], "same_outputs": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-lib", default="",
                    help="libtdoa_b200.so of another build for the config 5 and windowed comparisons")
    ap.add_argument("--cfg5-reps", type=int, default=21)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_window_grid.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    if args.parent_lib:
        lines.append(cfg5_ab(args.parent_lib, args.cfg5_reps))
    delays, _ = configs_bench.delays_for(bench.STATION_LLH)
    caps = configs_bench.synth(dev, 3, BLOCK, delays)
    def case(name, stations, caps, grid, **kw):
        with T.Engine(T.MODE_EXTENDED, **kw) as e:
            for k, c in enumerate(caps):
                e.load_u8_device(k, c.data_ptr(), c.numel(), keep=c)
            lines.append(run_case(name, e, stations, caps, grid, args.reps, bench.TX_LLH))
            if args.parent_lib:
                with engine_on(args.parent_lib, T.MODE_EXTENDED, **kw) as p:
                    for k, c in enumerate(caps):
                        p.load_u8_device(k, c.data_ptr(), c.numel(), keep=c)
                    lines.append(windows_ab(name, {"branch": e, "parent": p}, stations, grid, args.reps))

    case("config 3: 3 stations, Mode B FM, EXTENDED, +-50000 lags", bench.STATION_LLH, caps, around(bench.STATION_LLH, 400),
         max_lag=50_000)
    del caps
    torch.cuda.empty_cache()
    stations = S.ring_stations(16)
    caps, _ = S.simulate_weak(stations, tuple(bench.TX_LLH), 92300000.0, 10.0, 1000.0, BLOCK, seed=4242, device=dev)
    case("configs[3]: 16 stations, weak_signal_simulator.go content, EXTENDED, +-2000 lags", np.asarray(stations), caps,
         around(stations, 1000), n_stations=16, max_lag=2000)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    with out.open("a") as f:
        for ln in lines:
            ln["card"] = info
            s = json.dumps(ln)
            print(s)
            f.write(s + "\n")


if __name__ == "__main__":
    main()
