#!/usr/bin/env python
"""Times the station check of the windowed fixes: the fix stage with the check off and on (same run, alternating;
ms_fix of each), and tdoa_exclude_stations alone per set, with k_window_exclude's device time from a profiled pass
of its own.

    python tools/exclusion_bench.py [--reps K] [--out profiles/r8_exclusion.jsonl]

  6 stations   ring_stations(6) with tools/configs_bench.py's Mode-B generator, 100 s at 2 Msps, +-2000 lags,
               EXTENDED; 66 REF and 33 TGT windows of 2e6.  tdoa_process_windows off / on (nothing to exclude: every
               window's rms is far below max_rms), then tdoa_window_fixes off / on on the same tables with station 4's
               TGT lags 20 samples (3 km) long, so that the check runs and excludes station 4 in every window
  16 stations  BASELINE configs[3]'s stations (ring_stations(16)), the same generator and windows; off / on, and the
               same with station 11's TGT lags 20 samples long
  alone        tdoa_exclude_stations on exact range differences (+ 2 m noise) at 16 stations (1024 sets) and 64 stations
               (64 sets), with no bad station (the check stops at once) and with one (3..20 km)
The windowed cases pass the transmitter as ref_tx_llh: the generator's REF and TGT come from the same place, so
without its geometric term every range difference would be 0 and no fix would fit.

One JSON line per case (stdout and --out) with the card name, power limit and max SM clock read in the same run."""
import argparse
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
import tdoa_b200 as T  # noqa: E402
import window_oracle as WO  # noqa: E402
from retimed_bench import BLOCK, W, card  # noqa: E402

EXCLUSION = {"max_rms": 50.0, "max_exclude": 1}
TX = bench.TX_LLH   # the generator's REF and TGT transmitter: its geometric term is added back


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_window_exclude" in ev.key:
            us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return us / 1e3, int(ev.count)
    return float("nan"), 0


def alternate(e, off, on, reps):
    for _ in range(2):
        off(); on()
    t_off, t_on, f_off, f_on = [], [], [], []
    for _ in range(reps):
        torch.cuda.synchronize(); t0 = time.perf_counter(); a = off(); t_off.append(time.perf_counter() - t0)
        f_off.append(e.stats()["ms_fix"])
        torch.cuda.synchronize(); t0 = time.perf_counter(); b = on(); t_on.append(time.perf_counter() - t0)
        f_on.append(e.stats()["ms_fix"])
    ms_k, n_k = kernel_ms(on)
    return a, b, {"reps": reps, "off_ms": 1e3 * float(np.median(t_off)), "on_ms": 1e3 * float(np.median(t_on)),
                  "off_ms_all": [1e3 * t for t in t_off], "on_ms_all": [1e3 * t for t in t_on],
                  "ms_fix_off": float(np.median(f_off)), "ms_fix_on": float(np.median(f_on)),
                  "k_window_exclude_ms": ms_k, "k_window_exclude_launches": n_k}


def windows_cases(name, e, st, bad, reps):
    nw_r, nw_t = 2 * BLOCK // W, BLOCK // W
    a, b, r = alternate(e, lambda: e.process_windows(st, 0, W, nw_r, nw_t, W, ref_tx_llh=TX),
                        lambda: e.process_windows(st, 0, W, nw_r, nw_t, W, ref_tx_llh=TX, exclusion=EXCLUSION), reps)
    same = all(np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes() for k in ("ref", "tgt", "position", "rms"))
    out = [{"case": f"tdoa_process_windows, {name}, nothing to exclude", "pairs": e.n_pairs,
            "windows": {"ref": [nw_r, W], "tgt": [nw_t, W]}, "exclusion": EXCLUSION, **r, "outputs_equal": same,
            "stations_excluded": int(b["excluded"].sum()), "rms_max_m": float(a["rms"].max())}]
    tgt = a["tgt"].copy()
    S = st.shape[0]
    p = 0
    for i in range(S):
        for j in range(i + 1, S):
            tgt["lag"][:, p] += 20 if j == bad else (-20 if i == bad else 0)
            p += 1
    c, d, r = alternate(e, lambda: e.window_fixes(st, 0, W, a["ref"], tgt, W, ref_tx_llh=TX),
                        lambda: e.window_fixes(st, 0, W, a["ref"], tgt, W, ref_tx_llh=TX, exclusion=EXCLUSION), reps)
    out.append({"case": f"tdoa_window_fixes, {name}, station {bad}'s TGT lags 20 samples long", "pairs": e.n_pairs,
                "windows": {"ref": [nw_r, W], "tgt": [nw_t, W]}, "exclusion": EXCLUSION, **r,
                "windows_excluding_the_station": int((d["station_excluded"][:, bad] == 1).sum()),
                "stations_excluded": int(d["excluded"].sum()), "rms_off_median_m": float(np.median(c["rms"])),
                "rms_on_median_m": float(np.median(d["rms"]))})
    return out


def alone_case(S, n_sets, n_bad, reps, seed=7):
    rng = np.random.default_rng(seed)
    st = np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), 350.0] for _ in range(S)])
    P = S * (S - 1) // 2
    rd, init = np.zeros((n_sets, P)), np.zeros((n_sets, 3))
    for k in range(n_sets):
        tx = (41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0)
        x = WO.llh_to_ecef(*tx)
        r = [float(np.linalg.norm(np.subtract(x, WO.llh_to_ecef(*s)))) for s in st]
        rd[k] = [r[j] - r[i] for i in range(S) for j in range(i + 1, S)]
        rd[k] += rng.normal(0, 2.0, P)
        init[k] = tx
        init[k, :2] += 0.02
        for s in rng.choice(S, n_bad, replace=False):
            d = rng.choice([-1, 1]) * rng.uniform(3e3, 2e4)
            rd[k] += [d if j == s else (-d if i == s else 0.0) for i in range(S) for j in range(i + 1, S)]
    used = np.ones((n_sets, P), np.uint8)
    with T.Engine(T.MODE_BINARY) as e:
        def run():
            return e.exclude_stations(st, rd, used, init, 2, **EXCLUSION)
        run()
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize(); t0 = time.perf_counter(); out = run(); ts.append(time.perf_counter() - t0)
        ms_k, n_k = kernel_ms(run)
    return {"case": f"tdoa_exclude_stations alone, {S} stations, {n_sets} sets, {n_bad} bad station per set", "reps": reps,
            "call_ms": 1e3 * float(np.median(ts)), "k_window_exclude_ms": ms_k, "k_window_exclude_launches": n_k,
            "kernel_us_per_set": 1e3 * ms_k / n_sets, "mean_excluded_per_set": float(np.mean(out["excluded"])),
            "mean_iters_final_fix": float(np.mean(out["iters"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r8_exclusion.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    for S, bad, name in ((6, 4, "ring_stations(6), 6 stations, EXTENDED, +-2000 lags"),
                         (16, 11, "configs[3] stations, 16 stations, EXTENDED, +-2000 lags")):
        st = np.asarray(configs_bench.ring_stations(S))
        delays, _ = configs_bench.delays_for(st)
        caps = configs_bench.synth(dev, S, BLOCK, delays)
        with T.Engine(T.MODE_EXTENDED, n_stations=S, max_lag=2000) as e:
            for k in range(S):
                e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
            lines += windows_cases(name, e, st, bad, args.reps)
        del caps
        torch.cuda.empty_cache()
    for S, n_sets in ((16, 1024), (64, 64)):
        for n_bad in (0, 1):
            lines.append(alone_case(S, n_sets, n_bad, args.reps))
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
