#!/usr/bin/env python
"""Times the closure check of the windowed fixes: tdoa_process_windows with the check off and on (same run,
alternating; ms_fix of each), and tdoa_closure alone per set, with k_window_closure's device time from a profiled
pass of its own.

    python tools/closure_bench.py [--reps K] [--out profiles/r7_closure.jsonl]

  cfg2      3 stations, config 2 content (tools/configs_bench.py's Mode-B generator), 100 s at 2 Msps, +-50 000 lags,
            EXTENDED; 66 REF and 33 TGT windows of 2e6 (three stations are one cycle: the check never drops there)
  configs3  BASELINE configs[3]'s 16 stations (ring_stations(16)) with the same generator, +-2000 lags; same windows
  alone     tdoa_closure on exact range differences at 16 stations (1024 sets) and 64 stations (64 sets), the latter
            with no wrong pair and with 200 wrong pairs per set (errors of 2..40 km)

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

CLOSURE = {"max_residual": 300.0}


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_window_closure" in ev.key:
            us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return us / 1e3, int(ev.count)
    return float("nan"), 0


def windows_case(name, e, stations, reps):
    nw_r, nw_t = 2 * BLOCK // W, BLOCK // W

    def off():
        return e.process_windows(stations, 0, W, nw_r, nw_t, W)

    def on():
        return e.process_windows(stations, 0, W, nw_r, nw_t, W, closure=CLOSURE)

    for _ in range(2):
        off(); on()
    t_off, t_on, f_off, f_on = [], [], [], []
    for _ in range(reps):   # alternating
        torch.cuda.synchronize(); t0 = time.perf_counter(); a = off(); t_off.append(time.perf_counter() - t0)
        f_off.append(e.stats()["ms_fix"])
        torch.cuda.synchronize(); t0 = time.perf_counter(); b = on(); t_on.append(time.perf_counter() - t0)
        f_on.append(e.stats()["ms_fix"])
    ms_k, n_k = kernel_ms(on)
    same = all(np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes() for k in ("ref", "tgt", "range_differences"))
    return {"case": name, "pairs": e.n_pairs, "reps": reps, "windows": {"ref": [nw_r, W], "tgt": [nw_t, W]},
            "closure": CLOSURE, "off_ms": 1e3 * float(np.median(t_off)), "on_ms": 1e3 * float(np.median(t_on)),
            "off_ms_all": [1e3 * t for t in t_off], "on_ms_all": [1e3 * t for t in t_on],
            "ms_fix_off": float(np.median(f_off)), "ms_fix_on": float(np.median(f_on)),
            "k_window_closure_ms": ms_k, "k_window_closure_launches": n_k, "tables_equal": same,
            "pairs_dropped": int(b["dropped"].sum()), "status_off": a["status"].tolist(), "status_on": b["status"].tolist()}


def alone_case(S, n_sets, n_bad, reps, seed=7):
    rng = np.random.default_rng(seed)
    st = np.array([[41.26 + rng.uniform(-0.3, 0.3), -96.02 + rng.uniform(-0.4, 0.4), 350.0] for _ in range(S)])
    P = S * (S - 1) // 2
    rd = np.zeros((n_sets, P))
    for k in range(n_sets):
        x = WO.llh_to_ecef(41.26 + rng.uniform(-0.1, 0.1), -96.02 + rng.uniform(-0.1, 0.1), 350.0)
        r = [float(np.linalg.norm(np.subtract(x, WO.llh_to_ecef(*s)))) for s in st]
        rd[k] = [r[j] - r[i] for i in range(S) for j in range(i + 1, S)]
        if n_bad:
            bad = rng.choice(P, n_bad, replace=False)
            rd[k, bad] += rng.choice([-1, 1], n_bad) * rng.uniform(2e3, 4e4, n_bad)
    used = np.ones((n_sets, P), np.uint8)
    with T.Engine(T.MODE_BINARY) as e:
        def run():
            return e.closure(S, rd, used, max_residual=CLOSURE["max_residual"])
        run()
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize(); t0 = time.perf_counter(); out = run(); ts.append(time.perf_counter() - t0)
        ms_k, n_k = kernel_ms(run)
    return {"case": f"tdoa_closure alone, {S} stations, {n_sets} sets, {n_bad} wrong pairs per set", "reps": reps,
            "call_ms": 1e3 * float(np.median(ts)), "k_window_closure_ms": ms_k, "k_window_closure_launches": n_k,
            "kernel_us_per_set": 1e3 * ms_k / n_sets, "mean_drops_per_set": float(np.mean(out[2]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r7_closure.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    for S, max_lag, st, name in ((3, 50_000, np.asarray(bench.STATION_LLH), "config 2 content, 3 stations, EXTENDED, +-50000 lags"),
                                 (16, 2000, np.asarray(configs_bench.ring_stations(16)),
                                  "configs[3] stations, 16 stations, EXTENDED, +-2000 lags")):
        delays, _ = configs_bench.delays_for(st)
        caps = configs_bench.synth(dev, S, BLOCK, delays)
        with T.Engine(T.MODE_EXTENDED, n_stations=S, max_lag=max_lag) as e:
            for k in range(S):
                e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
            lines.append(windows_case(name, e, st, args.reps))
        del caps
        torch.cuda.empty_cache()
    lines.append(alone_case(16, 1024, 0, args.reps))
    lines.append(alone_case(64, 64, 0, args.reps))
    lines.append(alone_case(64, 64, 200, args.reps))
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
