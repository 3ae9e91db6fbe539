#!/usr/bin/env python
"""Times tdoa_process_windows (one fix per TGT window, REF drift fitted across blocks 1 and 3) on the two
windowed workloads of BASELINE.json, beside tdoa_xcorr_windows over the same windows (same run, alternating),
and gives each case an oracle verdict: the fix stage's plain restatement (tests/window_oracle.py) on the returned
tables for one sampled TGT window.

    python tools/windows_bench.py [--n-devices N] [--reps K] [--out profiles/r3_windows.jsonl]

  cfg3      3 stations, 66 REF + 33 TGT windows of 2e6 samples, +-50 000 lags, EXTENDED (SURVEY 8d config 3)
  configs3  16 stations (120 pairs), weak_signal_simulator.go content (tools/simulators.py), 66 + 33 windows,
            +-2000 lags, EXTENDED; n_devices = N deals the windows over N GPUs of this process

One JSON line per case (stdout and --out) with the card name and power limit read in the same run."""
import argparse
import json
import subprocess
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
import window_oracle as WO  # noqa: E402  (the checker; never on the measured path)
from oracle import oracle  # noqa: E402

W = 2_000_000
BLOCK = 66_666_666   # 100 s capture at 2 Msps: 33 TGT windows, 66 REF windows


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def verdict(e, stations, res, w):
    """the fix stage's statement on the engine's own tables, TGT window w"""
    want = WO.window_fixes(stations, res["nsamp"], 0, 0, W, W, res["ref"], res["tgt"], fs=2e6, dims=2)
    u = want["pair_used"][w]
    ok = bool(np.array_equal(u, res["pair_used"][w]))
    drd = float(np.abs(want["range_differences"][w][u] - res["range_differences"][w][u]).max()) if u.any() else 0.0
    dfit = float(np.abs(want["ref_fit"] - res["ref_fit"]).max())
    dpos = float(np.linalg.norm(oracle.llh_to_ecef(*want["position"][w]) - oracle.llh_to_ecef(*res["position"][w])))
    rms, want_rms = float(res["rms"][w]), float(want["rms"][w])
    # the fix: within 1e-4 m of the statement's, or -- on a flat least-squares valley, where CUDA's and the C library's
    # sin / cos / sqrt rounding moves the stopping point along the valley -- at the same rms to 1e-9
    same_fix = dpos <= 1e-4 or abs(rms - want_rms) <= 1e-9 * max(want_rms, 1.0)
    ok = ok and drd <= 1e-6 and dfit <= 1e-9 and same_fix and int(want["status"][w]) == int(res["status"][w])
    return {"tgt_window": w, "pairs_used": int(u.sum()), "max_abs_rd_diff_m": drd, "max_abs_ref_fit_diff": dfit,
            "fix_diff_m": dpos, "rms_m": rms, "oracle_rms_m": want_rms, "status": int(res["status"][w]),
            "ok": "ok" if ok else "MISMATCH"}


def run_case(name, e, stations, caps, reps):
    nw_t, nw_r = BLOCK // W, 2 * BLOCK // W

    def pw():
        return e.process_windows(stations, 0, W, nw_r, nw_t, W)

    def xw():
        return e.xcorr_windows(0, W, nw_r, nw_t, W)

    for _ in range(2):   # warm every shape
        pw(); xw()
    t_pw, t_xw, fix_ms = [], [], []
    for _ in range(reps):   # alternating
        torch.cuda.synchronize(); t0 = time.perf_counter(); res = pw(); t_pw.append(time.perf_counter() - t0)
        fix_ms.append(e.stats()["ms_fix"])
        torch.cuda.synchronize(); t0 = time.perf_counter(); ref, tgt = xw(); t_xw.append(time.perf_counter() - t0)
    res["nsamp"] = [c.numel() // 2 for c in caps]
    same = res["ref"].tobytes() == ref.tobytes() and res["tgt"].tobytes() == tgt.tobytes()
    ms_pw, ms_xw = 1e3 * float(np.median(t_pw)), 1e3 * float(np.median(t_xw))
    return {"case": name, "n_devices": e.cfg.n_devices or 1, "windows": {"ref": nw_r, "tgt": nw_t, "samples": W},
            "pairs": e.n_pairs, "reps": reps,
            "process_windows_ms": ms_pw, "process_windows_ms_all": [1e3 * t for t in t_pw],
            "fixes_per_s": nw_t / (ms_pw * 1e-3),
            "fix_stage_device_ms": float(np.median(fix_ms)), "fix_stage_device_ms_all": fix_ms,
            "xcorr_windows_ms": ms_xw, "xcorr_windows_ms_all": [1e3 * t for t in t_xw],
            "fix_stage_share_of_call": float(np.median(fix_ms)) / ms_pw,
            "tables_equal_xcorr_windows": bool(same), "status_counts": np.bincount(res["status"], minlength=3).tolist(),
            "oracle": verdict(e, stations, res, nw_t // 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-devices", type=int, default=1)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_windows.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    # config 3 as SURVEY 8d defines it (Mode-B FM content with injected delays, tools/configs_bench.py's generator)
    delays, _ = configs_bench.delays_for(bench.STATION_LLH)
    caps = configs_bench.synth(dev, 3, BLOCK, delays)
    with T.Engine(T.MODE_EXTENDED, max_lag=50_000) as e:
        for k in range(3):
            e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
        lines.append(run_case("config 3: 3 stations, Mode B FM, EXTENDED, +-50000 lags", e, bench.STATION_LLH, caps, args.reps))
    del caps
    torch.cuda.empty_cache()
    # BASELINE configs[3] as fixes
    stations = S.ring_stations(16)
    caps, _ = S.simulate_weak(stations, tuple(bench.TX_LLH), 92300000.0, 10.0, 1000.0, BLOCK, seed=4242, device=dev)
    with T.Engine(T.MODE_EXTENDED, n_stations=16, max_lag=2000, n_devices=args.n_devices) as e:
        for k in range(16):   # a multi-device engine forwards host captures to its peers (not device pointers)
            if args.n_devices > 1:
                e.load_u8(k, caps[k].cpu().numpy())
            else:
                e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
        lines.append(run_case("configs[3]: 16 stations, weak_signal_simulator.go content, EXTENDED, +-2000 lags", e,
                              np.asarray(stations), caps, args.reps))
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
