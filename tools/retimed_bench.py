#!/usr/bin/env python
"""Times tdoa_process_windows_retimed (station clock rates from the REF windows, every TGT plane re-timed, one TGT
window of the whole block) on captures with injected clock drift, beside tdoa_process_windows over 33 TGT windows of
2e6 samples on the same captures (same run, alternating), and measures k_retime's device time in a profiled pass of
its own.

    python tools/retimed_bench.py [--reps K] [--out profiles/r6_retimed.jsonl]

  cfg2      3 stations, config 2 content (tools/configs_bench.py's Mode-B generator), 100 s at 2 Msps, drift
            0 / +40 / -40 ppm, +-50 000 lags, EXTENDED; 66 REF windows of 2e6, the TGT block as one window
  configs3  BASELINE configs[3]'s 16 stations (ring_stations(16)) with the same generator, drift within +-3 ppm,
            +-2000 lags, EXTENDED; same windows

Drift is injected on the device: station k's sample n is the undrifted capture's sample n - round(eps_k n).  k_retime's
algorithmic bytes are 8 per plane sample (4 read, 4 written), S planes of one TGT block; its share is of the 6557.4
GB/s HBM copy rate DESIGN uses.  The verdict: the rates against the restatement's fit of the returned REF slopes
(tests/retime_oracle.py), the REF fit's restatement (tests/window_oracle.py) and the range differences it gives for the whole-block window.
One JSON line per case (stdout and --out) with the card name, power limit and max SM clock read in the same run."""
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
import retime_oracle as RO  # noqa: E402  (the checkers; never on the measured path)
import tdoa_b200 as T  # noqa: E402
import window_oracle as WO  # noqa: E402

W = 2_000_000
BLOCK = 66_666_666
HBM_GBPS = 6557.4


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def drifted(cap, eps_ppm):
    n = cap.numel() // 2
    t = torch.arange(n, device=cap.device, dtype=torch.float64)
    idx = (t - torch.round(t * (eps_ppm * 1e-6))).clamp_(0, n - 1).long()
    return cap.view(n, 2)[idx].reshape(-1).contiguous()


def retime_device_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_retime" in ev.key:
            us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return us / 1e3, int(ev.count)
    return float("nan"), 0


def verdict(stations, res, nsamp):
    S = len(stations)
    _, clock = RO.station_rates(res["ref_fit"][:, 1], res["ref_fit"][:, 2], S)
    fin = np.isfinite(clock)
    d_rate = float(np.abs(res["clock_rate"][fin] - clock[fin]).max() / max(np.abs(clock[fin]).max(), 1e-300))
    # the REF fit restated on the REF windows; the TGT window is the block, whose centre is block 2's centre, where
    # ref_fit[p][0] evaluates the REF line: rd = (y_tgt / fs - ref_fit[p][0] / fs) * c
    want = WO.window_fixes(stations, nsamp, 0, 0, W, W, res["ref"], res["tgt"], fs=2e6, dims=2)
    dfit = float(np.abs(want["ref_fit"] - res["ref_fit"]).max())
    y = res["tgt"][0]["lag"].astype(np.float64) + res["tgt"][0]["frac"].astype(np.float64)
    rd = (y / 2e6 - res["ref_fit"][:, 0] / 2e6) * WO.C_LIGHT
    u = res["pair_used"][0]
    drd = float(np.abs(rd[u] - res["range_differences"][0][u]).max()) if u.any() else 0.0
    ok = d_rate <= 1e-12 and dfit <= 1e-9 and drd <= 1e-6
    return {"rel_rate_diff": d_rate, "max_abs_ref_fit_diff": dfit, "pairs_used": int(u.sum()), "max_abs_rd_diff_m": drd,
            "ok": "ok" if ok else "MISMATCH"}


def run_case(name, e, stations, caps, eps, reps):
    nw_r, nw_t = 2 * BLOCK // W, BLOCK // W

    def rt():
        return e.process_windows_retimed(stations, ref=(0, W, nw_r, W), tgt=(0, BLOCK, 1, BLOCK))

    def pw():
        return e.process_windows(stations, 0, W, nw_r, nw_t, W)

    for _ in range(2):   # warm every shape
        rt(); pw()
    t_rt, t_pw = [], []
    for _ in range(reps):   # alternating
        torch.cuda.synchronize(); t0 = time.perf_counter(); res = rt(); t_rt.append(time.perf_counter() - t0)
        torch.cuda.synchronize(); t0 = time.perf_counter(); pw(); t_pw.append(time.perf_counter() - t0)
    ms_k, n_k = retime_device_ms(rt)
    nbytes = 8 * len(stations) * BLOCK
    c = res["clock_rate"] - np.nanmean(res["clock_rate"])
    e0 = (np.asarray(eps) - np.mean(eps)) * 1e-6
    return {"case": name, "pairs": e.n_pairs, "reps": reps, "windows": {"ref": [nw_r, W], "tgt": [1, BLOCK]},
            "eps_ppm": list(map(float, eps)),
            "retimed_ms": 1e3 * float(np.median(t_rt)), "retimed_ms_all": [1e3 * t for t in t_rt],
            "process_windows_33_ms": 1e3 * float(np.median(t_pw)), "process_windows_33_ms_all": [1e3 * t for t in t_pw],
            "k_retime_ms": ms_k, "k_retime_launches": n_k, "k_retime_bytes": nbytes,
            "k_retime_gbps": nbytes / (ms_k * 1e-3) / 1e9, "k_retime_share_of_6557": nbytes / (ms_k * 1e-3) / 1e9 / HBM_GBPS,
            "max_abs_rate_err_ppm": float(np.abs(c - e0).max() * 1e6), "status": int(res["status"][0]),
            "oracle": verdict(stations, res, [cp.numel() // 2 for cp in caps])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r6_retimed.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    st3 = bench.STATION_LLH
    eps3 = [0.0, 40.0, -40.0]
    delays, _ = configs_bench.delays_for(st3)
    caps = [drifted(c, eps3[k]) for k, c in enumerate(configs_bench.synth(dev, 3, BLOCK, delays))]
    with T.Engine(T.MODE_EXTENDED, max_lag=50_000) as e:
        for k in range(3):
            e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
        lines.append(run_case("config 2 content, 3 stations, drift 0/+40/-40 ppm, EXTENDED, +-50000 lags", e, np.asarray(st3),
                              caps, eps3, args.reps))
    del caps
    torch.cuda.empty_cache()
    st16 = configs_bench.ring_stations(16)
    eps16 = list(np.random.default_rng(6).uniform(-3.0, 3.0, 16))
    delays, _ = configs_bench.delays_for(st16)
    caps = [drifted(c, eps16[k]) for k, c in enumerate(configs_bench.synth(dev, 16, BLOCK, delays))]
    with T.Engine(T.MODE_EXTENDED, n_stations=16, max_lag=2000) as e:
        for k in range(16):
            e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
        lines.append(run_case("configs[3] stations, 16 stations, drift within +-3 ppm, EXTENDED, +-2000 lags", e,
                              np.asarray(st16), caps, eps16, args.reps))
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
