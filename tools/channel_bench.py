#!/usr/bin/env python
"""Times the channel filter (tdoa_set_channel).

    python tools/channel_bench.py [--quick] [--reps K] [--out profiles/r9_channel.jsonl]

  fused      k_channel_demod (the strong branch's filter + discriminator) over config 2's content: 3 stations, blocks of
             66 666 666 samples (2e8 per station, both kinds), tdoa_process with serial_kinds = 1; kernel time from the
             engine's device events (ms_demod over demod_samples), at T = 31 / 63 / 127 with real and complex taps, and
             without a channel (k_demod_df) for comparison.  The FP32 floor is 4 T FMA per sample for complex taps and
             2 T for real ones, at 148 SMs x 128 lanes x the max SM clock nvidia-smi reports.
  plane      the same content scaled to the moderate branch (amplitude 0.05): the filter runs to planes (k_channel),
             then k_power and the envelope chain; ms_preprocess with and without a 63-tap channel, alternating.
  per call   config 3 (100 s, 33 TGT windows of 2e6, +-50k lags, xcorr + solve) with and without a 63-tap channel,
             alternating, medians.
  scenarios  the adjacent-channel and off-centre captures of tests/test_gpu_channel.py: TGT lag errors and fix errors
             with and without the channel.

One JSON line per case (stdout and --out) with the card name, power limit and max SM clock read in the same run."""
import argparse
import json
import re
import statistics
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
from retimed_bench import card  # noqa: E402

FS, CL = 2e6, 299792458.0


def max_clock_mhz(c):
    m = re.findall(r"(\d+)\s*MHz", c["nvidia_smi"])
    return float(m[-1]) if m else float("nan")


def load(e, caps):
    for k, cap in enumerate(caps):
        e.load_u8_device(k, cap.data_ptr(), cap.numel(), keep=cap)


def taps_of(n, cplx):
    # the content is FM at 0 Hz with 75 kHz deviation: a pass band offset by 20 kHz keeps it on the strong branch and
    # makes the taps complex
    h = T.channel_taps(20e3 if cplx else 0.0, 100e3, n)
    return h if cplx else h.real.astype(np.float32)


def fused(args, caps, clock, out):
    with T.Engine(T.MODE_EXTENDED, max_lag=2000, chunk_samples=0, serial_kinds=1) as e:
        load(e, caps)
        for n_taps, cplx in [(0, False)] + [(n, c) for n in (31, 63, 127) for c in (False, True)]:
            e.set_channel(T.KIND_REF, taps_of(n_taps, cplx) if n_taps else None)
            e.set_channel(T.KIND_TGT, taps_of(n_taps, cplx) if n_taps else None)
            e.process(bench.STATION_LLH)   # warm-up; the branch memo then says strong
            ms, samples = [], 0
            for _ in range(args.reps):
                e.process(bench.STATION_LLH)
                st = e.stats()
                ms.append(st["ms_demod"])
                samples = st["demod_samples"]
            t = statistics.median(ms)
            if not t > 0:   # no discriminator ran: the filtered signal left the strong branch
                out({"case": "fused", "n_taps": n_taps, "taps": "complex" if cplx else "real", "error": "not on the strong branch"})
                continue
            gs = samples / (t * 1e-3) / 1e9
            row = {"case": "fused", "kernel": "k_channel_demod" if n_taps else "k_demod_df (no channel)", "n_taps": n_taps,
                   "taps": "complex" if cplx else "real", "samples": int(samples), "ms_demod_median": t, "gsample_per_s": gs}
            if n_taps:
                floor = 148 * 128 * clock * 1e6 / ((4 if cplx else 2) * n_taps) / 1e9
                row.update({"fp32_floor_gsample_per_s": floor, "frac_of_floor": gs / floor})
            out(row)


def plane(args, caps, out):
    moderate = [(((c.float() - 127.5) * 0.1) + 127.5).round().to(torch.uint8) for c in caps]
    with T.Engine(T.MODE_EXTENDED, max_lag=2000, chunk_samples=0, serial_kinds=1) as e:
        load(e, moderate)
        res = {0: [], 63: []}
        for rep in range(args.reps + 1):
            for n_taps in (0, 63):
                e.set_channel(T.KIND_REF, taps_of(63, True) if n_taps else None)
                e.set_channel(T.KIND_TGT, taps_of(63, True) if n_taps else None)
                e.process(bench.STATION_LLH)
                e.process(bench.STATION_LLH)
                if rep:
                    res[n_taps].append(e.stats()["ms_preprocess"])
        info, _ = e.xcorr_info(T.KIND_TGT)
    out({"case": "plane", "branch": [s["branch"] for s in info], "ms_preprocess_median_no_channel": statistics.median(res[0]),
         "ms_preprocess_median_63_complex": statistics.median(res[63]),
         "note": "k_channel + k_power replace k_raw_stats; the difference is the plane path's cost"})


def per_call(args, dev, out):
    delays, _ = configs_bench.delays_for(bench.STATION_LLH)
    block = 8_000_000 if args.quick else 66_666_666
    caps = configs_bench.synth(dev, 3, block, delays)
    W, L = 2_000_000, 50_000
    nw = block // W
    with T.Engine(T.MODE_EXTENDED, max_lag=L) as e:
        load(e, caps)
        ms = {0: [], 63: []}
        lags = {}
        for rep in range(args.reps + 1):
            for n_taps in (0, 63):
                e.set_channel(T.KIND_TGT, taps_of(63, True) if n_taps else None)
                t0 = time.perf_counter()
                pk = e.xcorr(T.KIND_TGT, 0, W, nw, W)
                e.solve(bench.STATION_LLH, pk["lag"].astype(np.float64) / FS * CL)
                torch.cuda.synchronize()
                if rep:
                    ms[n_taps].append((time.perf_counter() - t0) * 1e3)
                lags[n_taps] = pk["lag"].copy()
    out({"case": "per_call", "config": f"3 ({nw} TGT windows of {W}, +-{L} lags, xcorr + solve)",
         "ms_median_no_channel": statistics.median(ms[0]), "ms_median_63_complex": statistics.median(ms[63]),
         "ms_all_no_channel": ms[0], "ms_all_63_complex": ms[63],
         "lags_equal": bool(np.array_equal(lags[0], lags[63]))})


def scenarios(out):
    import channel_oracle as CH
    import closure_oracle as CO
    from test_gpu_closure import ST6, TX6
    from test_gpu_window_grid import REF_TX, metres
    other = np.array([41.50, -96.40, 300.0])
    BE = 1_000_000
    for kind in ("adjacent", "off_centre"):
        raws, dT, f_tgt = CH.scenario(kind, ST6, TX6, REF_TX, other, BE, 4)
        row = {"case": "scenario", "scenario": kind}
        with T.Engine(T.MODE_EXTENDED, max_lag=600, n_stations=6) as e:
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            for name, taps in (("plain", None), ("channel", f_tgt)):
                if taps is not None:
                    e.set_channel(T.KIND_REF, T.channel_taps(0.0, 100e3))
                    e.set_channel(T.KIND_TGT, T.channel_taps(f_tgt, 100e3))
                r = e.process_windows(ST6, 0, BE // 2, 4, 2, BE // 2, ref_tx_llh=REF_TX, init_llh=TX6 + [0.03, 0.03, 0.0])
                err = [[int(r["tgt"]["lag"][w, p] - (dT[j] - dT[i])) for p, (i, j) in enumerate(CO.pairs(6))] for w in range(2)]
                row[name] = {"tgt_lag_errors": err, "fix_error_m": [metres(r["position"][w], TX6) for w in range(2)]}
        out(row)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("channel_bench: no GPU")
    dev = torch.device("cuda")
    c = card()
    clock = max_clock_mhz(c)
    f = open(args.out, "w") if args.out else None

    def out(row):
        row = {**row, "card": c}
        line = json.dumps(row)
        print(line, flush=True)
        if f:
            f.write(line + "\n")
            f.flush()

    delays, _ = configs_bench.delays_for(bench.STATION_LLH)
    block = 8_000_000 if args.quick else 66_666_666
    caps = configs_bench.synth(dev, 3, block, delays)
    fused(args, caps, clock, out)
    plane(args, caps, out)
    del caps
    torch.cuda.empty_cache()
    per_call(args, dev, out)
    scenarios(out)
    if f:
        f.close()


if __name__ == "__main__":
    main()
