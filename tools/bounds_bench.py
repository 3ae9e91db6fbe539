#!/usr/bin/env python
"""Times the bounded TGT search of the windowed calls: tdoa_process_windows with tdoa_set_tgt_bounds off and on
(guard 5 samples; same engine, alternating; medians), with ms_fix, ms_exact of the TGT pass and the candidate counts
(TDOA_PEAK_NCAND) of the TGT records.

    python tools/bounds_bench.py [--reps K] [--out profiles/r10_bounds.jsonl]

  cfg3      3 stations (bench.STATION_LLH), Mode-B FM content (tools/configs_bench.py's generator), 100 s at 2 Msps,
            +-50 000 lags, EXTENDED; 66 REF and 33 TGT windows of 2e6
  configs3  BASELINE configs[3]'s 16 stations (ring_stations(16)), the same content and windows, +-2000 lags
  weak      the same 16 stations on weak_signal_simulator.go's content (tools/simulators.py)
  oracle    the weak-target scenario of tests/bounds_oracle.py on the CPU oracle, window 0: unbounded and bounded
            lag errors per pair; and the same target without its repeats over a range of amplitudes

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
import simulators as SIM  # noqa: E402
import tdoa_b200 as T  # noqa: E402
from retimed_bench import BLOCK, W, card  # noqa: E402

GUARD = 5.0


def ncand(tgt):
    return ((np.asarray(tgt["flags"]) >> 16) & 0xff).astype(np.int64)


def windows_case(name, e, stations, reps):
    nw_r, nw_t = 2 * BLOCK // W, BLOCK // W

    def run(on):
        e.set_tgt_bounds(GUARD if on else None)
        r = e.process_windows(stations, 0, W, nw_r, nw_t, W)
        return r, e.stats()

    for _ in range(2):
        run(False); run(True)
    t = {False: [], True: []}
    fix = {False: [], True: []}
    exact = {False: [], True: []}
    out = {}
    for _ in range(reps):   # alternating
        for on in (False, True):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            r, st = run(on)
            t[on].append(time.perf_counter() - t0)
            fix[on].append(st["ms_fix"]); exact[on].append(st["ms_exact"])
            out[on] = r
    a, b = out[False], out[True]
    med = lambda v: float(np.median(v))
    return {"case": name, "pairs": e.n_pairs, "reps": reps, "windows": {"ref": [nw_r, W], "tgt": [nw_t, W]}, "guard": GUARD,
            "off_ms": 1e3 * med(t[False]), "on_ms": 1e3 * med(t[True]),
            "off_ms_all": [1e3 * x for x in t[False]], "on_ms_all": [1e3 * x for x in t[True]],
            "ms_fix_off": med(fix[False]), "ms_fix_on": med(fix[True]),
            "ms_exact_tgt_off": med(exact[False]), "ms_exact_tgt_on": med(exact[True]),
            "ncand_tgt_off": {"sum": int(ncand(a["tgt"]).sum()), "max": int(ncand(a["tgt"]).max())},
            "ncand_tgt_on": {"sum": int(ncand(b["tgt"]).sum()), "max": int(ncand(b["tgt"]).max())},
            "ref_equal": a["ref"].tobytes() == b["ref"].tobytes(),
            "tgt_lags_changed": int(np.count_nonzero(a["tgt"]["lag"] != b["tgt"]["lag"])),
            "status_off": np.bincount(a["status"], minlength=3).tolist(),
            "status_on": np.bincount(b["status"], minlength=3).tolist()}


def oracle_case():
    """The weak-target scenario of tests/bounds_oracle.py on the CPU oracle, TGT window 0 (where the two searches
    differ), and a sweep of the same target without its repeats (period 0): per amplitude, the unbounded lags more than
    5 samples off and the largest bounded lag error over the three windows."""
    import bounds_oracle as B
    import lag_edges as E
    from oracle import oracle
    oracle.set_seq_dc_limit(0)
    st, L, S = B.SCN_LLH, B.SCN_MAX_LAG, len(B.SCN_LLH)

    def errors(raws, d, w):
        s0 = w * B.SCN_HOP
        ys = [oracle.preprocess_binary(E.split(r)[1][s0:s0 + B.SCN_WIN])[0] for r in raws]
        free, bnd = [], []
        for i in range(S):
            for j in range(i + 1, S):
                c = oracle.xcorr_two_sided(ys[i], ys[j], L)
                lo, hi = B.interval(0.0, 0.0, 0.0, 0.0, 0.0, B.baseline(st[i], st[j]), False, B.SCN_GUARD)
                free.append(B.bounded_peak(c, -L, L)["lag"] - (d[j] - d[i]))
                r = B.bounded_peak(c, lo, hi)
                bnd.append(round(r["lag"] + float(r["frac"]) - (d[j] - d[i]), 3))
        return free, bnd

    raws, d = B.scenario_captures()
    free, bnd = errors(raws, d, 0)
    sweep = []
    for amp in (0.0035, 0.005, 0.007, 0.01, 0.015):
        raws, d = B.scenario_captures(amp, 0.018, period=0)
        e = [errors(raws, d, w) for w in range(B.SCN_NT)]
        sweep.append({"amp": amp, "noise": 0.018, "unbounded_off_gt5": sum(sum(abs(x) > 5 for x in f) for f, _ in e),
                      "bounded_max_err": max(max(abs(x) for x in b) for _, b in e)})
    return {"case": f"oracle: weak-target scenario (tests/bounds_oracle.py: amp {B.SCN_AMP}, noise {B.SCN_NOISE}, "
                    f"period {B.SCN_PERIOD}), TGT window 0, 10 pairs", "lag_error_unbounded": free, "lag_error_bounded": bnd,
            "sweep_without_repeats": sweep,
            "sweep_note": "30 lags per amplitude (3 windows x 10 pairs); at no amplitude of this sweep does a weak-branch "
                          "target without repeats give bounded lags within 1 sample: its peak is ~10 samples wide"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r10_bounds.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    st16 = np.asarray(configs_bench.ring_stations(16))
    cases = ((3, 50_000, np.asarray(bench.STATION_LLH), "cfg3: config 3 stations, FM content, EXTENDED, +-50000 lags", "fm"),
             (16, 2000, st16, "configs3: 16 stations, FM content, EXTENDED, +-2000 lags", "fm"),
             (16, 2000, st16, "configs3: 16 stations, weak_signal_simulator.go content, EXTENDED, +-2000 lags", "weak"))
    for S, max_lag, st, name, content in cases:
        if content == "fm":
            delays, _ = configs_bench.delays_for(st)
            caps = configs_bench.synth(dev, S, BLOCK, delays)
        else:
            caps = SIM.simulate_weak([tuple(x) for x in st], tuple(bench.TX_LLH), 92300000.0, 10.0, 1000.0, BLOCK,
                                     seed=4242, device=dev)[0]
        with T.Engine(T.MODE_EXTENDED, n_stations=S, max_lag=max_lag) as e:
            for k in range(S):
                e.load_u8_device(k, caps[k].data_ptr(), caps[k].numel(), keep=caps[k])
            lines.append(windows_case(name, e, st, args.reps))
        del caps
        torch.cuda.empty_cache()
    lines.append(oracle_case())
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
