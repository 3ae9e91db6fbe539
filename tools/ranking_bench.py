"""Worst error of the FFT search's f32 ranking plane per path and content, against an f64 correlation of the engine's
own planes (tdoa_xcorr_ranking; tests/ranking_oracle.py), and the timing rows of the ranking transforms' change.

    python tools/ranking_bench.py --label after [--full] [--out profiles/r11_ranking.jsonl]
        the cases of tests/test_gpu_ranking.py on every path (default tiles = 1, one transform per pair = 2, no
        2^21-point transform = 3, no parked spectra = 4): one row per case and path, then one per (path, content)
    python tools/ranking_bench.py --label timing --timing DIR
        DIR holds bench.py outputs bench_<version>_<k>.json (version parent / change, alternating runs k) and
        configs_bench.py outputs cfg4_<version>_<k>.json: one row of medians per version

Rows are appended to --out, each with the card's name and power limit."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def card():
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else ""}


def measure(raws, mode, start, W, paths, **cfg):
    """{path: worst |approx - exact| over the records that have a ranking}, max / min power1 of the stations."""
    import tdoa_b200 as T
    import ranking_oracle as R
    import torch
    dev = torch.device("cuda", 0)
    S = len(raws)
    pairs = [(i, j) for i in range(S) for j in range(i + 1, S)]
    ext = mode == T.MODE_EXTENDED
    D = max(1, cfg.get("decimate", 1)) if ext else 1
    with T.Engine(mode, n_stations=S, use_fft=0, **cfg) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        e.xcorr(T.KIND_TGT, start, W, 1, 0)
        info, _ = e.xcorr_info(T.KIND_TGT)
        n = [W if W else x["n"] for x in info]
        planes = [e.preprocess(k, T.KIND_TGT, start, n[k])[0] for k in range(S)]
    p1 = np.array([x["power1"] for x in info])
    if ext:
        exact = [R.exact_extended(planes[i], planes[j], cfg.get("max_lag", 2000) // D, dev) for i, j in pairs]
    else:
        exact = [R.exact_binary(planes[i], planes[j], cfg.get("max_lag", 2000), 10000, dev) for i, j in pairs]
    out = {}
    for u in paths:
        with T.Engine(mode, n_stations=S, use_fft=u, **cfg) as e:
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            _, rk = e.xcorr_ranking(T.KIND_TGT, start, W, 1, 0)
        errs = [np.max(np.abs(rk[0, p, :c.size] - c)) for p, c in enumerate(exact) if not np.isnan(rk[0, p, 0])]
        out[u] = float(max(errs)) if errs else None
    return out, float(p1.max() / p1.min())


def cases(full):
    import tdoa_b200 as T
    import test_gpu_ranking as G
    from helpers import fm_capture
    for name, S, L, n_t, D, content in G.EXT_CASES:
        W = D * (n_t + 2 * (L // D))
        yield name, content, G.capture(content, W + 400, S, seed=len(name)), T.MODE_EXTENDED, 200, W, \
            dict(max_lag=L, decimate=D)
    for name, S, L, n_t in G.WEAK_GEOMETRIES:
        W = n_t + 2 * L
        yield "weak_" + name, "weak", G.capture("noise", W + 400, S, seed=11, weak=[(2, 1, 1)]), T.MODE_EXTENDED, \
            200, W, dict(max_lag=L)
    W = 100000 + 2048
    for flips, step in ((25000, 4), (3000, 1)):
        yield f"weak_sweep_{flips}x{step}", "weak", G.capture("noise", W + 400, 3, seed=12, weak=[(2, flips, step)]), \
            T.MODE_EXTENDED, 200, W, dict(max_lag=1024)
    raws = fm_capture(W + 400, [0, 5, 10], [0, 7, 15], seed=12)
    raws[2] = fm_capture(W + 400, [0, 5, 10], [0, 7, 15], seed=12, dev_tgt=4e3, noise=0.005)[2]
    yield "fm_low_dev", "fm_low_dev", raws, T.MODE_EXTENDED, 200, W, dict(max_lag=1024)
    yield "binary", "fm", G.capture("fm", 250000, 3, seed=2), T.MODE_BINARY, 0, 0, {}
    if full:
        import bench
        import configs_bench as cb
        import torch
        delays, _ = cb.delays_for(bench.STATION_LLH)
        caps = [c.cpu().numpy() for c in cb.synth(torch.device("cuda", 0), 3, 66_666_666, delays)]
        yield "binary_full", "fm_full", caps, T.MODE_BINARY, 0, 0, dict(chunk_samples=0)


def timing(d: Path):
    rows = {}
    for f in sorted(d.glob("bench_*.json")):
        version = f.stem.split("_")[1]
        lines = [json.loads(x) for x in f.read_text().splitlines() if x.startswith("{")]
        head = next(x for x in lines if "ms_per_step" in x)
        shard = next((x["sharded"] for x in lines if "sharded" in x), {})
        r = rows.setdefault(version, {"bench_ms_per_step": [], "sharded": []})
        r["bench_ms_per_step"].append(head["ms_per_step"])
        r["sharded"].append({k: v for k, v in shard.items() if "ms" in k and isinstance(v, (int, float))})
    for f in sorted(d.glob("cfg4_*.json")):
        version = f.stem.split("_")[1]
        lines = [json.loads(x) for x in f.read_text().splitlines() if x.startswith("{")]
        rows.setdefault(version, {}).setdefault("config4", []).append(
            [{k: v for k, v in x.items() if "ms" in k or k in ("config", "content")} for x in lines])
    for r in rows.values():
        if r.get("bench_ms_per_step"):
            r["bench_median_ms"] = float(np.median(r["bench_ms_per_step"]))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--label", required=True, help="what the library is (e.g. before / after the change)")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r11_ranking.jsonl"))
    ap.add_argument("--full", action="store_true", help="also configs[1]'s full TGT size (BINARY, default path)")
    ap.add_argument("--timing", metavar="DIR", help="summarise bench.py / configs_bench.py outputs instead")
    args = ap.parse_args()
    c = card()
    rows = []
    if args.timing:
        for version, r in timing(Path(args.timing)).items():
            rows.append({"label": args.label, "version": version, **r, "card": c})
    else:
        worst = {}
        for name, content, raws, mode, start, W, cfg in cases(args.full):
            paths = (1,) if name == "binary_full" else (1, 2, 3, 4)
            err, ratio = measure(raws, mode, start, W, paths, **cfg)
            rows.append({"label": args.label, "case": name, "content": content, "power_ratio": ratio,
                         "worst_err": {str(u): v for u, v in err.items()}, "card": c})
            for u, v in err.items():
                if v is not None:
                    key = (u, content)
                    worst[key] = max(worst.get(key, 0.0), v)
            print(json.dumps(rows[-1]), flush=True)
        for (u, content), v in sorted(worst.items()):
            rows.append({"label": args.label, "path": u, "content": content, "worst_err": v, "card": c})
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    for r in rows[-12:]:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
