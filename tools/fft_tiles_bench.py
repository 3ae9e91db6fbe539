#!/usr/bin/env python
"""Times tdoa_process on bench.py's headline workload (configs[1]: 3 stations, 100 s at 2 Msps, BINARY, FFT path)
with this tree's library and with a second library (e.g. built from the parent commit), alternating in one process,
and reports k_fft_tiles' mean device time per launch for both.

    python tools/fft_tiles_bench.py --parent-lib PATH [--calls 21] [--warmup 3] [--out profiles/r5_fft_tiles.jsonl]

The captures are bench.synth_captures_gpu's (seed 0, bench.py's default block), so inputs_sha256 equals the one
bench.py prints.  Per build:
  - tdoa_process wall time: a host clock from a device synchronise to the returned host arrays, one call of each build
    in turn (the build that goes first alternates), --calls calls each;
  - k_fft_tiles ms per launch: the engine's CUDA events around each tile launch (stats() ms_fft_seg / fft_launches)
    on a serial_kinds = 1 twin, where the REF and TGT pair loops share one stream and a launch's duration is its own;
  - every array tdoa_process returns, compared byte for byte between the builds (resident and serial engines).
One JSON line (stdout and --out) with the card's name, power limit and max SM clock read in the same run."""
import argparse
import ctypes
import hashlib
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402

import bench  # noqa: E402
import tdoa_b200 as T  # noqa: E402
from windows_bench import card  # noqa: E402

_N = sys.modules[T.Engine.__module__]
BLOCK = 66_666_666   # bench.py --block default


def engine_on(lib_path, *args, **kw):
    """an Engine bound to another build of the library"""
    other, cur = ctypes.CDLL(str(lib_path)), _N.load_library()
    for name in ("tdoa_default_config", "tdoa_create", "tdoa_destroy", "tdoa_last_error", "tdoa_get_stats",
                 "tdoa_load_u8_device", "tdoa_process", "tdoa_set_stream", "tdoa_stream", "tdoa_synchronize"):
        getattr(other, name).argtypes = getattr(cur, name).argtypes
        getattr(other, name).restype = getattr(cur, name).restype
    saved = _N._lib
    try:
        _N._lib = other
        return T.Engine(*args, **kw)
    finally:
        _N._lib = saved


def differing(a, b):
    """names of the returned arrays (and peak-record fields) whose bytes differ"""
    out = []
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.tobytes() == y.tobytes():
            continue
        if x.dtype.names:
            out += [f"{k}.{f}" for f in x.dtype.names if x[f].tobytes() != y[f].tobytes()]
        else:
            out.append(k)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libtdoa_b200.so of the build to compare against")
    ap.add_argument("--calls", type=int, default=21, help="timed tdoa_process calls per build (at least 21)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r5_fft_tiles.jsonl"))
    args = ap.parse_args()
    if args.calls < 21:
        ap.error("--calls must be at least 21")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = card()
    caps, _ = bench.synth_captures_gpu(torch, dev, BLOCK, seed=0)
    digest = hashlib.sha256()
    for c in caps:
        digest.update(c.cpu().numpy())
    nbytes = caps[0].numel()
    stream = torch.cuda.current_stream().cuda_stream

    def make(lib, **kw):
        e = (T.Engine(T.MODE_BINARY, chunk_samples=0, use_fft=1, **kw) if lib is None else
             engine_on(lib, T.MODE_BINARY, chunk_samples=0, use_fft=1, **kw))
        e.set_stream(stream)
        for k in range(3):
            e.load_u8_device(k, caps[k].data_ptr(), nbytes, keep=caps[k])
        return e

    builds = {"branch": None, "parent": args.parent_lib}
    resident = {k: make(v) for k, v in builds.items()}
    serial = {k: make(v, serial_kinds=1) for k, v in builds.items()}

    outs, times = {}, {k: [] for k in builds}
    for _ in range(args.warmup):
        for k, e in resident.items():
            e.process(bench.STATION_LLH)
    for i in range(args.calls):
        for k in (("branch", "parent") if i % 2 == 0 else ("parent", "branch")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[k] = resident[k].process(bench.STATION_LLH)
            times[k].append(1e3 * (time.perf_counter() - t0))

    seg_ms, launches, serial_outs = {k: [] for k in builds}, {k: [] for k in builds}, {}
    for _ in range(args.warmup):
        for k, e in serial.items():
            e.process(bench.STATION_LLH)
    for i in range(args.calls):
        for k in (("branch", "parent") if i % 2 == 0 else ("parent", "branch")):
            serial_outs[k] = serial[k].process(bench.STATION_LLH)
            st = serial[k].stats()
            seg_ms[k].append(st["ms_fft_seg"])
            launches[k].append(st["fft_launches"])
    for e in (*resident.values(), *serial.values()):
        e.close()

    med = {k: float(np.median(v)) for k, v in times.items()}
    per_launch = {k: float(np.sum(seg_ms[k]) / np.sum(launches[k])) for k in builds}
    diff = differing(outs["branch"], outs["parent"]) + [f"serial.{d}" for d in
                                                        differing(serial_outs["branch"], serial_outs["parent"])]
    line = {"case": "configs[1]: tdoa_process, 3 stations, block %d, BINARY, FFT path; branch vs parent build" % BLOCK,
            "inputs_sha256": digest.hexdigest(), "calls": args.calls,
            "branch_ms": med["branch"], "parent_ms": med["parent"], "delta_ms": med["parent"] - med["branch"],
            "branch_calls_below_parent_median": float(np.mean(np.array(times["branch"]) < med["parent"])),
            "branch_ms_all": times["branch"], "parent_ms_all": times["parent"],
            "fft_tiles_ms_per_launch": per_launch,
            "fft_tiles_speedup": per_launch["parent"] / per_launch["branch"],
            "fft_launches_per_call": {k: float(np.mean(v)) for k, v in launches.items()},
            "fft_seg_ms_per_call_all": seg_ms,
            "same_outputs": not diff, "differing": diff, "card": info}
    s = json.dumps(line)
    print(s)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    with out.open("a") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
