"""Builds libtdoa_b200.so (sm_100a only) in-tree with nvcc.

    python tdoa-geolocation_b200/build.py [--force]

The parity-critical translation units are compiled with -fmad=false: the reference is
Go on amd64, which never contracts a*b+c (SURVEY.md appendix A); the FFT kernels keep
FMA contraction.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
INCLUDE = HERE.parent / "include"
OUT = HERE / "libtdoa_b200.so"
OBJ = HERE / "build"

# (source, extra flags)
UNITS = [
    ("preprocess.cu", ["-fmad=false"]),
    ("preprocess_fast.cu", []),
    ("preprocess_weak.cu", ["-fmad=false"]),
    ("seqsum.cu", ["-fmad=false"]),
    ("xcorr_exact.cu", ["-fmad=false"]),
    ("solve.cu", ["-fmad=false"]),
    ("window_fix.cu", ["-fmad=false"]),
    ("retime.cu", ["-fmad=false"]),
    ("exclude.cu", ["-fmad=false"]),
    ("analyze.cu", ["-fmad=false"]),
    ("xcorr_fft.cu", []),
    ("xcorr_tile.cu", []),
    ("xcorr_big.cu", []),
    ("xcorr_spec.cu", []),
    ("engine.cu", []),
    ("engine_pipeline.cu", []),
    ("engine_multi.cu", []),
]

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-Xptxas", "-v",
          "-I", str(INCLUDE), "-I", str(CSRC)]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    headers = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + list(INCLUDE.glob("*.h")) + [Path(__file__)]
    objs = []
    todo = []
    for src, extra in UNITS:
        s = CSRC / src
        if not s.exists():
            continue
        o = OBJ / (s.stem + ".o")
        objs.append(o)
        if force or _stale(o, [s] + headers):
            todo.append((src, s, o, extra))

    def compile_unit(item):
        src, s, o, extra = item
        cmd = [nvcc(), *ARCH, *COMMON, *extra, "-c", str(s), "-o", str(o)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        (OBJ / (s.stem + ".ptxas.log")).write_text(res.stderr)
        return src, res

    if todo:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 4)) as pool:
            results = list(pool.map(compile_unit, todo))   # translation units are independent
        for src, res in results:
            if verbose or res.returncode:
                sys.stderr.write(res.stderr)
            if res.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
    if force or _stale(OUT, objs):
        cmd = [nvcc(), *ARCH, "-shared", "-o", str(OUT), *map(str, objs), "-cudart", "static", "-ldl", "-lpthread"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode:
            sys.stderr.write(res.stderr)
            raise RuntimeError("link failed")
    build_host(force)
    return OUT


HOST_PROGRAMS = ["processor_b200", "fast_analyzer_b200", "analyzer_b200"]
HOST_OUT = HERE / "processor_b200"


def build_host(force: bool = False) -> Path:
    """The reference's commands over the C ABI (host/*.cpp: processor, fast_analyzer): plain g++,
    linked against libtdoa_b200.so, which they find next to themselves at run time."""
    for name in HOST_PROGRAMS:
        src, out = HERE / "host" / f"{name}.cpp", HERE / name
        if force or _stale(out, [src, OUT, *INCLUDE.glob("*.h")]):
            cxx = shutil.which("g++") or "g++"
            cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-I", str(INCLUDE), str(src), "-o", str(out),
                   "-L", str(HERE), "-ltdoa_b200", "-Wl,-rpath,$ORIGIN"]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if res.returncode:
                sys.stderr.write(res.stderr)
                raise RuntimeError(f"g++ failed on {name}.cpp")
    return HOST_OUT


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
