"""channel.cu's two kernels against the statement's restatement (tests/channel_oracle.py), bit for bit, launched
directly through tests/native/channel_probe.cu:

  - k_channel's planes against orc_channel at T = 1, 3, 31, 63, 127, with complex and real taps, real taps passed
    with zero imaginary parts against taps_im = NULL, at lengths around the 2048-output tile and the halo, on
    two-run views with the joint at several positions, and several jobs in one launch;
  - k_channel_demod's plane against k_demod on k_channel's planes, bit for bit, its power and output sum within
    1e-14 of the terms' magnitudes (the same terms, added in another tree).

The probe puts 64 canary words on both sides of every output array and fills the array itself with a NaN pattern
before each launch, so a write past either end and a sample left unwritten are both findings."""
import ctypes
import importlib.util
import subprocess
from pathlib import Path

import numpy as np
import pytest

import channel_oracle as CH
import tdoa_b200 as T
from oracle import oracle

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tdoa-geolocation_b200"
ST_COUNT, ST_POWER0, ST_SUM_RE, ST_DC_RE = 8, 0, 1, 3

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """the probe compiled with the library's flags and channel.cu's own, linked with preprocess.cu"""
    spec = importlib.util.spec_from_file_location("tdoa_b200_build_flags", PKG / "build.py")
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    so = tmp_path_factory.mktemp("channel_probe") / "channel_probe.so"
    extra = dict(b.UNITS)["channel.cu"]
    assert extra == dict(b.UNITS)["preprocess.cu"]
    cmd = [b.nvcc(), *b.ARCH, *b.COMMON, *extra, "-shared", "-Xcompiler", "-fPIC",
           str(ROOT / "tests" / "native" / "channel_probe.cu"), str(PKG / "csrc" / "preprocess.cu"), "-o", str(so)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = ctypes.CDLL(str(so))
    lib.probe_channel.restype = ctypes.c_int
    lib.probe_demod_planes.restype = ctypes.c_int
    return lib


def _p(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None


def view(raw, n, run0_start, run0_len, run1_start):
    """the unpacked samples of a view, as SigSrc maps them"""
    x = oracle.unpack_u8(raw)
    i = np.arange(n)
    idx = np.where(i < run0_len, run0_start + i, run1_start + (i - run0_len))
    return x[idx]


def run(lib, jobs, taps, real_kernel=False, demod=False):
    """jobs: (raw, n, (run0_start, run0_len, run1_start)); taps complex64 (real_kernel: taps_im = NULL)"""
    k = len(jobs)
    raws = [np.ascontiguousarray(j[0], np.uint8) for j in jobs]
    n = np.array([j[1] for j in jobs], np.int64)
    runs = np.array([r for j in jobs for r in j[2]], np.int64)
    nbytes = np.array([r.size for r in raws], np.int64)
    re_out = [np.empty(max(int(m), 1), np.float32) for m in n]
    im_out = [np.empty(max(int(m), 1), np.float32) for m in n]
    stats = np.zeros(k * ST_COUNT, np.float64)
    hr = np.ascontiguousarray(np.real(taps), np.float32)
    hi = None if real_kernel else np.ascontiguousarray(np.imag(taps), np.float32)
    bad = ctypes.c_longlong(-1)
    err = lib.probe_channel(ctypes.c_int(k), _p(n), (ctypes.c_void_p * k)(*[r.ctypes.data for r in raws]), _p(nbytes), _p(runs),
                            _p(hr), _p(hi), ctypes.c_int(hr.size), ctypes.c_int(int(demod)),
                            (ctypes.c_void_p * k)(*[o.ctypes.data for o in re_out]),
                            (ctypes.c_void_p * k)(*[o.ctypes.data for o in im_out]), _p(stats), ctypes.byref(bad))
    assert err == 0, f"CUDA error {err}"
    assert bad.value == 0, "canary words changed"
    if demod:
        return [o[:m] for o, m in zip(re_out, n)], stats.reshape(k, ST_COUNT)
    return [(o[:m], p[:m]) for o, p, m in zip(re_out, im_out, n)]


def same_bits(planes, want, what):
    re, im = planes
    w = np.ascontiguousarray(want, np.complex64)
    assert re.view(np.uint32).tolist() == w.real.copy().view(np.uint32).tolist(), what + " re"
    assert im.view(np.uint32).tolist() == w.imag.copy().view(np.uint32).tolist(), what + " im"


def capture(n_samp, seed):
    return np.random.default_rng(seed).integers(0, 256, 2 * n_samp, dtype=np.uint8)


def taps_for(T_, seed, real):
    if T_ == 63 and not real:
        return T.channel_taps(300e3, 100e3, 63)
    rng = np.random.default_rng(seed)
    h = rng.standard_normal(T_) + (0 if real else 1j * rng.standard_normal(T_))
    return (h / np.abs(h).sum()).astype(np.complex64)


LENGTHS = [0, 1, 2, 3, 31, 63, 127, 4095, 4096, 4097, 1_000_003]


@pytest.mark.parametrize("T_", [1, 3, 31, 63, 127])
@pytest.mark.parametrize("real", [False, True])
def test_k_channel_bits(probe, T_, real):
    taps = taps_for(T_, T_, real)
    c = (T_ - 1) // 2
    lengths = sorted({m for m in LENGTHS + [c, T_] if m <= 1_000_003})
    raw = capture(1_000_003 + 5000, T_)
    jobs = [(raw, m, (17, m, 0)) for m in lengths]
    want = [CH.channel(view(raw, *j[1:2], *j[2]), taps) for j in jobs]
    got = run(probe, jobs, taps)
    for m, g, w in zip(lengths, got, want):
        same_bits(g, w, f"T={T_} n={m}")
    if real:
        # the real-tap kernel (taps_im = NULL) against the same taps with zero imaginary parts
        got_r = run(probe, jobs, taps, real_kernel=True)
        for m, g, w in zip(lengths, got_r, want):
            same_bits(g, w, f"real kernel T={T_} n={m}")


@pytest.mark.parametrize("T_", [3, 63, 127])
def test_k_channel_two_run_views(probe, T_):
    """REF views across the block 1 | block 3 joint: the filter runs in view order across it"""
    taps = taps_for(T_, 100 + T_, False)
    b = 300_000
    raw = capture(3 * b + 2, 50 + T_)
    jobs = []
    for start, ln in [(0, 2 * b), (b - 1, 2), (b - 10, 5000), (b - 4096, 8193), (b - 63, 127), (b - 2048 * 37 - 5, 2048 * 80)]:
        r0 = min(ln, b - start)
        jobs.append((raw, ln, (start, r0, 2 * b)))
    got = run(probe, jobs, taps)
    for j, g in zip(jobs, got):
        same_bits(g, CH.channel(view(raw, j[1], *j[2]), taps), f"view {j[1:]}")


def test_k_channel_demod_equals_k_demod_on_the_planes(probe):
    for T_, real in [(1, True), (31, True), (63, False), (127, False)]:
        taps = taps_for(T_, 7 * T_, real)
        b = 200_000
        raw = capture(3 * b, T_)
        jobs = [(raw, m, (5, m, 0)) for m in (2, 3, 2047, 2048, 2049, 4097, 100_001)]
        jobs.append((raw, 2 * b - 100, (100, b - 100, 2 * b)))   # across the joint
        planes = run(probe, jobs, taps, real_kernel=real)
        outs, stats = run(probe, jobs, taps, real_kernel=real, demod=True)
        for j, (re, im), o, st in zip(jobs, planes, outs, stats):
            m = j[1]
            want = np.empty(m, np.float32)
            ws = np.zeros(ST_COUNT, np.float64)
            err = probe.probe_demod_planes(ctypes.c_longlong(m), _p(np.ascontiguousarray(re)), _p(np.ascontiguousarray(im)),
                                           _p(want), _p(ws))
            assert err == 0
            assert o.view(np.uint32).tolist() == want.view(np.uint32).tolist(), f"T={T_} n={m}"
            # the two kernels add the same f64 terms in different trees: 1e-14 of the sum of the terms' magnitudes
            mags = {ST_POWER0: ws[ST_POWER0], ST_SUM_RE: np.abs(want.astype(np.float64)).sum()}
            for slot in (ST_POWER0, ST_SUM_RE):
                assert abs(st[slot] - ws[slot]) <= 1e-14 * mags[slot], (T_, m, slot)
            assert st[ST_DC_RE] == np.float64(np.float32(np.float32(st[ST_SUM_RE]) / np.float32(m)))


def test_several_jobs_in_one_launch(probe):
    taps = T.channel_taps(-250e3, 80e3, 127)
    raws = [capture(n_s, 900 + k) for k, n_s in enumerate([5000, 70_000, 3, 1_000_003])]
    jobs = [(raws[0], 4000, (1000, 4000, 0)), (raws[1], 60_000, (2, 30_000, 40_000)), (raws[2], 3, (0, 3, 0)),
            (raws[3], 1_000_003, (0, 1_000_003, 0)), (raws[1], 0, (0, 0, 0))]
    got = run(probe, jobs, taps)
    for j, g in zip(jobs, got):
        same_bits(g, CH.channel(view(j[0], j[1], *j[2]), taps), f"job {j[1:]}")
