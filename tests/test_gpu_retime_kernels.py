"""retime.cu's two kernels against their restatement (tests/retime_oracle.py), bit for bit, launched directly through
tests/native/retime_probe.cu:

  - k_retime on planes of distinct finite floats (a misplaced index never matches, a written 0 shows), at lengths
    around the 4096-sample tile and up to the 4 M-sample block, at rates that take the identity, the staged path
    with 0 to 32 change points per tile, and the per-sample fall-back (|c| past about 1/128, and the 2^40 guard of a
    one-sample tail tile), from source planes 0 to 3 floats past a 16-byte boundary (the vector and scalar loads);
  - k_station_rates at 3 to 64 stations over every shape of the fitted-pair graph, both outputs as f64 bits.

The probe puts 64 canary words on both sides of every output array and fills the array itself with a NaN pattern
before each launch, so a write past either end and a sample left unwritten are both findings."""
import ctypes
import importlib.util
import subprocess
from pathlib import Path

import numpy as np
import pytest

import retime_oracle as RO

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tdoa-geolocation_b200"

pytestmark = pytest.mark.gpu


def _build_module():
    spec = importlib.util.spec_from_file_location("tdoa_b200_build_flags", PKG / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """the probe compiled with the library's flags and retime.cu's own"""
    b = _build_module()
    so = tmp_path_factory.mktemp("retime_probe") / "retime_probe.so"
    extra = dict(b.UNITS)["retime.cu"]
    cmd = [b.nvcc(), *b.ARCH, *b.COMMON, *extra, "-shared", "-Xcompiler", "-fPIC",
           str(ROOT / "tests" / "native" / "retime_probe.cu"), "-o", str(so)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = ctypes.CDLL(str(so))
    lib.probe_retime.restype = ctypes.c_int
    lib.probe_station_rates.restype = ctypes.c_int
    return lib


def _ptr(a, t=ctypes.c_void_p):
    return ctypes.cast(a.ctypes.data, t)


def run_retime(lib, planes, offsets, stations, rates):
    """one launch: job k re-times planes[k] (float32) read offsets[k] floats past a 16-byte boundary by
    rates[stations[k]]; returns the outputs and the canary words that changed"""
    k = len(planes)
    planes = [np.ascontiguousarray(p, np.float32) for p in planes]
    outs = [np.empty(p.size, np.float32) for p in planes]
    n = np.array([p.size for p in planes], np.int64)
    st = np.array(stations, np.int32)
    off = np.array(offsets, np.int32)
    xs = (ctypes.c_void_p * k)(*[p.ctypes.data for p in planes])
    ys = (ctypes.c_void_p * k)(*[o.ctypes.data for o in outs])
    r = np.ascontiguousarray(rates, np.float64)
    bad = ctypes.c_longlong(-1)
    err = lib.probe_retime(ctypes.c_int(k), _ptr(n), _ptr(st), _ptr(off), xs, ys, _ptr(r), ctypes.c_int(r.size),
                           ctypes.byref(bad))
    assert err == 0, f"CUDA error {err}"
    return outs, bad.value


def distinct_plane(n):
    """0x3f800000 + k as f32: distinct, finite, nonzero"""
    return (np.uint32(0x3F800000) + np.arange(n, dtype=np.uint32)).view(np.float32)


def assert_same_bits(got, want, what):
    g, w = got.view(np.uint32), want.view(np.uint32)
    if not np.array_equal(g, w):
        bad = np.flatnonzero(g != w)
        raise AssertionError(f"{what}: {bad.size} samples differ, first at {bad[:8].tolist()}: "
                             f"got {[hex(v) for v in g[bad[:4]]]} want {[hex(v) for v in w[bad[:4]]]}")


LENGTHS = [1, 2, 3, 4, 5, 7, 4095, 4096, 4097, 8191, 8193, 3 * 4096 + 3, 2 ** 21 + 3, 4_000_000]
# magnitudes; every one is taken with both signs
RATES = [
    4e-5, 1e-3,                                   # clock rates: 0 or 1 change point per tile, then a few
    2.0 ** -12,                                   # c (n - n_c) + 0.5 lands exactly on integers
    2.0 ** -7, 31.9 / 4095, 32 / 4095, 32.1 / 4095,   # about 32 change points per tile: staged and fall-back tiles
    0.3, 0.999, 1.5, 1e20,                        # the per-sample fall-back; 1e20 also the 2^40 guard
]


def rate_set(n):
    """0, the rates above, and 1 / (n - 1) -- about where the first samples move (at n = 4096 exactly: its lower
    neighbour copies the plane) -- with its two f64 neighbours"""
    mags = list(RATES)
    if n > 1:
        t = 1.0 / (n - 1)
        mags += [np.nextafter(t, 0.0), t, np.nextafter(t, np.inf)]
    return np.array([0.0] + [s * m for m in mags for s in (1.0, -1.0)], np.float64)


@pytest.mark.parametrize("n", LENGTHS)
def test_retime_matches_restatement_bit_for_bit(probe, n):
    """every rate of the set as one job of one launch, from each source alignment"""
    x = distinct_plane(n)
    rates = rate_set(n)
    want = [RO.retime(x, c) for c in rates]
    for off in (0, 1, 2, 3):
        outs, bad = run_retime(probe, [x] * rates.size, [off] * rates.size, range(rates.size), rates)
        assert bad == 0, (n, off, bad)
        for c, got, w in zip(rates, outs, want):
            assert_same_bits(got, w, f"n={n} offset={off} c={c!r}")


def test_retime_jobs_of_different_lengths_and_stations_in_one_launch(probe):
    """a 4 M plane, a 999 999 plane, a 3-sample plane and an empty one: the tiles past a short job's end return
    early, and each job takes its own station's rate"""
    rates = np.array([-31.9 / 4095, 1e-3, 0.0, -4e-5, 0.3, 2.0 ** -7])
    lens = [4_000_000, 999_999, 3, 0, 12_291]
    stations = [1, 3, 4, 0, 5]
    offsets = [0, 3, 1, 2, 1]
    g = np.random.default_rng(1)
    planes = [(np.uint32(0x3F800000) + g.permutation(m).astype(np.uint32)).view(np.float32) for m in lens]
    outs, bad = run_retime(probe, planes, offsets, stations, rates)
    assert bad == 0
    for m, s, p, got in zip(lens, stations, planes, outs):
        assert_same_bits(got, RO.retime(p, rates[s]), f"n={m} station={s}")


# ------------------------------------------------------------------ k_station_rates
def run_rates(lib, beta, count, S, seed):
    """fit rows with beta at [1] and the window count at [3]; the other three slots carry noise the kernel must not
    read"""
    P = S * (S - 1) // 2
    g = np.random.default_rng(seed)
    fit = g.standard_normal((P, 5))
    fit[:, 1] = beta
    fit[:, 3] = count
    fit = np.ascontiguousarray(fit)
    rate = np.empty(S, np.float64)
    clock = np.empty(S, np.float64)
    bad = ctypes.c_longlong(-1)
    err = lib.probe_station_rates(_ptr(fit), ctypes.c_int(S), _ptr(rate), _ptr(clock), ctypes.byref(bad))
    assert err == 0, f"CUDA error {err}"
    return rate, clock, bad.value


def fitted_pattern(kind, S, g):
    """which pairs (i < j, in RO.pairs order) carry a fit"""
    pp = RO.pairs(S)
    if kind == "all":
        return np.ones(len(pp), bool)
    if kind == "none":
        return np.zeros(len(pp), bool)
    if kind == "tree":
        order = g.permutation(S)
        edges = {tuple(sorted((int(order[k]), int(order[g.integers(k)])))) for k in range(1, S)}
        return np.array([p in edges for p in pp])
    if kind in ("two", "three"):
        labels = g.integers(0, 2 if kind == "two" else 3, S)
        labels[:3 if kind == "three" else 2] = np.arange(3 if kind == "three" else 2)   # every component present
        dense = g.random(len(pp)) < 0.6
        use = np.array([labels[i] == labels[j] for i, j in pp]) & dense
        # each component connected: a chain through its members
        for c in np.unique(labels):
            m = np.flatnonzero(labels == c)
            for a, b in zip(m[:-1], m[1:]):
                use[pp.index((int(a), int(b)))] = True
        return use
    if kind == "isolated":
        alone = set(g.choice(S, size=max(1, S // 4), replace=False).tolist()) | {S - 1}
        return np.array([i not in alone and j not in alone for i, j in pp])
    raise ValueError(kind)


RATE_S = [3, 4, 16, 63, 64]
PATTERNS = ["all", "tree", "two", "three", "isolated", "none"]


@pytest.mark.parametrize("S", RATE_S)
@pytest.mark.parametrize("kind", PATTERNS)
def test_station_rates_match_restatement_bit_for_bit(probe, S, kind):
    g = np.random.default_rng(1000 * S + PATTERNS.index(kind))
    P = S * (S - 1) // 2
    use = fitted_pattern(kind, S, g)
    # betas over 1e-9 .. 1e-3 in both signs, not consistent with any station rates (a real least-squares residual)
    beta = g.choice([-1.0, 1.0], P) * 10.0 ** g.uniform(-9.0, -3.0, P)
    count = np.where(use, g.choice([2.0, 7.0], P), g.choice([1.0, np.nan, 0.0], P))
    # an unfitted pair's beta is anything, NaN included: it must not enter
    beta = np.where(use, beta, g.choice([1.0, -1e3, np.nan], P))
    rate, clock, bad = run_rates(probe, beta, count, S, seed=S)
    assert bad == 0
    want_rate, want_clock = RO.station_rates(beta, count, S)
    assert rate.view(np.uint64).tolist() == want_rate.view(np.uint64).tolist(), (rate, want_rate)
    assert np.array_equal(np.isnan(clock), np.isnan(want_clock))
    assert clock.view(np.uint64).tolist() == want_clock.view(np.uint64).tolist(), (clock, want_clock)
    # what the patterns are for: a station without a fitted pair has rate 0 and clock NaN, the others a number
    pp = RO.pairs(S)
    has = np.zeros(S, bool)
    for p in np.flatnonzero(use):
        has[list(pp[p])] = True
    assert np.array_equal(np.isnan(clock), ~has)
    assert (rate[~has] == 0.0).all() and np.isfinite(rate).all()


def test_station_rates_nan_and_count_two(probe):
    """a NaN window count is unfitted and exactly 2.0 is fitted: four stations, pairs (0,1) count 2, (2,3) NaN"""
    S = 4
    pp = RO.pairs(S)
    beta = np.full(len(pp), 5e-6)
    count = np.ones(len(pp))
    count[pp.index((0, 1))] = 2.0
    count[pp.index((2, 3))] = np.nan
    rate, clock, bad = run_rates(probe, beta, count, S, seed=4)
    assert bad == 0
    assert abs(rate[0] + 2.5e-6) <= 1e-18 and abs(rate[1] - 2.5e-6) <= 1e-18
    assert (rate[2:] == 0.0).all() and np.isnan(clock[2:]).all()
