"""The FFT search's f32 ranking plane against an f64 correlation, on every path that produces it: the 2 x 2 tiles
(default; TDOA_FFT_TILE16 in a subprocess), one transform per pair (use_fft = 2), the parked station spectra (>= 10
pairs), the 2^21-point transform (>= 8192 lags; segmented when the template is longer than one transform), with
use_fft = 3 and 4 moving cases off the last two.  k_select_candidates keeps every lag within TOL = 2e-5 of the
maximum |approx| and evaluates only those exactly, so an error over TOL / 2 at two lags can drop the true maximum
without any flag.  Each record is checked for
 (a) max |approx - exact| <= TOL / 4, and the exact plane at the record's lag equal to corr;
 (b) TDOA_PEAK_NCAND = |select(approx)|, and lag, corr, frac equal to the every-lag record;
 (c) margin bit for bit the statement's on the dumped plane;
 (d) NaN exactly where no ranking exists, the probe's records equal to xcorr's, xcorr's launches unchanged by it.
Contents: FM, white-noise bytes, a carrier off-centre, and a weak-branch station of near-constant bytes beside
strong ones -- in the same tile, the same packed spectra transform and the same big-transform pair -- whose plane
power (xcorr_info's power1) is 1e8 and more times smaller than theirs."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import tdoa_b200 as T
from helpers import fm_capture, fm_signal, quantise
import ranking_oracle as R

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
RESEARCHED, EDGE, BRUTE, EMPTY, OVERFLOW = 0x1, 0x2, 0x4, 0x8, 0x10
ERR_BOUND = R.TOL / 4
PATHS = (1, 2, 3, 4)


def ncand(flags):
    return (np.asarray(flags) >> 16) & 0xff


def device():
    import torch
    return torch.device("cuda", 0)


# ------------------------------------------------------------------ contents (uint8 captures, 3 blocks each)
def noise_capture(block, S, seed):
    g = np.random.default_rng(500 + seed)
    return [g.integers(0, 256, 6 * block, dtype=np.uint8) for _ in range(S)]


def carrier_capture(block, S, seed, f_off=300e3, delays=None):
    """FM tuned f_off off-centre: the discriminator output carries a DC of 2 pi f_off / fs."""
    d = delays or [3 * k for k in range(S)]
    n = block + max(d) + 16
    tgt = fm_signal(n, 2000 + seed, 60e3) * np.exp(2j * np.pi * f_off / 2e6 * np.arange(n))
    ref = fm_signal(n, 1000 + seed, 75e3)
    raws = []
    for k, dk in enumerate(d):
        g = np.random.default_rng(900 + k + seed)
        cut = lambda x: x[16 + max(d) - dk:][:block] + 0.02 * (g.standard_normal(block) + 1j * g.standard_normal(block))
        raws.append(quantise(np.concatenate([cut(ref), cut(tgt), cut(ref)])))
    return raws


def near_constant(block, flips, seed, step=1):
    """A capture of the constant byte 127 (a receiver with its gain at zero) but for `flips` I bytes of 127 + step
    per block: the weak branch, with a plane power of about 1e-9 per flip per 1e5 samples (step 1)."""
    raw = np.full(6 * block, 127, np.uint8)
    g = np.random.default_rng(700 + seed)
    for b in range(3):
        raw[2 * (b * block + g.choice(block, flips, replace=False))] = 127 + step
    return raw


def capture(content, block, S, seed=0, weak=()):
    """weak: (station, flips, step) triples replaced by near-constant captures."""
    if content == "fm":
        raws = fm_capture(block, [5 * k for k in range(S)], [7 * k + (k % 3) for k in range(S)], seed=seed)
    elif content == "noise":
        raws = noise_capture(block, S, seed)
    elif content == "carrier":
        raws = carrier_capture(block, S, seed)
    else:
        raise ValueError(content)
    for s, flips, step in weak:
        raws[s] = near_constant(block, flips, seed + s, step)
    return raws


# ------------------------------------------------------------------ one engine run, every record checked
def probe(raws, mode, kind, start, W, use_fft, **cfg):
    with T.Engine(mode, n_stations=len(raws), use_fft=use_fft, **cfg) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        e.xcorr(kind, start, W, 1, 0)   # a first call may redo a window whose branch it guessed wrong
        plain = e.xcorr(kind, start, W, 1, 0)
        launches = e.stats()["launches_last"]
        rec, rk = e.xcorr_ranking(kind, start, W, 1, 0)
        again = e.xcorr(kind, start, W, 1, 0)
        assert e.stats()["launches_last"] == launches                                 # (d) xcorr unchanged
        assert rec.tobytes() == plain.tobytes() == again.tobytes()
        info, first = e.xcorr_info(kind)
        planes = [e.preprocess(k, kind, start, W)[0] if W else None for k in range(len(raws))]
        if not W:
            n = [x["n"] for x in info]
            planes = [e.preprocess(k, kind, 0, n[k])[0] for k in range(len(raws))]
    return rec[0], rk[0], info, first, planes


def check(raws, mode, kind=T.KIND_TGT, start=0, W=0, paths=PATHS, content="fm", min_ratio=None, **cfg):
    """Runs every path and use_fft = 0; returns the power ratio max power1 / min power1 of the stations."""
    S = len(raws)
    pairs = [(i, j) for i in range(S) for j in range(i + 1, S)]
    ext = mode == T.MODE_EXTENDED
    D = max(1, cfg.get("decimate", 1)) if ext else 1
    L = cfg.get("max_lag", 2000) // D
    ref, rk0, info0, _, planes = probe(raws, mode, kind, start, W, 0, **cfg)
    assert np.all(np.isnan(rk0))                                                       # (d) every-lag: no ranking
    p1 = np.array([x["power1"] for x in info0])
    ratio = float(p1.max() / p1.min())
    dev = device()
    if ext:
        exact = [R.exact_extended(planes[i], planes[j], L, dev) for i, j in pairs]
    else:
        exact = [R.exact_binary(planes[i], planes[j], cfg.get("max_lag", 2000), 10000, dev) for i, j in pairs]
    sanity = 0 if ext else cfg.get("sanity_lag", 120)
    for u in paths:
        rec, rk, info, first, _ = probe(raws, mode, kind, start, W, u, **cfg)
        for p, (i, j) in enumerate(pairs):
            r, c = rec[p], exact[p]
            n_lags = c.size
            a = rk[p, :n_lags]
            assert np.all(np.isnan(rk[p, n_lags:])), (u, p)                           # (d) NaN past the lags
            assert not np.any(np.isnan(a)), (u, p)
            err = float(np.max(np.abs(a - c)))
            print(f"ranking: path {u} {content} pair {p} ratio {ratio:.3g} max|approx - exact| = {err:.3e}")
            assert err <= ERR_BOUND, (u, p, err, ratio)                                # (a)
            if r["flags"] & BRUTE:                                                     # the cap's redo keeps the plane
                assert len(R.select(a, neighbours=ext, sanity=sanity)) > E_MAX_CAND, (u, p)
                assert r.tobytes() == ref[p].tobytes(), (u, p)
                continue
            cand = R.select(a, neighbours=ext, sanity=sanity)
            assert ncand(r["flags"]) == min(len(cand), 255), (u, p, ncand(r["flags"]), len(cand))   # (b)
            for name in ("lag", "first_lag", "n_blocks"):                             # (b) the every-lag record
                assert r[name] == ref[p][name], (u, p, name)
            assert r["flags"] & (RESEARCHED | EDGE | EMPTY) == ref[p]["flags"] & (RESEARCHED | EDGE | EMPTY), (u, p)
            assert abs(r["corr"] - ref[p]["corr"]) <= 1e-12 and abs(r["frac"] - ref[p]["frac"]) <= 1e-6, (u, p)
            best = int(r["first_lag"]) // D + (L if ext else 0)
            c1 = float(first[p]) if r["flags"] & RESEARCHED else float(r["corr"])
            assert r["margin"] == R.margin(a, best, c1), (u, p, r["margin"], R.margin(a, best, c1))   # (c)
            if ext:
                assert abs(c[best] - c1) <= 1e-12, (u, p)                              # (a) corr on the plane
            else:
                assert abs(R.binary_at(planes[i], planes[j], cfg.get("max_lag", 2000), 10000, int(r["lag"]))
                           - float(r["corr"])) <= 1e-12, (u, p)
    if min_ratio is not None:
        assert ratio >= min_ratio, ratio
    return ratio


E_MAX_CAND = 64


# ------------------------------------------------------------------ EXTENDED geometries
# (name, stations, max_lag, template W - 2L, decimate, content)
EXT_CASES = [
    ("L1024_t100", 3, 1024, 100, 1, "noise"),          # 2049 lags: a 1-lag last chunk
    ("L1024_t6143", 3, 1024, 6143, 1, "fm"),
    ("L1024_t6144", 3, 1024, 6144, 1, "carrier"),
    ("L1024_t6145", 3, 1024, 6145, 1, "fm"),
    ("L3000", 3, 3000, 40000, 1, "noise"),
    ("L4095_spectra", 5, 4095, 30000, 1, "fm"),        # 10 pairs, 8191 lags: the spectra's chunk joint
    ("L4096_big", 3, 4096, 30000, 1, "carrier"),
    ("L5000_big", 3, 5000, 40000, 1, "fm"),
    ("dec4", 3, 1200, 20000, 4, "fm"),
    ("spectra16", 16, 1024, 20000, 1, "noise"),
    ("segments_2001", 3, 1024, 2001 * 6144 - 7, 1, "fm"),   # >= 2000 segments, not a multiple of the CTAs
    ("big_segmented", 3, 4096, (1 << 21) + 3000, 1, "fm"),  # template > 2^21 - n_lags
]


@pytest.mark.parametrize("case", EXT_CASES, ids=lambda c: c[0])
def test_extended_ranking_on_every_path(case):
    name, S, L, n_t, D, content = case
    W = D * (n_t + 2 * (L // D))
    raws = capture(content, W + 400, S, seed=len(name))
    check(raws, T.MODE_EXTENDED, start=200, W=W, content=content, max_lag=L, decimate=D)


def test_binary_ranking_with_sanity():
    raws = capture("fm", 250000, 3, seed=2)
    check(raws, T.MODE_BINARY, content="fm")


def test_binary_ranking_unequal_lengths():
    """Station 1's capture is 30 001 samples per block shorter: its signals are the template of its pairs, with
    n_lags = min(2000, sl - tl) < 2000 for the pair with station 0."""
    raws = capture("noise", 250000, 3, seed=3)
    raws[1] = raws[1][:6 * 250000 - 6 * 30001]     # blocks of 219 999 samples
    check(raws, T.MODE_BINARY, content="noise")


# ------------------------------------------------------------------ the weak station beside strong ones
# strong stations of white-noise bytes beside station 2 of near-constant bytes: in one tile (3 stations), one
# packed spectra transform (5 stations, 10 pairs), one big-transform pair (8193 lags)
WEAK_GEOMETRIES = [("tile", 3, 1024, 100000), ("spectra", 5, 1024, 100000), ("big", 3, 4096, 100000)]


@pytest.mark.parametrize("geo", WEAK_GEOMETRIES, ids=lambda g: g[0])
def test_weak_station_at_a_power_ratio_of_1e8(geo):
    name, S, L, n_t = geo
    W = n_t + 2 * L
    raws = capture("noise", W + 400, S, seed=11, weak=[(2, 1, 1)])
    ratio = check(raws, T.MODE_EXTENDED, start=200, W=W, content="weak", min_ratio=1e8, max_lag=L)
    print(f"ranking: weak station in a {name}: power ratio {ratio:.3g}")


@pytest.mark.parametrize("flips, step, lo, hi", [(None, 0, 0.1, 10), (25000, 4, 2e3, 5e4), (3000, 1, 2e5, 5e6)])
def test_weak_station_power_sweep(flips, step, lo, hi):
    """Ratios about 1, 1e4 and 1e6 (flips of `step` per block of the near-constant station; None: all strong)."""
    W = 100000 + 2048
    raws = capture("noise", W + 400, 3, seed=12, weak=[(2, flips, step)] if flips else [])
    ratio = check(raws, T.MODE_EXTENDED, start=200, W=W, content="weak", max_lag=1024)
    print(f"ranking: weak sweep {flips} flips: power ratio {ratio:.3g}")
    assert lo <= ratio <= hi, ratio


def test_unscaled_planes_just_under_the_pack_ratio():
    """Station 2 is FM at a fifteenth of the others' deviation: a plane power about 190 times smaller, scales about
    14x apart, just under kRankPackRatio = 16 -- the largest disparity the transforms pack without scaling."""
    W = 100000 + 2048
    raws = fm_capture(W + 400, [0, 5, 10], [0, 7, 15], seed=12)
    raws[2] = fm_capture(W + 400, [0, 5, 10], [0, 7, 15], seed=12, dev_tgt=4e3, noise=0.005)[2]
    ratio = check(raws, T.MODE_EXTENDED, start=200, W=W, content="fm_low_dev", max_lag=1024)
    print(f"ranking: unscaled pack: power ratio {ratio:.3g}")
    assert 120 <= ratio < 256, ratio


# ------------------------------------------------------------------ several windows in one call
def test_windows_map_to_their_own_planes():
    """3 windows with a hop: the two-stream split of tdoa_xcorr (windows 0-1 and 2 on two streams) and the record
    index of every plane; each window's plane against its own f64 plane."""
    L, W, hop, start = 1024, 30000, 7001, 300
    raws = capture("fm", start + 2 * hop + W + 400, 3, seed=21)
    pairs = [(0, 1), (0, 2), (1, 2)]
    for u in (1, 2):
        with T.Engine(T.MODE_EXTENDED, use_fft=u, max_lag=L) as e:
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            plain = e.xcorr(T.KIND_TGT, start, W, 3, hop)
            rec, rk = e.xcorr_ranking(T.KIND_TGT, start, W, 3, hop)
            assert rec.tobytes() == plain.tobytes() and rk.shape == (3, 3, 2 * L + 1)
            for w in range(3):
                y = [e.preprocess(k, T.KIND_TGT, start + w * hop, W)[0] for k in range(3)]
                for p, (i, j) in enumerate(pairs):
                    c = R.exact_extended(y[i], y[j], L, device())
                    err = float(np.max(np.abs(rk[w, p] - c)))
                    assert err <= ERR_BOUND, (u, w, p, err)
                    assert abs(c[int(rec[w, p]["lag"]) + L] - rec[w, p]["corr"]) <= 1e-12, (u, w, p)
            # a window's plane is not its neighbour's: the mapping is by record
            assert np.max(np.abs(rk[0] - rk[1])) > 10 * ERR_BOUND


# ------------------------------------------------------------------ records without a ranking, and the cap's redo
def test_nan_where_no_ranking_exists():
    # BINARY with max_lag 1000 on 31 500-sample signals: the sanity re-search's template (tl - 2000) has fewer
    # whole blocks than the first pass's (tl - 1000), so every pair is evaluated lag by lag (need2)
    raws = capture("fm", 31500, 3, seed=5)
    with T.Engine(T.MODE_BINARY, max_lag=1000) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        rec, rk = e.xcorr_ranking(T.KIND_TGT)
        assert rec.tobytes() == e.xcorr(T.KIND_TGT).tobytes()
    assert rk.shape == (1, 3, 1000) and np.all(rec["flags"] & BRUTE) and np.all(np.isnan(rk))
    # <= 8 lags: EXTENDED with max_lag 3 (7 lags) is evaluated lag by lag
    with T.Engine(T.MODE_EXTENDED, max_lag=3) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        rec, rk = e.xcorr_ranking(T.KIND_TGT, 0, 20000)
    assert rk.shape == (1, 3, 7) and np.all(rec["flags"] & BRUTE) and np.all(np.isnan(rk))
    # an empty capture: its pairs are EMPTY and have no plane, the pair of the other two has one
    from helpers import load_golden
    raws, _ = load_golden("empty_third")
    with T.Engine(T.MODE_BINARY) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        rec, rk = e.xcorr_ranking(T.KIND_TGT)
    empty = (rec[0]["flags"] & EMPTY) != 0
    assert empty.tolist() == [False, True, True]
    assert np.all(np.isnan(rk[0, empty])) and not rec[0][0]["flags"] & BRUTE
    assert ncand(rec[0][0]["flags"]) > 0 and not np.any(np.isnan(rk[0, 0]))   # 2000 lags: the whole row


def test_cap_redo_keeps_its_plane():
    """lag_edges' 22-tie capture: 66 candidates on every pair, over the cap of 64, so every record comes back redone
    lag by lag (BRUTE, the every-lag record) and keeps the FFT plane that overflowed."""
    import lag_edges as E
    raws = E.tie_captures()[:3]
    check(raws, T.MODE_EXTENDED, start=E.TIE_START, W=E.TIE_W, paths=(1, 2), content="ties", max_lag=E.TIE_L[22])
    with T.Engine(T.MODE_EXTENDED, max_lag=E.TIE_L[22]) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        rec, rk = e.xcorr_ranking(T.KIND_TGT, E.TIE_START, E.TIE_W)
    assert np.all(rec["flags"] & BRUTE) and not np.any(np.isnan(rk))


# ------------------------------------------------------------------ the f64 statement's device FFT
def test_device_statement_equals_the_oracle():
    """The torch f64 FFT the tests above use for the exact plane, against the oracle's time-domain correlators on
    one medium case (the CPU tests check the numpy FFT the same way)."""
    from oracle import oracle
    rng = np.random.default_rng(8)
    y = [(rng.standard_normal(60000) + 1j * rng.standard_normal(60000)).astype(np.complex64) for _ in range(2)]
    L = 3000
    want = oracle.xcorr_two_sided(y[0], y[1], L)
    assert np.max(np.abs(R.exact_extended(y[0], y[1], L, device()) - want)) <= 1e-12
    want = oracle.tdcorr_binary_lags_mt(y[0], y[1], y[0].size - 2000, 2000)
    assert np.max(np.abs(R.exact_binary(y[0], y[1], 2000, 10000, device()) - want)) <= 1e-9   # f32 products there
    assert np.max(np.abs(R.exact_binary(y[0], y[1], 2000, 10000, device())
                         - R.exact_binary(y[0], y[1], 2000, 10000))) <= 1e-12


# ------------------------------------------------------------------ configs[1]'s full TGT size
def test_full_size_binary_tgt():
    """3 x 66 666 666-sample TGT signals, whole-signal BINARY correlation (about 10 850 segments per pair)."""
    sys.path.insert(0, str(ROOT / "tools"))
    import torch
    import bench
    import configs_bench as cb
    dev = device()
    delays, _ = cb.delays_for(bench.STATION_LLH)
    caps = [c.cpu().numpy() for c in cb.synth(dev, 3, 66_666_666, delays)]
    torch.cuda.empty_cache()
    check(caps, T.MODE_BINARY, paths=(1,), content="fm_full", chunk_samples=0)


# ------------------------------------------------------------------ the 16-row tile kernel (read once per process)
def test_tile16_in_a_subprocess():
    env = dict(os.environ, TDOA_FFT_TILE16="1")
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_ranking as G, tdoa_b200 as T; "
            "c = G.EXT_CASES; [G.test_extended_ranking_on_every_path(x) for x in (c[2], c[5], c[10])]; "
            "G.test_weak_station_at_a_power_ratio_of_1e8(G.WEAK_GEOMETRIES[0])"
            % (str(ROOT / "tests"), str(ROOT)))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-3000:], r.stderr[-3000:])
    assert r.returncode == 0


# ------------------------------------------------------------------ refusals
def test_probe_refuses_multi_device_engines():
    import torch
    raws = capture("fm", 30000, 3)
    if torch.cuda.device_count() >= 2:
        with T.Engine(T.MODE_EXTENDED, max_lag=300, n_devices=2) as e:
            for k, r in enumerate(raws):
                e.load_u8(k, r)
            with pytest.raises(T.TdoaError, match="one GPU"):
                e.xcorr_ranking(T.KIND_TGT, 0, 20000)
    with T.Engine(T.MODE_EXTENDED, max_lag=300) as e:
        for k, r in enumerate(raws):
            e.load_u8(k, r)
        e.comm_init(T.comm_unique_id(), 0, 1)
        with pytest.raises(T.TdoaError, match="one GPU"):
            e.xcorr_ranking(T.KIND_TGT, 0, 20000)
    with T.Engine(T.MODE_SOURCE) as e:
        with pytest.raises(T.TdoaError, match="SOURCE"):
            e.xcorr_ranking(T.KIND_TGT)
