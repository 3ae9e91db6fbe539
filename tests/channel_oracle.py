"""The channel filter (tdoa_set_channel) restated on the CPU, and captures of several FM programmes in one 2 MHz band.

channel(x, taps): include/tdoa_b200.h's statement with explicit fmaf (tests/native/channel_oracle.c, compiled here with
the oracle's flags).  window_record: one filtered TGT window of a pair through the oracle chain -- channel ->
oracle.preprocess_binary(_dec) -> oracle.xcorr_two_sided -> oracle.peak_parabolic.

fm_band_captures: one uint8 capture per station (quantised as simulator.go), block 1 = REF, block 2 = TGT, block 3 =
REF, each the sum of FM programmes at chosen offsets, amplitudes and per-station delays.  Unlike the closure tests'
interfered_captures, which replace the target on the same frequency (co-channel, which no channel filter can help),
the programmes here sit in other channels of the band."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import oracle
from helpers import quantise

FS = 2e6
CL = 299792458.0
_SRC = Path(__file__).resolve().parent / "native" / "channel_oracle.c"
_lib = None


def _load():
    global _lib
    if _lib is None:
        src = _SRC.read_bytes()
        d = Path(tempfile.gettempdir()) / f"tdoa_channel_oracle_{os.getuid()}"
        d.mkdir(exist_ok=True)
        so = d / f"channel_oracle_{hashlib.sha256(src).hexdigest()[:16]}.so"
        if not so.exists():
            cc = "/usr/bin/gcc" if Path("/usr/bin/gcc").exists() else "gcc"
            tmp = so.with_suffix(f".{os.getpid()}.tmp")
            subprocess.run([cc, "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o", str(tmp), str(_SRC),
                            "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(str(so))
        _lib.orc_channel.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        _lib.orc_channel.restype = None
    return _lib


def channel(x, taps):
    """the filtered signal y (complex64) of x under taps (real: passed with NULL imaginary parts)"""
    x = np.ascontiguousarray(x, np.complex64)
    t = np.asarray(taps)
    hr = np.ascontiguousarray(t.real, np.float32)
    hi = np.ascontiguousarray(t.imag, np.float32) if np.iscomplexobj(t) else None
    y = np.empty_like(x)
    _load().orc_channel(x.ctypes.data, x.size, hr.ctypes.data, hi.ctypes.data if hi is not None else None, t.size,
                        y.ctypes.data)
    return y


def window_record(sig_i, sig_j, taps, max_lag, D=1):
    """(lag, frac, corr, branch_i, branch_j) of one window of pair (i, j) in EXTENDED mode with the channel filter;
    sig_*: the two stations' samples of the window (complex, as oracle.extract_target gives them)"""
    if taps is not None:
        sig_i, sig_j = channel(sig_i, taps), channel(sig_j, taps)
    yi, bi = oracle.preprocess_binary_dec(sig_i, D) if D > 1 else oracle.preprocess_binary(sig_i)
    yj, bj = oracle.preprocess_binary_dec(sig_j, D) if D > 1 else oracle.preprocess_binary(sig_j)
    L = max_lag // D
    idx, frac, val = oracle.peak_parabolic(oracle.xcorr_two_sided(yi, yj, L))
    return idx - L, frac, val, bi, bj


def fm_programme(n: int, seed: int, dev: float = 75e3, taps: int = 11) -> np.ndarray:
    """unit-amplitude FM of a band-limited random programme (11-sample box-car: an audio band well inside the
    deviation), n samples"""
    a = np.random.default_rng(seed).standard_normal(n + 4 * taps)
    a = np.convolve(a, np.ones(taps) / taps, "same")[:n]
    a /= np.abs(a).max()
    return np.exp(1j * 2 * np.pi * np.cumsum(a) * dev / FS)


def delays(stations_llh, tx_llh) -> np.ndarray:
    """integer sample delays of a transmitter at the stations, the nearest at 0"""
    d = np.round([np.linalg.norm(oracle.llh_to_ecef(*tx_llh) - oracle.llh_to_ecef(*s)) / CL * FS for s in stations_llh])
    return (d - d.min()).astype(np.int64)


def fm_band_captures(block: int, programmes, n_stations: int, seed: int = 0, noise: float = 0.02):
    """programmes: dicts with
      seed       the programme's random stream
      offset     its carrier's offset from the tuned frequency (Hz)
      amp        its amplitude
      blocks     "ref" (blocks 1 and 3), "tgt" (block 2) or "all"
      delays     per-station integer sample delays
      stations   the stations that receive it (default: all)
    Returns one uint8 capture of 3 block samples per station."""
    n = 3 * block
    t = np.arange(n)
    in_tgt = (t >= block) & (t < 2 * block)
    pad = max(int(np.max(p["delays"])) for p in programmes) + 16
    sigs = [fm_programme(n + pad, p["seed"], p.get("dev", 75e3)) for p in programmes]
    raws = []
    for k in range(n_stations):
        x = np.zeros(n, np.complex128)
        for p, s in zip(programmes, sigs):
            if k not in p.get("stations", range(n_stations)):
                continue
            on = {"ref": ~in_tgt, "tgt": in_tgt, "all": np.ones(n, bool)}[p["blocks"]]
            v = p["amp"] * s[pad + t - int(p["delays"][k])] * np.exp(2j * np.pi * p["offset"] / FS * t)
            x += np.where(on, v, 0.0)
        g = np.random.default_rng(7000 + 31 * seed + k)
        raws.append(quantise(x + noise * (g.standard_normal(n) + 1j * g.standard_normal(n))))
    return raws


def scenario(kind: str, stations_llh, tx_llh, ref_tx_llh, other_tx_llh, block: int, bad: int, seed: int = 0,
             other_amp: float = 0.75):
    """The two failures a channel filter recovers, at station `bad` (TGT block only):
      "adjacent":   the target at 0 Hz, a 3x stronger FM station at +500 kHz;
      "off_centre": the target tuned to +300 kHz, a 3x stronger FM station at 0 Hz.
    The REF programme sits at 0 Hz in blocks 1 and 3 of every station; other_amp = 0 gives the same captures without
    the interferer (the same noise).  Returns (captures, TGT delays, target offset)."""
    S = len(stations_llh)
    dR, dT, dO = delays(stations_llh, ref_tx_llh), delays(stations_llh, tx_llh), delays(stations_llh, other_tx_llh)
    f_tgt, f_other = (0.0, 500e3) if kind == "adjacent" else (300e3, 0.0)
    progs = [
        dict(seed=100 + seed, offset=0.0, amp=0.25, blocks="ref", delays=dR),
        dict(seed=200 + seed, offset=f_tgt, amp=0.25, blocks="tgt", delays=dT),
        dict(seed=300 + seed, offset=f_other, amp=other_amp, blocks="tgt", delays=dO, stations=[bad]),
    ]
    return fm_band_captures(block, progs, S, seed), dT, f_tgt
