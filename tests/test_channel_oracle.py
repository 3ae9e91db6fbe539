"""The channel filter's CPU restatement (tests/channel_oracle.py) on simple inputs, the response of channel_taps, and
the two failures the filter recovers -- a stronger station in an adjacent channel, and a target tuned off-centre
beside a stronger one at DC -- through the oracle chain on five stations."""
import numpy as np
import pytest

import channel_oracle as CH
import tdoa_b200 as T
from oracle import oracle

FS = 2e6
ST5 = np.array([[41.1866, -95.9606, 355.7], [41.2467, -96.0837, 329.0], [41.3292, -96.0351, 373.2],
                [41.42, -95.80, 330.0], [41.10, -96.30, 360.0]])
TX = np.array([41.28, -96.05, 350.0])
REF_TX = np.array([41.30, -95.95, 400.0])
OTHER_TX = np.array([41.50, -96.40, 300.0])


def samples(n, seed=0):
    """unpacked capture samples (every value loadIQData can give)"""
    raw = np.random.default_rng(seed).integers(0, 256, 2 * n, dtype=np.uint8)
    return oracle.unpack_u8(raw)


def bits(a):
    return np.ascontiguousarray(a, np.complex64).view(np.uint32)


def test_one_unit_tap_is_the_identity():
    x = samples(1000)
    assert (bits(CH.channel(x, np.ones(1, np.float32))) == bits(x)).all()
    assert (bits(CH.channel(x, np.ones(1, np.complex64))) == bits(x)).all()


@pytest.mark.parametrize("T_", [1, 3, 31, 63, 127])
def test_unit_tap_shifts_with_zero_edges(T_):
    x = samples(500, T_)
    c = (T_ - 1) // 2
    for k in sorted({0, c, T_ - 1, T_ // 3}):
        h = np.zeros(T_, np.float32)
        h[k] = 1.0
        y = CH.channel(x, h)
        want = np.zeros_like(x)
        s = k - c   # y[i] = x[i + c - k]
        idx = np.arange(x.size) - s
        ok = (idx >= 0) & (idx < x.size)
        want[ok] = x[idx[ok]]
        assert (bits(y) == bits(want)).all(), k


@pytest.mark.parametrize("T_", list(range(1, 128, 2)))
def test_every_length_against_f64_convolution(T_):
    rng = np.random.default_rng(T_)
    x = samples(300, T_)
    h = (rng.standard_normal(T_) + 1j * rng.standard_normal(T_)).astype(np.complex64)
    y = CH.channel(x, h)
    c = (T_ - 1) // 2
    xp = np.concatenate([np.zeros(T_), x.astype(np.complex128), np.zeros(T_)])
    want = np.array([sum(h[k] * xp[T_ + i + c - k] for k in range(T_)) for i in range(x.size)])
    assert np.abs(y - want).max() <= 1e-5 * max(1.0, np.abs(want).max())


def test_real_taps_equal_complex_taps_with_zero_imaginary_parts():
    x = samples(4000)
    h = T.channel_taps(0.0, 100e3).real.astype(np.float32)
    assert (bits(CH.channel(x, h)) == bits(CH.channel(x, h.astype(np.complex64)))).all()


def response_db(h, f):
    c = (h.size - 1) // 2
    H = np.exp(-2j * np.pi * np.outer(f, np.arange(h.size) - c) / FS) @ h.astype(np.complex128)
    return 20 * np.log10(np.maximum(np.abs(H), 1e-30))


@pytest.mark.parametrize("n_taps", [31, 63, 127])
@pytest.mark.parametrize("offset", [0.0, 300e3, -400e3])
def test_channel_taps_response(n_taps, offset):
    hw = 100e3
    h = T.channel_taps(offset, hw, n_taps)
    assert h.dtype == np.complex64 and h.size == n_taps
    d = np.linspace(0, 500e3, 5001)   # distance from the channel's centre
    for sign in (1, -1):
        db = response_db(h, offset + sign * d)
        edge = hw - 2.75 * FS / n_taps
        if edge > 0:
            assert np.abs(db[d <= edge]).max() <= 0.01
        assert db[(d >= hw + 2.75 * FS / n_taps) & (np.abs(offset + sign * d) <= 1e6)].max() <= -60.0
        if n_taps >= 63:
            f6 = d[np.argmin(np.abs(db + 20 * np.log10(2)))]
            assert abs(f6 - hw) <= 0.01 * hw


def test_channel_taps_refuses_bad_lengths():
    for n in (0, 2, 128, 129):
        with pytest.raises(ValueError):
            T.channel_taps(0.0, 100e3, n)


def tgt_lags(raws, taps, max_lag=200):
    sig = [oracle.extract_target(oracle.unpack_u8(r)) for r in raws]
    S = len(raws)
    return {(i, j): CH.window_record(sig[i], sig[j], taps, max_lag)[0] for i in range(S) for j in range(i + 1, S)}


@pytest.mark.parametrize("kind", ["adjacent", "off_centre"])
def test_scenarios_through_the_oracle(kind):
    bad = 3
    raws, dT, f_tgt = CH.scenario(kind, ST5, TX, REF_TX, OTHER_TX, 200_000, bad)
    plain = tgt_lags(raws, None)
    filt = tgt_lags(raws, T.channel_taps(f_tgt, 100e3))
    for (i, j), lag in plain.items():
        want = dT[j] - dT[i]
        if bad in (i, j):
            assert abs(lag - want) > 5, (i, j)
        assert abs(filt[(i, j)] - want) <= 1, (i, j)
