"""The channel filter end to end (EXTENDED mode, tdoa_set_channel): a stronger station in an adjacent channel and a
target tuned off-centre, recovered on six stations; one window's records against the oracle chain on the strong,
moderate and weak branches; identity taps; clearing; the filter with decimation, guard samples, the re-timed call and
a lazily pinned load; more than one GPU; the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import channel_oracle as CH
import closure_oracle as CO
import tdoa_b200 as T
from oracle import oracle
from test_gpu_closure import ST6, TX6
from test_gpu_window_grid import REF_TX, metres

pytestmark = pytest.mark.gpu

OTHER_TX = np.array([41.50, -96.40, 300.0])
BE = 1_000_000
BAD = 4
ARGS = (ST6, 0, BE // 2, 4, 2, BE // 2)
INIT = TX6 + [0.03, 0.03, 0.0]
FIX_KEYS = ("position", "rms", "status", "iters")


def engine(**kw):
    return T.Engine(T.MODE_EXTENDED, max_lag=600, n_stations=6, **kw)


def load(e, raws):
    for k, r in enumerate(raws):
        e.load_u8(k, r)


def set_channels(e, f_tgt):
    e.set_channel(T.KIND_REF, T.channel_taps(0.0, 100e3))
    e.set_channel(T.KIND_TGT, T.channel_taps(f_tgt, 100e3))


def tgt_lag_errors(res, dT):
    lags = res["tgt"]["lag"]
    return np.array([[lags[w, p] - (dT[j] - dT[i]) for p, (i, j) in enumerate(CO.pairs(6))] for w in range(lags.shape[0])])


def same(a, b, keys):
    for k in keys:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


@pytest.fixture(scope="module", params=["adjacent", "off_centre"])
def scene(request):
    raws, dT, f_tgt = CH.scenario(request.param, ST6, TX6, REF_TX, OTHER_TX, BE, BAD)
    clean, _, _ = CH.scenario(request.param, ST6, TX6, REF_TX, OTHER_TX, BE, BAD, other_amp=0.0)
    return request.param, raws, clean, dT, f_tgt


def test_interfered_station_recovered(scene):
    kind, raws, clean, dT, f_tgt = scene
    ex = {"max_rms": 300.0}
    with engine() as e:
        load(e, raws)
        plain = e.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT, exclusion=ex)
        set_channels(e, f_tgt)
        filt = e.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT, exclusion=ex)
        load(e, clean)
        want = e.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT, exclusion=ex)
    err = tgt_lag_errors(plain, dT)
    bad_pairs = [p for p, (i, j) in enumerate(CO.pairs(6)) if BAD in (i, j)]
    assert (np.abs(err[:, bad_pairs]) > 5).all(), err
    assert plain["station_excluded"].tolist() == [[0, 0, 0, 0, 1, 0]] * 2
    assert (np.abs(tgt_lag_errors(filt, dT)) <= 1).all(), tgt_lag_errors(filt, dT)
    assert filt["excluded"].tolist() == [0, 0] and filt["pair_used"].all()
    for w in range(2):
        assert metres(filt["position"][w], want["position"][w]) <= 1.0


def test_oracle_parity_on_every_branch():
    """one TGT window of three stations, each with an FM station 3x stronger at +500 kHz, against channel ->
    preprocess_binary -> xcorr_two_sided -> peak_parabolic; the target's amplitude puts the filtered signal on the
    strong, moderate or weak branch"""
    L, W, B = 300, 100_000, 120_000
    taps = T.channel_taps(0.0, 100e3)
    st3 = ST6[:3]
    oracle.set_seq_dc_limit(0)
    oracle.set_wide_boxcar_f64(33)
    try:
        for amp, branch in ((0.25, 0), (0.06, 1), (0.02, 2)):
            dR, dT = CH.delays(st3, REF_TX), CH.delays(st3, TX6)
            raws = CH.fm_band_captures(B, [dict(seed=11, offset=0.0, amp=amp, blocks="ref", delays=dR),
                                           dict(seed=12, offset=0.0, amp=amp, blocks="tgt", delays=dT),
                                           dict(seed=13, offset=500e3, amp=3 * amp, blocks="all", delays=dT)], 3, seed=5)
            with T.Engine(T.MODE_EXTENDED, max_lag=L) as e:
                load(e, raws)
                e.set_channel(T.KIND_TGT, taps)
                got = e.xcorr(T.KIND_TGT, 500, W, 1, 0)[0]
                info, _ = e.xcorr_info(T.KIND_TGT)
            sig = [oracle.extract_target(oracle.unpack_u8(r))[500:500 + W] for r in raws]
            for p, (i, j) in enumerate([(0, 1), (0, 2), (1, 2)]):
                lag, frac, val, bi, bj = CH.window_record(sig[i], sig[j], taps, L)
                assert (info[i]["branch"], info[j]["branch"]) == (bi, bj) == (branch, branch)
                assert int(got[p]["lag"]) == lag, (amp, p)
                assert abs(float(got[p]["frac"]) - frac) <= 1e-3
                assert abs(float(got[p]["corr"]) - val) <= 1e-6
    finally:
        oracle.set_seq_dc_limit(-1)
        oracle.set_wide_boxcar_f64(0)


@pytest.fixture(scope="module")
def adjacent():
    return CH.scenario("adjacent", ST6, TX6, REF_TX, OTHER_TX, BE, BAD)[0]


def test_identity_taps(adjacent):
    one = np.ones(1, np.float32)
    with engine() as a, engine() as b:
        load(a, adjacent)
        load(b, adjacent)
        want = a.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        b.set_channel(T.KIND_REF, one)
        b.set_channel(T.KIND_TGT, one)
        got = b.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
    for k in ("ref", "tgt"):
        assert np.array_equal(got[k]["lag"], want[k]["lag"])
        np.testing.assert_allclose(got[k]["corr"], want[k]["corr"], rtol=1e-12, atol=0)
    assert np.array_equal(got["position"], want["position"])


def test_clearing_restores_a_fresh_engine(adjacent):
    with engine() as fresh, engine() as e:
        load(fresh, adjacent)
        load(e, adjacent)
        want = fresh.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        n_want = fresh.stats()["launches_last"]
        set_channels(e, 0.0)
        e.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        e.set_channel(T.KIND_REF, None)
        e.set_channel(T.KIND_TGT, None)
        got = e.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        assert e.stats()["launches_last"] == n_want
    same(want, got, FIX_KEYS + ("ref", "tgt", "range_differences"))


def test_decimated_guarded_retimed_and_pinned(adjacent):
    taps = T.channel_taps(0.0, 100e3)
    dT = CH.delays(ST6, TX6)
    # decimate 2 with guard samples: the TGT lags still land on the delays
    with engine(decimate=2, guard_samples=2000) as e:
        load(e, adjacent)
        e.set_channel(T.KIND_REF, taps)
        e.set_channel(T.KIND_TGT, taps)
        got = e.process_windows(ST6, 0, 400_000, 4, 2, 400_000, ref_tx_llh=REF_TX, init_llh=INIT)
    assert (np.abs(tgt_lag_errors(got, dT)) <= 2).all()
    # the re-timed call filters before it re-times
    with engine() as e:
        load(e, adjacent)
        e.set_channel(T.KIND_REF, taps)
        e.set_channel(T.KIND_TGT, taps)
        rt = e.process_windows_retimed(ST6, (0, 250_000, 8, 250_000), (0, 0, 1, 1_000_000), ref_tx_llh=REF_TX, init_llh=INIT)
    assert (np.abs(tgt_lag_errors(rt, dT)) <= 1).all()
    # a lazily pinned load gives the synchronous load's results
    bufs = []
    for r in adjacent:
        b = T.host_alloc(r.size)
        b.array[:] = r
        bufs.append(b)
    with engine() as a, engine(copy_chunk=1 << 20) as b:
        load(a, adjacent)
        for k, buf in enumerate(bufs):
            b.load_u8_pinned(k, buf)
        for x in (a, b):
            x.set_channel(T.KIND_REF, taps)
            x.set_channel(T.KIND_TGT, taps)
        want = a.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        got = b.process_windows(*ARGS, ref_tx_llh=REF_TX, init_llh=INIT)
        b.synchronize()
    same(want, got, FIX_KEYS + ("ref", "tgt"))


def test_more_than_one_gpu(adjacent):
    taps = T.channel_taps(0.0, 100e3)
    with engine() as a:
        load(a, adjacent)
        a.set_channel(T.KIND_TGT, taps)
        want = a.xcorr_windows(0, BE // 2, 4, 2, BE // 2)
    with engine() as c:
        c.comm_init(T.comm_unique_id(), 0, 1)
        load(c, adjacent)
        c.set_channel(T.KIND_TGT, taps)
        got = c.xcorr_windows(0, BE // 2, 4, 2, BE // 2)
    for g, w in zip(got, want):
        assert g.tobytes() == w.tobytes()
    if torch.cuda.device_count() >= 2:
        with engine(n_devices=2) as d:
            load(d, adjacent)
            d.set_channel(T.KIND_TGT, taps)
            got = d.xcorr_windows(0, BE // 2, 4, 2, BE // 2)
        for g, w in zip(got, want):
            assert g.tobytes() == w.tobytes()


def test_refusals():
    lib = T.load_library()
    ok = np.ones(3, np.float32)

    def call(e, kind, re, im, n):
        return lib.tdoa_set_channel(e._h, kind, re.ctypes.data if re is not None else None,
                                    im.ctypes.data if im is not None else None, n)

    for mode in (T.MODE_BINARY, T.MODE_SOURCE):
        with T.Engine(mode) as e:
            assert call(e, T.KIND_TGT, ok, None, 3) == -1
    with T.Engine(T.MODE_EXTENDED) as e:
        assert call(e, 2, ok, None, 3) == -1
        assert call(e, -1, ok, None, 3) == -1
        for n in (-1, 2, 128, 129):
            assert call(e, T.KIND_REF, np.ones(130, np.float32), None, n) == -1
        assert call(e, T.KIND_REF, None, ok, 3) == -1
        for bad in (math.nan, math.inf, -math.inf, 1e-40):
            h = np.array([0.5, bad, 0.5], np.float32)
            assert call(e, T.KIND_REF, h, None, 3) == -1
            assert call(e, T.KIND_REF, ok, h, 3) == -1
        assert call(e, T.KIND_REF, ok, None, 3) == 0
        assert call(e, T.KIND_REF, None, None, 0) == 0
        with pytest.raises(ValueError):
            e.set_channel(T.KIND_REF, np.ones((3, 1)))
