"""The captures of tests/test_gpu_lag_edges.py, checked on the CPU oracle before any GPU run: every planted lag is
the oracle's arg-max, the tie counts are what each case intends and stand more than 5 x TOL clear of the next lag
(so the f32 ranking's error cannot change the candidate count), and the I/Q-swapped station's preprocessed plane,
hence every correlation with it, is exactly the negation."""
import numpy as np
import pytest

from oracle import oracle
import lag_edges as E


@pytest.fixture(autouse=True)
def extended_dc():
    oracle.set_seq_dc_limit(0)   # EXTENDED mode: exactly rounded DC sum
    yield
    oracle.set_seq_dc_limit(-1)


def pair_corr(raws, i, j, L, start, W):
    yi, _ = oracle.preprocess_binary(E.split(raws[i])[1][start:start + W])
    yj, _ = oracle.preprocess_binary(E.split(raws[j])[1][start:start + W])
    return oracle.xcorr_two_sided(yi, yj, L)


@pytest.mark.parametrize("case", [c for c in E.EDGE_CASES if c[4] != 0 or c[1] > 2], ids=lambda c: c[0])
def test_planted_lag_is_the_oracle_argmax(case):
    name, S, L, W, lag, others = case
    raws, d = E.edge_capture(case)
    idx, frac, val = oracle.peak_parabolic(pair_corr(raws, 0, 1, L, E.START, W))
    want = int(np.clip(lag, -L, L))
    assert idx - L == want
    if abs(lag) >= L:
        assert frac == 0.0                          # on the edge: no vertex
    if S > 2:
        for k, x in enumerate(others, start=2):     # the spectra joint: pair (0, 2) at lag 1
            idx, _, _ = oracle.peak_parabolic(pair_corr(raws, 0, k, L, E.START, W))
            assert idx - L == x


@pytest.mark.parametrize("lag", E.BINARY_EDGE_LAGS)
def test_binary_planted_lag_is_the_first_pass_argmax(lag):
    raws, _ = E.planted(E.BINARY_BLOCK, lag, seed=lag % 53)
    c = E.binary_lags(raws)
    assert int(np.argmax(np.abs(c))) == lag
    for sanity in (E.SANITY, 0):
        ti, tj = E.split(raws[0])[1], E.split(raws[1])[1]
        yi, _ = oracle.preprocess_binary(ti)
        yj, _ = oracle.preprocess_binary(tj)
        d, _, researched = oracle.tdcorr_binary(yi, yj, sanity=sanity)
        if sanity and lag == E.SANITY + 1:
            # first pass at 121 > sanity: lag 119, two samples off the peak, holds more than half its
            # correlation, so the re-search over [0, 120) replaces it
            assert (d, researched) == (E.SANITY - 1, True)
        else:
            assert d == lag and not researched


def test_decimated_lag_at_the_range_edge():
    for lag in (E.DEC_L, -E.DEC_L):
        raws, _ = E.planted(E.START + E.DEC_W + 300, lag, seed=5, dev_tgt=20e3)
        yi, _ = oracle.preprocess_binary_dec(E.split(raws[0])[1][E.START:E.START + E.DEC_W], E.DEC_D)
        yj, _ = oracle.preprocess_binary_dec(E.split(raws[1])[1][E.START:E.START + E.DEC_W], E.DEC_D)
        Ld = E.DEC_L // E.DEC_D
        idx, frac, _ = oracle.peak_parabolic(oracle.xcorr_two_sided(yi, yj, Ld))
        assert idx - Ld == lag // E.DEC_D and frac == 0.0


@pytest.mark.parametrize("n_ties", sorted(E.TIE_L))
def test_extended_ties_count_and_gap(n_ties):
    L = E.TIE_L[n_ties]
    raws = E.tie_captures()
    S = len(E.TIE_DELAYS)
    for i in range(S):
        for j in range(i + 1, S):
            c = E.extended_ties(raws, E.TIE_START, E.TIE_W, L, i, j)
            a = np.abs(c)
            top = np.flatnonzero(a == a.max())
            assert len(top) == n_ties, (i, j)                                         # bit-exact ties
            assert np.all(np.diff(top) == E.TIE_PERIOD)
            assert top[0] >= 32 and top[-1] <= 2 * L - 32                             # >= 32 lags inside
            assert (top[0] - L - (E.TIE_DELAYS[j] - E.TIE_DELAYS[i])) % E.TIE_PERIOD == 0
            assert len(E.candidates(c, neighbours=True)) == 3 * n_ties                # 63 / 66
            assert E.selection_gap(c) > 5 * E.TOL


def test_binary_ties_count_and_gap():
    raws = E.tie_captures(binary=True)
    pairs = [(0, 1), (0, 2), (1, 2)]
    for (i, j), want in zip(pairs, E.BTIE_COUNT):
        c = E.binary_lags(raws, i, j)
        a = np.abs(c)
        top = np.flatnonzero(a == a.max())
        assert len(top) == want and top[0] >= 6 and top[0] < E.SANITY          # ties in [0, sanity): one set
        assert len(E.candidates(c, neighbours=False, sanity=E.SANITY)) == want  # 64: no overflow, 65: overflow
        assert E.selection_gap(c, sanity=E.SANITY) > 5 * E.TOL
        # the reference keeps the first of the tied lags and does not re-search
        yi, _ = oracle.preprocess_binary(E.split(raws[i])[1])
        yj, _ = oracle.preprocess_binary(E.split(raws[j])[1])
        d, _, researched = oracle.tdcorr_binary(yi, yj)
        assert d == top[0] and not researched


def test_swapped_iq_negates_the_plane():
    from helpers import fm_capture
    raws = fm_capture(30000, (0, 5, 12), (0, 9, 31), seed=3)
    for kind in (0, 1):
        for k in range(3):
            x = E.split(raws[k])[kind]
            xs = E.split(E.swap_iq(raws[k]))[kind]
            y, br = oracle.preprocess_binary(x)
            ys, brs = oracle.preprocess_binary(xs)
            assert br == brs == 0
            assert np.array_equal(ys.real.view(np.uint32), (-y.real).view(np.uint32))
    a = pair_corr(raws, 0, 1, 300, 200, 20000)
    sw = [raws[0], E.swap_iq(raws[1])]
    b = pair_corr(sw, 0, 1, 300, 200, 20000)
    assert np.array_equal(b, -a)


@pytest.mark.parametrize("extra", [1, 7, 3001])
def test_unequal_lengths_statement_keeps_the_planted_lag(extra):
    """Each station in turn is the longer one; the statement's lag is d_j - d_i whichever is longer."""
    L = 300
    d = (0, 17, 40)
    for longer in range(3):
        blocks = [30000 + (extra if k == longer else 0) for k in range(3)]
        raws = E.ragged(blocks, d, seed=extra)
        for kind in (0, 1):
            ys = [oracle.preprocess_binary(E.split(r)[kind])[0] for r in raws]
            for i, j in ((0, 1), (0, 2), (1, 2)):
                idx, _, _ = oracle.peak_parabolic(E.unequal_statement(ys[i], ys[j], L))
                assert idx - L == d[j] - d[i], (longer, kind, i, j)
