"""CPU checks of oracle/mc_oracle.py: the Philox restatement, the surrogate layout it rebuilds,
the histogram parity check and the replica of the direct-row split rule."""

import math

import numpy as np
import pytest

from oracle import mc_oracle as mo
from oracle import pycwt_oracle as po

DT = 1 / 12


@pytest.mark.parametrize("ctr,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, expect):
    """Random123's known-answer vectors for Philox4x32-10."""
    assert tuple(int(w) for w in mo.philox4x32_10(ctr, key)) == expect


def test_philox_vectorised_matches_scalar():
    blk = np.arange(5, dtype=np.uint64)
    words = mo.philox4x32_10((blk, 1, 0xFFFFFFFE, 7), (0x89ABCDEF, 0x01234567))
    for b in range(5):
        one = mo.philox4x32_10((b, 1, 0xFFFFFFFE, 7), (0x89ABCDEF, 0x01234567))
        assert [int(w[b]) for w in words] == [int(w) for w in one]


def test_device_innovations_layout():
    """Sample t comes from counter block t >> 2, words (x, y) for t & 3 < 2 and (z, w) after."""
    seed, real = 0x1234_5678_9ABC_DEF0, (1 << 32) + 5
    e = mo.device_innovations(10, 1, real, seed)
    x, y, z, w = mo.philox4x32_10((2, 1, real & 0xFFFFFFFF, real >> 32), (seed & 0xFFFFFFFF, seed >> 32))
    u1, u2 = ((np.float32(int(v) >> 8) + np.float32(0.5)) * np.float32(2.0 ** -24) for v in (x, y))
    r = math.sqrt(-2 * math.log(float(u1)))
    assert e[8] == pytest.approx(r * math.cos(2 * math.pi * float(u2)), abs=1e-15)
    assert e[9] == pytest.approx(r * math.sin(2 * math.pi * float(u2)), abs=1e-15)
    # the two series of a pair and neighbouring realisations are different streams
    assert not np.allclose(e, mo.device_innovations(10, 0, real, seed))
    assert not np.allclose(e, mo.device_innovations(10, 1, real + 1, seed))
    assert np.all(np.abs(e) < 6)


def test_device_surrogates_burn_in_and_white():
    g1, g2, n = 0.9, 0.0, 50
    red = mo.device_surrogates(g1, g2, n, 3, 2, 11)
    white = mo.device_surrogates(g1, g2, n, 3, 2, 11, white=True)
    tau = po.burn_in(g1)
    eps = mo.device_innovations(n + tau, 0, 4, 11)
    assert np.array_equal(white[1, 0], eps[tau:])
    assert np.allclose(red[1, 0], po.rednoise_from_eps(eps, g1, tau), rtol=0, atol=1e-14)
    # g = 0: no burn-in, red and white coincide
    assert np.array_equal(red[:, 1], white[:, 1])
    assert np.array_equal(white[0, 1], mo.device_innovations(n, 1, 3, 11))


def test_assert_hist_matches_band():
    rng = np.random.default_rng(3)
    samples = [rng.uniform(0, 1, 500), rng.uniform(0, 1, 20), np.empty(0)]
    hist = mo.samples_histogram(samples)
    mo.assert_hist_matches(hist, samples, 1e-10)
    assert mo.hist_delta(hist, samples) == 0.0
    # one sample moved one bin up: accepted only with a band that reaches it
    v = samples[0][samples[0] < 0.999][0]
    moved = hist.copy()
    b = int(v * 1000)
    moved[0, b] -= 1
    moved[0, b + 1] += 1
    need = (b + 1) / 1000 - v
    assert mo.hist_delta(moved, samples) == pytest.approx(need)
    mo.assert_hist_matches(moved, samples, need * 1.01)
    with pytest.raises(AssertionError):
        mo.assert_hist_matches(moved, samples, need * 0.99)
    # row totals are exact, rows the reference leaves empty must stay empty
    short = hist.copy()
    short[1, int(samples[1][0] * 1000)] -= 1
    with pytest.raises(AssertionError, match="row 1"):
        mo.assert_hist_matches(short, samples, 1.0)
    extra = hist.copy()
    extra[2, 500] = 1
    with pytest.raises(AssertionError, match="row 2"):
        mo.assert_hist_matches(extra, samples, 1.0)


def test_direct_split_cfg5():
    """cfg5 Monte-Carlo shape (dj 1/8, J 65, 3351 samples -> nfft 4096): the 28 largest scales are
    served by the direct kernel; the first of them has the widest band the kernel accepts."""
    assert mo.direct_split(DT, 1 / 8, 2 * DT, 65) == 38
    assert mo.row_bands(DT, 1 / 8, 2 * DT, 65)[38] == (9, 128, 68)
    assert mo.row_bands(DT, 1 / 8, 2 * DT, 65)[37][1] > 128
    # WTB_MC_DIRECT_B moves the split; values above the kernel's 128 bins are clamped
    assert mo.direct_split(DT, 1 / 8, 2 * DT, 65, bmax=0) == 66
    assert mo.direct_split(DT, 1 / 8, 2 * DT, 65, bmax=1000) == 38
    assert 38 < mo.direct_split(DT, 1 / 8, 2 * DT, 65, bmax=64) < mo.direct_split(DT, 1 / 8, 2 * DT, 65, bmax=16) < 66


def test_direct_split_band_shapes():
    """The band shapes the GPU fuzz relies on: B = 1 / kc = 0 rows at the end of the longest
    scale range of a 4096-sample series, and l0 = 0 for f0 = 5.3."""
    bands = mo.row_bands(DT, 1 / 8, 2 * DT, 88)
    assert bands[-2:] == [(1, 1, 0), (1, 1, 0)]
    assert mo.direct_split(DT, 1 / 8, 2 * DT, 88) <= 87
    s = mo.direct_split(DT, 1 / 8, 2 * DT, 88, f0=5.3)
    assert s <= 88 and all(b[0] == 0 for b in mo.row_bands(DT, 1 / 8, 2 * DT, 88, f0=5.3)[s:])
