"""CPU: the float64 references of the partial / multiple coherence Monte Carlo (oracle/pwct_mc_oracle.py).

The triple restatement of the device surrogates draws series 0 and 1 from the same Philox stream as the pair
restatement, and the banded histogram assertion accepts the oracle's own histogram and rejects one sample moved
across an edge its band does not reach (or in or out of a row where its band does not reach 0)."""

import numpy as np
import pytest

from oracle import mc_oracle as mo
from oracle import pwct_mc_oracle as pmo
from oracle import pycwt_oracle as po

SEED = 0x9E3779B9_00C0FFEE


@pytest.mark.parametrize("white", [False, True], ids=["red", "white"])
def test_triples_extend_the_pair_stream(white):
    """K = 2 is the first two series of K = 3: the counter of series `which` does not depend on how many series
    a realisation has.  first = 2^32 - 2 crosses the counter's high word."""
    for nsurr, first, count in [(5, 0, 3), (3351, 2**32 - 2, 4)]:
        tri = pmo.device_surrogate_triples(0.989, 0.966, 0.5, nsurr, first, count, SEED, white=white)
        pair = mo.device_surrogates(0.989, 0.966, nsurr, first, count, SEED, white=white)
        assert tri.shape == (count, 3, nsurr)
        assert np.array_equal(tri[:, :2], pair)
        # the third series is its own stream (series index 2), with its own coefficient and burn-in
        eps = mo.device_innovations(nsurr + po.burn_in(0.5), 2, first, SEED)
        ref = eps[po.burn_in(0.5):] if white else po.rednoise_from_eps(eps, 0.5, po.burn_in(0.5))
        assert np.array_equal(tri[0, 2], ref)


@pytest.fixture(scope="module")
def samples():
    """One realisation of a small geometry (dt 1, dj 1/4, s0 2, J 24: 768-sample surrogates, 25 rows)."""
    dt, dj, s0, J = 1.0, 1 / 4, 2.0, 24
    N, _, _, outside, maxscale = po.mc_geometry(dt, dj, s0, J, po.Morlet())
    sur = pmo.device_surrogate_triples(0.7, 0.5, 0.3, N, 17, 1, SEED)[0]
    values, bands = pmo.partial_coherence_samples(*sur, dt, dj, s0, J, pad_pow2=True, tol=1e-4)
    assert 0 < maxscale <= J and N == 768
    for half in (values, bands):
        assert len(half) == 2 and all(len(rows) == J + 1 for rows in half)
    for s in range(J + 1):
        assert values[0][s].size == (outside[s].sum() if s < maxscale else 0)
    return values, bands


def test_banded_assertion_accepts_the_oracle_histogram(samples):
    values, bands = samples
    for half in range(2):
        pmo.assert_hist_matches_banded(pmo.banded_histogram(values[half]), values[half], bands[half])


def _far_from_edges(v, d, move, nbins=po.NBINS):
    """Index of a sample whose band stays inside its bin, and its bin, such that no sample's band reaches the edge
    the sample is moved across."""
    b = np.floor(v * nbins)
    inside = (v - d > b / nbins) & (v + d < (b + 1) / nbins) & (b >= 1) & (b < nbins - 1)
    for i in np.nonzero(inside)[0]:
        E = (b[i] + (move > 0)) / nbins
        if not np.any((v - d < E) & (v + d >= E)):
            return int(i), int(b[i])
    raise AssertionError("no sample can be moved")


@pytest.mark.parametrize("half", [0, 1], ids=["pwc", "mwc"])
@pytest.mark.parametrize("move", [-1, 1])
def test_banded_assertion_rejects_a_sample_moved_outside_its_band(samples, half, move):
    values, bands = samples
    rows = [s for s in range(len(values[half])) if values[half][s].size]
    s = rows[len(rows) // 2]
    i, b = _far_from_edges(values[half][s], bands[half][s], move)
    hist = pmo.banded_histogram(values[half])
    hist[s, b] -= 1
    hist[s, b + move] += 1
    with pytest.raises(AssertionError, match=f"row {s}, edge"):
        pmo.assert_hist_matches_banded(hist, values[half], bands[half])
    # the same move is accepted once that sample's band reaches across the edge
    wide = [d.copy() for d in bands[half]]
    wide[s][i] = 2.0 / po.NBINS
    pmo.assert_hist_matches_banded(hist, values[half], wide)


def test_banded_assertion_rejects_a_sample_that_comes_or_goes(samples):
    values, bands = samples
    rows = [s for s in range(len(values[0])) if values[0][s].size]
    hist = pmo.banded_histogram(values[0])
    for delta in (-1, 1):
        h = hist.copy()
        b = int(np.nonzero(h[rows[0]])[0][0])
        h[rows[0], b] += delta
        with pytest.raises(AssertionError, match="samples in the histogram"):
            pmo.assert_hist_matches_banded(h, values[0], bands[0])


def test_banded_assertion_lets_a_sample_cross_zero_only_inside_its_band():
    v = [np.array([-1e-6, 0.25, 0.5])]
    h_skip = pmo.banded_histogram(v)
    h_kept = h_skip.copy()
    h_kept[0, 0] += 1                     # the device's value came out at +0 instead of -1e-6
    pmo.assert_hist_matches_banded(h_skip, v, [np.array([2e-6, 1e-9, 1e-9])])
    pmo.assert_hist_matches_banded(h_kept, v, [np.array([2e-6, 1e-9, 1e-9])])
    with pytest.raises(AssertionError, match="samples in the histogram"):
        pmo.assert_hist_matches_banded(h_kept, v, [np.array([1e-7, 1e-9, 1e-9])])
