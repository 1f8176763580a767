"""float64 references for the Monte-Carlo significance of partial and multiple coherence, one realisation at a time.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

* ``device_surrogate_triples``: the surrogate triples of ``wtb_partial_wct_mc_hist`` (noise.cu with three series
  per realisation) restated in NumPy: series ``which`` in {0, 1, 2} of realisation m draws the Philox counter
  (t >> 2, which, m lo, m hi) of ``mc_oracle.device_innovations``.
* ``partial_coherence_samples``: the PWC and MWC values one realisation adds to each histogram row (the reliable
  region of rows below maxscale), from ``pwct_oracle.spectra`` / ``closed_forms``, each with the half-width of
  its rounding band, ``tol * kappa * (1 + |v|)`` with kappa the conditioning of the ratio
  (``pwct_oracle.conditioning``, the gate of the partial-coherence plane tests).
* ``assert_hist_matches_banded``: ``mc_oracle.assert_hist_matches`` with one band per sample, and the skip edge at
  0 (NaN and negative values are not binned) as the only place where a sample may come or go.
"""

from __future__ import annotations

import numpy as np

from . import mc_oracle as mo
from . import pwct_oracle as pw
from . import pycwt_oracle as po


def device_surrogate_triples(ay, a1, a2, nsurr, first, count, seed, white=False):
    """float64 restatement of ``wtb_rednoise_triples``: [count, 3, nsurr] surrogates of realisations
    first .. first + count - 1, series 0, 1, 2 with coefficients ay, a1, a2 and burn-in ceil(-2 / ln|g|) each."""
    out = np.empty((count, 3, nsurr))
    for which, g in enumerate((ay, a1, a2)):
        tau = po.burn_in(g)
        for m in range(count):
            eps = mo.device_innovations(nsurr + tau, which, first + m, seed)
            out[m, which] = eps[tau:] if white else po.rednoise_from_eps(eps, g, tau)
    return out


def partial_coherence_samples(y, x1, x2, dt, dj, s0, J, pad_pow2=True, tol=1e-4):
    """(values, bands): per half (0: PWC, 1: MWC) a list of J + 1 float64 arrays, the values one realisation of
    surrogates y, x1, x2 adds to each row (reliable region of rows below maxscale; empty from maxscale on), and the
    half-widths ``tol * kappa * (1 + |v|)`` of their rounding bands."""
    _, _, _, outside, maxscale = po.mc_geometry(dt, dj, s0, J, po.Morlet())
    sp = pw.spectra(y, x1, x2, dt, dj, s0, J, pad_pow2)
    pwc, _, mwc = pw.closed_forms(sp)
    with np.errstate(divide="ignore", invalid="ignore"):
        kappas = pw.conditioning(sp)
    values, bands = [], []
    for v, kappa in zip((pwc, mwc), kappas):
        rows = [outside[s] if s < maxscale else np.zeros(v.shape[1], dtype=bool) for s in range(J + 1)]
        values.append([v[s, r] for s, r in enumerate(rows)])
        # a NaN kappa (a singular 2 x 2 minor) bounds nothing: its band is infinite
        bands.append([np.nan_to_num(tol * np.abs(kappa[s, r]) * (1 + np.abs(v[s, r])), nan=np.inf)
                      for s, r in enumerate(rows)])
    return values, bands


def banded_histogram(values, nbins=po.NBINS):
    """The histogram [S, nbins] of exact values, binned as the device bins: NaN and negative values skipped,
    bin = min(floor(v nbins), nbins - 1)."""
    hist = np.zeros((len(values), nbins), dtype=np.int64)
    for s, v in enumerate(values):
        v = np.asarray(v, dtype=float)
        v = v[v >= 0]
        idx = np.minimum(np.floor(np.minimum(v, 2.0) * nbins), nbins - 1).astype(np.int64)
        hist[s] = np.bincount(idx, minlength=nbins)[:nbins]
    return hist


def assert_hist_matches_banded(hist, samples, bands):
    """Per-row parity of a device histogram [S, nbins] with reference samples and their bands (lists of S arrays):
    a device value may lie anywhere in [v - d, v + d].

    * the row total lies between #(v - d >= 0) and #(v + d >= 0): a sample may be skipped (negative, NaN) or
      binned only where its band reaches across 0;
    * at every interior edge E = e / nbins the count below it, hist[s, :e].sum(), lies between
      #(v - d >= 0 and v + d < E) and #(v + d >= 0 and v - d < E): a sample may change bins only across an edge
      its band reaches.
    NaN reference values (0/0) may be binned nowhere: they count in neither bound."""
    hist = np.asarray(hist, dtype=np.int64)
    S, nbins = hist.shape
    assert len(samples) == S and len(bands) == S, (len(samples), len(bands), S)
    E = np.arange(1, nbins) / nbins
    for s, (v, d) in enumerate(zip(samples, bands)):
        v, d = np.asarray(v, dtype=float), np.asarray(d, dtype=float)
        assert v.shape == d.shape, (s, v.shape, d.shape)
        ok = ~np.isnan(v)
        v, d = v[ok], d[ok]
        sure, maybe = v - d >= 0, v + d >= 0
        total = int(hist[s].sum())
        assert int(sure.sum()) <= total <= int(maybe.sum()), \
            f"row {s}: {total} samples in the histogram, the reference puts {int(sure.sum())} .. {int(maybe.sum())}"
        C = np.cumsum(hist[s])[:-1]
        hi_sorted = np.sort((v + d)[sure])     # surely binned: below E when v + d < E
        lo_sorted = np.sort((v - d)[maybe])    # possibly binned: possibly below E when v - d < E
        lo = np.searchsorted(hi_sorted, E, side="left")
        hi = np.searchsorted(lo_sorted, E, side="left")
        bad = np.nonzero((C < lo) | (C > hi))[0]
        if bad.size:
            e = int(bad[0]) + 1
            raise AssertionError(
                f"row {s}, edge {e}/{nbins}: {int(C[e - 1])} samples below it, the reference puts "
                f"{int(lo[e - 1])} .. {int(hi[e - 1])} there; {bad.size} edges off in this row")
