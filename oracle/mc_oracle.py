"""float64 references for the Monte-Carlo coherence chain, one realisation at a time.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

* ``philox4x32_10`` / ``device_surrogates``: the device surrogate generator of
  ``wavelet_transformer_b200/csrc/noise.cu`` restated in NumPy -- the same
  Philox4x32-10 stream, the same counter layout, the same Box-Muller pairing
  and AR(1) burn-in -- so a device realisation can be rebuilt on the CPU.
* ``coherence_samples``: the per-row R^2 values one realisation contributes to
  ``pycwt.wct_significance``'s histogram (the reliable region, rows below
  maxscale), from ``pycwt_oracle``.
* ``assert_hist_matches``: exact histogram parity up to a rounding band: a
  sample may sit in another bin than the reference's only if the reference puts
  it within ``delta`` of that bin edge.
* ``direct_split``: the rule by which the FP32 nfft-4096 coherence pipeline
  (``wct_fast.cu``, ``fill_rows`` and ``wct_fast``) hands its largest
  scales to the direct band-limited kernel, so tests can choose and assert the
  band shapes they exercise.
"""

from __future__ import annotations

import math

import numpy as np

from oracle import pycwt_oracle as po

_MASK = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011, Random123) in uint64 NumPy arithmetic.

    ``ctr``: four arrays (or scalars) of 32-bit words, broadcast together;
    ``key``: two 32-bit words.  Returns the four output words as uint64 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) for c in ctr))
    k0, k1 = (np.uint64(int(k) & 0xFFFFFFFF) for k in key)
    for _ in range(10):
        p0 = _M0 * c0                   # < 2^64: the full 32 x 32 product
        p1 = _M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + _W0) & _MASK
        k1 = (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def _uniform(w):
    """``((w >> 8) + 0.5) / 2^24`` formed in float32 as the kernel forms it: for ``w >> 8 >= 2^23``
    the ``+ 0.5`` rounds (to even), and near u = 1 that moves -2 ln u by a large relative amount."""
    f = (w >> np.uint64(8)).astype(np.float32) + np.float32(0.5)
    return (f * np.float32(1.0 / 16777216.0)).astype(np.float64)


def _box_muller(a, b):
    r = np.sqrt(-2.0 * np.log(_uniform(a)))
    ang = 2.0 * np.pi * _uniform(b)
    return r * np.cos(ang), r * np.sin(ang)


def device_innovations(nsamples, which, real, seed):
    """The first ``nsamples`` standard normals of series ``which`` (0 / 1) of realisation ``real``
    (global index, any int64): Philox counter ``(t >> 2, which, real lo, real hi)``, key
    ``(seed lo, seed hi)``; words x, y give samples 4b, 4b+1 and words z, w samples 4b+2, 4b+3."""
    nblk = (nsamples + 3) // 4
    blk = np.arange(nblk, dtype=np.uint64)
    real = int(real)
    x, y, z, w = philox4x32_10((blk, which, real & 0xFFFFFFFF, real >> 32), (seed & 0xFFFFFFFF, seed >> 32))
    e = np.empty((nblk, 4))
    e[:, 0], e[:, 1] = _box_muller(x, y)
    e[:, 2], e[:, 3] = _box_muller(z, w)
    return e.reshape(-1)[:nsamples]


def device_surrogates(a1, a2, nsurr, first, count, seed, white=False):
    """float64 restatement of ``wtb_rednoise``: [count, 2, nsurr] surrogates of realisations
    first .. first + count - 1.  AR(1) y[t] = g y[t-1] + eps[t] over nsurr + tau innovations with
    tau = ceil(-2 / ln|g|) (0 for g = 0), the first tau samples dropped; ``white``: eps[tau:]."""
    out = np.empty((count, 2, nsurr))
    for which, g in enumerate((a1, a2)):
        tau = po.burn_in(g)
        for m in range(count):
            eps = device_innovations(nsurr + tau, which, first + m, seed)
            out[m, which] = eps[tau:] if white else po.rednoise_from_eps(eps, g, tau)
    return out


def coherence_samples(n1, n2, dt, dj, s0, J, pad_pow2=True):
    """The R^2 values one realisation adds to each row of pycwt.wct_significance's histogram:
    a list of S float64 arrays (reliable region of rows below maxscale; empty from maxscale on)."""
    wavelet = po.Morlet()
    _, sj, _, outsidecoi, maxscale = po.mc_geometry(dt, dj, s0, J, wavelet)
    W1 = po.cwt(n1, dt, dj, s0, J, wavelet, pad_pow2)[0]
    W2 = po.cwt(n2, dt, dj, s0, J, wavelet, pad_pow2)[0]
    S1, S2, S12, _ = po.smoothed_spectra(W1, W2, sj, dt, dj, wavelet, pad_pow2)
    R2 = np.abs(S12) ** 2 / (S1 * S2)
    return [R2[s, outsidecoi[s]] if s < maxscale else np.empty(0) for s in range(J + 1)]


def mc_samples(surrogates, dt, dj, s0, J, pad_pow2=True):
    """``coherence_samples`` of every realisation of [mc, 2, N] surrogates, concatenated per row."""
    per = [coherence_samples(p[0], p[1], dt, dj, s0, J, pad_pow2) for p in np.asarray(surrogates, dtype=float)]
    return [np.concatenate([r[s] for r in per]) for s in range(J + 1)]


def samples_histogram(samples, nbins=po.NBINS):
    """The histogram pycwt would build from these samples ([S, nbins] int64)."""
    hist = np.zeros((len(samples), nbins), dtype=np.int64)
    for s, v in enumerate(samples):
        idx = np.minimum(np.floor(v * nbins).astype(np.int64), nbins - 1)
        hist[s] = np.bincount(idx, minlength=nbins)[:nbins]
    return hist


def hist_delta(hist, samples):
    """Smallest rounding band ``delta`` for which ``assert_hist_matches`` accepts ``hist`` (inf when
    a row's total differs).  At edge E with C samples below it in ``hist`` and the reference sorted
    as v: #(v < E - delta) <= C needs delta >= E - v[C], C <= #(v < E + delta) needs delta > v[C-1] - E."""
    hist = np.asarray(hist, dtype=np.int64)
    nbins = hist.shape[1]
    worst = 0.0
    for s, v in enumerate(samples):
        v = np.sort(np.asarray(v, dtype=float))
        if hist[s].sum() != v.size:
            return math.inf
        C = np.cumsum(hist[s])[:-1]
        E = np.arange(1, nbins) / nbins
        above, below = C < v.size, C > 0
        worst = max(worst, float(np.max(E[above] - v[C[above]], initial=0.0)),
                    float(np.max(v[C[below] - 1] - E[below], initial=0.0)))
    return worst


def assert_hist_matches(hist, samples, delta):
    """Per-row parity of a device histogram [S, nbins] with reference samples (list of S arrays):

    * every row holds exactly as many samples as the reference row (so rows from maxscale on,
      which the reference leaves empty, hold none);
    * at every interior edge E = e / nbins the count below it, C(e) = hist[s, :e].sum(), satisfies
      #(v < E - delta) <= C(e) <= #(v < E + delta): a sample may change bins only if the
      reference puts it within ``delta`` of the edge it crosses."""
    hist = np.asarray(hist, dtype=np.int64)
    S, nbins = hist.shape
    assert len(samples) == S, (len(samples), S)
    E = np.arange(1, nbins) / nbins
    for s, v in enumerate(samples):
        v = np.sort(np.asarray(v, dtype=float))
        total = int(hist[s].sum())
        assert total == v.size, f"row {s}: {total} samples in the histogram, {v.size} in the reference"
        C = np.cumsum(hist[s])[:-1]
        lo = np.searchsorted(v, E - delta, side="left")
        hi = np.searchsorted(v, E + delta, side="left")
        bad = np.nonzero((C < lo) | (C > hi))[0]
        if bad.size:
            e = int(bad[0]) + 1
            raise AssertionError(
                f"row {s}, edge {e}/{nbins}: {int(C[e - 1])} samples below it, the reference puts "
                f"{int(lo[e - 1])} .. {int(hi[e - 1])} there (delta {delta:g}); {bad.size} edges off in this row, "
                f"smallest delta that would pass: {hist_delta(hist, samples):.3g}")


# ---- the direct-row split of the FP32 nfft-4096 coherence pipeline (wct_fast.cu)
NFFT_FAST = 4096
DIRECT_B = 128          # kDirB: widest band a direct row may have (WTB_MC_DIRECT_B is clamped to it)
DIRECT_KC = 72          # kDirKc: largest Gaussian cut-off bin of a direct row


def row_bands(dt, dj, s0, J, f0=6.0):
    """Per scale row: (l0, B, kc) -- first bin and width of the daughter's support on the 4096-point
    grid (|a k - f0| <= 5.3, a = 2 pi s / (dt N)) and the time filter's cut-off bin floor(5.68 / a)."""
    out = []
    for j in range(J + 1):
        a = s0 * 2.0 ** (j * dj) / dt * 2.0 * math.pi / NFFT_FAST
        lo = max(math.ceil((f0 - 5.3) / a), 0)
        hi = min(math.floor((f0 + 5.3) / a), NFFT_FAST // 2 - 1)
        kc = min(math.floor(5.68 / a), NFFT_FAST // 2)
        out.append((lo, hi - lo + 1, kc))
    return out


def direct_split(dt, dj, s0, J, f0=6.0, bmax=DIRECT_B):
    """First row served by the direct kernel (J + 1: none).  Rows are taken from the largest scale
    down while the band is 1 .. bmax bins wide and kc <= DIRECT_KC; ``bmax`` is WTB_MC_DIRECT_B."""
    bmax = min(int(bmax), DIRECT_B)
    bands = row_bands(dt, dj, s0, J, f0)
    s_split = J + 1
    for q in range(J, -1, -1):
        _, B, kc = bands[q]
        if B < 1 or B > bmax or kc > DIRECT_KC or kc >= NFFT_FAST // 2:
            break
        s_split = q
    return s_split
