"""Long-series cross spectra and coherence (wct_long.cu) -- TEST INFRASTRUCTURE ONLY.

* ``wct_rows``: chosen scale rows of pycwt's WCT, its phase and W12 in float64.  Only the rows each row's
  scale boxcar reads are built (``cwt_long.cwt_rows``, then ``Morlet.smooth``'s time filter per row and the
  zero-filled 'same' boxcar), so a test at nfft = 2^22 never holds the whole [S, n0] plane;
* a replica of the host rules of the long coherence path: which transforms serve a ``wct_device`` call
  (``route``), its wave rule (``wave_rows``), its launches in the plane, W12-only and histogram modes
  (``launches``) and the chunk rule of ``wtb_xwt_wct`` (``xwt_chunk_rows``).
"""

import numpy as np

from oracle import cwt_long as cl
from oracle import pycwt_oracle as po

WAVE_BYTES = cl.WAVE_BYTES
XWT_BUDGET = 1 << 30
MODES = ("plane", "w12", "hist")


def boxcar(dj, wavelet=None):
    """Morlet.smooth's scale window: (weights, up) with out[i] = sum_k w[k] T[i + up - k], zero outside."""
    wavelet = wavelet or po.Morlet()
    w = po.rect(int(np.round(wavelet.deltaj0 / dj * 2)), normalize=True)
    return w, (w.size - 1) // 2


def wct_rows(y1, y2, dt, dj, s0, J, rows, wavelet=None, normalize=True, nfft=None, spectra=False):
    """(WCT, phase, W12) [len(rows), n0] of ``po.wct(y1, y2, dt, dj, s0, J, sig=False)`` (and pycwt.xwt's W12
    and angle) for the chosen scale rows, in float64; with ``spectra`` also the smoothed S1, S2 of those rows."""
    wavelet = wavelet or po.Morlet()
    y1 = np.asarray(y1, dtype=float)
    y2 = np.asarray(y2, dtype=float)
    n0 = y1.size
    if s0 == -1:
        s0 = 2 * dt / wavelet.flambda()
    if J == -1:
        J = int(np.round(np.log2(n0 * dt / s0) / dj))
    if normalize:
        y1, y2 = po._normalise(y1), po._normalise(y2)
    sj, _, _ = po.cwt_axes(n0, dt, dj, s0, J, wavelet)
    S = sj.size
    rows = np.asarray(rows, dtype=int)
    w, up = boxcar(dj, wavelet)
    need = sorted({r + up - k for r in rows for k in range(w.size) if 0 <= r + up - k < S})
    W1 = cl.cwt_rows(y1, dt, dj, s0, J, wavelet, need, nfft)
    W2 = cl.cwt_rows(y2, dt, dj, s0, J, wavelet, need, nfft)
    npad = nfft or po._pow2(n0)
    k = 2 * np.pi * np.fft.fftfreq(npad)
    T = {}
    for i, r in enumerate(need):
        g = np.exp(-0.5 * (sj[r] / dt) ** 2 * k ** 2)
        tf = lambda v: np.fft.ifft(g * np.fft.fft(v, n=npad))[:n0]
        T[r] = (tf(np.abs(W1[i]) ** 2 / sj[r]).real, tf(np.abs(W2[i]) ** 2 / sj[r]).real,
                tf(W1[i] * W2[i].conj() / sj[r]))
    wct = np.empty((rows.size, n0))
    w12 = np.empty((rows.size, n0), dtype=np.complex128)
    S1 = np.empty((rows.size, n0))
    S2 = np.empty((rows.size, n0))
    for j, r in enumerate(rows):
        s1 = np.zeros(n0)
        s2 = np.zeros(n0)
        s12 = np.zeros(n0, dtype=np.complex128)
        for kk in range(w.size):
            q = r + up - kk
            if 0 <= q < S:
                s1 += w[kk] * T[q][0]
                s2 += w[kk] * T[q][1]
                s12 += w[kk] * T[q][2]
        wct[j] = np.abs(s12) ** 2 / (s1 * s2)
        S1[j], S2[j] = s1, s2
        i = need.index(r)
        w12[j] = W1[i] * W2[i].conj()
    if spectra:
        return wct, np.angle(w12), w12, S1, S2
    return wct, np.angle(w12), w12


# ---- host rules ------------------------------------------------------------------------------------------
def route(nfft, f64):
    """'long', 'refused' (a power of two past 2^22) or 'generic' (every length wct_device served before)."""
    return cl.route(nfft, f64)


def wave_rows(nfft, f64, rows, smooth=True):
    """wct_long_wave_rows: (pair, scale) rows whose four (smoothed) or two N-point complex fields fit 64 MiB,
    at least 1, at most ``rows``."""
    per = (4 if smooth else 2) * 2 * cl._elem(f64) * nfft
    return min(rows, max(1, WAVE_BYTES // per))


def launches(nfft, f64, pairs, S, mode):
    """Kernel launches of one long-path wct_device call: two per forward wave of the 2 pairs series, five
    per row wave (two without smoothing), and the scale boxcar / coherence kernel when smoothed."""
    assert mode in MODES
    smooth = mode != "w12"
    fw = -(-(2 * pairs) // cl.wave_rows(nfft, f64, 2 * pairs))
    rw = -(-(pairs * S) // wave_rows(nfft, f64, pairs * S, smooth))
    return 2 * fw + (5 if smooth else 2) * rw + (1 if smooth else 0)


def pair_bytes(n0, nfft, S, f64):
    """wct.cu's pair_bytes: X^ of both series and an [S, nfft] vec4 plane (what a chunk rule counts)."""
    e = cl._elem(f64)
    return 2 * e * 2 * nfft + 4 * e * S * nfft


def xwt_chunk_rows(batch, n0, nfft, S, f64, wct=True, phase=True, w12=False):
    """Pairs per wtb_xwt_wct chunk: staging and intermediates within 1 GiB, at least one."""
    e = cl._elem(f64)
    plane = S * n0
    per_pair = e * (2 * n0 + (plane if wct else 0) + (plane if phase else 0) + (2 * plane if w12 else 0))
    return max(1, min(batch, XWT_BUDGET // (per_pair + pair_bytes(n0, nfft, S, f64))))


def xwt_launches(batch, n0, nfft, S, f64, wct=True, phase=True, w12=False):
    """Kernel launches of a long-path wtb_xwt_wct call over host buffers on one device."""
    rows = xwt_chunk_rows(batch, n0, nfft, S, f64, wct, phase, w12)
    mode = "plane" if wct else "w12"
    total, b0 = 0, 0
    while b0 < batch:
        nb = min(rows, batch - b0)
        total += launches(nfft, f64, nb, S, mode)
        b0 += nb
    return total


def mc_nfft(nsurr):
    """The padded transform length of a Monte-Carlo call (pycwt pads to the next power of two)."""
    return po._pow2(nsurr)
