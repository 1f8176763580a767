"""Partial and multiple wavelet coherence of three series (Aguiar-Conraria & Soares 2014; Ng & Chan 2012).

How coherent are y and x1 once a third series x2 is accounted for, and how much of y do x1 and x2 explain
together?  Both come from the 3x3 matrix of smoothed cross spectra S_ij = smooth(W_i conj(W_j) / s) that
pycwt's ``wct`` builds for two series (Morlet CWT, Gaussian in time, boxcar over scales); every transform and
ratio runs on the device (``wtb_partial_wct``).
"""

from __future__ import annotations

import numpy as np

from . import _shim

F0 = 6.0


def partial_wct(y, x1, x2, dt, dj=1 / 12, s0=-1, J=-1, normalize=True):
    """Partial wavelet coherence of y and x1 given x2, its phase, and the multiple wavelet coherence of y on
    (x1, x2), with a Morlet(6) mother.

    Returns ``(pwc, pphase, mwc, coi, freq, scales)``: three float64 [S, n0] planes, then the cone of
    influence [n0], Fourier frequencies [S] and scales [S] as pycwt's ``wct`` forms them.

    * ``pwc = |S_y1 S_22 - S_y2 conj(S_12)|^2 / ((S_yy S_22 - |S_y2|^2) (S_11 S_22 - |S_12|^2))``
    * ``pphase = angle(S_y1 S_22 - S_y2 conj(S_12))``
    * ``mwc = (|S_y1|^2 S_22 + |S_y2|^2 S_11 - 2 Re(S_y1 conj(S_y2) S_12)) / (S_yy (S_11 S_22 - |S_12|^2))``

    With ``normalize`` each series becomes ``(v - v.mean()) / v.std()`` first, as in ``wct(normalize=True)``.
    Precision and FFT padding follow ``set_precision`` and ``set_fft_padding``.  0/0 gives NaN, as in pycwt's
    coherence; nothing is clamped."""
    series = [np.asarray(v, dtype=float) for v in (y, x1, x2)]
    if series[0].ndim != 1 or not series[0].shape == series[1].shape == series[2].shape:
        raise ValueError("y, x1 and x2 must be 1-D series of the same length")
    if normalize:
        series = [(v - v.mean()) / v.std() for v in series]
    Jr, scales, freq, coi = _shim.cwt_axes(series[0].size, dt, dj, s0, J, F0)
    pwc, pphase, mwc = _shim.partial_wct(*series, dt, dj, s0, Jr, F0)
    return (np.asarray(pwc, dtype=float), np.asarray(pphase, dtype=float), np.asarray(mwc, dtype=float), coi, freq,
            scales)
