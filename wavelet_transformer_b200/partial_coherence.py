"""Partial and multiple wavelet coherence of three series (Aguiar-Conraria & Soares 2014; Ng & Chan 2012).

How coherent are y and x1 once a third series x2 is accounted for, and how much of y do x1 and x2 explain
together?  Both come from the 3x3 matrix of smoothed cross spectra S_ij = smooth(W_i conj(W_j) / s) that
pycwt's ``wct`` builds for two series (Morlet CWT, Gaussian in time, boxcar over scales); every transform and
ratio runs on the device (``wtb_partial_wct``).
"""

from __future__ import annotations

import os

import numpy as np

from . import _shim
from .pycwt_compat import ar1

F0 = 6.0


def partial_wct(y, x1, x2, dt, dj=1 / 12, s0=-1, J=-1, normalize=True, sig=False, significance_level=0.95,
                **mc_kwargs):
    """Partial wavelet coherence of y and x1 given x2, its phase, and the multiple wavelet coherence of y on
    (x1, x2), with a Morlet(6) mother.

    Returns ``(pwc, pphase, mwc, coi, freq, scales)``: three float64 [S, n0] planes, then the cone of
    influence [n0], Fourier frequencies [S] and scales [S] as pycwt's ``wct`` forms them.  With ``sig=True``
    the 95th-percentile (``significance_level``) thresholds ``sig_pwc, sig_mwc`` [S] of
    ``partial_wct_significance`` follow, for the AR(1) coefficients ``ar1`` estimates from the three series
    (its ``Warning`` for an unbounded estimate propagates); ``mc_kwargs`` go to ``partial_wct_significance``.

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
    out = (np.asarray(pwc, dtype=float), np.asarray(pphase, dtype=float), np.asarray(mwc, dtype=float), coi, freq,
           scales)
    if not sig:
        return out
    ay, a1, a2 = (ar1(v)[0] for v in series)
    return out + partial_wct_significance(ay, a1, a2, dt, dj, s0, Jr, significance_level=significance_level,
                                          **mc_kwargs)


def partial_wct_significance(ay, a1, a2, dt, dj, s0, J, significance_level=0.95, mc_count=300, seed=0, white=False,
                             surrogates=None, n_gpus=None, precision=None):
    """Monte-Carlo significance of partial and multiple wavelet coherence (Ng & Chan 2012): ``(sig_pwc,
    sig_mwc)``, one threshold per scale [J+1].

    ``mc_count`` triples of independent AR(1) series with coefficients ``(ay, a1, a2)`` (white noise with
    ``white``) of pycwt's ``wct_significance`` length are transformed on the device; the partial and multiple
    coherence inside the reliable region of each scale below pycwt's ``maxscale`` fill one histogram per scale,
    and its ``significance_level`` percentile is the threshold (NaN for larger scales that have reliable points,
    0 for those without).  ``J`` must be resolved (>= 0); ``s0 = -1`` means ``2 dt / flambda``.  The realisations
    are drawn from Philox streams keyed by ``seed`` and the global realisation index and spread over every GPU
    the library drives (``n_gpus`` here, or ``_shim.init_multi`` / ``WTB_GPUS`` beforehand): the thresholds do not
    depend on the number of GPUs.  ``surrogates`` ([mc_count, 3, nsurr]) injects ready-made series.

    ``precision``: "fp32" | "fp64" | None.  None keeps the global precision when surrogates are injected and runs
    FP32 with the device RNG, as ``pycwt_compat.wct_significance`` does (``WTB_MC_PRECISION=fp64`` restores the
    global setting).  Series past one CTA per transform (about 1365 samples in FP32 and 680 in FP64 with
    s0 = 2 dt, padded) are refused."""
    if precision is None and surrogates is None and os.environ.get("WTB_MC_PRECISION", "fp32").lower() != "fp64":
        precision = "fp32"
    f64 = None if precision is None else {"fp32": False, "fp64": True}[precision.lower()]
    if n_gpus is not None and int(n_gpus) != _shim.gpu_count():
        _shim.init_multi(int(n_gpus))
    return _shim.partial_wct_significance(ay, a1, a2, dt, dj, s0, int(J), F0, level=significance_level,
                                          mc_count=mc_count, seed=seed, surrogates=surrogates, f64=f64, white=white)
