"""float64 reference of partial and multiple wavelet coherence (Aguiar-Conraria & Soares 2014; Ng & Chan 2012).

TEST INFRASTRUCTURE ONLY.  The smoothed spectra S_ij = smooth(W_i conj(W_j) / s) are those of
``pycwt_oracle.wct`` (``cwt`` and ``Morlet.smooth``, both padding rules).  PWC and MWC are formed twice:

* ``closed_forms``: the expressions of ``wtb_partial_wct`` (include/wtb.h);
* ``inverse_forms``: from P = S^-1 of the 3x3 Hermitian matrix S at every point, independently:
  ``PWC = |P_y1|^2 / (P_yy P_11)`` and ``MWC = 1 - 1 / (S_yy P_yy)``.

The partial phase is defined by the closed form, ``angle(S_y1 S_22 - S_y2 conj(S_12))``.
"""

from __future__ import annotations

import numpy as np
from scipy.signal import lfilter

from . import pycwt_oracle as po


INPUTS = ("independent", "correlated", "built")


def triple(kind, n0, seed, a=0.7):
    """Test series (y, x1, x2), each normalised, from AR(1) processes with coefficient a:
    'independent': three independent series; 'correlated': x2 = 0.6 x1 + noise, y independent;
    'built': x2 = 0.6 x1 + noise and y = 0.7 x1 + 0.5 x2 + noise."""
    rng = np.random.default_rng(seed)
    ar = lambda: lfilter([1.0], [1.0, -a], rng.standard_normal(n0 + 500))[500:]
    y, x1, x2 = ar(), ar(), ar()
    if kind in ("correlated", "built"):
        x2 = 0.6 * x1 + 0.8 * x2
    if kind == "built":
        y = 0.7 * x1 + 0.5 * x2 + 0.5 * y
    elif kind != "independent" and kind != "correlated":
        raise ValueError(kind)
    return tuple((v - v.mean()) / v.std() for v in (y, x1, x2))


def spectra(y, x1, x2, dt, dj, s0, J, pad_pow2=True, f0=6.0):
    """Smoothed spectra of three already-normalised series: dict with Syy, S11, S22 (real) and Sy1, Sy2, S12
    (complex), each [S, n0], plus the scales."""
    wavelet = po.Morlet(f0)
    W = [po.cwt(v, dt, dj, s0, J, wavelet, pad_pow2)[0] for v in (y, x1, x2)]
    sj = po.cwt_axes(len(y), dt, dj, s0, J, wavelet)[0]
    s = sj[:, None]
    sm = lambda a: wavelet.smooth(a / s, dt, dj, sj, pad_pow2)
    return {"Syy": sm(np.abs(W[0]) ** 2), "S11": sm(np.abs(W[1]) ** 2), "S22": sm(np.abs(W[2]) ** 2),
            "Sy1": sm(W[0] * W[1].conj()), "Sy2": sm(W[0] * W[2].conj()), "S12": sm(W[1] * W[2].conj()),
            "scales": sj}


def closed_forms(sp):
    """(pwc, pphase, mwc) from the closed forms."""
    Syy, S11, S22, Sy1, Sy2, S12 = (sp[k] for k in ("Syy", "S11", "S22", "Sy1", "Sy2", "S12"))
    num = Sy1 * S22 - Sy2 * S12.conj()
    d12 = S11 * S22 - np.abs(S12) ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        pwc = np.abs(num) ** 2 / ((Syy * S22 - np.abs(Sy2) ** 2) * d12)
        mwc = (np.abs(Sy1) ** 2 * S22 + np.abs(Sy2) ** 2 * S11 - 2 * np.real(Sy1 * Sy2.conj() * S12)) / (Syy * d12)
    return pwc, np.angle(num), mwc


def matrix(sp):
    """The Hermitian 3x3 smoothed spectral matrix at every point: [S, n0, 3, 3], order (y, x1, x2)."""
    Syy, S11, S22, Sy1, Sy2, S12 = (sp[k] for k in ("Syy", "S11", "S22", "Sy1", "Sy2", "S12"))
    M = np.empty(Syy.shape + (3, 3), dtype=complex)
    M[..., 0, 0], M[..., 1, 1], M[..., 2, 2] = Syy, S11, S22
    M[..., 0, 1], M[..., 0, 2], M[..., 1, 2] = Sy1, Sy2, S12
    M[..., 1, 0], M[..., 2, 0], M[..., 2, 1] = Sy1.conj(), Sy2.conj(), S12.conj()
    return M


def inverse_forms(sp):
    """(pwc, mwc) from the inverse of the spectral matrix; NaN where it is singular in floating point (the
    largest scales of a short un-padded series can make the three rows proportional to rounding)."""
    M = matrix(sp)
    sign, _ = np.linalg.slogdet(M)
    ok = sign != 0
    P = np.full(M.shape, np.nan, dtype=complex)
    P[ok] = np.linalg.inv(M[ok])
    pwc = np.abs(P[..., 0, 1]) ** 2 / (P[..., 0, 0].real * P[..., 1, 1].real)
    mwc = 1.0 - 1.0 / (sp["Syy"] * P[..., 0, 0].real)
    return pwc, mwc


def rho2(sp, a, b):
    """Squared ordinary coherence |S_ab|^2 / (S_aa S_bb) of two of 'y', '1', '2'."""
    key = {("y", "1"): "Sy1", ("y", "2"): "Sy2", ("1", "2"): "S12"}[(a, b)]
    auto = {"y": "Syy", "1": "S11", "2": "S22"}
    return np.abs(sp[key]) ** 2 / (sp[auto[a]] * sp[auto[b]])


def conditioning(sp):
    """(kappa_pwc, kappa_mwc): 1 / ((1 - |rho_y2|^2)(1 - |rho_12|^2)) and 1 / (1 - |rho_12|^2), the
    amplification of relative errors in the spectra by the two ratios."""
    r12 = rho2(sp, "1", "2")
    return 1.0 / ((1.0 - rho2(sp, "y", "2")) * (1.0 - r12)), 1.0 / (1.0 - r12)


def smoothing_kernel(n0, dt, scales, pad_pow2=True):
    """The time kernel of Morlet.smooth per scale row: the inverse DFT of the Gaussian at the padded length,
    [S, npad] real.  Where it is non-negative the smoothed matrix of a row is positive semidefinite."""
    npad = po._pow2(n0) if pad_pow2 else n0
    k = 2 * np.pi * np.fft.fftfreq(npad)
    gauss = np.exp(-0.5 * (np.asarray(scales) / dt)[:, None] ** 2 * k ** 2)
    return np.fft.ifft(gauss, axis=1).real


def partial_wct(y, x1, x2, dt, dj=1 / 12, s0=-1, J=-1, normalize=True, pad_pow2=True):
    """(pwc, pphase, mwc, coi, freq, scales) of the public ``partial_wct``."""
    series = [np.asarray(v, dtype=float) for v in (y, x1, x2)]
    if normalize:
        series = [(v - v.mean()) / v.std() for v in series]
    wavelet = po.Morlet()
    if s0 == -1:
        s0 = 2 * dt / wavelet.flambda()
    if J == -1:
        J = int(np.round(np.log2(series[0].size * dt / s0) / dj))
    sp = spectra(*series, dt, dj, s0, J, pad_pow2)
    sj, freq, coi = po.cwt_axes(series[0].size, dt, dj, s0, J, wavelet)
    pwc, pphase, mwc = closed_forms(sp)
    return pwc, pphase, mwc, coi, freq, sj
