"""MODWT wavelet variance, covariance and cross-correlation by level, with confidence intervals (Percival & Walden
2000, ch. 8; Whitcher, Guttorp & Percival 2000).

How much variance does each time scale carry, and how correlated are two series at each scale and lag?  The MODWT
of ``modwt`` (``h~ = dec_hi / sqrt 2``, ``g~ = dec_lo / sqrt 2``) is taken on the device and reduced there over the
coefficients free of the circular wrap (``wtb_modwt_wavelet_stats``); only the per-level numbers come back.  For a
filter of length L, level j has ``L_j = (2^j - 1)(L - 1) + 1`` and ``M_j = n - L_j + 1`` such coefficients
(``t >= L_j - 1``):

* ``variance[j] = (1/M_j) sum_t W_{X,j}[t]^2``
* ``xcov[j, tau] = (1/M_j) sum_t W_{X,j}[t] W_{Y,j}[t + tau]`` over the t with t and t + tau both free of the wrap,
  the biased estimator (divisor M_j at every lag); lag 0 is the wavelet covariance
* ``xcorr[j, tau] = xcov[j, tau] / sqrt(var_x[j] var_y[j])``

NaN where M_j <= 0 and for lags |tau| >= M_j.  Confidence intervals, with ``p = (1 - significance_level) / 2``:

* variance (P&W eq. 313c, EDOF eta_3): ``[eta nu^2 / chi2_eta(1 - p), eta nu^2 / chi2_eta(p)]``,
  ``eta = max(M_j / 2^j, 1)``
* correlation, at every lag (Fisher's z): ``tanh(atanh rho -+ Phi^-1(1 - p) / sqrt(N_j - 3))`` with
  ``N_j = M_j / 2^j``; NaN where ``N_j <= 3``.
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import numpy.typing as npt

from . import _shim
from . import pywt_compat as pywt


def _bank(wavelet):
    w = wavelet if hasattr(wavelet, "dec_lo") else pywt.Wavelet(wavelet)
    return np.asarray(w.dec_lo, dtype=float), np.asarray(w.dec_hi, dtype=float)


def _levels(n, L, levels, dt):
    j = np.arange(1, int(levels) + 1)
    m = n - ((2 ** j - 1) * (L - 1) + 1) + 1
    return j, 2.0 ** (j - 1) * dt, m


def _series(x, name):
    a = np.asarray(x, dtype=float)
    if a.ndim not in (1, 2) or a.shape[-1] < 1:
        raise ValueError(f"{name} must be [n] or [batch, n]")
    return a


def _p(significance_level):
    if not 0.0 < significance_level < 1.0:
        raise ValueError("significance_level must lie in (0, 1)")
    return (1.0 - significance_level) / 2.0


def variance_ci(nu2, m, level_index, significance_level=0.95):
    """Chi-square interval of a wavelet variance with EDOF eta = max(M_j / 2^j, 1); ``level_index`` is j."""
    from scipy import stats  # host-side closed form only
    p = _p(significance_level)
    eta = np.maximum(np.asarray(m, dtype=float) / 2.0 ** np.asarray(level_index, dtype=float), 1.0)
    nu2 = np.asarray(nu2, dtype=float)
    return eta * nu2 / stats.chi2.ppf(1.0 - p, eta), eta * nu2 / stats.chi2.ppf(p, eta)


def correlation_ci(rho, n_hat, significance_level=0.95):
    """Fisher-z interval of a wavelet correlation with N_j = M_j / 2^j (broadcast against rho); NaN where
    N_j <= 3."""
    from scipy import stats
    z = stats.norm.ppf(1.0 - _p(significance_level))
    n_hat = np.asarray(n_hat, dtype=float)
    with np.errstate(invalid="ignore", divide="ignore"):
        half = np.where(n_hat > 3.0, z / np.sqrt(np.where(n_hat > 3.0, n_hat - 3.0, 1.0)), np.nan)
        at = np.arctanh(np.asarray(rho, dtype=float))
        return np.tanh(at - half), np.tanh(at + half)


@dataclass
class WaveletVariance:
    """Per-level MODWT wavelet variance of one series ([J]) or a batch ([batch, J])."""

    level: npt.NDArray          # [J] j = 1..J
    scale: npt.NDArray          # [J] 2^(j-1) dt
    m: npt.NDArray              # [J] M_j, coefficients free of the circular wrap (<= 0: none)
    edof: npt.NDArray           # [J] eta = max(M_j / 2^j, 1)
    variance: npt.NDArray       # [..., J]
    ci_low: npt.NDArray         # [..., J]
    ci_high: npt.NDArray        # [..., J]
    significance_level: float


@dataclass
class WaveletCorrelation:
    """Per-level MODWT wavelet covariance and correlation of two series, at lag 0 and at every lag -K..K."""

    level: npt.NDArray          # [J]
    scale: npt.NDArray          # [J] 2^(j-1) dt
    m: npt.NDArray              # [J] M_j
    edof: npt.NDArray           # [J] N_j = M_j / 2^j, the sample size of the correlation interval
    var_x: npt.NDArray          # [..., J]
    var_y: npt.NDArray          # [..., J]
    covariance: npt.NDArray     # [..., J] lag 0
    correlation: npt.NDArray    # [..., J] lag 0
    ci_low: npt.NDArray         # [..., J] lag 0
    ci_high: npt.NDArray        # [..., J]
    lags: npt.NDArray           # [2K+1] -K..K
    xcov: npt.NDArray           # [..., J, 2K+1]
    xcorr: npt.NDArray          # [..., J, 2K+1]
    xcorr_ci_low: npt.NDArray   # [..., J, 2K+1]
    xcorr_ci_high: npt.NDArray  # [..., J, 2K+1]
    significance_level: float


def wavelet_variance(x, wavelet="sym4", levels=6, significance_level=0.95, dt=1.0) -> WaveletVariance:
    """MODWT wavelet variance of ``x`` ([n] or [batch, n]) at levels 1..``levels`` with its chi-square interval.
    Precision follows ``set_precision``; the outputs are float64."""
    x = _series(x, "x")
    g, h = _bank(wavelet)
    var, _, _ = _shim.modwt_wavelet_stats(x, None, g, h, int(levels))
    j, scale, m = _levels(x.shape[-1], g.size, levels, dt)
    lo, hi = variance_ci(var, m, j, significance_level)
    return WaveletVariance(j, scale, m, np.maximum(m / 2.0 ** j, 1.0), var, lo, hi, float(significance_level))


def wavelet_correlation(x, y, wavelet="sym4", levels=6, max_lag=0, significance_level=0.95,
                        dt=1.0) -> WaveletCorrelation:
    """MODWT wavelet covariance and correlation of ``x`` and ``y`` ([n] or [batch, n], same shape) at levels
    1..``levels``, and their cross-covariance and cross-correlation at lags -``max_lag``..``max_lag`` (``y`` leads
    by tau: ``W_X[t] W_Y[t + tau]``), with Fisher-z intervals.  Precision follows ``set_precision``; the outputs
    are float64."""
    x, y = _series(x, "x"), _series(y, "y")
    if x.shape != y.shape:
        raise ValueError("x and y must have the same shape")
    g, h = _bank(wavelet)
    var_x, var_y, xcov = _shim.modwt_wavelet_stats(x, y, g, h, int(levels), int(max_lag))
    j, scale, m = _levels(x.shape[-1], g.size, levels, dt)
    n_hat = m / 2.0 ** j
    with np.errstate(invalid="ignore", divide="ignore"):
        xcorr = xcov / np.sqrt(var_x * var_y)[..., None]
    lo, hi = correlation_ci(xcorr, n_hat[:, None], significance_level)
    K = int(max_lag)
    return WaveletCorrelation(j, scale, m, n_hat, var_x, var_y, xcov[..., K], xcorr[..., K], lo[..., K], hi[..., K],
                              np.arange(-K, K + 1), xcov, xcorr, lo, hi, float(significance_level))
