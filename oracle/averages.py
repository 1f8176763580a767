"""Time- and scale-averaged wavelet spectra -- TEST INFRASTRUCTURE ONLY.

* ``significance``: pycwt.significance with the time-averaged (sigma_test=1, Torrence & Compo 1998
  eq. 23) and scale-averaged (sigma_test=2, eqs. 25-28) branches the pycwt sample uses next to the
  sigma_test=0 branch of ``pycwt_oracle.significance``, which serves sigma_test=0 unchanged and forms
  the red-noise spectrum all three branches start from.  The pycwt side of both branches is RECALLED,
  not checked against pycwt itself, and restated from the paper below.
* ``averages_gate``: the per-row gate of ``cwt_rows.row_gate`` carried through the two reductions of
  wtb_cwt_averages.
"""

import math

import numpy as np

from oracle.cwt_rows import ROW_FLOOR
from oracle.pycwt_oracle import Morlet
from oracle.pycwt_oracle import significance as _significance_0


def significance(signal, dt, scales, sigma_test=0, alpha=None, significance_level=0.95, dof=-1,
                 wavelet=None):
    """pycwt.significance for sigma_test 0, 1 and 2; returns (signif, fft_theor).

    sigma_test=1 [RECALLED]: the time average over n_a points (``dof``, a scalar or one value per scale,
    taken as at least 1) has nu = dofmin sqrt(1 + (n_a dt / (gamma s))^2) degrees of freedom, at least
    dofmin (eq. 23); signif = fft_theor chi2_nu(level) / nu.

    sigma_test=2 [RECALLED]: the average over the scales s1 <= s_j <= s2 (``dof = [s1, s2]``):
    S_avg = (sum_j 1/s_j)^-1 (eq. 25), S_mid = sqrt(s1 s2) (pycwt's power-of-two mid point),
    nu = dofmin n_a S_avg / S_mid sqrt(1 + (n_a dj / dj0)^2) (eq. 28), P = S_avg sum_j P_j / s_j
    (eq. 27) and signif = dj dt / (C_delta S_avg) P chi2_nu(level) / nu (eq. 26), with dj = log2(s_1 / s_0)
    of the scale axis; returns (signif, P).  pycwt raises a bare Exception for a ``dof`` that is not a pair
    and ValueError for an undefined C_delta or an empty band."""
    wavelet = wavelet or Morlet()
    fft_theor = _significance_0(signal, dt, scales, 0, alpha, significance_level, wavelet=wavelet)[1]
    scales = np.asarray(scales, dtype=float)
    if sigma_test == 0:
        return _significance_0(signal, dt, scales, 0, alpha, significance_level, dof, wavelet)
    from scipy.stats import chi2
    if sigma_test == 1:
        na = np.broadcast_to(np.asarray(dof, dtype=float), scales.shape)
        na = np.where(na < 1, 1.0, na)
        nu = wavelet.dofmin * np.sqrt(1 + (na * dt / (wavelet.gamma * scales)) ** 2)
        nu = np.where(nu < wavelet.dofmin, wavelet.dofmin, nu)
        return fft_theor * chi2.ppf(significance_level, nu) / nu, fft_theor
    if sigma_test != 2:
        raise NotImplementedError("oracle covers sigma_test=0, 1 and 2")
    if np.ndim(dof) != 1 or len(dof) != 2:
        raise Exception("DOF must be set to [s1, s2], the range of scale-averages")
    if wavelet.cdelta == -1:
        raise ValueError("Cdelta and dj0 not defined for this mother wavelet")
    s1, s2 = float(dof[0]), float(dof[1])
    inside = (scales >= s1) & (scales <= s2)
    band = scales[inside]
    if band.size == 0:
        raise ValueError(f"No valid scales between {s1} and {s2}.")
    dj = math.log2(scales[1] / scales[0])
    s_avg = 1.0 / np.sum(1.0 / band)
    nu = wavelet.dofmin * band.size * s_avg / math.sqrt(s1 * s2) * math.sqrt(1 + (band.size * dj / wavelet.deltaj0) ** 2)
    p_avg = s_avg * np.sum(fft_theor[inside] / band)
    return dj * dt / (wavelet.cdelta * s_avg) * p_avg * chi2.ppf(significance_level, nu) / nu, p_avg


def averages_gate(got_global, got_band, W_ref, scales, band, factor, tol, resolved):
    """The row gate carried through the two reductions of wtb_cwt_averages.  Each power entry may be off by
    tol (|b| + scale_row) (``cwt_rows.row_gate`` on b = |W_ref|^2, with the plane maximum in place of
    scale_row on the rows that are not ``resolved``), so
        |d global_s| <= tol (mean_t |b_s| + scale_row_s),
        |d band_t|   <= factor sum_{s=lo..hi} tol (|b_st| + scale_row_s) / s_s.
    got_global [S] and got_band [n0] may be None; band = (lo, hi), inclusive.  Returns the worst ratio to
    the bound and where it sits: ("global", s) or ("band", t)."""
    b = np.abs(np.asarray(W_ref)) ** 2
    mag_max = b.max()
    scale_row = np.where(resolved, np.maximum(b.max(axis=1), ROW_FLOOR * mag_max), mag_max)
    worst, where = 0.0, None
    if got_global is not None:
        ref = b.mean(axis=1)
        ratio = np.abs(np.asarray(got_global, dtype=np.float64) - ref) / (tol * (ref + scale_row) + 1e-300)
        worst, where = float(ratio.max()), ("global", int(np.argmax(ratio)))
    if got_band is not None:
        lo, hi = band
        inv = 1.0 / np.asarray(scales, dtype=np.float64)[lo:hi + 1, None]
        ref = factor * (b[lo:hi + 1] * inv).sum(axis=0)
        bound = abs(factor) * tol * ((b[lo:hi + 1] + scale_row[lo:hi + 1, None]) * inv).sum(axis=0)
        ratio = np.abs(np.asarray(got_band, dtype=np.float64) - ref) / (bound + 1e-300)
        if ratio.max() > worst:
            worst, where = float(ratio.max()), ("band", int(np.argmax(ratio)))
    return worst, where
