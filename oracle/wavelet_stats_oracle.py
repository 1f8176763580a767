"""float64 NumPy reference for the MODWT wavelet variance, covariance and cross-correlation by level
(Percival & Walden 2000, ch. 8; Whitcher, Guttorp & Percival 2000).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Built on ``modwt_oracle.modwt``, which is pinned to the
reference's own MODWT through the committed goldens.  Definitions (include/wtb.h, wtb_modwt_wavelet_stats):

* ``L_j = (2^j - 1)(L - 1) + 1``; ``W_j[t]`` is free of the circular wrap exactly for ``t >= L_j - 1``;
  ``M_j = n - L_j + 1``.
* ``var(j) = (1/M_j) sum_{t=L_j-1}^{n-1} W_j[t]^2`` for j = 1..J.
* ``xcov(j, tau) = (1/M_j) sum_t W_{X,j}[t] W_{Y,j}[t+tau]`` over t with t, t+tau in [L_j-1, n-1].
* NaN where M_j <= 0 and for |tau| >= M_j.
"""

from __future__ import annotations

import numpy as np
from scipy import stats as st

from . import modwt_oracle


def filter_length(filters):
    h, _ = modwt_oracle._taps(filters)
    return h.size


def width(j, L):
    """L_j, the width of the level-j equivalent wavelet filter."""
    return (2 ** int(j) - 1) * (int(L) - 1) + 1


def m_count(n, j, L):
    """M_j, the number of level-j coefficients free of the circular wrap (may be <= 0)."""
    return int(n) - width(j, L) + 1


def stats(x, y, filters, J, K=0):
    """(var_x [J], var_y [J] or None, xcov [J, 2K+1] or None) of one series or pair, float64."""
    x = np.asarray(x, dtype=float)
    n = x.size
    L = filter_length(filters)
    wx = modwt_oracle.modwt(x, filters, J)[:J]
    wy = None if y is None else modwt_oracle.modwt(np.asarray(y, dtype=float), filters, J)[:J]
    var_x, var_y = np.full(J, np.nan), np.full(J, np.nan)
    xcov = np.full((J, 2 * K + 1), np.nan)
    for j in range(1, J + 1):
        M = m_count(n, j, L)
        if M <= 0:
            continue
        a = width(j, L) - 1
        var_x[j - 1] = np.dot(wx[j - 1, a:], wx[j - 1, a:]) / M
        if wy is None:
            continue
        var_y[j - 1] = np.dot(wy[j - 1, a:], wy[j - 1, a:]) / M
        for tau in range(-K, K + 1):
            if abs(tau) >= M:
                continue
            lo, hi = max(a, a - tau), min(n - 1, n - 1 - tau)   # t and t + tau in [a, n-1]
            xcov[j - 1, tau + K] = np.dot(wx[j - 1, lo:hi + 1], wy[j - 1, lo + tau:hi + tau + 1]) / M
    if wy is None:
        return var_x, None, None
    return var_x, var_y, xcov


def correlation(var_x, var_y, xcov):
    return xcov / np.sqrt(var_x * var_y)[..., None]


def variance_ci(nu2, n, J, L, level=0.95):
    """P&W eq. 313c with EDOF eta_3 = max(M_j / 2^j, 1), by a direct scipy evaluation."""
    p = (1 - level) / 2
    lo, hi = np.empty(J), np.empty(J)
    for j in range(1, J + 1):
        eta = max(m_count(n, j, L) / 2 ** j, 1.0)
        lo[j - 1] = eta * nu2[j - 1] / st.chi2.ppf(1 - p, eta)
        hi[j - 1] = eta * nu2[j - 1] / st.chi2.ppf(p, eta)
    return lo, hi


def correlation_ci(rho, n, J, L, level=0.95):
    """Fisher z with N_j = M_j / 2^j at every lag of rho [J, ...]; NaN where N_j <= 3."""
    p = (1 - level) / 2
    rho = np.asarray(rho, dtype=float)
    lo, hi = np.full(rho.shape, np.nan), np.full(rho.shape, np.nan)
    for j in range(1, J + 1):
        nh = m_count(n, j, L) / 2 ** j
        if nh <= 3:
            continue
        half = st.norm.ppf(1 - p) / np.sqrt(nh - 3)
        lo[j - 1] = np.tanh(np.arctanh(rho[j - 1]) - half)
        hi[j - 1] = np.tanh(np.arctanh(rho[j - 1]) + half)
    return lo, hi
