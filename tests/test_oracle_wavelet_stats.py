"""CPU: the float64 reference for the MODWT wavelet variance, covariance and cross-correlation
(oracle/wavelet_stats_oracle.py), and the host-side interval formulas of wavelet_transformer_b200.wavelet_stats."""

import numpy as np
import pytest
from scipy import stats as st

from oracle import modwt_oracle as mo
from oracle import wavelet_stats_oracle as wo


@pytest.mark.parametrize("filters", ["haar", "db4", "sym4"])
def test_boundary_rule(filters):
    """W_j[t] depends on x[t - L_j + 1 .. t] only for t >= L_j - 1; below that the wrap reaches x[n-1]."""
    L = wo.filter_length(filters)
    rng = np.random.default_rng(L)
    for J in range(1, 9):
        Lj = wo.width(J, L)
        n = Lj + 40
        x = rng.standard_normal(n)
        w = mo.modwt(x, filters, J)[J - 1]
        for t in (Lj - 1, Lj + 7, n - 1):
            x2 = x.copy()
            keep = np.zeros(n, bool)
            keep[t - Lj + 1:t + 1] = True
            x2[~keep] += rng.standard_normal((~keep).sum())
            assert mo.modwt(x2, filters, J)[J - 1][t] == pytest.approx(w[t], abs=1e-12), (filters, J, t)
        x3 = x.copy()
        x3[n - 1] += 1.0
        changed = np.abs(mo.modwt(x3, filters, J)[J - 1] - w) > 1e-12
        assert changed[:Lj - 1].any(), (filters, J)
        assert not changed[Lj - 1:n - 1].any()


def test_white_noise_mean_and_chi2_coverage():
    """E nu^2(j) = sigma^2 / 2^j for white noise; the eta_3 interval covers the truth at least at about its
    nominal rate (eta_3 = M_j / 2^j is a lower bound on the EDOF, so the interval is conservative)."""
    rng = np.random.default_rng(2000)
    n, J, sigma2 = 512, 5, 2.25
    truth = sigma2 / 2.0 ** np.arange(1, J + 1)
    est, covered = [], np.zeros(J)
    for _ in range(2000):
        v, _, _ = wo.stats(np.sqrt(sigma2) * rng.standard_normal(n), None, "sym4", J)
        lo, hi = wo.variance_ci(v, n, J, 8, 0.95)
        covered += (lo <= truth) & (truth <= hi)
        est.append(v)
    est = np.array(est)
    se = est.std(axis=0) / np.sqrt(len(est))
    assert np.all(np.abs(est.mean(axis=0) - truth) <= 4 * se), (est.mean(axis=0), truth)
    rate = covered / len(est)
    assert np.all(rate >= 0.94) and np.all(rate <= 0.998), rate


def test_identities():
    rng = np.random.default_rng(5)
    x, y = rng.standard_normal((2, 700))
    vx, vy, cxy = wo.stats(x, y, "sym4", 5, 12)
    _, _, cyx = wo.stats(y, x, "sym4", 5, 12)
    assert np.array_equal(cxy, cyx[:, ::-1])             # gamma_XY(j, tau) = gamma_YX(j, -tau), exactly
    vxx, _, cxx = wo.stats(x, x, "sym4", 5, 12)
    rho = wo.correlation(vxx, vxx, cxx)
    assert np.allclose(rho[:, 12], 1.0, rtol=0, atol=1e-14)
    assert np.array_equal(vxx, vx)
    v_alone, none_y, none_c = wo.stats(x, None, "sym4", 5)
    assert np.array_equal(v_alone, vx) and none_y is None and none_c is None


def test_delayed_copy_peaks_at_the_delay():
    """y cut from the same longer series d samples later (y[t] = x[t - d]): W_Y[t] = W_X[t - d] past the
    boundary, so the cross-correlation W_X[t] W_Y[t + tau] peaks at tau = d on the levels whose scale resolves
    the delay."""
    rng = np.random.default_rng(9)
    n, d, K, J = 1200, 3, 10, 4
    z = np.cumsum(rng.standard_normal(n + d)) * 0.1 + rng.standard_normal(n + d)
    x, y = z[d:], z[:n]
    vx, vy, c = wo.stats(x, y, "db4", J, K)
    rho = wo.correlation(vx, vy, c)
    for j in (1, 2, 3):
        assert np.argmax(rho[j - 1]) - K == d, j
        assert rho[j - 1, K + d] > 0.99


def test_ci_formulas_match_scipy():
    from wavelet_transformer_b200 import wavelet_stats as ws
    n, J, L = 1333, 9, 8
    rng = np.random.default_rng(1)
    nu2 = rng.uniform(0.1, 2.0, J)
    j = np.arange(1, J + 1)
    m = np.array([wo.m_count(n, k, L) for k in j])
    for level in (0.9, 0.95, 0.99):
        lo, hi = ws.variance_ci(nu2, m, j, level)
        rlo, rhi = wo.variance_ci(nu2, n, J, L, level)
        assert np.allclose(lo, rlo, rtol=1e-14) and np.allclose(hi, rhi, rtol=1e-14)
        p = (1 - level) / 2
        eta = max(m[0] / 2, 1.0)
        assert lo[0] == pytest.approx(eta * nu2[0] / st.chi2.ppf(1 - p, eta), rel=1e-14)
        rho = rng.uniform(-0.95, 0.95, (J, 5))
        clo, chi = ws.correlation_ci(rho, (m / 2.0 ** j)[:, None], level)
        rlo, rhi = wo.correlation_ci(rho, n, J, L, level)
        assert np.array_equal(np.isnan(clo), np.isnan(rlo))
        ok = ~np.isnan(rlo)
        assert np.allclose(clo[ok], rlo[ok], rtol=1e-14) and np.allclose(chi[ok], rhi[ok], rtol=1e-14)
    with pytest.raises(ValueError):
        ws.variance_ci(nu2, m, j, 1.0)


def test_nan_rules():
    """NaN where M_j <= 0 and for |tau| >= M_j; the correlation interval is NaN where N_j <= 3."""
    rng = np.random.default_rng(3)
    n, J, K = 60, 4, 40        # sym4: M_j = 53, 39, 11, -45
    x, y = rng.standard_normal((2, n))
    vx, vy, c = wo.stats(x, y, "sym4", J, K)
    M = [wo.m_count(n, j, 8) for j in range(1, J + 1)]
    assert M == [53, 39, 11, -45]
    assert np.isnan(vx[3]) and np.isnan(vy[3]) and np.isnan(c[3]).all()
    assert np.isfinite(vx[:3]).all()
    for j in range(3):
        lags = np.arange(-K, K + 1)
        assert np.array_equal(np.isnan(c[j]), np.abs(lags) >= M[j])
    lo, hi = wo.correlation_ci(wo.correlation(vx, vy, c), n, J, 8)
    assert np.isfinite(lo[0, K]) and np.isnan(lo[2]).all()        # N_3 = 11 / 8 <= 3
