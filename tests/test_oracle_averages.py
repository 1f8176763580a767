"""CPU checks of the averaged-spectrum pieces that need no GPU: pycwt_compat.significance for the time-
(sigma_test=1) and scale-averaged (sigma_test=2) tests against the float64 oracle, the error cases of
both, the averages gate of oracle/averages.py, and the argument checks of _shim.cwt_averages."""

import numpy as np
import pytest
from scipy.signal import lfilter

from oracle import averages as oa
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

DT = 1 / 12
MOTHERS = [("morlet", 6), ("paul", 4), ("dog", 2), ("dog", 6)]


def _pair(name, param):
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    if name == "morlet":
        return wavelet.Morlet(param), po.Morlet(param)
    if name == "paul":
        return wavelet.Paul(param), po.Paul(param)
    return wavelet.DOG(param), po.DOG(param)


def _scales(dj=1 / 12, J=84):
    return 2 * DT * 2.0 ** (np.arange(J + 1) * dj)


@pytest.mark.parametrize("name,param", MOTHERS)
def test_time_averaged_significance_matches_oracle(name, param):
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    m, ref_m = _pair(name, param)
    sj = _scales()
    n0 = 1346
    for dof in (n0 - sj, 40.0, 0.2, np.linspace(-3, 900, sj.size)):
        for var, alpha, level in ((1.0, 0.72, 0.95), (3.7, 0.0, 0.9), (0.02, 0.989, 0.99)):
            a = wavelet.significance(var, DT, sj, 1, alpha, significance_level=level, dof=dof, wavelet=m)
            b = oa.significance(var, DT, sj, 1, alpha, significance_level=level, dof=dof, wavelet=ref_m)
            assert np.allclose(a[0], b[0], rtol=1e-12, atol=0) and np.allclose(a[1], b[1], rtol=1e-12, atol=0)
    # sigma_test=1 keeps the unsmoothed spectrum as its second output, and more points mean a lower threshold
    s_lo = wavelet.significance(1.0, DT, sj, 1, 0.5, dof=10.0, wavelet=m)[0]
    s_hi = wavelet.significance(1.0, DT, sj, 1, 0.5, dof=1000.0, wavelet=m)[0]
    assert (s_hi < s_lo).all()


@pytest.mark.parametrize("name,param", MOTHERS)
@pytest.mark.parametrize("band", ["one_scale", "interior", "full_axis"])
def test_scale_averaged_significance_matches_oracle(name, param, band):
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    m, ref_m = _pair(name, param)
    sj = _scales()
    lo, hi = {"one_scale": (30, 30), "interior": (24, 48), "full_axis": (0, sj.size - 1)}[band]
    for var, alpha, level in ((1.0, 0.72, 0.95), (3.7, 0.0, 0.9), (0.02, 0.989, 0.99)):
        a = wavelet.significance(var, DT, sj, 2, alpha, significance_level=level, dof=[sj[lo], sj[hi]], wavelet=m)
        b = oa.significance(var, DT, sj, 2, alpha, significance_level=level, dof=[sj[lo], sj[hi]], wavelet=ref_m)
        assert np.ndim(a[0]) == 0 and np.ndim(a[1]) == 0
        assert a[0] == pytest.approx(b[0], rel=1e-12, abs=0) and a[1] == pytest.approx(b[1], rel=1e-12, abs=0)
    if band == "one_scale":
        # one scale: S_avg = S_mid = s, so P is that scale's red-noise spectrum
        fft0 = wavelet.significance(1.0, DT, sj, 0, 0.72, wavelet=m)[1]
        p = wavelet.significance(1.0, DT, sj, 2, 0.72, dof=[sj[lo], sj[hi]], wavelet=m)[1]
        assert p == pytest.approx(fft0[lo], rel=1e-13)


def test_scale_averaged_significance_by_hand():
    """Torrence & Compo (1998) eqs. 25-28 written out once for a three-scale band of Morlet(6)."""
    from scipy.stats import chi2
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    sj = _scales(1 / 4, 20)
    s = sj[5:8]
    fft_theor = (1 - 0.5 ** 2) / (1 + 0.5 ** 2 - 2 * 0.5 * np.cos(2 * np.pi * DT / (sj * wavelet.Morlet().flambda())))
    savg = 1 / (1 / s).sum()
    nu = 2 * 3 * savg / np.sqrt(s[0] * s[2]) * np.sqrt(1 + (3 * 0.25 / 0.6) ** 2)
    p = savg * (fft_theor[5:8] / s).sum()
    want = 0.25 * DT / (0.776 * savg) * p * chi2.ppf(0.95, nu) / nu
    got = wavelet.significance(1.0, DT, sj, 2, 0.5, dof=[s[0], s[2]])
    assert got[0] == pytest.approx(want, rel=1e-13) and got[1] == pytest.approx(p, rel=1e-13)


def test_significance_error_cases():
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    sj = _scales()
    for sig in (wavelet.significance, oa.significance):
        mk = (lambda cls, *a: getattr(wavelet, cls)(*a)) if sig is wavelet.significance else \
             (lambda cls, *a: getattr(po, cls)(*a))
        with pytest.raises(Exception, match="DOF must be set"):
            sig(1.0, DT, sj, 2, 0.5, dof=[sj[3]], wavelet=mk("Morlet", 6))
        with pytest.raises(Exception, match="DOF must be set"):
            sig(1.0, DT, sj, 2, 0.5, dof=-1, wavelet=mk("Morlet", 6))
        with pytest.raises(Exception, match="DOF must be set"):
            sig(1.0, DT, sj, 2, 0.5, dof=[sj[1], sj[2], sj[3]], wavelet=mk("Morlet", 6))
        for m in (mk("Morlet", 5), mk("Paul", 3), mk("DOG", 4)):
            with pytest.raises(ValueError):
                sig(1.0, DT, sj, 2, 0.5, dof=[sj[3], sj[9]], wavelet=m)
        with pytest.raises(ValueError, match="No valid scales"):
            sig(1.0, DT, sj, 2, 0.5, dof=[sj[3] * 1.01, sj[3] * 1.02], wavelet=mk("Morlet", 6))
        with pytest.raises(ValueError, match="No valid scales"):
            sig(1.0, DT, sj, 2, 0.5, dof=[sj[9], sj[3]], wavelet=mk("Morlet", 6))
    with pytest.raises(NotImplementedError):
        wavelet.significance(1.0, DT, sj, 3, 0.5)


def test_sigma_test_0_unchanged():
    from wavelet_transformer_b200 import pycwt_compat as wavelet
    sj = _scales()
    for m, ref_m in (_pair("morlet", 6), _pair("dog", 2)):
        a = wavelet.significance(1.0, DT, sj, 0, 0.72, significance_level=0.9, wavelet=m)
        b = oa.significance(1.0, DT, sj, 0, 0.72, significance_level=0.9, wavelet=ref_m)
        assert np.allclose(a[0], b[0], rtol=1e-13) and np.allclose(a[1], b[1], rtol=1e-13)


# ---- the averages gate ---------------------------------------------------------------------------
DJ5, J5 = 1 / 8, 65


def _ar1_coef(n0=3351, g=0.989, seed=5):
    rng = np.random.default_rng(seed)
    x = lfilter([1.0], [1.0, -g], rng.standard_normal(n0 + 3000))[3000:]
    x -= x.mean()
    W, sj = po.cwt(x, DT, DJ5, 2 * DT, J5)[:2]
    return W, sj


def _reduce(P, sj, band, factor):
    lo, hi = band
    return P.mean(axis=1), factor * (P[lo:hi + 1] / sj[lo:hi + 1, None]).sum(axis=0)


def test_averages_gate_accepts_float32_round_off():
    W, sj = _ar1_coef()
    resolved = cr.resolved_rows(3351, 4096, DT, DJ5, 2 * DT, J5)
    P32 = (np.abs(W) ** 2).astype(np.float32).astype(np.float64)        # the plane rounded to float32
    factor = DJ5 * DT / 0.776
    for band in ((0, J5), (20, 40), (7, 7)):
        g, b = _reduce(P32, sj, band, factor)
        ratio, _ = oa.averages_gate(g.astype(np.float32), b.astype(np.float32), W, sj, band, factor, 1e-4, resolved)
        assert ratio < 0.01
        g, b = _reduce(np.abs(W) ** 2, sj, band, factor)
        assert oa.averages_gate(g, b, W, sj, band, factor, 1e-4, resolved)[0] < 1e-9
    assert oa.averages_gate(None, b, W, sj, (7, 7), factor, 1e-4, resolved)[1][0] == "band"


def test_averages_gate_rejects_a_gain_on_one_row():
    """A 3e-4 gain on a row at 1e-3 of the plane maximum: the band over that row is rejected at 1e-4, where
    the plane maximum in place of scale_row (unresolved rows) lets it through."""
    W, sj = _ar1_coef()
    P = np.abs(W) ** 2
    resolved = cr.resolved_rows(3351, 4096, DT, DJ5, 2 * DT, J5)
    share = P.max(axis=1) / P.max()
    s = int(np.argmin(np.abs(np.log(share / 1e-3))))
    assert 5e-4 < share[s] < 2e-3 and resolved[s]
    bad = P.copy()
    bad[s] *= 1 + 3e-4
    factor = DJ5 * DT / 0.776
    g, b = _reduce(bad, sj, (s, s), factor)
    ratio, where = oa.averages_gate(g, b, W, sj, (s, s), factor, 1e-4, resolved)
    assert ratio > 1.0 and where[0] == "band"
    assert oa.averages_gate(g, b, W, sj, (s, s), factor, 1e-4, np.zeros_like(resolved))[0] < 1.0
    # a larger gain shows in the global spectrum of that row too
    bad[s] = P[s] * (1 + 3e-3)
    g, _ = _reduce(bad, sj, (s, s), factor)
    ratio, where = oa.averages_gate(g, None, W, sj, (s, s), factor, 1e-4, resolved)
    assert ratio > 1.0 and where == ("global", s)


# ---- _shim.cwt_averages refuses bad arguments before any transform -------------------------------------
def test_cwt_averages_refuses_bad_bands_without_a_gpu():
    from wavelet_transformer_b200 import _shim
    x = np.zeros((2, 64))
    S = 9                                    # dj = 1/4, J = 8
    for band in ((-1, 3), (4, 3), (0, S), (2, S + 5), (1,), (0.0, 3), (True, 3), "ab"):
        with pytest.raises(ValueError):
            _shim.cwt_averages(x, DT, 0.25, 2 * DT, 8, band=band)
    with pytest.raises(ValueError):
        _shim.cwt_averages(x, DT, 0.25, 2 * DT, 8, band=(0, 3), band_factor=float("nan"))
    with pytest.raises(ValueError):
        _shim.cwt_averages(x, DT, 0.25, 2 * DT, 8, band=None, want_global=False)
    with pytest.raises(ValueError):
        _shim.cwt_averages_device(0, 2, 64, DT, 0.25, 2 * DT, 8, _shim.MORLET, 6.0, 0, 1, band=None)
