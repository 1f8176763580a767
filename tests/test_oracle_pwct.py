"""CPU: the float64 reference of partial and multiple wavelet coherence (oracle/pwct_oracle.py).

The closed forms of wtb_partial_wct are checked against an independent formulation (the inverse of the 3x3
smoothed spectral matrix), against the bounds that hold wherever the smoothing kernel keeps that matrix positive
semidefinite, against the Desnanot-Jacobi identity 1 - MWC = (1 - |rho_y2|^2)(1 - PWC) and against the x1 <-> x2
symmetry of MWC, in both padding modes."""

import numpy as np
import pytest

from oracle import pwct_oracle as pw

DT = 1.0
TOL = 1e-12
# (n0, dj): the cfg3 shape, the cfg1 length, and a Bluestein length
SHAPES = [(565, 1 / 8), (1346, 1 / 12), (2047, 1 / 8)]


def _case(kind, n0, dj, pad):
    sp = pw.spectra(*pw.triple(kind, n0, seed=n0 + len(kind)), DT, dj, -1, -1, pad_pow2=pad)
    pwc, _, mwc = pw.closed_forms(sp)
    kp, km = pw.conditioning(sp)
    return sp, pwc, mwc, kp, km


@pytest.mark.parametrize("pad", [True, False], ids=["pow2", "unpadded"])
@pytest.mark.parametrize("n0,dj", SHAPES)
@pytest.mark.parametrize("kind", pw.INPUTS)
def test_closed_forms_equal_the_inverse_forms(kind, n0, dj, pad):
    """Agreement within TOL times the worse of the two conditionings: kappa for the closed forms, cond(S) for the
    inverse.  Points where S is singular to working precision (cond > 1e12: the largest scales, where the three
    smoothed rows become nearly proportional) carry no digits in the inverse form and are left out."""
    sp, pwc, mwc, kp, km = _case(kind, n0, dj, pad)
    ipwc, imwc = pw.inverse_forms(sp)
    cond = np.linalg.cond(pw.matrix(sp))
    ok = cond < 1e12
    assert ok.mean() > 0.9
    for got, ref, kappa, what in ((ipwc, pwc, kp, "pwc"), (imwc, mwc, km, "mwc")):
        ratio = np.abs(got - ref)[ok] / (TOL * np.maximum(kappa, cond)[ok] * (1 + np.abs(ref[ok])))
        assert ratio.max() <= 1.0, f"{what}: {ratio.max():.3g}"
    print(f"PWCTORACLE {kind} {n0} {'pow2' if pad else 'none'}: singular points left out {(~ok).sum()} of {ok.size}")


@pytest.mark.parametrize("pad", [True, False], ids=["pow2", "unpadded"])
@pytest.mark.parametrize("n0,dj", SHAPES)
@pytest.mark.parametrize("kind", pw.INPUTS)
def test_bounds_on_rows_with_a_non_negative_kernel(kind, n0, dj, pad):
    """0 <= PWC, MWC <= 1 and MWC >= max(|rho_y1|^2, |rho_y2|^2) to rounding.  Both need a positive semidefinite
    smoothed matrix, which holds on a row whose time kernel is non-negative; the kernel is the inverse DFT of the
    Gaussian truncated at Nyquist and rings at the smallest scales."""
    sp, pwc, mwc, kp, km = _case(kind, n0, dj, pad)
    ker = pw.smoothing_kernel(n0, DT, sp["scales"], pad)
    nonneg = ker.min(axis=1) >= -1e-14 * ker.max(axis=1)      # below that: the rounding of the inverse DFT
    assert nonneg.mean() > 0.9
    print(f"PWCTBOUNDS {kind} {n0} {'pow2' if pad else 'none'}: rows with a ringing kernel "
          f"{np.flatnonzero(~nonneg).tolist()}")
    rows = np.flatnonzero(nonneg)
    for v, kappa in ((pwc, kp), (mwc, km)):
        v, slack = v[rows], TOL * kappa[rows]
        assert np.all(v >= -slack) and np.all(v <= 1 + slack)
    dom = np.maximum(pw.rho2(sp, "y", "1"), pw.rho2(sp, "y", "2"))[rows]
    assert np.all(mwc[rows] >= dom - TOL * km[rows])


@pytest.mark.parametrize("pad", [True, False], ids=["pow2", "unpadded"])
@pytest.mark.parametrize("n0,dj", SHAPES)
@pytest.mark.parametrize("kind", pw.INPUTS)
def test_multiple_and_partial_coherence_identity(kind, n0, dj, pad):
    """1 - MWC = (1 - |rho_y2|^2)(1 - PWC): algebraic (Desnanot-Jacobi), so it holds on every row."""
    sp, pwc, mwc, kp, km = _case(kind, n0, dj, pad)
    err = np.abs((1 - mwc) - (1 - pw.rho2(sp, "y", "2")) * (1 - pwc))
    assert np.all(err <= TOL * kp * (1 + np.abs(pwc)))


@pytest.mark.parametrize("pad", [True, False], ids=["pow2", "unpadded"])
@pytest.mark.parametrize("kind", pw.INPUTS)
def test_multiple_coherence_is_symmetric_in_the_predictors(kind, pad):
    n0, dj = 565, 1 / 8
    y, x1, x2 = pw.triple(kind, n0, seed=5)
    _, _, m12 = pw.closed_forms(pw.spectra(y, x1, x2, DT, dj, -1, -1, pad_pow2=pad))
    sp21 = pw.spectra(y, x2, x1, DT, dj, -1, -1, pad_pow2=pad)
    _, _, m21 = pw.closed_forms(sp21)
    _, km = pw.conditioning(sp21)
    assert np.all(np.abs(m12 - m21) <= TOL * km * (1 + np.abs(m21)))


def test_unpadded_transforms_run_at_the_series_length():
    """pad_pow2=False transforms at n0 itself: the spectra differ from the padded ones."""
    y, x1, x2 = pw.triple("built", 565, seed=6)
    a = pw.spectra(y, x1, x2, DT, 1 / 8, -1, -1, pad_pow2=True)
    b = pw.spectra(y, x1, x2, DT, 1 / 8, -1, -1, pad_pow2=False)
    assert a["Syy"].shape == b["Syy"].shape == (a["scales"].size, 565)
    assert np.abs(a["Syy"] - b["Syy"]).max() > 1e-6
