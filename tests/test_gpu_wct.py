"""GPU parity: XWT / WCT / Monte Carlo significance vs the pycwt oracle."""

import numpy as np
import pytest

from conftest import normwise_close
from oracle import mc_oracle as mo
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1 / 12


def _norm(y):
    return (y - y.mean()) / y.std()


def test_wct_fp64_cfg3_pair(shim, series):
    """BASELINE cfg3 transform: inflation vs expectation, n0=565, dj=1/8, s0=2dt, 66 scales."""
    y1, y2 = series["pair_inflation"], series["pair_expectation"]
    WCT, aWCT, coi, freq, _ = po.wct(y1, y2, DT, dj=1 / 8, s0=2 * DT, J=-1, sig=False)
    wct, phase, w12 = shim.xwt_wct(_norm(y1), _norm(y2), DT, 1 / 8, 2 * DT, -1, f64=True, want_w12=True)
    assert wct.shape == WCT.shape == (66, 565)
    assert np.abs(wct - WCT).max() <= 1e-10
    # phase of the unsmoothed cross spectrum (compare on the circle)
    d = np.angle(np.exp(1j * (phase - aWCT)))
    assert np.abs(d).max() <= 1e-8
    assert 0 <= wct.min() and wct.max() <= 1 + 1e-12


def test_xwt_fp64(shim, series):
    y1, y2 = series["pair_expectation"], series["pair_expectation"][::-1].copy()
    W1 = po.cwt(_norm(y1), DT, 1 / 8, 2 * DT, -1)[0]
    W2 = po.cwt(_norm(y2), DT, 1 / 8, 2 * DT, -1)[0]
    ref = W1 * W2.conj()
    _, _, w12 = shim.xwt_wct(_norm(y1), _norm(y2), DT, 1 / 8, 2 * DT, -1, f64=True, want_wct=False,
                             want_phase=False, want_w12=True)
    assert np.abs(w12 - ref).max() <= 1e-10 * np.abs(ref).max()


@pytest.mark.parametrize("dj", [1 / 8, 1 / 12, 1 / 4])
def test_wct_fp32_batch(shim, dj):
    rng = np.random.default_rng(17)
    n0 = 700
    y1 = rng.standard_normal((4, n0)).cumsum(axis=1)
    y2 = y1 * 0.3 + rng.standard_normal((4, n0)) * 3
    y1 = np.stack([_norm(r) for r in y1])
    y2 = np.stack([_norm(r) for r in y2])
    wct, phase, _ = shim.xwt_wct(y1, y2, DT, dj, 2 * DT, -1, f64=False)
    for b in range(4):
        WCT = po.wct(y1[b], y2[b], DT, dj=dj, s0=2 * DT, J=-1, sig=False, normalize=False)[0]
        ok, worst = normwise_close(wct[b], WCT, 1e-4)      # BASELINE.md FP32 gate: 1e-4 |b| + 1e-4 max|b|
        assert ok, worst
        assert np.abs(wct[b] - WCT).mean() <= 2e-6        # measured 2e-7 .. 5e-7 (profiles/r2_wct_fp32_error.jsonl)


def test_wct_self_coherence_is_one(shim):
    x = _norm(np.random.default_rng(2).standard_normal(1000))
    wct, _, _ = shim.xwt_wct(x, x, DT, 1 / 8, 2 * DT, -1, f64=True)
    assert np.abs(wct - 1).max() <= 1e-10


def test_mc_geometry_matches_oracle(shim):
    for dj, J in [(1 / 8, 65), (1 / 12, 60), (1 / 4, 20)]:
        N, sj, freq, outside, maxscale = po.mc_geometry(DT, dj, 2 * DT, J, po.Morlet())
        assert shim.wct_mc_geometry(DT, dj, 2 * DT, J) == (N, maxscale)
        assert np.array_equal(shim.row_has_points(DT, dj, 2 * DT, J), outside.any(axis=1))


def test_mc_injected_surrogates_fp64_exact(shim):
    """Per-realisation parity: same surrogates in, same histogram out (FP64)."""
    dj, s0, J = 1 / 8, 2 * DT, 40
    N = shim.wct_mc_geometry(DT, dj, s0, J)[0]
    rng = np.random.default_rng(99)
    mc = 6
    sur = np.empty((mc, 2, N))
    for m in range(mc):
        sur[m, 0] = po.rednoise(N, 0.989, 1, rng)
        sur[m, 1] = po.rednoise(N, 0.966, 1, rng)
    sig_ref, hist_ref = po.wct_significance(0.989, 0.966, DT, dj, s0, J, mc_count=mc, surrogates=sur,
                                            return_hist=True)
    hist = shim.wct_mc_hist(0.989, 0.966, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=True)
    assert hist.sum() == hist_ref.sum()
    # a value within 1e-12 of a bin edge may land on either side
    assert np.abs(hist.astype(np.int64) - hist_ref).sum() <= 4
    _, maxscale = shim.wct_mc_geometry(DT, dj, s0, J)
    sig = shim.wct_sig_from_hist(hist, maxscale, 0.95, shim.row_has_points(DT, dj, s0, J))
    assert np.allclose(sig[:maxscale], sig_ref[:maxscale], atol=2e-3)
    assert np.isnan(sig[maxscale]) and np.isnan(sig_ref[maxscale])


def test_mc_injected_surrogates_fp32(shim):
    dj, s0, J = 1 / 8, 2 * DT, 40
    N = shim.wct_mc_geometry(DT, dj, s0, J)[0]
    rng = np.random.default_rng(100)
    mc = 8
    sur = np.stack([np.stack([po.rednoise(N, 0.9, 1, rng), po.rednoise(N, 0.5, 1, rng)]) for _ in range(mc)])
    hist = shim.wct_mc_hist(0.9, 0.5, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=False)
    # exact row totals; an FP32 value may cross a bin edge only within the FP32 gate (2e-4 at v <= 1)
    mo.assert_hist_matches(hist, mo.mc_samples(sur, DT, dj, s0, J), 2e-4)


def test_mc_partition_invariance(shim):
    """Sharding realisations (the multi-GPU split) must not change the histogram."""
    dj, s0, J = 1 / 4, 2 * DT, 24
    full = shim.wct_mc_hist(0.8, 0.6, DT, dj, s0, J, mc_first=0, mc_count=10, seed=7, f64=False)
    a = shim.wct_mc_hist(0.8, 0.6, DT, dj, s0, J, mc_first=0, mc_count=4, seed=7, f64=False)
    b = shim.wct_mc_hist(0.8, 0.6, DT, dj, s0, J, mc_first=4, mc_count=6, seed=7, f64=False)
    assert np.array_equal(full, a + b)
    other = shim.wct_mc_hist(0.8, 0.6, DT, dj, s0, J, mc_first=0, mc_count=10, seed=8, f64=False)
    assert not np.array_equal(full, other)


def test_device_rednoise_statistics(shim):
    """Device Philox AR(1): unit innovations, lag-1 autocorrelation g, stationarity."""
    g1, g2, n = 0.9, 0.3, 4000
    y = shim.rednoise(g1, g2, n, 0, 64, 2024, f64=True)
    for which, g in ((0, g1), (1, g2)):
        s = y[:, which, :]
        var = s.var()
        assert abs(var - 1 / (1 - g * g)) / (1 / (1 - g * g)) < 0.08
        r1 = (s[:, 1:] * s[:, :-1]).mean() / var
        assert abs(r1 - g) < 0.02
        eps = s[:, 1:] - g * s[:, :-1]
        assert abs(eps.std() - 1) < 0.01 and abs(eps.mean()) < 0.01
    # different realisations and the two series of a pair are independent streams
    assert abs(np.corrcoef(y[0, 0], y[1, 0])[0, 1]) < 0.2
    w = shim.rednoise(g1, g2, n, 0, 4, 2024, f64=True, white=True)
    assert abs(w.std() - 1) < 0.02


def test_mc_device_rng_distribution(shim):
    """Distribution-level parity: 95 % thresholds from device surrogates agree with
    the oracle's NumPy-RNG thresholds within Monte Carlo error."""
    dj, s0, J = 1 / 4, 2 * DT, 24
    _, maxscale = shim.wct_mc_geometry(DT, dj, s0, J)
    hist = shim.wct_mc_hist(0.8, 0.6, DT, dj, s0, J, mc_count=400, seed=1, f64=False)
    sig = shim.wct_sig_from_hist(hist, maxscale, 0.95, shim.row_has_points(DT, dj, s0, J))
    ref = po.wct_significance(0.8, 0.6, DT, dj, s0, J, mc_count=120, rng=np.random.default_rng(5))
    m = maxscale - 2  # the last rows have very few reliable samples
    assert np.abs(sig[:m] - ref[:m]).max() < 0.05, np.abs(sig[:m] - ref[:m])


def test_wct_fp32_n4096_fast_path(shim):
    """nfft = 4096 takes the register-FFT row kernel (wct_fast.cu); check it against the
    oracle and against the generic kernels on the cfg5 surrogate shape (n0 = 3351)."""
    rng = np.random.default_rng(41)
    n0 = 3351
    y1 = np.stack([_norm(po.rednoise(n0, 0.989, 1, rng)) for _ in range(2)])
    y2 = np.stack([_norm(po.rednoise(n0, 0.966, 1, rng)) for _ in range(2)])
    wct, phase, w12 = shim.xwt_wct(y1, y2, DT, 1 / 8, 2 * DT, 65, f64=False, want_w12=True)
    wct_g, phase_g, w12_g = shim.xwt_wct(y1, y2, DT, 1 / 8, 2 * DT, 65, f64=False, want_w12=True,
                                         generic_only=True)
    for b in range(2):
        WCT, aWCT, _, _, _ = po.wct(y1[b], y2[b], DT, dj=1 / 8, s0=2 * DT, J=65, sig=False, normalize=False)
        W1 = po.cwt(y1[b], DT, 1 / 8, 2 * DT, 65)[0]
        W2 = po.cwt(y2[b], DT, 1 / 8, 2 * DT, 65)[0]
        ref12 = W1 * W2.conj()
        for got in (w12[b], w12_g[b]):
            assert np.abs(got - ref12).max() <= 1e-4 * np.abs(ref12).max()
        for got in (wct[b], wct_g[b]):
            ok, worst = normwise_close(got, WCT, 1e-4)     # measured max 6e-6 on this shape
            assert ok, worst
            assert np.abs(got - WCT).mean() <= 2e-6
    assert np.abs(wct - wct_g).max() <= 1e-4


def test_mc_cfg5_shape_fast_vs_generic_vs_oracle(shim):
    """cfg5 / cfg3 Monte Carlo shape (J=65, dj=1/8 -> 3351 samples, FFT 4096), injected surrogates."""
    dj, s0, J = 1 / 8, 2 * DT, 65
    N, maxscale = shim.wct_mc_geometry(DT, dj, s0, J)
    assert (N, maxscale) == (3351, 65)
    rng = np.random.default_rng(77)
    mc = 3
    sur = np.stack([np.stack([po.rednoise(N, 0.989, 1, rng), po.rednoise(N, 0.966, 1, rng)]) for _ in range(mc)])
    ref = mo.mc_samples(sur, DT, dj, s0, J)
    hist_ref = mo.samples_histogram(ref)
    fast = shim.wct_mc_hist(0.989, 0.966, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=False)
    gen = shim.wct_mc_hist(0.989, 0.966, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=False, generic_only=True)
    f64 = shim.wct_mc_hist(0.989, 0.966, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=True)
    assert np.abs(f64.astype(np.int64) - hist_ref).sum() <= 6
    mo.assert_hist_matches(f64, ref, 1e-10)
    for h in (fast, gen):
        mo.assert_hist_matches(h, ref, 2e-4)


@pytest.mark.parametrize("dj,J,taps", [(1 / 12, 97, 14), (1 / 4, 33, 5), (1 / 6, 49, 7), (1 / 10, 82, 12)])
def test_mc_fast_path_other_scale_resolutions(shim, dj, J, taps):
    """The register-FFT Monte-Carlo kernels at other dj (surrogates still 2049..4096 samples):
    the scale boxcar has rect(round(1.2/dj)) taps -- 14 and 5 take the register-ring
    instantiations, 7 and 12 the shared-memory ring.  Injected surrogates, per-row oracle parity."""
    s0 = 2 * DT
    N, maxscale = shim.wct_mc_geometry(DT, dj, s0, J)
    assert 2048 < N <= 4096 and int(round(0.6 / dj * 2)) == taps
    rng = np.random.default_rng(J)
    mc = 2
    sur = np.stack([np.stack([po.rednoise(N, 0.9, 1, rng), po.rednoise(N, 0.7, 1, rng)]) for _ in range(mc)])
    ref = mo.mc_samples(sur, DT, dj, s0, J)
    fast = shim.wct_mc_hist(0.9, 0.7, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=False)
    gen = shim.wct_mc_hist(0.9, 0.7, DT, dj, s0, J, mc_count=mc, surrogates=sur, f64=False, generic_only=True)
    for h in (fast, gen):
        mo.assert_hist_matches(h, ref, 2e-4)


def test_wct_fp32_fast_path_fuzz(shim):
    """Random parameters through the nfft = 4096 coherence kernels (other f0, sampling steps, dj,
    smallest scales): the pruned bands of the daughters and of the Gaussian time filter move with
    them.  Reference = the FP64 generic kernels (oracle-gated above)."""
    rng = np.random.default_rng(4096)
    for _ in range(6):
        n0 = int(rng.integers(2049, 4097))
        dt = float(rng.choice([1 / 12, 0.5, 2.0]))
        dj = float(rng.choice([1 / 4, 1 / 8, 1 / 10, 1 / 12]))
        s0 = dt * float(rng.choice([1.0, 2.0, 4.0]))
        f0 = float(rng.choice([6.0, 6.0, 7.5, 10.0]))
        jmax = int(np.floor(np.log2(n0 * dt / s0) / dj))
        J = int(rng.integers(jmax // 2, min(jmax, 110) + 1))
        y1 = _norm(po.rednoise(n0, 0.8, 1, rng))
        y2 = _norm(0.5 * y1 + po.rednoise(n0, 0.5, 1, rng))
        wct, phase, w12 = shim.xwt_wct(y1, y2, dt, dj, s0, J, f0, f64=False, want_w12=True)
        ref, _, ref12 = shim.xwt_wct(y1, y2, dt, dj, s0, J, f0, f64=True, want_w12=True, generic_only=True)
        tag = f"n0={n0} dt={dt} dj={dj:.4f} s0={s0} f0={f0} J={J}"
        assert np.abs(w12 - ref12).max() <= 1e-4 * np.abs(ref12).max(), tag
        # Rows whose daughter peaks beyond the Nyquist frequency (s / dt < f0 / pi; the fuzz draws
        # s0 = dt, the reference never goes below s0 = 2 dt with f0 = 6) see only the wavelet's tail:
        # their coefficients are rounding-level and the coherence is a ratio of noise.  They are held
        # to 2e-3, every resolvable row to BASELINE.md's gate.
        sj = s0 * 2.0 ** (np.arange(J + 1) * dj)
        resolvable = sj / dt >= f0 / np.pi
        ok, worst = normwise_close(wct[resolvable], ref[resolvable], 1e-4)
        assert ok, (tag, worst)
        assert np.abs(wct - ref).max() <= 2e-3, tag
        assert np.abs(wct[resolvable] - ref[resolvable]).mean() <= 5e-6, (tag, np.abs(wct - ref).mean())
