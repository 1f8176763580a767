"""GPU: MODWT wavelet variance, covariance and cross-correlation by level (wtb_modwt_wavelet_stats).

Every MODWT kernel class feeds the reduction (blocked haar / db4 / sym4, k_modwt<T, 0> for db3, the generic kernels,
the level-by-level long path), and each case is held to the float64 oracle (oracle/wavelet_stats_oracle.py):
FP64 within 1e-10 (1 + |ref|) on variances and correlations; FP32 within 1e-4 nu^2 on variances,
1e-4 sqrt(nu_X^2 nu_Y^2) on covariances and 1e-4 absolute on correlations.  NaN exactly where the oracle has it.
Results are bit-identical across batch sizes, pool sizes and host vs device pointers; the x-only call gives the
pair call's var_x bits; writes stay inside their outputs; refusals launch nothing."""

import ctypes as C
import os

import numpy as np
import pytest

from oracle import modwt_oracle as mo
from oracle import wavelet_stats_oracle as wo

pytestmark = pytest.mark.gpu


def _pair(n, seed, batch=None):
    """A pair sharing a random-walk component (correlated at the coarse levels) plus independent noise."""
    rng = np.random.default_rng(seed)
    shape = (n,) if batch is None else (batch, n)
    common = np.cumsum(rng.standard_normal(shape), axis=-1) * 0.05
    return common + rng.standard_normal(shape), 0.5 * common + rng.standard_normal(shape)


def _gate(shim, x, y, wavelet, J, K, f64, generic=False, label=""):
    """Run one case and hold every row to the oracle; returns the outputs."""
    w = mo.Wavelet(wavelet)
    vx, vy, xc = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, J, K, f64=f64, generic_only=generic)
    x2, y2 = np.atleast_2d(x), np.atleast_2d(y)
    gx, gy, gc = np.atleast_2d(vx), np.atleast_2d(vy), xc.reshape(-1, J, 2 * K + 1)
    worst = {"var": 0.0, "cov": 0.0, "corr": 0.0}
    for i in sorted({0, x2.shape[0] - 1}):
        rx, ry, rc = wo.stats(x2[i], y2[i], wavelet, J, K)
        for got, ref in ((gx[i], rx), (gy[i], ry), (gc[i], rc)):
            assert np.array_equal(np.isnan(got), np.isnan(ref)), f"{label}: NaN pattern"
        ok = ~np.isnan(rc)
        rho, rrho = wo.correlation(gx[i], gy[i], gc[i]), wo.correlation(rx, ry, rc)
        if f64:
            bound = lambda ref: 1e-10 * (1 + np.abs(ref))
            ratios = {"var": np.abs(np.r_[gx[i] - rx, gy[i] - ry]) / bound(np.r_[rx, ry]),
                      "cov": np.abs(gc[i] - rc)[ok] / bound(rc[ok]),
                      "corr": np.abs(rho - rrho)[ok] / bound(rrho[ok])}
        else:
            scale = np.sqrt(rx * ry)[:, None] * np.ones_like(rc)
            ratios = {"var": np.abs(np.r_[gx[i] - rx, gy[i] - ry]) / (1e-4 * np.r_[rx, ry]),
                      "cov": np.abs(gc[i] - rc)[ok] / (1e-4 * scale[ok]),
                      "corr": np.abs(rho - rrho)[ok] / 1e-4}
        for k, r in ratios.items():
            r = r[~np.isnan(r)]
            worst[k] = max(worst[k], float(r.max()) if r.size else 0.0)
    print(f"WSTATSGATE {label} {'fp64' if f64 else 'fp32'}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, (label, worst)
    return vx, vy, xc


@pytest.mark.parametrize("f64", [False, True])
def test_inflation_against_expectation(shim, series, f64):
    """The cfg2 pair: inflation against the overlapping stretch of expectation, sym4, J = 6, K = 36."""
    x, y = series["pair_inflation"], series["pair_expectation"]
    vx, vy, xc = _gate(shim, x, y, "sym4", 6, 36, f64, label="cfg2")
    assert vx.shape == (6,) and xc.shape == (6, 73)


# (wavelet, n, batch, J, K, generic): blocked kernels, k_modwt<T, 0>, the generic kernels, odd n
SHAPES = [("haar", 1001, 3, 6, 20, False), ("db4", 1001, 3, 6, 20, False), ("sym4", 1333, 5, 6, 36, False),
          ("db3", 1001, 3, 5, 17, False), ("sym4", 1001, 3, 6, 36, True), ("db4", 4096, 2, 8, 64, False)]


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("case", SHAPES, ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}-J{c[3]}-K{c[4]}" + ("-generic" if c[5] else ""))
def test_kernel_classes(shim, case, f64):
    wavelet, n, batch, J, K, generic = case
    x, y = _pair(n, n + J, batch)
    _gate(shim, x, y, wavelet, J, K, f64, generic, label=f"{wavelet}-{n}x{batch}")


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n,J,K", [(40000, 8, 64), (1 << 20, 10, 256)])
def test_long_path(shim, n, J, K, f64):
    """Lengths past one CTA's MODWT run the level-by-level kernels; several t-blocks per level."""
    x, y = _pair(n, 7)
    _gate(shim, x, y, "sym4", J, K, f64, label=f"long-{n}")


@pytest.mark.parametrize("f64", [False, True])
def test_levels_past_the_series_and_lags_past_m(shim, f64):
    """sym4 at n = 60: M_j = 53, 39, 11, -45; lags up to 40 reach past M_3 and the whole of level 4 is NaN."""
    x, y = _pair(60, 3)
    vx, vy, xc = _gate(shim, x, y, "sym4", 4, 40, f64, label="short-60")
    assert np.isnan(vx[3]) and np.isnan(xc[3]).all() and np.isnan(xc[2, :40 - 11 + 1]).all()


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n", [565, 40000])
def test_univariate_equals_the_pair_bits(shim, n, f64):
    w = mo.Wavelet("sym4")
    x, y = _pair(n, 21, 3)
    vx, _, _ = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, 6, 12, f64=f64)
    v1, none_y, none_c = shim.modwt_wavelet_stats(x, None, w.dec_lo, w.dec_hi, 6, f64=f64)
    assert none_y is None and none_c is None
    assert np.array_equal(v1, vx)


# ---- invariance ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n", [1333, 40000])
def test_batch_and_pointer_invariance(shim, n, f64):
    import torch
    w = mo.Wavelet("sym4")
    J, K = 6, 36
    x, y = _pair(n, 33, 7)
    v7 = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, J, K, f64=f64)
    for i in (0, 6):
        v1 = shim.modwt_wavelet_stats(x[i], y[i], w.dec_lo, w.dec_hi, J, K, f64=f64)
        for a, b in zip(v1, v7):
            assert np.array_equal(a, b[i], equal_nan=True)
    dtype = torch.float64 if f64 else torch.float32
    xd, yd = (torch.as_tensor(v, dtype=dtype, device="cuda").contiguous() for v in (x, y))
    outs = [torch.empty(7, J, dtype=torch.float64, device="cuda") for _ in range(2)]
    outs.append(torch.empty(7, J, 2 * K + 1, dtype=torch.float64, device="cuda"))
    shim.modwt_wavelet_stats_device(xd.data_ptr(), yd.data_ptr(), 7, n, w.dec_lo, w.dec_hi, J, K,
                                    *(o.data_ptr() for o in outs), f64=f64,
                                    stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for a, b in zip(outs, v7):
        assert np.array_equal(a.cpu().numpy(), b, equal_nan=True)


def test_across_a_chunk_boundary(shim):
    """2^20 samples, J = 10 in FP64: 184 MB of planes per pair, five pairs per 1 GiB chunk, so seven pairs take two
    chunks; every pair has the bits of its own call."""
    w = mo.Wavelet("sym4")
    x, y = _pair(1 << 20, 55, 7)
    v7 = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, 10, 16, f64=True)
    for i in (4, 5, 6):
        v1 = shim.modwt_wavelet_stats(x[i], y[i], w.dec_lo, w.dec_hi, 10, 16, f64=True)
        for a, b in zip(v1, v7):
            assert np.array_equal(a, b[i], equal_nan=True)


@pytest.fixture()
def pool(shim):
    """A pool of two workers: two GPUs when the box has them, one shared GPU otherwise."""
    os.environ["WTB_POOL_SHARE_DEVICES"] = "1"
    n = shim.init_multi(2)
    assert n == 2
    yield shim
    shim.init_multi(1)
    assert shim.gpu_count() == 1


@pytest.mark.parametrize("f64", [False, True])
def test_split_over_the_pool(shim, pool, f64):
    w = mo.Wavelet("db4")
    x, y = _pair(2000, 44, 9)
    v2 = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, 7, 30, f64=f64)
    shim.init_multi(1)
    v1 = shim.modwt_wavelet_stats(x, y, w.dec_lo, w.dec_hi, 7, 30, f64=f64)
    for a, b in zip(v1, v2):
        assert np.array_equal(a, b, equal_nan=True)


# ---- guard writes ----------------------------------------------------------------------------------------
GUARD = 4096


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n,batch,J,K", [(565, 3, 6, 36), (40000, 2, 9, 100), (60, 5, 4, 40)])
def test_outputs_stay_inside(shim, n, batch, J, K, f64):
    import torch
    w = mo.Wavelet("sym4")
    dtype = torch.float64 if f64 else torch.float32
    x, y = (torch.as_tensor(v, dtype=dtype, device="cuda").contiguous() for v in _pair(n, 5, batch))
    shapes = [(batch, J), (batch, J), (batch, J, 2 * K + 1)]
    bufs = [torch.full((int(np.prod(s)) + 2 * GUARD,), -7.0e33, dtype=torch.float64, device="cuda") for s in shapes]
    views = [b[GUARD:GUARD + int(np.prod(s))] for b, s in zip(bufs, shapes)]
    shim.modwt_wavelet_stats_device(x.data_ptr(), y.data_ptr(), batch, n, w.dec_lo, w.dec_hi, J, K,
                                    *(v.data_ptr() for v in views), f64=f64)
    torch.cuda.synchronize()
    for b, v in zip(bufs, views):
        assert bool((b[:GUARD] == -7.0e33).all()) and bool((b[GUARD + v.numel():] == -7.0e33).all())
        assert not bool((v == -7.0e33).any())
    ref = shim.modwt_wavelet_stats(x.cpu().numpy(), y.cpu().numpy(), w.dec_lo, w.dec_hi, J, K, f64=f64)
    for v, r, s in zip(views, ref, shapes):
        assert np.array_equal(v.cpu().numpy().reshape(s), r, equal_nan=True)


# ---- refusals ------------------------------------------------------------------------------------------
def test_refusals(shim):
    lib = shim.lib()
    w = mo.Wavelet("sym4")
    g, h = (np.ascontiguousarray(v, dtype=np.float64) for v in (w.dec_lo, w.dec_hi))
    x, y = (np.ascontiguousarray(v) for v in _pair(100, 1, 2))
    vx, vy, xc = np.zeros((2, 4)), np.zeros((2, 4)), np.zeros((2, 4, 11))
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))

    def call(x=x, y=y, batch=2, n=100, L=8, J=4, K=5, ox=vx, oy=vy, oc=xc):
        return lib.wtb_modwt_wavelet_stats(p(x), p(y), batch, n, dp(g), dp(h), L, J, K, shim.F64, p(ox), p(oy),
                                           p(oc), None)

    launches = shim.kernel_launches()
    for kwargs in ({"ox": None, "oy": None, "oc": None}, {"y": None}, {"y": None, "oy": None},
                   {"y": None, "oc": None}, {"J": 0}, {"J": 31}, {"K": -1}, {"K": 100}, {"n": 10000, "K": 8193},
                   {"x": None}, {"batch": -1}, {"n": 0}):
        assert call(**kwargs) == -1, kwargs
        assert lib.wtb_last_error()
    for L in (1, 33):
        assert call(L=L) == -3, L
    assert call(batch=0) == 0
    assert shim.kernel_launches() == launches, "a refusal launched a kernel"
    assert call() == 0
    assert call(y=None, oy=None, oc=None) == 0
    rx, ry, rc = wo.stats(x[1], y[1], "sym4", 4, 5)
    assert np.allclose(vx[1], rx, rtol=1e-10, equal_nan=True) and np.allclose(xc[1], rc, rtol=1e-10, atol=1e-12, equal_nan=True)


# ---- public functions ----------------------------------------------------------------------------------
def test_public_functions(shim, series):
    import wavelet_transformer_b200 as wtb
    from wavelet_transformer_b200 import _shim
    x, y = series["pair_inflation"], series["pair_expectation"]
    before = _shim.get_precision()
    try:
        _shim.set_precision("fp64")
        r = wtb.wavelet_correlation(x, y, "sym4", 6, max_lag=36, dt=1 / 12)
        v = wtb.wavelet_variance(x, "sym4", 6, dt=1 / 12)
    finally:
        _shim.set_precision(before)
    rx, ry, rc = wo.stats(x, y, "sym4", 6, 36)
    n, L = x.size, 8
    assert np.array_equal(r.level, np.arange(1, 7)) and np.allclose(r.scale, 2.0 ** np.arange(6) / 12)
    assert list(r.m) == [wo.m_count(n, j, L) for j in range(1, 7)]
    assert np.allclose(v.variance, rx, rtol=1e-10) and np.array_equal(v.variance, r.var_x)
    lo, hi = wo.variance_ci(rx, n, 6, L)
    assert np.allclose(v.ci_low, lo, rtol=1e-9) and np.allclose(v.ci_high, hi, rtol=1e-9)
    rho = wo.correlation(rx, ry, rc)
    assert np.allclose(r.xcorr, rho, atol=1e-10, equal_nan=True) and np.array_equal(r.lags, np.arange(-36, 37))
    assert np.allclose(r.correlation, rho[:, 36], atol=1e-10)
    clo, chi = wo.correlation_ci(rho, n, 6, L)
    assert np.allclose(r.xcorr_ci_low, clo, atol=1e-9, equal_nan=True)
    assert np.allclose(r.xcorr_ci_high, chi, atol=1e-9, equal_nan=True)
    b = wtb.wavelet_correlation(np.stack([x, y]), np.stack([y, x]), "sym4", 6, max_lag=4)
    assert b.xcorr.shape == (2, 6, 9) and b.correlation.shape == (2, 6)
    with pytest.raises(ValueError):
        wtb.wavelet_correlation(x, y[:-1])
