"""GPU: cross spectra, coherence and its Monte-Carlo significance for long series (wct_long.cu), the
power-of-two lengths past one CTA's shared memory up to nfft = 2^22.

Coherence, W12 and the phase are held row by row to the float64 reference of oracle/wct_long.py (1e-10 in FP64;
in FP32 the norm-wise plane gate for the coherence and the per-row gate on resolved rows for W12 and the phasor
|W12| e^{i phase}), from the first newly covered lengths up to 3 000 000 samples.  Launch counts show which path
served a call.  W12 is the product of wtb_cwt's own coefficients; results are bit-identical across batch sizes,
pool sizes and device pointers; writes stay inside their outputs.  The Monte Carlo, the one-call significance
and the façades work at these lengths."""

import ctypes as C
import os

import numpy as np
import pytest
from scipy.signal import lfilter

from conftest import normwise_close
from oracle import cwt_long as cl
from oracle import cwt_rows as cr
from oracle import mc_oracle as mo
from oracle import pycwt_oracle as po
from oracle import wct_long as wl

pytestmark = pytest.mark.gpu

DT = 1.0
INPUTS = ["white", "ar1_0.989", "two_tone"]
EUNSUPPORTED = -3


def _inputs(kind, batch, n0, seed):
    """[batch, 2, n0] pairs: the second series of a pair is the first plus independent noise of the same kind."""
    rng = np.random.default_rng(seed)
    if kind == "white":
        x = rng.standard_normal((batch, 2, n0))
    elif kind == "ar1_0.989":
        x = lfilter([1.0], [1.0, -0.989], rng.standard_normal((batch, 2, n0 + 2000)), axis=2)[:, :, 2000:]
    elif kind == "two_tone":
        t = np.arange(n0)
        period = rng.uniform(20.0, 60.0, size=(batch, 2, 1))
        ph = rng.uniform(0, 2 * np.pi, size=(batch, 2, 2))
        x = np.sin(2 * np.pi * t / period + ph[..., :1]) + 1e-3 * np.sin(2 * np.pi * t / 3.0 + ph[..., 1:])
    else:
        raise ValueError(kind)
    x[:, 1] += 0.5 * x[:, 0]
    x = x - x.mean(axis=2, keepdims=True)
    return x / x.std(axis=2, keepdims=True)


def _nfft(n0):
    return 1 << (n0 - 1).bit_length()


def _xwt(shim, y, dj, J, f64, wct=True, phase=True, w12=True):
    before = shim.kernel_launches()
    out = shim.xwt_wct(y[:, 0], y[:, 1], DT, dj, -1, J, f64=f64, want_wct=wct, want_phase=phase, want_w12=w12)
    return out, shim.kernel_launches() - before


def _check(shim, y, dj, J, f64, rows, out):
    """wct / phase / w12 [S, n0] of one pair against the float64 rows of the reference; worst gate ratio.
    The coherence is held where both smoothed spectra exceed COND (1e-3 in FP32, 1e-4 in FP64) of their row's
    maximum: below that they sit at the rounding level of the row's smoothing transforms (a pure tone has
    such rows), and |S12|^2 / (S1 S2) is ill-conditioned in any implementation."""
    wct, phase, w12 = out
    n0 = y.shape[1]
    Jr, sj, _, _ = shim.cwt_axes(n0, DT, dj, -1, J)
    yr = y.astype(np.float64) if f64 else y.astype(np.float32).astype(np.float64)
    rwct, rph, rw12, s1, s2 = wl.wct_rows(yr[0], yr[1], DT, dj, -1, Jr, rows, normalize=False, spectra=True)
    tol = 1e-10 if f64 else 1e-4
    cond = 1e-4 if f64 else 1e-3
    ok = (s1 > cond * s1.max(axis=1, keepdims=True)) & (s2 > cond * s2.max(axis=1, keepdims=True))
    assert ok.mean() > 0.5, f"only {ok.mean():.3g} of the plane is well conditioned"
    got = np.where(ok, wct[rows], 0.0)
    want = np.where(ok, rwct, 0.0)
    if f64:
        assert np.abs(got - want).max() <= tol, "coherence"
        resolved = np.ones(len(rows), bool)
    else:
        good, worst = normwise_close(got, want, tol)
        assert good, f"coherence: plane gate, worst {worst:.3g}"
        resolved = cr.resolved_rows(n0, _nfft(n0), DT, dj, sj[0], Jr)[rows]
    if not ok.all():
        print(f"ill-conditioned coherence points skipped: {(~ok).sum()} of {ok.size}")
    worst = 0.0
    ph = np.abs(w12[rows]) * np.exp(1j * phase[rows].astype(np.float64))
    for got, want, what in ((w12[rows], rw12, "w12"), (ph, np.abs(rw12) * np.exp(1j * rph), "phase")):
        ratio, where = cr.row_gate(got, want, tol, resolved)
        assert ratio <= 1.0, f"{what}: {ratio:.3g} of the row bound at row {rows[where[0]]}, t = {where[1]}"
        worst = max(worst, ratio)
        if not resolved.all():
            b = np.abs(want[~resolved])
            assert np.all(np.abs(got[~resolved] - want[~resolved]) <= tol * b + tol * np.abs(want).max()), what
    return worst


# ---- against the reference ---------------------------------------------------------------------------
@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("f64", [False, True], ids=["fp32-8193", "fp64-4097"])
def test_first_new_lengths(shim, f64, inp):
    n0 = 4097 if f64 else 8193
    y = _inputs(inp, 1, n0, seed=n0 + len(inp))
    (wct, phase, w12), launches = _xwt(shim, y, 1 / 4, -1, f64)
    S = wct.shape[1]
    assert launches == wl.xwt_launches(1, n0, _nfft(n0), S, f64, w12=True), "the long path did not serve the call"
    worst = _check(shim, y[0], 1 / 4, -1, f64, np.arange(S), (wct[0], phase[0], w12[0]))
    print(f"WCTLONG {'fp64' if f64 else 'fp32'} {n0} {inp}: {worst:.3g}")


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("n0,inp", [(1 << 17, "ar1_0.989"), (1 << 20, "white")])
def test_longer_series(shim, n0, inp, f64):
    y = _inputs(inp, 1, n0, seed=7)
    (wct, phase, w12), launches = _xwt(shim, y, 1 / 2, -1, f64)
    S = wct.shape[1]
    assert launches == wl.xwt_launches(1, n0, n0, S, f64, w12=True)
    rows = np.arange(S) if n0 <= 1 << 17 else np.unique(np.r_[0, np.arange(1, S, 4), S - 1])
    worst = _check(shim, y[0], 1 / 2, -1, f64, rows, (wct[0], phase[0], w12[0]))
    print(f"WCTLONG {'fp64' if f64 else 'fp32'} {n0} {inp}: {worst:.3g}")


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_three_million_samples(shim, f64):
    n0, J = 3_000_000, 16
    y = _inputs("ar1_0.989", 1, n0, seed=8)
    (wct, phase, w12), launches = _xwt(shim, y, 1.0, J, f64)
    assert wct.shape == (1, J + 1, n0) and launches == wl.xwt_launches(1, n0, 1 << 22, J + 1, f64, w12=True)
    worst = _check(shim, y[0], 1.0, J, f64, np.array([0, 5, 10, 13, 16]), (wct[0], phase[0], w12[0]))
    print(f"WCTLONG {'fp64' if f64 else 'fp32'} {n0} ar1: {worst:.3g}")


@pytest.mark.parametrize("f64,n0", [(False, 8193), (True, 4097), (False, 1 << 17)])
def test_w12_is_the_product_of_the_cwt_coefficients(shim, f64, n0):
    """Same forward transforms and daughter arithmetic as wtb_cwt: W12 is W1 conj(W2) of its coefficients up to
    the rounding of one complex product."""
    y = _inputs("white", 1, n0, seed=20)
    (_, _, w12), _ = _xwt(shim, y, 1 / 4, -1, f64, wct=False, phase=False)
    _, W = shim.cwt(y[0], DT, 1 / 4, -1, -1, 0, 6.0, f64=f64, want_power=False, want_coef=True)
    W = W.astype(np.complex128)
    ref = W[0] * np.conj(W[1])
    eps = np.finfo(np.float64 if f64 else np.float32).eps
    err = np.abs(w12[0].astype(np.complex128) - ref) / (np.abs(W[0]) * np.abs(W[1]) * eps + 1e-300)
    assert err.max() <= 4.0, f"{err.max():.3g} ulp"


# ---- dispatch and refusals -----------------------------------------------------------------------------
@pytest.mark.parametrize("f64,n0", [(False, 8192), (True, 4096)])
def test_largest_one_cta_lengths_keep_the_generic_path(shim, f64, n0):
    y = _inputs("white", 1, n0, seed=10)
    _, launches = _xwt(shim, y, 1 / 4, -1, f64, w12=False)
    assert wl.route(n0, f64) == "generic" and wl.route(2 * n0, f64) == "long"
    assert launches == 3          # forward transforms, k_wct_rows, k_wct_scale


@pytest.mark.parametrize("f64", [False, True])
def test_refusals(shim, f64):
    lib = shim.lib()
    rt = np.float64 if f64 else np.float32
    x = np.random.default_rng(3).standard_normal((1, 5000)).astype(rt)
    out = np.zeros((1, 9, 5000), rt)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    flags = shim.F64 if f64 else 0
    before = shim.kernel_launches()
    assert lib.wtb_xwt_wct(p(x), p(x), 1, 5000, 1 << 23, DT, 1.0, 2.0, 8, 6.0, flags, p(out), None, None,
                           None) == EUNSUPPORTED
    assert b"2^22" in lib.wtb_last_error()
    # un-padded lengths past the one-CTA limit: the refusal and message are unchanged
    assert lib.wtb_xwt_wct(p(x), p(x), 1, 5000, 5000, DT, 1.0, 2.0, 8, 6.0, flags, p(out), None, None,
                           None) == EUNSUPPORTED
    B = 3 * (16 if f64 else 8) * 16384
    assert lib.wtb_last_error() == (f"nfft=5000 needs {B} B of shared memory per CTA (limit 227 KB): a power of two "
                                    f"up to {4096 if f64 else 8192}, any other length up to {2048 if f64 else 4096} "
                                    f"for {'double' if f64 else 'float'}").encode()
    assert shim.kernel_launches() == before


# ---- invariance ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("f64,n0", [(False, 1 << 17), (True, 1 << 16)])
def test_bits_do_not_depend_on_the_batch(shim, f64, n0):
    """16 rows per wave: in batches of 3 and 1 the wave boundaries fall on different scales of a pair."""
    y = _inputs("ar1_0.989", 3, n0, seed=11)
    o3, _ = _xwt(shim, y, 1 / 2, -1, f64)
    S = o3[0].shape[1]
    assert wl.wave_rows(n0, f64, 3 * S) == 16 and S % 16
    for i in (0, 2):
        o1, _ = _xwt(shim, y[i:i + 1], 1 / 2, -1, f64)
        for a, b in zip(o1, o3):
            assert np.array_equal(a[0], b[i], equal_nan=True)


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
    y = _inputs("two_tone", 5, 1 << 15 if f64 else 1 << 16, seed=12)
    o2, _ = _xwt(shim, y, 1 / 2, -1, f64)
    shim.init_multi(1)
    o1, _ = _xwt(shim, y, 1 / 2, -1, f64)
    for a, b in zip(o1, o2):
        assert np.array_equal(a, b, equal_nan=True)


def _device_call(shim, torch, y1, y2, dj, J, f64, wct, phase, w12):
    batch, n0 = y1.shape
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    rc = shim.lib().wtb_xwt_wct(ptr(y1), ptr(y2), batch, n0, _nfft(n0), DT, dj, -1.0, J, 6.0, flags, ptr(wct),
                                ptr(phase), ptr(w12), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, shim.lib().wtb_last_error()


@pytest.mark.parametrize("f64", [False, True])
def test_device_pointers_equal_host_buffers(shim, f64):
    import torch
    n0 = 20001
    y = _inputs("two_tone", 2, n0, seed=13)
    o, _ = _xwt(shim, y, 1 / 4, -1, f64)
    dtype = torch.float64 if f64 else torch.float32
    y1 = torch.as_tensor(y[:, 0], dtype=dtype, device="cuda").contiguous()
    y2 = torch.as_tensor(y[:, 1], dtype=dtype, device="cuda").contiguous()
    wct = torch.empty(o[0].shape, dtype=dtype, device="cuda")
    phase = torch.empty_like(wct)
    w12 = torch.empty(o[0].shape, dtype=torch.complex128 if f64 else torch.complex64, device="cuda")
    _device_call(shim, torch, y1, y2, 1 / 4, o[0].shape[1] - 1, f64, wct, phase, w12)
    torch.cuda.synchronize()
    for a, b in zip((wct, phase, w12), o):
        assert np.array_equal(a.cpu().numpy(), b, equal_nan=True)


GUARD = 4096


def _guarded(torch, n, dtype):
    buf = torch.full((n + 2 * GUARD,), -7.0e33, dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n]


def _intact(buf, n):
    return bool((buf[:GUARD] == -7.0e33).all()) and bool((buf[GUARD + n:] == -7.0e33).all())


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n0", [8193, 70001])
def test_writes_stay_inside_their_outputs(shim, n0, f64):
    import torch
    dtype = torch.float64 if f64 else torch.float32
    batch, J = 3, 20                      # largest scale ~2000 samples: finite coherence in FP32 as well
    g = torch.Generator("cuda").manual_seed(n0)
    y1 = torch.randn(batch, n0, dtype=dtype, device="cuda", generator=g)
    y2 = torch.randn(batch, n0, dtype=dtype, device="cuda", generator=g)
    n = batch * (J + 1) * n0
    bufs = [_guarded(torch, m, dtype) for m in (n, n, 2 * n)]
    _device_call(shim, torch, y1, y2, 1 / 2, J, f64, *(v for _, v in bufs))
    torch.cuda.synchronize()
    for (buf, v), m in zip(bufs, (n, n, 2 * n)):
        assert _intact(buf, m) and bool(torch.isfinite(v).all())


# ---- Monte Carlo ---------------------------------------------------------------------------------------
# run_wct's geometry for a 2000-sample pair: dt 1/12, dj 1/8, s0 2 dt, J 80 -> 12288-sample surrogates
MC_DT, MC_DJ, MC_J = 1 / 12, 1 / 8, 80
MC_S0 = 2 * MC_DT
A1, A2 = 0.72, 0.55


def _mc(shim, **kw):
    return shim.wct_mc_hist(A1, A2, MC_DT, MC_DJ, MC_S0, MC_J, **kw).astype(np.int64)


def test_mc_geometry_takes_the_long_path(shim):
    nsurr, _ = shim.wct_mc_geometry(MC_DT, MC_DJ, MC_S0, MC_J)
    assert nsurr == 12288 and wl.route(wl.mc_nfft(nsurr), False) == "long"


def test_mc_fp32_device_rng(shim):
    nsurr, _ = shim.wct_mc_geometry(MC_DT, MC_DJ, MC_S0, MC_J)
    count, seed = 3, 17
    hist = _mc(shim, mc_count=count, seed=seed, f64=False)
    samples = mo.mc_samples(mo.device_surrogates(A1, A2, nsurr, 0, count, seed), MC_DT, MC_DJ, MC_S0, MC_J)
    print(f"MCLONG fp32 smallest passing delta {mo.hist_delta(hist, samples):.3g}")
    mo.assert_hist_matches(hist, samples, 2e-4)


def test_mc_fp64_device_surrogates(shim):
    nsurr, _ = shim.wct_mc_geometry(MC_DT, MC_DJ, MC_S0, MC_J)
    count, seed = 2, 23
    hist = _mc(shim, mc_count=count, seed=seed, f64=True)
    sur = shim.rednoise(A1, A2, nsurr, 0, count, seed, f64=True)
    samples = mo.mc_samples(sur, MC_DT, MC_DJ, MC_S0, MC_J)
    print(f"MCLONG fp64 smallest passing delta {mo.hist_delta(hist, samples):.3g}")
    mo.assert_hist_matches(hist, samples, 1e-10)


@pytest.mark.parametrize("f64", [False, True])
def test_mc_injected_chunks_equal_one_chunk(shim, f64):
    nsurr, _ = shim.wct_mc_geometry(MC_DT, MC_DJ, MC_S0, MC_J)
    count = 5
    sur = np.random.default_rng(31).standard_normal((count, 2, nsurr))
    one = _mc(shim, mc_count=count, surrogates=sur, f64=f64)
    per = wl.pair_bytes(nsurr, wl.mc_nfft(nsurr), MC_J + 1, f64) + (16 if f64 else 8) * nsurr
    os.environ["WTB_MC_CHUNK_MB"] = str(-(-2 * per // (1 << 20)))       # two realisations per chunk: 3 chunks
    try:
        chunked = _mc(shim, mc_count=count, surrogates=sur, f64=f64)
    finally:
        del os.environ["WTB_MC_CHUNK_MB"]
    assert np.array_equal(one, chunked) and one.sum() > 0


def test_mc_first_split_sums_to_the_whole(shim):
    whole = _mc(shim, mc_count=5, seed=41, f64=False)
    parts = _mc(shim, mc_first=0, mc_count=2, seed=41, f64=False) + _mc(shim, mc_first=2, mc_count=3, seed=41,
                                                                         f64=False)
    assert np.array_equal(whole, parts)


def test_one_call_significance(shim):
    nsurr, maxscale = shim.wct_mc_geometry(MC_DT, MC_DJ, MC_S0, MC_J)
    count = 2
    rng = np.random.default_rng(43)
    sur = np.stack([np.stack([po.rednoise(nsurr, A1, 1, rng), po.rednoise(nsurr, A2, 1, rng)]) for _ in range(count)])
    sig, hist = shim.wct_significance(A1, A2, MC_DT, MC_DJ, MC_S0, MC_J, mc_count=count, surrogates=sur, f64=True,
                                      return_hist=True)
    ref_sig, ref_hist = po.wct_significance(A1, A2, MC_DT, MC_DJ, MC_S0, MC_J, mc_count=count, surrogates=sur,
                                            return_hist=True)
    samples = mo.mc_samples(sur, MC_DT, MC_DJ, MC_S0, MC_J)
    mo.assert_hist_matches(hist.astype(np.int64), samples, 1e-10)
    assert np.array_equal(hist.astype(np.int64)[:maxscale], np.asarray(ref_hist, dtype=np.int64)[:maxscale])
    both = np.isfinite(ref_sig[:maxscale])
    assert np.array_equal(np.isfinite(sig[:maxscale]), both)
    assert np.allclose(sig[:maxscale][both], ref_sig[:maxscale][both], rtol=1e-12, atol=1e-12)


# ---- façades -------------------------------------------------------------------------------------------
def _real_pair(n0, seed):
    y = _inputs("ar1_0.989", 1, n0, seed)[0]
    return y[0] * 3.0 + 1.0, y[1] - 2.0


def test_pycwt_compat_wct_with_significance(shim):
    from wavelet_transformer_b200 import pycwt_compat as pc
    y1, y2 = _real_pair(2000, 50)
    dt, dj, s0 = 1 / 12, 1 / 8, 2 / 12
    WCT, aWCT, coi, freq, sig = pc.wct(y1, y2, dt, dj, s0, -1, sig=True, mc_count=8, cache=False)
    ref = po.wct(y1, y2, dt, dj=dj, s0=s0, J=-1, sig=False)
    assert WCT.shape == ref[0].shape and sig.shape == (WCT.shape[0],)
    assert np.abs(WCT - ref[0]).max() <= 1e-10
    assert np.allclose(coi, ref[2], rtol=1e-13) and np.allclose(freq, ref[3], rtol=1e-13)
    _, maxscale = shim.wct_mc_geometry(dt, dj, s0, WCT.shape[0] - 1)
    assert np.all(np.isfinite(sig[:maxscale])) and np.all((sig[:maxscale] > 0) & (sig[:maxscale] <= 1))


def test_pycwt_compat_wct_and_xwt_of_10000_samples(shim):
    from wavelet_transformer_b200 import pycwt_compat as pc
    y1, y2 = _real_pair(10000, 51)
    WCT, aWCT, _, _, _ = pc.wct(y1, y2, 1.0, 1 / 12, -1, -1, sig=False)
    ref = po.wct(y1, y2, 1.0, dj=1 / 12, s0=-1, J=-1, sig=False)
    assert np.abs(WCT - ref[0]).max() <= 1e-10
    W12, _, _, signif = pc.xwt(y1, y2, 1.0, 1 / 12, -1, -1)
    rW12, _, _, rsignif = po.xwt(y1, y2, 1.0, dj=1 / 12, s0=-1, J=-1)
    ratio, where = cr.row_gate(W12, rW12, 1e-10)
    assert ratio <= 1.0, f"{ratio:.3g} of the row bound at {where}"
    ph = np.abs(W12) * np.exp(1j * aWCT)
    ratio, where = cr.row_gate(ph, rW12, 1e-10)
    assert ratio <= 1.0, f"phase: {ratio:.3g} of the row bound at {where}"
    assert np.allclose(signif, rsignif, rtol=1e-12)


def test_run_wct_of_a_2000_sample_pair(shim):
    from wavelet_transformer_b200.api import wct as api
    y1, y2 = _real_pair(2000, 52)
    d = api.DataForWCT(y1, y2, api.MOTHER, api.DT, api.DJ, api.S0, api.WCT_LEVELS)
    os.environ["WTB_CACHE_DIR"] = os.environ.get("TMPDIR", "/tmp") + "/wtb_wct_long_test_cache"
    try:
        res = api.run_wct(d, calculate_signficance=True)
    finally:
        del os.environ["WTB_CACHE_DIR"]
    ref = po.wct(y1, y2, api.DT, dj=api.DJ, s0=api.S0, J=-1, sig=False)
    assert np.abs(res.coherence - ref[0]).max() <= 1e-10
    assert np.allclose(res.period, 1 / ref[3], rtol=1e-13)
    assert res.significance_levels.shape == ref[0].shape and np.isfinite(res.significance_levels).any()


def test_engine_wct_batch_resident_at_8193(shim):
    import torch
    from wavelet_transformer_b200 import engine
    n0 = 8193
    y = _inputs("white", 2, n0, seed=53)
    o, launches = _xwt(shim, y, 1 / 8, -1, False, w12=False)
    assert launches == wl.xwt_launches(2, n0, _nfft(n0), o[0].shape[1], False)
    y1 = torch.as_tensor(y[:, 0], dtype=torch.float32, device="cuda").contiguous()
    y2 = torch.as_tensor(y[:, 1], dtype=torch.float32, device="cuda").contiguous()
    res = engine.wct_batch_resident(y1, y2, DT, 1 / 8, -1, -1)
    torch.cuda.synchronize()
    assert np.array_equal(res["coherence"].cpu().numpy(), o[0], equal_nan=True)
    assert np.array_equal(res["phase"].cpu().numpy(), o[1])
