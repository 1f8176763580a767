"""GPU: Monte-Carlo significance of partial and multiple wavelet coherence (wtb_partial_wct_mc_hist,
wtb_partial_wct_significance, wtb_rednoise_triples).

The surrogate triples are held to the Philox restatement and leave the pair generator as it was; the histograms of
device-RNG runs are held per realisation to the float64 closed forms, each sample within its own rounding band
tol * kappa * (1 + |v|) (tol 1e-4 FP32, 1e-10 FP64, kappa the conditioning of the ratio, the gate of
test_gpu_pwct.py); injected surrogates, chunk sizes and a pool of two give the same bits; the one-call thresholds
are the percentile step of each half; refusals come before any launch and leave the histogram untouched."""

import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from oracle import mc_oracle as mo
from oracle import pwct_mc_oracle as pmo
from oracle import pwct_oracle as pw
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1 / 12
CFG3 = (1 / 8, 65)                         # dj, J with s0 = 2 dt: 3351-sample surrogates, padded to 4096
SEED = 0x9E3779B9_00C0FFEE                 # non-zero high word: both key words matter
FIRST = 2**32 - 2                          # four realisations cross the counter's high word
COEFS = [(0.7, 0.7, 0.7), (0.989, 0.966, 0.5), (-0.3, 0.0, 0.9)]
TOL = {False: 1e-4, True: 1e-10}
EINVAL, EUNSUPPORTED = -1, -3


def _geometry(dj, J):
    N, _, _, outside, maxscale = po.mc_geometry(DT, dj, 2 * DT, J, po.Morlet())
    return N, maxscale, outside.any(axis=1)


def _reference(sur, dj, J, pad, f64):
    """Per half, the samples and bands of every realisation of [mc, 3, N] surrogates, concatenated per row."""
    per = [pmo.partial_coherence_samples(*np.asarray(t, dtype=np.float64), DT, dj, 2 * DT, J, pad_pow2=pad,
                                         tol=TOL[f64]) for t in sur]
    cat = lambda k, h: [np.concatenate([p[k][h][s] for p in per]) for s in range(J + 1)]
    return [(cat(0, h), cat(1, h)) for h in range(2)]


def _assert_matches(hist, ref):
    assert hist.shape[0] == 2
    for h, (values, bands) in enumerate(ref):
        try:
            pmo.assert_hist_matches_banded(hist[h], values, bands)
        except AssertionError as e:
            raise AssertionError(f"{('PWC', 'MWC')[h]} half: {e}") from None


def _padding(shim, mode):
    old = shim.get_fft_padding()
    shim.set_fft_padding(mode)
    return old


# ---------------------------------------------------------------- surrogates
def test_pairs_are_untouched(shim):
    """wtb_rednoise keeps its stream (the restatement of noise.cu as it was), its triples extend it (series 0 and
    1 of a triple are the pair, bit for bit), and the cfg5 job of bench.py -- 100 000 realisations, FP32, seed
    2024 -- still bins to the histogram recorded in profiles/r2_scale_n*_mc.json."""
    for f64 in (False, True):
        pair = shim.rednoise(0.989, 0.966, 3351, FIRST, 4, SEED, f64=f64)
        tri = shim.rednoise_triples(0.989, 0.966, 0.5, 3351, FIRST, 4, SEED, f64=f64)
        assert np.array_equal(tri[:, :2], pair)
        ref = mo.device_surrogates(0.989, 0.966, 3351, FIRST, 4, SEED)
        assert np.abs(pair - ref).max() <= 1e-5 * np.abs(ref).max() + (0 if f64 else np.abs(ref).max() * 2.0**-24)
    hist = shim.wct_mc_hist(0.989, 0.966, DT, 1 / 8, 2 * DT, 65, mc_first=0, mc_count=100_000, seed=2024, f64=False)
    assert hashlib.sha256(hist.tobytes()).hexdigest()[:16] == "aa520ec808fadc82"


@pytest.mark.parametrize("white", [False, True], ids=["red", "white"])
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_triples_are_the_philox_stream(shim, white, f64):
    """The tolerances of test_rednoise_is_the_philox_stream."""
    for (ay, a1, a2), (nsurr, first, count) in zip(COEFS, [(5, 99_996, 4), (3351, FIRST, 4), (1, 0, 3)]):
        dev = shim.rednoise_triples(ay, a1, a2, nsurr, first, count, SEED, f64=f64, white=white).astype(np.float64)
        ref = pmo.device_surrogate_triples(ay, a1, a2, nsurr, first, count, SEED, white=white)
        err = np.abs(dev - ref)
        if white:
            bound = 1e-6 * (1 + np.abs(ref))
        else:
            bound = 1e-5 * np.abs(ref).max(axis=-1, keepdims=True)
        if not f64:
            bound = bound + np.abs(ref) * 2.0**-24
        bad = np.argwhere(err > bound)
        assert bad.size == 0, (nsurr, first, count, bad[:4].tolist(), float(err.max()))


# ---------------------------------------------------------------- histograms against the oracle
def _device_rng_case(shim, coefs, dj, J, f64, pad, generic=False, mc=4):
    N, _, _ = _geometry(dj, J)
    old = _padding(shim, "pow2" if pad else "none")
    try:
        hist = shim.partial_wct_mc_hist(*coefs, DT, dj, 2 * DT, J, mc_first=FIRST, mc_count=mc, seed=SEED, f64=f64,
                                        generic_only=generic)
    finally:
        shim.set_fft_padding(old)
    # FP64: the device's own FP64 triples (its float32 Box-Muller normals are ~1e-7 off the float64 restatement,
    # far outside the 1e-10 band; the triples themselves are held to the restatement above)
    sur = (shim.rednoise_triples(*coefs, N, FIRST, mc, SEED, f64=True) if f64
           else pmo.device_surrogate_triples(*coefs, N, FIRST, mc, SEED))
    _assert_matches(hist, _reference(sur, dj, J, pad, f64))
    return hist


@pytest.mark.parametrize("coefs", COEFS, ids=["a0.7", "red", "mixed"])
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_device_rng_cfg3(shim, coefs, f64):
    hist = _device_rng_case(shim, coefs, *CFG3, f64, pad=True)
    assert hist.sum() > 0


def test_device_rng_unpadded_fp32(shim):
    """914-sample surrogates transformed at their own length (Bluestein), set_fft_padding('none')."""
    dj, J = 1 / 8, 50
    assert _geometry(dj, J)[0] == 914
    _device_rng_case(shim, COEFS[1], dj, J, False, pad=False)


def test_device_rng_generic_only(shim):
    _device_rng_case(shim, COEFS[0], *CFG3, False, pad=True, generic=True)


# ---------------------------------------------------------------- the same bits every way
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_injected_device_surrogates_give_the_device_rng_histogram(shim, f64):
    dj, J = CFG3
    N, _, _ = _geometry(dj, J)
    rng = shim.partial_wct_mc_hist(*COEFS[1], DT, dj, 2 * DT, J, mc_first=FIRST, mc_count=3, seed=SEED, f64=f64)
    sur = shim.rednoise_triples(*COEFS[1], N, FIRST, 3, SEED, f64=f64)
    inj = shim.partial_wct_mc_hist(*COEFS[1], DT, dj, 2 * DT, J, mc_count=3, surrogates=sur, f64=f64)
    assert np.array_equal(inj, rng)


# cfg3 costs 13 310 172 B of staging per triple in FP32 and twice that in FP64 (pwct.cu, per_triple): 26 / 52 MB
# budgets hold two triples, so seven realisations run as chunks of 2, 2, 2 and 1; 1 MB holds none (one per chunk).
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_bits_do_not_depend_on_the_chunks(shim, monkeypatch, f64):
    dj, J = CFG3
    args = (*COEFS[0], DT, dj, 2 * DT, J)
    N, _, _ = _geometry(dj, J)
    sur = shim.rednoise_triples(*COEFS[0], N, 4242, 7, SEED, f64=f64)
    whole = shim.partial_wct_mc_hist(*args, mc_first=4242, mc_count=7, seed=SEED, f64=f64)
    for mb in ({False: "26", True: "52"}[f64], "1"):
        monkeypatch.setenv("WTB_MC_CHUNK_MB", mb)
        assert np.array_equal(shim.partial_wct_mc_hist(*args, mc_first=4242, mc_count=7, seed=SEED, f64=f64), whole)
        assert np.array_equal(shim.partial_wct_mc_hist(*args, mc_count=7, surrogates=sur, f64=f64), whole)
    monkeypatch.delenv("WTB_MC_CHUNK_MB")


@pytest.fixture()
def pool(shim):
    """A pool of two workers: two GPUs when the box has them, one shared GPU otherwise."""
    os.environ["WTB_POOL_SHARE_DEVICES"] = "1"
    n = shim.init_multi(2)
    assert n == 2
    yield shim
    shim.init_multi(1)
    assert shim.gpu_count() == 1


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_split_over_the_pool(shim, pool, f64):
    dj, J = CFG3
    N, _, _ = _geometry(dj, J)
    args = (*COEFS[2], DT, dj, 2 * DT, J)
    sur = shim.rednoise_triples(*COEFS[2], N, 0, 5, SEED, f64=f64)
    two = shim.partial_wct_significance(*args, mc_count=5, seed=SEED, f64=f64, return_hist=True)
    two_inj = shim.partial_wct_significance(*args, mc_count=5, surrogates=sur, f64=f64, return_hist=True)
    shim.init_multi(1)
    one = shim.partial_wct_significance(*args, mc_count=5, seed=SEED, f64=f64, return_hist=True)
    hist = shim.partial_wct_mc_hist(*args, mc_count=5, seed=SEED, f64=f64)
    assert np.array_equal(one[2], hist)
    for got in (two, two_inj):
        assert np.array_equal(got[2], hist)
        for a, b in zip(got[:2], one[:2]):
            assert np.array_equal(a, b, equal_nan=True)


def test_thresholds_are_the_percentile_step_of_each_half(shim):
    dj, J = CFG3
    _, maxscale, rows_any = _geometry(dj, J)
    sig_pwc, sig_mwc, hist = shim.partial_wct_significance(*COEFS[1], DT, dj, 2 * DT, J, level=0.9, mc_count=6,
                                                           seed=SEED, f64=False, return_hist=True)
    has = shim.row_has_points(DT, dj, 2 * DT, J)
    assert np.array_equal(has, rows_any)
    for h, sig in enumerate((sig_pwc, sig_mwc)):
        assert sig.shape == (J + 1,)
        assert np.array_equal(sig, shim.wct_sig_from_hist(hist[h], maxscale, 0.9, has), equal_nan=True)
        assert np.all(np.isfinite(sig[:maxscale])) and np.all((sig[:maxscale] > 0) & (sig[:maxscale] < 1))
    assert np.array_equal(hist, shim.partial_wct_mc_hist(*COEFS[1], DT, dj, 2 * DT, J, mc_count=6, seed=SEED,
                                                         f64=False))


# ---------------------------------------------------------------- refusals and bounds
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_refusals_leave_the_histogram_untouched(shim, f64):
    lib = shim.lib()
    dj, J = CFG3
    # a 1346-sample series at dj 1/12 (J 113): 8202-sample surrogates, padded to 16384: past one CTA in both
    # precisions; FP64 also refuses cfg3 un-padded (3351 > 2048)
    refused = [(1 / 12, 113, "pow2")] + ([(dj, J, "none")] if f64 else [])
    pow2, other = (4096, 2048) if f64 else (8192, 4096)
    limit = f"a power of two up to {pow2}, any other length up to {other} for {'double' if f64 else 'float'}"
    before = shim.kernel_launches()
    hist = np.full((2, J + 1, shim.NBINS), 7, dtype=np.uint64)
    for rdj, rJ, pad in refused:
        old = _padding(shim, pad)
        try:
            h = np.full((2, rJ + 1, shim.NBINS), 7, dtype=np.uint64)
            with pytest.raises(shim.WaveletEngineError, match="past one CTA"):
                shim.partial_wct_mc_hist(0.5, 0.5, 0.5, DT, rdj, 2 * DT, rJ, mc_count=2, f64=f64, hist=h)
            assert limit in lib.wtb_last_error().decode()
            assert (h == 7).all()
            with pytest.raises(shim.WaveletEngineError, match="past one CTA"):
                shim.partial_wct_significance(0.5, 0.5, 0.5, DT, rdj, 2 * DT, rJ, mc_count=2, f64=f64)
        finally:
            shim.set_fft_padding(old)
    for coefs in [(1.0, 0.5, 0.5), (0.5, -1.0, 0.5), (0.5, 0.5, 1.5), (0.5, 0.5, float("nan")),
                  (float("nan"), 0.5, 0.5)]:
        with pytest.raises(ValueError, match="AR\\(1\\) coefficients"):
            shim.partial_wct_mc_hist(*coefs, DT, dj, 2 * DT, J, mc_count=2, f64=f64, hist=hist)
        with pytest.raises(ValueError, match="AR\\(1\\) coefficients"):
            shim.partial_wct_significance(*coefs, DT, dj, 2 * DT, J, mc_count=2, f64=f64)
    flags = shim.F64 if f64 else 0
    p = hist.ctypes.data_as(C.c_void_p)
    assert lib.wtb_partial_wct_mc_hist(0.5, 0.5, 0.5, DT, dj, 2 * DT, -1, 6.0, 0, 2, 0, None, flags, p, None) == EINVAL
    sig = np.zeros(J + 1)
    assert lib.wtb_partial_wct_significance(0.5, 0.5, 0.5, DT, dj, 2 * DT, -1, 6.0, 0.95, 2, 0, None, flags,
                                            sig.ctypes.data_as(shim._pd), sig.ctypes.data_as(shim._pd), None) == EINVAL
    N, _, _ = _geometry(dj, J)
    for shape in [(2, 2, N), (2, 3, N - 1), (3, 3, N)]:
        with pytest.raises(ValueError, match="surrogates must have shape"):
            shim.partial_wct_mc_hist(0.5, 0.5, 0.5, DT, dj, 2 * DT, J, mc_count=2, f64=f64, hist=hist,
                                     surrogates=np.zeros(shape))
    # mc_count == 0 is a no-op
    assert lib.wtb_partial_wct_mc_hist(0.5, 0.5, 0.5, DT, dj, 2 * DT, J, 6.0, 0, 0, 0, None, flags, p, None) == 0
    assert shim.kernel_launches() == before and (hist == 7).all()


GUARD = 4096


@pytest.mark.parametrize("f64,dj,J", [(False, 1 / 8, 65), (True, 1 / 4, 24)])
def test_writes_stay_inside_the_histogram(shim, f64, dj, J):
    """A device histogram in the middle of a pattern-filled buffer: the surroundings come back untouched, and
    the counts equal the host-buffer call's."""
    import torch
    n = 2 * (J + 1) * shim.NBINS
    buf = torch.full((n + 2 * GUARD,), -77, dtype=torch.int64, device="cuda")
    view = buf[GUARD:GUARD + n]
    view.zero_()
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    rc = shim.lib().wtb_partial_wct_mc_hist(*COEFS[0], DT, dj, 2 * DT, J, 6.0, 5, 3, SEED, None, flags,
                                            C.c_void_p(view.data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, shim.lib().wtb_last_error()
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == -77).all()) and bool((buf[GUARD + n:] == -77).all())
    host = shim.partial_wct_mc_hist(*COEFS[0], DT, dj, 2 * DT, J, mc_first=5, mc_count=3, seed=SEED, f64=f64)
    assert np.array_equal(view.cpu().numpy().astype(np.uint64).reshape(host.shape), host) and host.sum() > 0


# ---------------------------------------------------------------- façade
def test_partial_wct_sig(shim):
    """sig=True appends the thresholds of partial_wct_significance for the ar1 coefficients of the normalised
    series (FP32 with the device RNG) and leaves the planes as they are."""
    import wavelet_transformer_b200 as wtb
    from wavelet_transformer_b200.pycwt_compat import ar1
    y, x1, x2 = (3.0 * v + c for v, c in zip(pw.triple("built", 565, seed=21), (1.0, -2.0, 0.5)))
    dj = 1 / 8
    plain = wtb.partial_wct(y, x1, x2, DT, dj, 2 * DT)
    out = wtb.partial_wct(y, x1, x2, DT, dj, 2 * DT, sig=True, significance_level=0.9, mc_count=12, seed=3)
    assert len(plain) == 6 and len(out) == 8
    for a, b in zip(out[:6], plain):
        assert np.array_equal(a, b, equal_nan=True)
    J = len(plain[5]) - 1
    assert J == CFG3[1]
    norm = [(v - v.mean()) / v.std() for v in (y, x1, x2)]
    coefs = [ar1(v)[0] for v in norm]
    ref = wtb.partial_wct_significance(*coefs, DT, dj, 2 * DT, J, significance_level=0.9, mc_count=12, seed=3)
    direct = shim.partial_wct_significance(*coefs, DT, dj, 2 * DT, J, level=0.9, mc_count=12, seed=3, f64=False)
    for a, b, c in zip(out[6:], ref, direct):
        assert a.shape == (J + 1,)
        assert np.array_equal(a, b, equal_nan=True) and np.array_equal(a, c, equal_nan=True)
    trend = np.arange(565, dtype=float) ** 2
    with pytest.raises(Warning, match="upperbound"):
        wtb.partial_wct(trend, x1, x2, DT, dj, 2 * DT, sig=True, mc_count=2)
