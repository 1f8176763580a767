"""GPU: the one-CTA generic CWT and coherence kernels held row by row to float64 references.

k_fwd_fft + k_cwt_rows (cwt.cu) and k_fwd_fft + k_wct_rows + k_wct_scale (wct.cu), over plan_fft of
fft_block.cuh, serve every un-padded transform (Bluestein's chirp-z transform at a work length
M = 2^ceil(log2(2 nfft - 1))), every Paul and DOG transform and every Morlet with f0 < 5.3 up to one CTA's
shared memory, every power of two below 512 and every FP64 transform.  Each case proves by its launch count
that these kernels served it, runs a batch of three distinct series and checks the first and the last:

* the CWT at both ends of every Bluestein work-length class (M = 8 .. 8192, so every thread count 64 / 128 /
  256 of the plan), at powers of two from 2 to the largest one-CTA length, and at explicit lengths that are
  neither n0 nor the next power of two, for Morlet 6, Paul 4, DOG 2 and DOG 3 (odd order: imaginary
  prefactor), power and coefficients, against ``cwt_long.cwt_rows`` at the transform length itself;
* Morlet with f0 = 4 and 5.29, which the FP32 plan sends to the generic kernels;
* the cross spectrum, its phase and the coherence for boxcar widths K = 1, 2, 5, 10 and 14;
* ``wtb_cwt_averages`` and ``wtb_icwt`` on top of the same transforms;
* the limits of the un-padded transforms: the longest accepted length, the refusal past it, and writes that
  stay inside their outputs.

Gates (oracle/cwt_rows.row_gate): 1e-10 in FP64 and 1e-4 in FP32 on every scale row, Morlet included.  The
generic kernels evaluate the whole daughter at every bin (no one-sided band cut), so the rows that
``resolved_rows`` excludes for the fast kernels are held to the same per-row bound; their worst ratio is
printed as ``tail``.  The FP32 references are computed from the FP32-rounded inputs.  ``wtb_icwt`` also takes
more than 65535 series in one call (one launch per 65535)."""

import ctypes as C

import numpy as np
import pytest
from scipy.signal import lfilter

from conftest import normwise_close
from oracle import averages as oa
from oracle import cwt_long as cl
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1.0
DJ = 1 / 4
EUNSUPPORTED = -3
MOTHERS = {"morlet": (0, 6.0, po.Morlet(6)), "paul4": (1, 4.0, po.Paul(4)), "dog2": (2, 2.0, po.DOG(2)),
           "dog3": (2, 3.0, po.DOG(3))}
INPUTS = ["white", "ar1_0.989", "two_tone"]


def _inputs(kind, batch, n0, seed):
    rng = np.random.default_rng(seed)
    if kind == "white":
        x = rng.standard_normal((batch, n0))
    elif kind == "ar1_0.989":
        x = lfilter([1.0], [1.0, -0.989], rng.standard_normal((batch, n0 + 2000)), axis=1)[:, 2000:]
    elif kind == "two_tone":
        t = np.arange(n0)
        period = rng.uniform(20.0, 60.0, size=(batch, 1))
        ph = rng.uniform(0, 2 * np.pi, size=(batch, 2))
        x = np.sin(2 * np.pi * t / period + ph[:, :1]) + 1e-3 * np.sin(2 * np.pi * t / 3.0 + ph[:, 1:])
    else:
        raise ValueError(kind)
    return x - x.mean(axis=1, keepdims=True)


def _pow2(n):
    return 1 << (n - 1).bit_length()


def _work_length(nfft):
    """plan_fft's work length: nfft for a power of two, else the Bluestein convolution length."""
    return nfft if nfft & (nfft - 1) == 0 else _pow2(2 * nfft - 1)


def _generic_only(f64, mother, f0, nfft):
    """FP32 Morlet with f0 >= 5.3 at nfft 512 .. 4096 has fast kernels; the flag keeps it on the generic ones."""
    return not f64 and mother == "morlet" and f0 >= cr.ZCUT_F32 and nfft in (512, 1024, 2048, 4096)


def _other_two_launch_plan(f64, mother, f0, nfft, generic):
    """cwt_plan's FP32 Morlet plans that also take two launches, so that a launch count of 2 alone would not
    prove k_fwd_fft + k_cwt_rows served a call: k_fwd_fft_pair2048 + k_cwt_dif<2> (nfft 2048, f0 >= 5.3) and
    the radix-16 forward kernel + k_cwt_rows_4096 or k_cwt_rows (nfft 4096, any f0).  Every case must stay
    off them."""
    if f64 or mother != "morlet" or generic:
        return False
    return (nfft == 2048 and f0 >= cr.ZCUT_F32) or nfft == 4096


def _gate(got, ref, tol, tail, what):
    """row_gate on every row; returns (worst ratio, worst ratio on the ``tail`` rows)."""
    ratio, where = cr.row_gate(got, ref, tol)
    assert ratio <= 1.0, f"{what}: {ratio:.3g} of the per-row bound at (row, t) = {where}"
    return ratio, cr.row_gate(got, ref, tol, tail)[0]


def _icwt_factor(wl, dj):
    """pycwt.icwt's factor dj dt^0.5 / (C_delta psi_0); odd DOG orders have psi_0 = 0 (no inverse in pycwt),
    where the sum itself is checked (factor 1)."""
    psi0 = np.pi ** -0.25 if isinstance(wl, po.Morlet) else wl.psi0()
    return dj * np.sqrt(DT) / (wl.cdelta * psi0) if psi0 != 0 else None


def _icwt_ref(W, sj, dj, wl):
    factor = _icwt_factor(wl, dj)
    if factor is None:
        return 1.0, (np.real(W) / np.sqrt(sj)[:, None]).sum(axis=0)
    return factor, po.icwt(W, sj, DT, dj, wl)


def _plane_close(got, ref, f64, what):
    if f64:
        err = np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-300)
        assert err <= 1e-10, f"{what}: {err:.3e}"
    else:
        ok, err = normwise_close(got, ref, 1e-4)
        assert ok, f"{what}: {err:.3e}"
    return err


# ---- the CWT ---------------------------------------------------------------------------------------------
def _cwt_case(shim, f64, n0, nfft, mother, inp, dj=DJ, f0=None, seed=0, power_only_call=False):
    code, param, wl = MOTHERS[mother]
    if f0 is not None:
        param, wl = f0, po.Morlet(f0)
    rt = np.float64 if f64 else np.float32
    x = _inputs(inp, 3, n0, seed).astype(rt)
    generic = _generic_only(f64, mother, param, nfft)
    assert not _other_two_launch_plan(f64, mother, param, nfft, generic), "the launch count would not prove the path"
    before = shim.kernel_launches()
    if power_only_call:
        # power alone is the call the fast kernels take when they can: its routing is what is under test
        p, _ = shim.cwt(x, DT, dj, -1, -1, code, param, nfft=nfft, f64=f64, generic_only=generic)
        assert shim.kernel_launches() - before == 2, "another kernel served the call"
        _, c = shim.cwt(x, DT, dj, -1, -1, code, param, nfft=nfft, f64=f64, want_power=False, want_coef=True,
                        generic_only=generic)
        assert shim.kernel_launches() - before == 4, "another kernel served the call"
    else:
        p, c = shim.cwt(x, DT, dj, -1, -1, code, param, nfft=nfft, f64=f64, want_power=True, want_coef=True,
                        generic_only=generic)
        assert shim.kernel_launches() - before == 2, "another kernel served the call"
    Jr, sj, _, _ = shim.cwt_axes_mother(n0, DT, dj, -1, -1, code, param)
    S = Jr + 1
    assert p.shape == (3, S, n0) and c.shape == (3, S, n0)
    tol = 1e-10 if f64 else 1e-4
    tail = ~cr.resolved_rows(n0, nfft, DT, dj, sj[0], Jr, f0=param) if code == 0 else np.zeros(S, bool)
    worst, worst_tail, worst_inv = 0.0, 0.0, 0.0
    # wtb_icwt on the kernel's own coefficients against pycwt.icwt of the same coefficients
    factor = _icwt_factor(wl, dj) or 1.0
    rec = shim.icwt(c, sj, factor, f64=f64)
    assert np.array_equal(rec[2], shim.icwt(c[2], sj, factor, f64=f64))
    for b in (0, 2):
        ref = cl.cwt_rows(x[b].astype(np.float64), DT, dj, -1, -1, wl, range(S), nfft=nfft)
        what = f"{mother} n0={n0} nfft={nfft} series {b}"
        want_p = np.abs(ref) ** 2
        if not f64:
            # the power as FP32 holds it (rounding: 6e-8 relative): a Morlet row of n0 = nfft = 2 is the daughter at
            # the Nyquist bin alone, exp(-72), whose power (1e-63) is below FP32's range and comes out 0
            want_p = want_p.astype(np.float32).astype(np.float64)
        for got, want, kind in ((p[b], want_p, "power"), (c[b], ref, "coef")):
            r, rt_ = _gate(got, want, tol, tail, f"{what} {kind}")
            worst, worst_tail = max(worst, r), max(worst_tail, rt_)
        _, inv_ref = _icwt_ref(c[b].astype(np.complex128), sj, dj, wl)
        worst_inv = max(worst_inv, _plane_close(rec[b], inv_ref, f64, f"{what} icwt"))
    return worst, worst_tail, worst_inv, int(tail.sum())


def _report(tag, f64, n0, nfft, worst, worst_tail, worst_inv, ntail):
    M = _work_length(nfft)
    print(f"ROWGATE cwt {'fp64' if f64 else 'fp32'} {tag} n0={n0} nfft={nfft} M={M}: {worst:.3g} "
          f"(tail {worst_tail:.3g} over {ntail} rows), icwt {worst_inv:.3g}")


BLUESTEIN_N0 = [3, 5, 7, 9, 15, 17, 31, 33, 63, 65, 127, 129, 255, 257, 511, 513, 1023, 1025, 2047]
# (n0, nfft): powers of two at the series' length and padded, up to the largest one-CTA length
POW2 = [(2, 2), (4, 4), (5, 8), (16, 16), (50, 64), (256, 256), (1000, 1024)]


def _length_cases():
    cases = []
    for f64 in (True, False):
        lengths = [(n, n) for n in BLUESTEIN_N0 + ([] if f64 else [2049, 4095])]
        lengths += POW2 + [(4096, 4096) if f64 else (8192, 8192)]
        for i, (n0, nfft) in enumerate(lengths):
            for j, mother in enumerate(MOTHERS):
                cases.append((f64, n0, nfft, mother, INPUTS[(i + j) % 3]))
    return cases


def _cid(c):
    return f"{'fp64' if c[0] else 'fp32'}-{c[1]}-{c[2]}-{c[3]}-{c[4]}"


@pytest.mark.parametrize("case", _length_cases(), ids=_cid)
def test_cwt_length_classes(shim, case):
    f64, n0, nfft, mother, inp = case
    res = _cwt_case(shim, f64, n0, nfft, mother, inp, seed=n0 * 7 + len(mother))
    _report(f"{mother} {inp}", f64, n0, nfft, *res)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("mother", list(MOTHERS))
@pytest.mark.parametrize("n0,nfft", [(1000, 1500), (700, 4096), (33, 100)])
def test_cwt_explicit_transform_length(shim, n0, nfft, mother, f64):
    """pycwt's formula at a transform length N that is neither n0 nor the next power of two."""
    inp = INPUTS[(n0 + len(mother)) % 3]
    res = _cwt_case(shim, f64, n0, nfft, mother, inp, seed=nfft + len(mother))
    _report(f"{mother} {inp}", f64, n0, nfft, *res)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("f0", [4.0, 5.29])
@pytest.mark.parametrize("n0", [1024, 1346])
def test_cwt_morlet_small_f0(shim, n0, f0, f64):
    """f0 < 5.3: the daughter's negative-frequency tail (pycwt's Morlet has no Heaviside step) is above the
    fast kernels' band cut, so the FP32 plan sends even a power-only call to the generic kernels."""
    inp = INPUTS[(n0 + int(f0)) % 3]
    res = _cwt_case(shim, f64, n0, _pow2(n0), "morlet", inp, f0=f0, seed=n0 + int(100 * f0), power_only_call=True)
    _report(f"morlet f0={f0} {inp}", f64, n0, _pow2(n0), *res)


# ---- cross spectrum and coherence -----------------------------------------------------------------------
# dj -> boxcar width K = round(1.2 / dj) of Morlet.smooth: 1, 2, 5, 10, 14
DJS = [1.0, 1 / 2, 1 / 4, 1 / 8, 1 / 12]


def _wct_cases():
    cases = []
    for f64 in (True, False):
        shapes = [(n, n) for n in (33, 257, 1000, 2047) + (() if f64 else (4095,))]
        shapes += [(100, None), (4096, None) if f64 else (8192, None)]
        for n0, nfft in shapes:
            for dj in DJS:
                cases.append((f64, n0, nfft, dj))
    return cases


def _pairs(n0, kind, seed):
    """Three pairs (y1, y2 = 0.6 y1 + 0.8 z) of unit variance.  White and AR(1) 0.989 only: the smoothed spectra
    of a pure line (the two-tone series) underflow FP32 far from the line, where even the float64 coherence
    is 0 / 0."""
    y1 = _inputs(kind, 3, n0, seed)
    y2 = 0.6 * y1 + 0.8 * _inputs(kind, 3, n0, seed + 1)
    norm = lambda y: (y - y.mean(axis=1, keepdims=True)) / y.std(axis=1, keepdims=True)
    return norm(y1), norm(y2)


@pytest.mark.parametrize("case", _wct_cases(),
                         ids=lambda c: f"{'fp64' if c[0] else 'fp32'}-{c[1]}-{'pad' if c[2] is None else 'nopad'}"
                                       f"-K{int(round(1.2 / c[3]))}")
def test_xwt_wct_rows(shim, case):
    f64, n0, nfft, dj = case
    pad = nfft is None
    N = _pow2(n0) if pad else nfft
    kind = ["white", "ar1_0.989"][(n0 + int(round(1 / dj))) % 2]
    rt = np.float64 if f64 else np.float32
    y1, y2 = (y.astype(rt) for y in _pairs(n0, kind, seed=n0 * 13 + int(round(1 / dj))))
    Jr, sj, _, _ = shim.cwt_axes(n0, DT, dj, -1, -1)
    # FP32 at nfft 4096 takes the radix-16 forward kernel of wct_fast.cu, also three launches with k_wct_rows +
    # k_wct_scale: the launch counts below prove the generic pipeline only away from that length
    assert f64 or N != 4096, "the launch count would not prove the path"
    before = shim.kernel_launches()
    wct, phase, w12 = shim.xwt_wct(y1, y2, DT, dj, -1, Jr, nfft=N, f64=f64, want_w12=True)
    assert shim.kernel_launches() - before == 3, "another kernel served the coherence"
    _, _, w12_only = shim.xwt_wct(y1, y2, DT, dj, -1, Jr, nfft=N, f64=f64, want_wct=False, want_phase=False,
                                  want_w12=True)
    assert shim.kernel_launches() - before == 5, "another kernel served the cross spectrum"
    assert np.array_equal(w12_only, w12)
    tol = 1e-10 if f64 else 1e-4
    worst_w12 = worst_ph = worst_wct = 0.0
    for b in (0, 2):
        a1, a2 = y1[b].astype(np.float64), y2[b].astype(np.float64)
        W1 = cl.cwt_rows(a1, DT, dj, -1, Jr, po.Morlet(6), range(Jr + 1), nfft=N)
        W2 = cl.cwt_rows(a2, DT, dj, -1, Jr, po.Morlet(6), range(Jr + 1), nfft=N)
        ref12 = W1 * W2.conj()
        what = f"{kind} n0={n0} nfft={N} dj={dj:.4g} pair {b}"
        r, _ = _gate(w12[b], ref12, tol, None, f"{what} w12")
        worst_w12 = max(worst_w12, r)
        # the phase as the phasor |W12| e^{i phase}: a near-zero cross spectrum's phase does not count
        r, _ = _gate(np.abs(ref12) * np.exp(1j * phase[b].astype(np.float64)), ref12, tol, None, f"{what} phase")
        worst_ph = max(worst_ph, r)
        WCT = po.wct(a1, a2, DT, dj=dj, s0=-1, J=Jr, sig=False, normalize=False, pad_pow2=pad)[0]
        worst_wct = max(worst_wct, _plane_close(wct[b], WCT, f64, f"{what} wct"))
    print(f"ROWGATE xwt {'fp64' if f64 else 'fp32'} {kind} n0={n0} nfft={N} M={_work_length(N)} "
          f"K={int(round(1.2 / dj))}: w12 {worst_w12:.3g}, phase {worst_ph:.3g}, wct plane {worst_wct:.3g}")


# ---- averages over the same first pass ------------------------------------------------------------------
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("mother,n0,nfft", [("morlet", 1025, 1025), ("morlet", 2047, 2047), ("paul4", 1346, 2048),
                                            ("dog2", 3000, 4096)])
def test_averages(shim, mother, n0, nfft, f64):
    code, param, wl = MOTHERS[mother]
    rt = np.float64 if f64 else np.float32
    x = _inputs("ar1_0.989", 3, n0, seed=n0 + 5).astype(rt)
    Jr, sj, _, _ = shim.cwt_axes_mother(n0, DT, DJ, -1, -1, code, param)
    S = Jr + 1
    band = (S // 3, 2 * S // 3)
    factor = DJ * DT / 0.776
    assert not _other_two_launch_plan(f64, mother, param, nfft, False), "the launch count would not prove the path"
    before = shim.kernel_launches()
    g, bnd = shim.cwt_averages(x, DT, DJ, -1, -1, code, param, band=band, band_factor=factor, nfft=nfft, f64=f64)
    assert shim.kernel_launches() - before == 3, "another kernel served the first pass"
    tol = 1e-10 if f64 else 1e-4
    worst = 0.0
    for b in (0, 2):
        W = cl.cwt_rows(x[b].astype(np.float64), DT, DJ, -1, -1, wl, range(S), nfft=nfft)
        ratio, where = oa.averages_gate(g[b], bnd[b], W, sj, band, factor, tol, np.ones(S, bool))
        assert ratio <= 1.0, f"series {b}: {ratio:.3g} of the bound at {where}"
        worst = max(worst, ratio)
    print(f"ROWGATE averages {'fp64' if f64 else 'fp32'} {mother} n0={n0} nfft={nfft}: {worst:.3g}")


# ---- limits of the un-padded transforms -----------------------------------------------------------------
def _refusal(nfft, f64, buffers):
    elem = 16 if f64 else 8
    return (f"nfft={nfft} needs {buffers * elem * _work_length(nfft)} B of shared memory per CTA (limit 227 KB): "
            f"a power of two up to {4096 if f64 else 8192}, any other length up to {2048 if f64 else 4096} for "
            f"{'double' if f64 else 'float'}")


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_unpadded_limit_is_refused(shim, f64):
    """The longest un-padded length is served (test_cwt_length_classes, test_xwt_wct_rows); the next one is
    refused by wtb_cwt, wtb_cwt_averages and wtb_xwt_wct with WTB_EUNSUPPORTED, before any launch.  So are lengths
    whose Bluestein work length (2^31, 2^32) does not fit an int, for a series of 100 samples."""
    n0 = 2049 if f64 else 4097
    before = shim.kernel_launches()
    for n, nfft in ((n0, n0), (100, 600_000_001), (100, 1_500_000_001)):
        x = _inputs("white", 2, n, seed=1)
        for call, buffers in ((lambda: shim.cwt(x, DT, DJ, -1, -1, 2, 2.0, nfft=nfft, f64=f64), 2),
                              (lambda: shim.cwt_averages(x, DT, DJ, -1, -1, 0, 6.0, nfft=nfft, f64=f64), 2),
                              (lambda: shim.xwt_wct(x, x[::-1], DT, DJ, -1, -1, nfft=nfft, f64=f64), 3)):
            with pytest.raises(shim.WaveletEngineError) as err:
                call()
            assert f"(status {EUNSUPPORTED}): {_refusal(nfft, f64, buffers)}" in str(err.value)
    assert shim.kernel_launches() == before
    x = _inputs("white", 2, n0, seed=1)
    shim.cwt(x[:, :-2], DT, DJ, -1, -1, 2, 2.0, nfft=n0 - 2, f64=f64)        # and the longest accepted length


GUARD = 4096


def _guarded(torch, n, dtype):
    buf = torch.full((n + 2 * GUARD,), -7.0e33, dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n]


def _intact(buf, n):
    return bool((buf[:GUARD] == -7.0e33).all()) and bool((buf[GUARD + n:] == -7.0e33).all())


@pytest.mark.parametrize("f64,n0", [(False, 3), (True, 3), (False, 2047), (True, 2047), (False, 4095)])
def test_unpadded_writes_stay_inside_their_outputs(shim, f64, n0):
    """Device-pointer wtb_cwt (power and coefficients), wtb_xwt_wct (coherence, phase, cross spectrum) and
    wtb_icwt at un-padded lengths write into the middle of guarded buffers; the guards come back untouched."""
    import torch
    dtype = torch.float64 if f64 else torch.float32
    lib = shim.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    batch = 3
    x = torch.randn(batch, n0, dtype=dtype, device="cuda")
    y = torch.randn(batch, n0, dtype=dtype, device="cuda")
    Jr, sj, _, _ = shim.cwt_axes_mother(n0, DT, DJ, -1, -1, 1, 4.0)
    n = batch * (Jr + 1) * n0
    pbuf, pw = _guarded(torch, n, dtype)
    cbuf, cf = _guarded(torch, 2 * n, dtype)              # complex as interleaved reals
    assert lib.wtb_cwt(ptr(x), batch, n0, n0, DT, DJ, -1.0, Jr, 1, 4.0, flags, ptr(pw), ptr(cf), stream) == 0, \
        lib.wtb_last_error()
    ibuf, rec = _guarded(torch, batch * n0, dtype)
    assert lib.wtb_icwt(ptr(cf), batch, Jr + 1, n0, sj.ctypes.data_as(C.POINTER(C.c_double)), 1.0, flags, ptr(rec),
                        stream) == 0, lib.wtb_last_error()
    Jm, _, _, _ = shim.cwt_axes(n0, DT, DJ, -1, -1)
    m = batch * (Jm + 1) * n0
    wbuf, wc = _guarded(torch, m, dtype)
    hbuf, ph = _guarded(torch, m, dtype)
    xbuf, xw = _guarded(torch, 2 * m, dtype)
    assert lib.wtb_xwt_wct(ptr(x), ptr(y), batch, n0, n0, DT, DJ, -1.0, Jm, 6.0, flags, ptr(wc), ptr(ph), ptr(xw),
                           stream) == 0, lib.wtb_last_error()
    torch.cuda.synchronize()
    for buf, t, size in ((pbuf, pw, n), (cbuf, cf, 2 * n), (ibuf, rec, batch * n0), (wbuf, wc, m), (hbuf, ph, m),
                         (xbuf, xw, 2 * m)):
        assert _intact(buf, size)
        assert bool(torch.isfinite(t).all())


# ---- wtb_icwt past 65535 series ---------------------------------------------------------------------------
ICWT_S, ICWT_N0 = 4, 64        # 2 KiB of FP32 coefficients per series: 70 000 series are one host chunk


@pytest.fixture(scope="module")
def many_coefs():
    rng = np.random.default_rng(70000)
    W = rng.standard_normal((70000, ICWT_S, ICWT_N0, 2), dtype=np.float32).view(np.complex64)
    W = W.reshape(70000, ICWT_S, ICWT_N0)
    sj = 2.0 * 2.0 ** (np.arange(ICWT_S) / 4)
    return W, sj


@pytest.mark.parametrize("where", ["host", "device"])
@pytest.mark.parametrize("batch", [65535, 65536, 70000])
def test_icwt_more_than_65535_series(shim, many_coefs, batch, where):
    W, sj = many_coefs
    wl = po.Morlet(6)
    factor = _icwt_factor(wl, DJ)
    before = shim.kernel_launches()
    if where == "host":
        rec = shim.icwt(W[:batch], sj, factor, f64=False)
    else:
        import torch
        wd = torch.from_numpy(W[:batch]).to("cuda")
        out = torch.empty((batch, ICWT_N0), dtype=torch.float32, device="cuda")
        lib = shim.lib()
        rc = lib.wtb_icwt(C.c_void_p(wd.data_ptr()), batch, ICWT_S, ICWT_N0, sj.ctypes.data_as(C.POINTER(C.c_double)),
                          factor, shim.DEVICE_PTRS, C.c_void_p(out.data_ptr()),
                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, lib.wtb_last_error()
        torch.cuda.synchronize()
        rec = out.cpu().numpy()
    assert shim.kernel_launches() - before == -(-batch // 65535)       # one launch per 65535 series
    assert rec.shape == (batch, ICWT_N0)
    for b in sorted({0, 1, 65534, min(65535, batch - 1), batch - 1}):
        ok, err = normwise_close(rec[b], po.icwt(W[b].astype(np.complex128), sj, DT, DJ, wl), 1e-4)
        assert ok, f"series {b}: {err:.3e}"
        assert np.array_equal(rec[b], shim.icwt(W[b], sj, factor, f64=False))
