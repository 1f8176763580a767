"""GPU: partial and multiple wavelet coherence of three series (wtb_partial_wct, pwct.cu).

Every point of PWC, the partial phase and MWC is held to the float64 closed forms of oracle/pwct_oracle.py with
|got - ref| <= tol * kappa * (1 + |ref|), tol the project's coherence gates (1e-4 FP32, 1e-10 FP64) and kappa the
conditioning of each ratio in the oracle; the phase through the complex partial coherency sqrt(PWC) e^{i phase}.
The outputs satisfy the MWC / PWC identity and the x1 <-> x2 symmetry of MWC within the same gate.  The call
costs cwt_device's launches plus two, refuses what it cannot do before any launch, and its bits do not depend on
the batch, the pool or the pointers."""

import ctypes as C
import os

import numpy as np
import pytest

from oracle import pwct_oracle as pw

pytestmark = pytest.mark.gpu

DT = 1.0
EINVAL, EUNSUPPORTED = -1, -3


def _tol(f64):
    return 1e-10 if f64 else 1e-4


def _rounded(series, f64):
    """The inputs as the device sees them, in float64: the reference starts from the same numbers."""
    return [np.asarray(v, dtype=np.float64 if f64 else np.float32).astype(np.float64) for v in series]


def _run(shim, series, dj, f64, nfft, **kw):
    before = shim.kernel_launches()
    out = shim.partial_wct(*series, DT, dj, -1, -1, f64=f64, nfft=nfft, **kw)
    return out, shim.kernel_launches() - before


def _gate(got, ref, kappa, tol):
    """Worst |got - ref| / (tol kappa (1 + |ref|)); NaN in both counts as equal."""
    got = np.asarray(got, dtype=np.complex128 if np.iscomplexobj(got) else np.float64)
    both_nan = np.isnan(got) & np.isnan(ref)
    r = np.abs(got - ref) / (tol * kappa * (1 + np.abs(ref)))
    r = np.where(both_nan, 0.0, r)
    assert not np.isnan(r).any(), "NaN in one of the two only"
    return float(r.max())


def _coherency(pwc, phase):
    return np.sqrt(np.asarray(pwc, dtype=np.float64)) * np.exp(1j * np.asarray(phase, dtype=np.float64))


def _check(shim, series, dj, f64, pad, label):
    n0 = series[0].size
    (pwc, phase, mwc), _ = _run(shim, series, dj, f64, None if pad else n0)
    sp = pw.spectra(*_rounded(series, f64), DT, dj, -1, -1, pad_pow2=pad)
    rp, rph, rm = pw.closed_forms(sp)
    kp, km = pw.conditioning(sp)
    tol = _tol(f64)
    worst = {"pwc": _gate(pwc, rp, kp, tol), "phase": _gate(_coherency(pwc, phase), _coherency(rp, rph), kp, tol),
             "mwc": _gate(mwc, rm, km, tol)}
    print(f"PWCTGATE {label}: worst ratio pwc {worst['pwc']:.3g} phase {worst['phase']:.3g} mwc {worst['mwc']:.3g}; "
          f"max kappa pwc {kp.max():.3g} mwc {km.max():.3g}")
    for what, r in worst.items():
        assert r <= 1.0, f"{what}: {r:.3g} of the gate"
    return (pwc, phase, mwc), kp, km


# ---- against the reference ---------------------------------------------------------------------------
# (n0, dj) per padding mode and precision: the cfg3 shape, the cfg1 length, the largest one-CTA length
def _shapes(f64, pad):
    largest = (4096 if f64 else 8192) if pad else (2047 if f64 else 4095)
    return [(565, 1 / 8), (1346, 1 / 12), (largest, 1 / 8)]


PARITY = [(f64, pad, n0, dj) for f64 in (False, True) for pad in (True, False) for n0, dj in _shapes(f64, pad)]


@pytest.mark.parametrize("kind", pw.INPUTS)
@pytest.mark.parametrize("f64,pad,n0,dj", PARITY,
                         ids=[f"{'fp64' if f else 'fp32'}-{'pow2' if p else 'none'}-{n}" for f, p, n, _ in PARITY])
def test_parity_with_the_reference(shim, f64, pad, n0, dj, kind):
    series = pw.triple(kind, n0, seed=n0 + len(kind))
    _check(shim, series, dj, f64, pad, f"{'fp64' if f64 else 'fp32'} {'pow2' if pad else 'none'} {n0} {kind}")


# ---- identities on the device's outputs ------------------------------------------------------------------
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("pad", [True, False], ids=["pow2", "none"])
def test_identity_and_symmetry(shim, f64, pad):
    """1 - MWC = (1 - |rho_y2|^2)(1 - PWC), with |rho_y2|^2 the device's own coherence of y and x2
    (wtb_xwt_wct), and MWC(y; x1, x2) = MWC(y; x2, x1)."""
    n0, dj = 565, 1 / 8
    y, x1, x2 = pw.triple("built", n0, seed=77)
    nfft = None if pad else n0
    (pwc, _, mwc), _ = _run(shim, (y, x1, x2), dj, f64, nfft)
    (_, _, mwc21), _ = _run(shim, (y, x2, x1), dj, f64, nfft)
    wct, _, _ = shim.xwt_wct(y, x2, DT, dj, -1, -1, f64=f64, nfft=nfft, want_phase=False)
    sp = pw.spectra(*_rounded((y, x1, x2), f64), DT, dj, -1, -1, pad_pow2=pad)
    kp, km = pw.conditioning(sp)
    tol = _tol(f64)
    lhs = 1 - mwc.astype(np.float64)
    rhs = (1 - wct.astype(np.float64)) * (1 - pwc.astype(np.float64))
    r_id = _gate(lhs, rhs, kp, tol)
    r_sym = _gate(mwc, mwc21.astype(np.float64), km, tol)
    print(f"PWCTIDENT {'fp64' if f64 else 'fp32'} {'pow2' if pad else 'none'}: identity {r_id:.3g} "
          f"symmetry {r_sym:.3g}")
    assert r_id <= 1.0 and r_sym <= 1.0


# ---- dispatch and refusals -----------------------------------------------------------------------------
@pytest.mark.parametrize("f64,n0,pad,generic", [(False, 3351, True, False), (False, 3351, True, True),
                                                (False, 1346, False, False), (True, 1346, True, False)])
def test_launches_are_the_cwt_launches_plus_two(shim, f64, n0, pad, generic):
    """The coefficients come from cwt_device (the same plan as wtb_cwt of the 3 x batch series), then the
    smoothing and the scale pass."""
    series = pw.triple("correlated", n0, seed=3)
    nfft = None if pad else n0
    _, launches = _run(shim, series, 1 / 8, f64, nfft, generic_only=generic)
    before = shim.kernel_launches()
    shim.cwt(np.stack(series), DT, 1 / 8, -1, -1, shim.MORLET, 6.0, f64=f64, nfft=nfft, want_power=False,
             want_coef=True, generic_only=generic)
    assert launches == shim.kernel_launches() - before + 2


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_refusals(shim, f64):
    lib = shim.lib()
    rt = np.float64 if f64 else np.float32
    n = 20000
    x = np.random.default_rng(4).standard_normal(n).astype(rt)
    out = np.zeros((9, n), rt)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    flags = shim.F64 if f64 else 0
    call = lambda n0, nfft, dj, o: lib.wtb_partial_wct(p(x), p(x), p(x), 1, n0, nfft, DT, dj, 2.0, 8, 6.0, flags,
                                                      o, None, None, None)
    before = shim.kernel_launches()
    assert lib.wtb_partial_wct(p(x), p(x), p(x), 1, 565, 1024, DT, 0.5, 2.0, 8, 6.0, flags, None, None, None,
                               None) == EINVAL
    assert b"no output" in lib.wtb_last_error()
    pow2, other = (4096, 2048) if f64 else (8192, 4096)
    limit = f"a power of two up to {pow2}, any other length up to {other} for {'double' if f64 else 'float'}"
    for n0, nfft in ((2 * pow2 - 1, 2 * pow2), (other + 1, other + 1), (n, 1 << 23)):
        assert call(n0, nfft, 0.5, p(out)) == EUNSUPPORTED, (n0, nfft)
        msg = lib.wtb_last_error().decode()
        assert f"nfft={nfft}" in msg and limit in msg, msg
    assert call(565, 1024, 0.01, p(out)) == EUNSUPPORTED          # 120 boxcar taps
    assert b"scale window" in lib.wtb_last_error()
    # the length is checked before the scale window and before an empty batch returns
    assert call(other + 1, other + 1, 0.01, p(out)) == EUNSUPPORTED
    assert limit in lib.wtb_last_error().decode()
    assert lib.wtb_partial_wct(p(x), p(x), p(x), 0, 565, 1_500_000_001, DT, 0.5, 2.0, 8, 6.0, flags, p(out), None,
                               None, None) == EUNSUPPORTED
    assert limit in lib.wtb_last_error().decode()
    assert lib.wtb_partial_wct(p(x), p(x), p(x), 0, 565, 1024, DT, 0.5, 2.0, 8, 6.0, flags, p(out), None, None,
                               None) == 0
    assert shim.kernel_launches() == before and not out.any()


# ---- invariance ----------------------------------------------------------------------------------------
def _batch(n0, count, seed):
    tri = [pw.triple(k, n0, seed=seed + i) for i, k in enumerate(pw.INPUTS * count)][:count]
    return [np.stack([t[i] for t in tri]) for i in range(3)]


@pytest.mark.parametrize("f64,n0", [(False, 1346), (False, 3351), (True, 565)])
def test_bits_do_not_depend_on_the_batch(shim, f64, n0):
    ys = _batch(n0, 3, seed=11)
    o3, _ = _run(shim, ys, 1 / 8, f64, None)
    for i in (0, 2):
        o1, _ = _run(shim, [v[i:i + 1] for v in ys], 1 / 8, f64, None)
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
    ys = _batch(1346, 5, seed=12)
    o2, _ = _run(shim, ys, 1 / 12, f64, None)
    shim.init_multi(1)
    o1, _ = _run(shim, ys, 1 / 12, f64, None)
    for a, b in zip(o1, o2):
        assert np.array_equal(a, b, equal_nan=True)


def _device_call(shim, torch, ys, dj, J, nfft, f64, outs):
    batch, n0 = ys[0].shape
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    rc = shim.lib().wtb_partial_wct(*(ptr(v) for v in ys), batch, n0, nfft, DT, dj, -1.0, J, 6.0, flags,
                                    *(ptr(o) for o in outs), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, shim.lib().wtb_last_error()


@pytest.mark.parametrize("f64,pad", [(False, True), (True, False)])
def test_device_pointers_equal_host_buffers(shim, f64, pad):
    import torch
    n0 = 1346
    ys = _batch(n0, 2, seed=13)
    nfft = shim.next_pow2(n0) if pad else n0
    o, _ = _run(shim, ys, 1 / 8, f64, nfft)
    dtype = torch.float64 if f64 else torch.float32
    dys = [torch.as_tensor(v, dtype=dtype, device="cuda").contiguous() for v in ys]
    outs = [torch.empty(o[0].shape, dtype=dtype, device="cuda") for _ in range(3)]
    _device_call(shim, torch, dys, 1 / 8, o[0].shape[1] - 1, nfft, f64, outs)
    torch.cuda.synchronize()
    for a, b in zip(outs, o):
        assert np.array_equal(a.cpu().numpy(), b, equal_nan=True)


GUARD = 4096


@pytest.mark.parametrize("f64", [False, True])
def test_writes_stay_inside_their_outputs(shim, f64):
    import torch
    dtype = torch.float64 if f64 else torch.float32
    batch, n0, J = 3, 1346, 28
    ys = [torch.as_tensor(v, dtype=dtype, device="cuda").contiguous() for v in _batch(n0, batch, seed=14)]
    n = batch * (J + 1) * n0
    bufs = [torch.full((n + 2 * GUARD,), -7.0e33, dtype=dtype, device="cuda") for _ in range(3)]
    views = [b[GUARD:GUARD + n] for b in bufs]
    _device_call(shim, torch, ys, 1 / 4, J, 2048, f64, views)
    torch.cuda.synchronize()
    for b, v in zip(bufs, views):
        assert bool((b[:GUARD] == -7.0e33).all()) and bool((b[GUARD + n:] == -7.0e33).all())
        assert bool(torch.isfinite(v).all())


@pytest.mark.parametrize("want", [(True, False, False), (False, True, False), (False, False, True)])
def test_each_output_alone_equals_the_full_call(shim, want):
    ys = _batch(565, 2, seed=15)
    full, _ = _run(shim, ys, 1 / 8, True, None)
    part, _ = _run(shim, ys, 1 / 8, True, None, want_pwc=want[0], want_phase=want[1], want_mwc=want[2])
    for a, b, w in zip(part, full, want):
        assert (a is None) != w and (a is None or np.array_equal(a, b, equal_nan=True))


# ---- façade --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("padding", ["pow2", "none"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_facade_equals_the_shim_after_normalisation(shim, padding, precision):
    import wavelet_transformer_b200 as wtb
    from oracle import pycwt_oracle as po
    rng = np.random.default_rng(16)
    y, x1, x2 = (3.0 * v + c for v, c in zip(pw.triple("built", 565, seed=16), (1.0, -2.0, 0.5)))
    y = y + 0.1 * rng.standard_normal(565)
    dt, dj = 1 / 12, 1 / 8
    old = (wtb.get_precision(), wtb.get_fft_padding())
    wtb.set_precision(precision)
    wtb.set_fft_padding(padding)
    try:
        pwc, pphase, mwc, coi, freq, scales = wtb.partial_wct(y, x1, x2, dt, dj, 2 * dt)
        norm = [(v - v.mean()) / v.std() for v in (y, x1, x2)]
        ref = shim.partial_wct(*norm, dt, dj, 2 * dt, len(scales) - 1)
    finally:
        wtb.set_precision(old[0])
        wtb.set_fft_padding(old[1])
    for a, b in zip((pwc, pphase, mwc), ref):
        assert a.dtype == np.float64 and np.array_equal(a, b.astype(np.float64), equal_nan=True)
    sj, rfreq, rcoi = po.cwt_axes(565, dt, dj, 2 * dt, len(scales) - 1, po.Morlet())
    assert np.allclose(scales, sj, rtol=1e-13) and np.allclose(freq, rfreq, rtol=1e-13)
    assert np.allclose(coi, rcoi, rtol=1e-13)
    if precision == "fp64":
        rp, rph, rm, *_ = pw.partial_wct(y, x1, x2, dt, dj, 2 * dt, pad_pow2=padding == "pow2")
        assert np.nanmax(np.abs(pwc - rp)) < 1e-6 and np.nanmax(np.abs(mwc - rm)) < 1e-6
