"""GPU: MODWT, inverse MODWT, MRA and DWT of long series (filterbank_long.cu), past one CTA's shared memory.

Every entry point in both precisions is held to the float64 references of oracle/filterbank_long.py (1e-10 of
max(1, max|x|) in FP64, 1e-4 of max|x| in FP32) from the first long length up to 3 000 000 samples; at 2^22 the
transforms invert and conserve energy.  Launch counts show which path served a call.  Results are bit-identical
across batch sizes, host chunks, pool sizes and device pointers; writes stay inside their outputs; the Python
façades work at these lengths."""

import ctypes as C
import os

import numpy as np
import pytest

from oracle import filterbank_long as fl
from oracle import modwt_oracle as mo
from oracle import pywt_oracle as po

pytestmark = pytest.mark.gpu


def _x(batch, n, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((batch, n + 64)).cumsum(axis=1)[:, 64:] * 0.05 + rng.standard_normal((batch, n))
    return x[0] if batch == 1 else x


def _gate(got, ref, x, f64):
    """FP64: 1e-10 max(1, max|x|); FP32: 1e-4 max|x| (ref from the FP32-rounded input)."""
    scale = np.abs(x).max()
    bound = 1e-10 * max(1.0, scale) if f64 else 1e-4 * scale
    err = np.abs(np.asarray(got, np.float64) - ref).max()
    assert err <= bound, f"error {err:.3g} > {bound:.3g}"
    return err / bound


def _as(x, f64):
    return x if f64 else x.astype(np.float32).astype(np.float64)


def _taps(wavelet):
    w = po.Wavelet(wavelet)
    return np.array(w.dec_lo), np.array(w.dec_hi), np.array(w.rec_lo), np.array(w.rec_hi)


def _counted(shim, fn, *a, **k):
    before = shim.kernel_launches()
    out = fn(*a, **k)
    return out, shim.kernel_launches() - before


def _launches(entry, n, f64, L, J):
    """Launches of a one-series call: the replica's on the long path, one below it (every FP64 case and every
    FP32 one from 29 053 samples is long; 20 001 samples in FP32 is one-CTA but for imodwt)."""
    if fl.route(entry, n, f64, L=L, J=J, level=J) == "long":
        return fl.launches(entry, n, f64, 1, L=L, J=J, level=J)
    assert not f64 and n < 29053
    return 1


# ---- against the references -------------------------------------------------------------------------------------
def _first(entry, f64, L, J):
    return fl.first_long_n(entry, f64, L=L, J=J, level=J)


CASES = [("first", "db4", 6), ("first", "db5", 4), (20001, "haar", 8), (20001, "db2", "max"), (20001, "db4", 14),
         (65537, "sym4", 9), (65537, "db5", "max"), (1 << 20, "db4", 10), (3_000_000, "db4", 6)]
IDS = [f"{c[0]}-{c[1]}-J{c[2]}" for c in CASES]


def _shape(entry, case, f64):
    n, wavelet, J = case
    L = po.Wavelet(wavelet).dec_len
    if n == "first":
        n = _first(entry, f64, L, J if J != "max" else 1)
    if J == "max":
        J = po.dwt_max_level(n, L)
    return n, wavelet, L, J


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_modwt_and_inverse(shim, case, f64):
    n, wavelet, L, J = _shape("modwt", case, f64)
    g, h, _, _ = _taps(wavelet)
    x = _x(1, n, seed=n + J)
    w, k = _counted(shim, shim.modwt, x, g, h, J, f64=f64)
    assert k == _launches("modwt", n, f64, L, J)
    ref = mo.modwt(_as(x, f64), wavelet, J)
    _gate(w, ref, x, f64)
    n_i = n if case[0] != "first" else _first("imodwt", f64, L, J)   # imodwt's limit comes first
    xi = x if n_i == n else _x(1, n_i, seed=3)
    wi = mo.modwt(xi, wavelet, J)
    xr, k = _counted(shim, shim.imodwt, wi, g, h, f64=f64)
    assert k == _launches("imodwt", n_i, f64, L, J)
    _gate(xr, mo.imodwt(_as(wi, f64), wavelet), xi, f64)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("case", [c for c in CASES if c[0] != 3_000_000], ids=[i for c, i in zip(CASES, IDS)
                                                                             if c[0] != 3_000_000])
def test_mra(shim, case, f64):
    n, wavelet, L, J = _shape("modwtmra_taps", case, f64)
    J = min(J, 14 if n < 1 << 20 else 8)
    g, h, _, _ = _taps(wavelet)
    w = mo.modwt(_x(1, n, seed=n), wavelet, J)
    ref = fl.modwtmra(_as(w, f64), wavelet)
    got, k = _counted(shim, shim.modwtmra_taps, w, g, h, f64=f64)
    assert k == _launches("modwtmra_taps", n, f64, L, J)
    _gate(got, ref, w, f64)
    if n <= 65537 and J <= 9:                   # explicit periodised filters (wtb_modwtmra): one launch per wave
        filt = np.vstack(mo.mra_filters(wavelet, J, n))
        got, k = _counted(shim, shim.modwtmra, w, filt, f64=f64)
        assert k == _launches("modwtmra", n, f64, L, J)
        _gate(got, ref, w, f64)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_wavedec_waverec(shim, case, f64):
    n, wavelet, L, level = _shape("wavedec", case, f64)
    level = min(level, po.dwt_max_level(n, L))
    lo, hi, rlo, rhi = _taps(wavelet)
    x = _x(1, n, seed=n + 1)
    (packed, lens), k = _counted(shim, shim.wavedec, x, lo, hi, level, f64=f64)
    assert k == _launches("wavedec", n, f64, L, level)
    ref = fl.wavedec(_as(x, f64), wavelet, level=level)
    assert list(lens) == [r.size for r in ref]
    _gate(packed, np.concatenate(ref), x, f64)
    n_r = n if case[0] != "first" else _first("waverec", f64, L, level)
    xr = x if n_r == n else _x(1, n_r, seed=5)
    coeffs = fl.wavedec(xr, wavelet, level=level)
    rec, k = _counted(shim, shim.waverec, np.concatenate(coeffs), [c.size for c in coeffs], rlo, rhi, f64=f64)
    assert k == _launches("waverec", n_r, f64, L, level)
    _gate(rec, fl.waverec([_as(c, f64) for c in coeffs], wavelet), xr, f64)


# ---- identities at 2^22 in FP64 ---------------------------------------------------------------------------------
def test_identities_at_2_22(shim):
    n, J = 1 << 22, 10
    lo, hi, rlo, rhi = _taps("db4")
    x = _x(1, n, seed=22)
    w = shim.modwt(x, lo, hi, J, f64=True)
    scale = max(1.0, np.abs(x).max())
    assert np.abs(shim.imodwt(w, lo, hi, f64=True) - x).max() <= 1e-10 * scale
    assert abs((w ** 2).sum() - (x ** 2).sum()) <= 1e-10 * (x ** 2).sum()
    mra = shim.modwtmra_taps(w, lo, hi, f64=True)
    assert np.abs(mra.sum(axis=0) - x).max() <= 1e-10 * scale
    del w, mra
    packed, lens = shim.wavedec(x, lo, hi, po.dwt_max_level(n, 8), f64=True)
    assert np.abs(shim.waverec(packed, lens, rlo, rhi, f64=True) - x).max() <= 1e-10 * scale


# ---- routing ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("wavelet", ["db4", "db5"])
def test_last_one_cta_length_keeps_its_kernel(shim, f64, wavelet):
    """At the last one-CTA length each entry point runs its one-CTA kernel (one launch); one sample more runs the
    long path with the replica's launch count."""
    lo, hi, rlo, rhi = _taps(wavelet)
    L, J = lo.size, 5
    for entry in ("modwt", "imodwt", "modwtmra_taps", "wavedec", "waverec"):
        n1 = _first(entry, f64, L, J)
        for n, long in ((n1 - 1, False), (n1, True)):
            x = _x(1, n, seed=n)
            assert fl.route(entry, n, f64, L=L, J=J, level=J) == ("long" if long else "one-cta")
            if entry == "modwt":
                got, k = _counted(shim, shim.modwt, x, lo, hi, J, f64=f64)
                ref = mo.modwt(_as(x, f64), wavelet, J)
            elif entry == "imodwt":
                wi = mo.modwt(x, wavelet, J)
                got, k = _counted(shim, shim.imodwt, wi, lo, hi, f64=f64)
                ref = mo.imodwt(_as(wi, f64), wavelet)
            elif entry == "modwtmra_taps":
                wi = mo.modwt(x, wavelet, J)
                got, k = _counted(shim, shim.modwtmra_taps, wi, lo, hi, f64=f64)
                ref = fl.modwtmra(_as(wi, f64), wavelet)
            elif entry == "wavedec":
                (got, _), k = _counted(shim, shim.wavedec, x, lo, hi, J, f64=f64)
                ref = np.concatenate(fl.wavedec(_as(x, f64), wavelet, J))
            else:
                c = fl.wavedec(x, wavelet, J)
                got, k = _counted(shim, shim.waverec, np.concatenate(c), [a.size for a in c], rlo, rhi, f64=f64)
                ref = fl.waverec([_as(a, f64) for a in c], wavelet)
            want = fl.launches(entry, n, f64, 1, L=L, J=J, level=J) if long else 1
            assert k == want, f"{entry} n={n}: {k} launches, expected {want}"
            _gate(got, ref, x, f64)


def test_generic_only_does_not_stop_the_long_path(shim):
    lo, hi, _, _ = _taps("db4")
    x = _x(1, 20001, seed=1)
    w = shim.modwt(x, lo, hi, 6, f64=True)
    assert np.array_equal(shim.modwt(x, lo, hi, 6, f64=True, generic_only=True), w)
    assert np.array_equal(shim.modwtmra_taps(w, lo, hi, f64=True, generic_only=True),
                          shim.modwtmra_taps(w, lo, hi, f64=True))


# ---- invariance -------------------------------------------------------------------------------------------------
def _all_entries(shim, x, f64, J=6, wavelet="db4"):
    lo, hi, rlo, rhi = _taps(wavelet)
    w = shim.modwt(x, lo, hi, J, f64=f64)
    packed, lens = shim.wavedec(x, lo, hi, J, f64=f64)
    n = x.shape[-1]
    filt = np.vstack(mo.mra_filters(wavelet, J, n))
    return {"modwt": w, "imodwt": shim.imodwt(w, lo, hi, f64=f64), "mra": shim.modwtmra_taps(w, lo, hi, f64=f64),
            "mra_filt": shim.modwtmra(w, filt, f64=f64), "wavedec": packed,
            "waverec": shim.waverec(packed, lens, rlo, rhi, f64=f64)}


@pytest.mark.parametrize("f64,n", [(False, 1 << 21), (True, 1 << 20), (True, 65537)])
def test_bits_do_not_depend_on_the_batch(shim, f64, n):
    """At 2^20 in FP64 a wave holds 4 series (1 for the MRAs), so batches of 7, 3 and 1 cut the waves differently."""
    x = _x(7, n, seed=31)
    full = _all_entries(shim, x, f64)
    part = _all_entries(shim, x[2:5], f64)
    for k in full:
        assert np.array_equal(part[k], full[k][2:5]), k
    for i in (0, 4, 6):
        one = _all_entries(shim, x[i:i + 1], f64)
        for k in full:
            assert np.array_equal(one[k][0], full[k][i]), (k, i)


def test_bits_across_host_chunks(shim):
    """64 series of 2^20 samples, FP64, J = 6: four 1 GiB host chunks of 16 series, waves of 4."""
    n, J, batch = 1 << 20, 6, 64
    lo, hi, _, _ = _taps("db4")
    x = np.random.default_rng(41).standard_normal((batch, n))
    w, k = _counted(shim, shim.modwt, x, lo, hi, J, f64=True)
    assert k == fl.launches("modwt", n, True, batch, J=J) == 16 * J
    for i in (0, 15, 16, 63):
        assert np.array_equal(shim.modwt(x[i], lo, hi, J, f64=True), w[i]), i
    xr = shim.imodwt(w[:20], lo, hi, f64=True)
    assert np.array_equal(shim.imodwt(w[17], lo, hi, f64=True), xr[17])


def _dev_entries(shim, torch, x, f64, J=6, wavelet="db4"):
    lo, hi, rlo, rhi = _taps(wavelet)
    dt = torch.float64 if f64 else torch.float32
    batch, n = x.shape
    s = torch.cuda.current_stream().cuda_stream
    xd = torch.as_tensor(x, dtype=dt, device="cuda").contiguous()
    wd = torch.empty(batch, J + 1, n, dtype=dt, device="cuda")
    shim.modwt_device(xd.data_ptr(), batch, n, lo, hi, J, wd.data_ptr(), f64=f64, stream=s)
    xr = torch.empty(batch, n, dtype=dt, device="cuda")
    shim.imodwt_device(wd.data_ptr(), batch, n, lo, hi, J, xr.data_ptr(), f64=f64, stream=s)
    md = torch.empty_like(wd)
    shim.modwtmra_taps_device(wd.data_ptr(), batch, n, lo, hi, J, md.data_ptr(), f64=f64, stream=s)
    lens = shim.dwt_coeff_lens(n, lo.size, J)
    pd = torch.empty(batch, int(lens.sum()), dtype=dt, device="cuda")
    shim.wavedec_device(xd.data_ptr(), batch, n, lo, hi, J, pd.data_ptr(), f64=f64, stream=s)
    rd = torch.empty(batch, shim.waverec_len(lens, lo.size), dtype=dt, device="cuda")
    shim.waverec_device(pd.data_ptr(), batch, lens, rlo, rhi, rd.data_ptr(), f64=f64, stream=s)
    torch.cuda.synchronize()
    return {"modwt": wd, "imodwt": xr, "mra": md, "wavedec": pd, "waverec": rd}


@pytest.mark.parametrize("f64", [False, True])
def test_device_pointers_equal_host_buffers(shim, f64):
    import torch
    x = _x(3, 70001, seed=51)
    host = _all_entries(shim, x, f64)
    dev = _dev_entries(shim, torch, x, f64)
    for k, v in dev.items():
        assert np.array_equal(v.cpu().numpy(), host[k]), k


@pytest.fixture()
def pool(shim):
    """A pool of two workers: two GPUs when the box has them, one shared GPU otherwise."""
    os.environ["WTB_POOL_SHARE_DEVICES"] = "1"
    assert shim.init_multi(2) == 2
    yield shim
    shim.init_multi(1)
    assert shim.gpu_count() == 1


@pytest.mark.parametrize("f64", [False, True])
def test_split_over_the_pool(shim, pool, f64):
    x = _x(5, 40001, seed=61)
    two = _all_entries(shim, x, f64)
    shim.init_multi(1)
    one = _all_entries(shim, x, f64)
    for k in one:
        assert np.array_equal(one[k], two[k]), k


# ---- guards -----------------------------------------------------------------------------------------------------
GUARD = 4096


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n,batch", [(29057, 3), (65537, 1), (100003, 2)])
def test_writes_stay_inside_their_outputs(shim, n, batch, f64):
    import torch
    J, wavelet = 7, "db5"
    lo, hi, rlo, rhi = _taps(wavelet)
    dt = torch.float64 if f64 else torch.float32
    s = torch.cuda.current_stream().cuda_stream
    pattern = -7.0e33

    def guarded(count):
        buf = torch.full((count + 2 * GUARD,), pattern, dtype=dt, device="cuda")
        return buf, buf[GUARD:GUARD + count]

    def intact(buf, count):
        return bool((buf[:GUARD] == pattern).all()) and bool((buf[GUARD + count:] == pattern).all())

    xd = torch.randn(batch, n, dtype=dt, device="cuda")
    wbuf, wd = guarded(batch * (J + 1) * n)
    shim.modwt_device(xd.data_ptr(), batch, n, lo, hi, J, wd.data_ptr(), f64=f64, stream=s)
    xbuf, xr = guarded(batch * n)
    shim.imodwt_device(wd.data_ptr(), batch, n, lo, hi, J, xr.data_ptr(), f64=f64, stream=s)
    mbuf, md = guarded(batch * (J + 1) * n)
    shim.modwtmra_taps_device(wd.data_ptr(), batch, n, lo, hi, J, md.data_ptr(), f64=f64, stream=s)
    fbuf, fd = guarded(batch * (J + 1) * n)
    filt = np.ascontiguousarray(np.vstack(mo.mra_filters(wavelet, J, n)))
    rc = shim.lib().wtb_modwtmra(C.c_void_p(wd.data_ptr()), batch, n, filt.ctypes.data_as(C.POINTER(C.c_double)), J,
                                 shim.DEVICE_PTRS | (shim.F64 if f64 else 0), C.c_void_p(fd.data_ptr()), C.c_void_p(s))
    assert rc == 0, shim.lib().wtb_last_error()
    lens = shim.dwt_coeff_lens(n, lo.size, J)
    pbuf, pd = guarded(batch * int(lens.sum()))
    shim.wavedec_device(xd.data_ptr(), batch, n, lo, hi, J, pd.data_ptr(), f64=f64, stream=s)
    nout = shim.waverec_len(lens, lo.size)
    rbuf, rd = guarded(batch * nout)
    shim.waverec_device(pd.data_ptr(), batch, lens, rlo, rhi, rd.data_ptr(), f64=f64, stream=s)
    torch.cuda.synchronize()
    for name, buf, view in (("modwt", wbuf, wd), ("imodwt", xbuf, xr), ("mra", mbuf, md), ("mra_filt", fbuf, fd),
                            ("wavedec", pbuf, pd), ("waverec", rbuf, rd)):
        assert intact(buf, view.numel()), name
        assert bool(torch.isfinite(view).all()), name
    x = xd.double().cpu().numpy()
    assert np.abs(xr.double().cpu().numpy().reshape(batch, n) - x).max() <= (1e-9 if f64 else 1e-3) * np.abs(x).max()


# ---- façades ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [10_000, 100_000])
def test_modwt_facades(shim, n):
    from wavelet_transformer_b200.api import modwt as api
    x = _x(1, n, seed=n)
    J = 8
    w = api.modwt(x, "db4", J)
    ref = mo.modwt(x, "db4", J)
    _gate(w, ref, x, True)
    _gate(api.imodwt(ref, "db4"), x, x, True)
    _gate(api.modwtmra(ref, "db4"), fl.modwtmra(ref, "db4"), ref, True)
    sm = api.smooth_signal(ref, "db4", 4)
    for lev in range(4, 0, -1):
        c = ref.copy()
        c[:lev] = 0.0
        _gate(sm[lev]["signal"], mo.imodwt(c, "db4"), x, True)
    g, h = np.array(po.Wavelet("db4").dec_lo), np.array(po.Wavelet("db4").dec_hi)
    if n > 14528:                              # past the generic kernel's limit in FP64
        j = 5
        v = ref[J]
        d = api.circular_convolve_d(h / np.sqrt(2), v, j)
        _gate(d, mo._circ_gather(v, h / np.sqrt(2), 2 ** (j - 1), -1), v, True)
        s = api.circular_convolve_s(h / np.sqrt(2), g / np.sqrt(2), ref[j - 1], v, j)
        want = mo._circ_gather(ref[j - 1], h / np.sqrt(2), 2 ** (j - 1), 1) + mo._circ_gather(v, g / np.sqrt(2),
                                                                                             2 ** (j - 1), 1)
        _gate(s, want, v, True)


@pytest.mark.parametrize("n", [10_000, 100_000])
def test_dwt_facades(shim, n):
    from src import dwt as sdwt
    from wavelet_transformer_b200 import pywt_compat as pywt
    x = _x(1, n, seed=n + 7)
    w = pywt.Wavelet("db4")
    coeffs = pywt.wavedec(x, w)
    ref = fl.wavedec(x, "db4")
    assert len(coeffs) == len(ref)
    _gate(np.concatenate(coeffs), np.concatenate(ref), x, True)
    _gate(pywt.waverec(ref, w), fl.waverec(ref, "db4"), x, True)
    res = sdwt.run_dwt(sdwt.DataForDWT(x, w, None))
    assert res.levels == po.dwt_max_level(n, 8)
    _gate(np.concatenate(res.coeffs), np.concatenate(ref), x, True)
    for level in (0, 3, len(ref) - 1):
        only = [c if i == level else np.zeros_like(c) for i, c in enumerate(ref)]
        _gate(sdwt.reconstruct_signal_component(res.coeffs, w, level), fl.waverec(only, "db4"), x, True)
