"""GPU: the CWT of long series (cwt_long.cu), power-of-two transforms past one CTA's shared memory.

Every mother wavelet and both precisions are held row by row to the float64 reference of oracle/cwt_long.py
(1e-10 in FP64; in FP32 1e-4 on the resolved rows and the plane gate elsewhere, as test_gpu_cwt_rows.py),
from the first newly covered lengths up to nfft = 2^22.  Launch counts show which path served a call.
Results are bit-identical across batch sizes, pool sizes and device pointers; writes stay inside their
outputs; wtb_cwt_averages and the pycwt façade work at these lengths."""

import ctypes as C
import os

import numpy as np
import pytest
from scipy.signal import lfilter

from oracle import averages as oa
from oracle import cwt_long as cl
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1.0
MOTHERS = {"morlet": (0, 6.0, po.Morlet(6)), "paul4": (1, 4.0, po.Paul(4)), "dog2": (2, 2.0, po.DOG(2)),
           "dog6": (2, 6.0, po.DOG(6))}
INPUTS = ["white", "ar1_0.989", "two_tone"]
EUNSUPPORTED = -3


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


def _nfft(n0):
    return 1 << (n0 - 1).bit_length()


def _check_rows(shim, x, dj, J, mother, f64, rows, power, coef):
    """power / coef [S, n0] of one series against the float64 rows of the reference."""
    code, param, wl = MOTHERS[mother]
    n0 = x.size
    Jr, sj, _, _ = shim.cwt_axes_mother(n0, DT, dj, -1, J, code, param)
    xr = x.astype(np.float64) if f64 else x.astype(np.float32).astype(np.float64)
    ref = cl.cwt_rows(xr, DT, dj, -1, J, wl, rows)
    if f64:
        resolved = np.ones(len(rows), bool)
    elif mother == "morlet":
        resolved = cr.resolved_rows(n0, _nfft(n0), DT, dj, sj[0], Jr)[rows]
    else:
        resolved = np.ones(len(rows), bool)
    tol = 1e-10 if f64 else 1e-4
    worst = 0.0
    for got, want, what in ((power, np.abs(ref) ** 2, "power"), (coef, ref, "coef")):
        g = got[rows]
        ratio, where = cr.row_gate(g, want, tol, resolved)
        assert ratio <= 1.0, f"{mother} {what}: {ratio:.3g} of the row bound at row {rows[where[0]]}, t = {where[1]}"
        worst = max(worst, ratio)
        if not resolved.all():                    # the plane gate on the daughter-tail rows
            b = np.abs(want[~resolved])
            err = np.abs(g[~resolved].astype(want.dtype) - want[~resolved])
            assert np.all(err <= tol * b + tol * np.abs(want).max()), f"{mother} {what}: plane gate"
    return worst


def _cwt(shim, x, dj, J, mother, f64, coi_mask=False):
    code, param, _ = MOTHERS[mother]
    before = shim.kernel_launches()
    p, c = shim.cwt(x, DT, dj, -1, J, code, param, f64=f64, want_power=True, want_coef=True, coi_mask=coi_mask)
    return p, c, shim.kernel_launches() - before


# ---- against the reference ---------------------------------------------------------------------------
@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("mother", list(MOTHERS))
@pytest.mark.parametrize("f64", [False, True], ids=["fp32-8193", "fp64-4097"])
def test_first_new_lengths(shim, f64, mother, inp):
    n0 = 4097 if f64 else 8193
    x = _inputs(inp, 1, n0, seed=n0 + len(inp))[0]
    p, c, launches = _cwt(shim, x, 1 / 4, -1, mother, f64)
    S = p.shape[0]
    assert launches == cl.launches(_nfft(n0), f64, 1, S), "the long path did not serve the call"
    worst = _check_rows(shim, x, 1 / 4, -1, mother, f64, np.arange(S), p, c)
    print(f"LONGGATE {'fp64' if f64 else 'fp32'} {n0} {mother} {inp}: {worst:.3g}")


CASES_POW2 = [(1 << 17, m, inp) for m, inp in zip(MOTHERS, ["white", "ar1_0.989", "two_tone", "ar1_0.989"])] + \
             [(1 << 20, "morlet", "ar1_0.989"), (1 << 20, "dog2", "white")]


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("case", CASES_POW2, ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}")
def test_unpadded_powers_of_two(shim, case, f64):
    n0, mother, inp = case
    x = _inputs(inp, 1, n0, seed=7)[0]
    p, c, launches = _cwt(shim, x, 1 / 2, -1, mother, f64)
    S = p.shape[0]
    assert launches == cl.launches(n0, f64, 1, S)
    rows = np.arange(S) if n0 <= 1 << 17 else np.unique(np.r_[np.arange(0, S, 3), S - 1])
    worst = _check_rows(shim, x, 1 / 2, -1, mother, f64, rows, p, c)
    print(f"LONGGATE {'fp64' if f64 else 'fp32'} {n0} {mother} {inp}: {worst:.3g}")


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_three_million_samples(shim, f64):
    n0, J = 3_000_000, 16
    x = _inputs("ar1_0.989", 1, n0, seed=8)[0]
    p, c, launches = _cwt(shim, x, 1.0, J, "morlet", f64)
    assert p.shape == (J + 1, n0) and launches == cl.launches(1 << 22, f64, 1, J + 1)
    worst = _check_rows(shim, x, 1.0, J, "morlet", f64, np.array([0, 5, 10, 13, 16]), p, c)
    print(f"LONGGATE {'fp64' if f64 else 'fp32'} {n0} morlet ar1: {worst:.3g}")


@pytest.mark.parametrize("f64", [False, True], ids=["fp32-8193", "fp64-4097"])
@pytest.mark.parametrize("mother", ["morlet", "paul4"])
def test_coi_mask(shim, f64, mother):
    n0 = 4097 if f64 else 8193
    x = _inputs("white", 1, n0, seed=9)[0]
    pm, _, _ = _cwt(shim, x, 1 / 4, -1, mother, f64, coi_mask=True)
    p, _, _ = _cwt(shim, x, 1 / 4, -1, mother, f64)
    code, param, wl = MOTHERS[mother]
    _, sj, _, _ = shim.cwt_axes_mother(n0, DT, 1 / 4, -1, -1, code, param)
    coi = wl.flambda() * wl.coi() * DT * (n0 / 2 - np.abs(np.arange(n0) - (n0 - 1) / 2))
    period = 1 / (1 / (wl.flambda() * sj))
    outside = period[:, None] > coi[None, :]
    assert np.array_equal(np.isnan(pm), outside) and outside.any() and (~outside).any()
    assert np.array_equal(pm[~outside], p[~outside])


# ---- dispatch and refusals -----------------------------------------------------------------------------
@pytest.mark.parametrize("f64,n0", [(False, 8192), (True, 4096)])
def test_largest_one_cta_lengths_keep_the_generic_path(shim, f64, n0):
    x = _inputs("white", 1, n0, seed=10)[0]
    before = shim.kernel_launches()
    shim.cwt(x, DT, 1 / 4, -1, -1, 0, 6.0, f64=f64, want_power=True, want_coef=True)
    assert shim.kernel_launches() - before == 2
    assert cl.route(n0, f64) == "generic" and cl.route(2 * n0, f64) == "long"


@pytest.mark.parametrize("f64", [False, True])
def test_refusals(shim, f64):
    lib = shim.lib()
    rt = np.float64 if f64 else np.float32
    x = np.random.default_rng(3).standard_normal((1, 5000)).astype(rt)
    out = np.zeros((1, 9, 5000), rt)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    flags = shim.F64 if f64 else 0
    before = shim.kernel_launches()
    assert lib.wtb_cwt(p(x), 1, 5000, 1 << 23, DT, 1.0, 2.0, 8, 0, 6.0, flags, p(out), None, None) == EUNSUPPORTED
    assert b"2^22" in lib.wtb_last_error()
    if not f64:
        # un-padded lengths past the Bluestein limit: the refusal and message are unchanged
        assert lib.wtb_cwt(p(x), 1, 5000, 5000, DT, 1.0, 2.0, 8, 0, 6.0, flags, p(out), None, None) == EUNSUPPORTED
        assert lib.wtb_last_error() == (b"nfft=5000 needs 262144 B of shared memory per CTA (limit 227 KB): a power of "
                                        b"two up to 8192, any other length up to 4096 for float")
    # an empty batch returns before the length is looked at, for wtb_cwt and wtb_cwt_averages alike
    glob = np.zeros((1, 9), rt)
    for nfft in (5000, 1 << 23, 1_500_000_001):
        assert lib.wtb_cwt(p(x), 0, 5000, nfft, DT, 1.0, 2.0, 8, 0, 6.0, flags, p(out), None, None) == 0, nfft
        assert lib.wtb_cwt_averages(p(x), 0, 5000, nfft, DT, 1.0, 2.0, 8, 0, 6.0, 0, 0, 1.0, flags, p(glob), None,
                                    None) == 0, nfft
    assert shim.kernel_launches() == before


@pytest.mark.parametrize("f64,n0", [(False, 8193), (True, 4097), (True, 20000)])
def test_morlet_entry_point_keeps_its_lengths(shim, f64, n0):
    """wtb_cwt_morlet refuses the lengths past one CTA, naming wtb_cwt, which serves them with the same
    Morlet arithmetic; engine.cwt_power_resident and run_cwt go through wtb_cwt."""
    import torch
    from wavelet_transformer_b200 import engine
    x = _inputs("white", 2, n0, seed=18)
    before = shim.kernel_launches()
    with pytest.raises(RuntimeError, match="wtb_cwt with WTB_MORLET"):
        shim.cwt_morlet(x, DT, 1 / 4, -1, -1, f64=f64)
    assert shim.kernel_launches() == before
    p, _ = shim.cwt(x, DT, 1 / 4, -1, -1, 0, 6.0, f64=f64)
    dtype = torch.float64 if f64 else torch.float32
    xd = torch.as_tensor(x, dtype=dtype, device="cuda").contiguous()
    pd = torch.empty(p.shape, dtype=dtype, device="cuda")
    engine.cwt_power_resident(xd, pd, DT, 1 / 4, -1, p.shape[1] - 1)
    torch.cuda.synchronize()
    assert np.array_equal(pd.cpu().numpy(), p)


def test_run_cwt_of_a_long_series(shim):
    from wavelet_transformer_b200.api import cwt as api
    y = _inputs("ar1_0.989", 1, 6000, seed=19)[0]
    t = np.arange(y.size).astype("datetime64[M]").astype("datetime64[D]")
    res = api.run_cwt(api.DataForCWT(t, y, api.MOTHER, api.DT, api.DJ, api.S0, api.LEVELS),
                      calculate_significance=False)
    W, _, freqs, _, _, _ = po.cwt(y, api.DT, api.DJ, api.S0, int(api.J), po.Morlet(6))
    ratio, where = cr.row_gate(res.power, np.abs(W) ** 2, 1e-10)
    assert ratio <= 1.0, f"{ratio:.3g} of the row bound at {where}"
    assert np.allclose(res.period, 1 / freqs, rtol=1e-13)


# ---- invariance ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("f64,n0", [(False, 1 << 19), (True, 1 << 18)])
def test_bits_do_not_depend_on_the_batch(shim, f64, n0):
    """16 rows per wave: in batches of 7, 3 and 1 the wave boundaries fall on different scales of a series."""
    x = _inputs("white", 7, n0, seed=11)
    p7, _ = shim.cwt(x, DT, 1 / 2, -1, -1, 0, 6.0, f64=f64)
    S = p7.shape[1]
    wave = cl.wave_rows(n0, f64, 7 * S)

    def cuts(first, batch):          # scales of series `first` at which a wave starts, in a batch from series 0
        return {r - first * S for r in range(0, batch * S, wave) if first * S <= r < (first + 1) * S}

    assert wave == 16 and cuts(4, 7) != cuts(2, 3) != cuts(0, 1) and cuts(4, 7) != cuts(0, 1)
    p3, _ = shim.cwt(x[2:5], DT, 1 / 2, -1, -1, 0, 6.0, f64=f64)
    assert np.array_equal(p3, p7[2:5])
    for i in (0, 4, 6):
        p1, _ = shim.cwt(x[i], DT, 1 / 2, -1, -1, 0, 6.0, f64=f64)
        assert np.array_equal(p1, p7[i])


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
    x = _inputs("ar1_0.989", 5, 1 << 17, seed=12)
    p2, c2 = shim.cwt(x, DT, 1 / 2, -1, -1, 2, 2.0, f64=f64, want_coef=True)
    shim.init_multi(1)
    p1, c1 = shim.cwt(x, DT, 1 / 2, -1, -1, 2, 2.0, f64=f64, want_coef=True)
    assert np.array_equal(p1, p2) and np.array_equal(c1, c2)


def _device_call(shim, torch, xd, dj, J, mother, f64, power, coef, coi_mask=False):
    code, param, _ = MOTHERS[mother]
    batch, n0 = xd.shape
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0) | (shim.COI_MASK if coi_mask else 0)
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    rc = shim.lib().wtb_cwt(ptr(xd), batch, n0, _nfft(n0), DT, dj, -1.0, J, code, param, flags, ptr(power), ptr(coef),
                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, shim.lib().wtb_last_error()


@pytest.mark.parametrize("f64", [False, True])
def test_device_pointers_equal_host_buffers(shim, f64):
    import torch
    x = _inputs("two_tone", 2, 70001, seed=13)
    p, c = shim.cwt(x, DT, 1 / 4, -1, -1, 1, 4.0, f64=f64, want_coef=True)
    dtype = torch.float64 if f64 else torch.float32
    xd = torch.as_tensor(x, dtype=dtype, device="cuda").contiguous()
    pd = torch.empty(p.shape, dtype=dtype, device="cuda")
    cd = torch.empty(c.shape, dtype=torch.complex128 if f64 else torch.complex64, device="cuda")
    _device_call(shim, torch, xd, 1 / 4, -1, "paul4", f64, pd, cd)
    torch.cuda.synchronize()
    assert np.array_equal(pd.cpu().numpy(), p) and np.array_equal(cd.cpu().numpy(), c)


# ---- guards and scratch --------------------------------------------------------------------------------
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
    batch, J = 3, 30
    x = torch.randn(batch, n0, dtype=dtype, device="cuda")
    n = batch * (J + 1) * n0
    pbuf, pw = _guarded(torch, n, dtype)
    cbuf, cf = _guarded(torch, 2 * n, dtype)              # complex as interleaved reals
    _device_call(shim, torch, x, 1 / 2, J, "morlet", f64, pw, cf)
    torch.cuda.synchronize()
    assert _intact(pbuf, n) and _intact(cbuf, 2 * n)
    assert bool(torch.isfinite(pw).all()) and bool(torch.isfinite(cf).all())


def test_scratch_after_a_long_call(shim):
    n0, dj = 1 << 20, 1 / 2
    x = _inputs("white", 1, n0, seed=14)
    shim.shutdown()
    shim.init(0)
    assert shim.scratch_bytes() == 0
    p, _ = shim.cwt(x, DT, dj, -1, -1, 0, 6.0, f64=False)
    S = p.shape[1]
    grown = lambda b: b + b // 8 + (1 << 20)        # the arenas' growth rule
    xhat, wave = 8 * n0, 8 * n0 * cl.wave_rows(n0, False, S)
    staging = 4 * (n0 + S * n0) + 1024
    assert shim.scratch_bytes() <= grown(256 + xhat + wave) + grown(staging)


# ---- averages ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n0,dj", [(20000, 1 / 4), (1 << 20, 1 / 2)])
def test_averages(shim, n0, dj, f64):
    batch = 2
    x = _inputs("ar1_0.989", batch, n0, seed=15)
    _, sj, _, _ = shim.cwt_axes_mother(n0, DT, dj, -1, -1, 0, 6.0)
    S = sj.size
    band = (S // 3, 2 * S // 3)
    factor = dj * DT / 0.776
    before = shim.kernel_launches()
    g, b = shim.cwt_averages(x, DT, dj, -1, -1, 0, 6.0, band=band, band_factor=factor, f64=f64)
    chunk = cl.averages_chunk_rows(batch, S, n0, f64)
    nchunks = -(-batch // chunk)
    assert shim.kernel_launches() - before == nchunks * (cl.launches(_nfft(n0), f64, chunk, S) + 1)
    tol = 1e-10 if f64 else 1e-4
    resolved = cr.resolved_rows(n0, _nfft(n0), DT, dj, sj[0], S - 1)
    for i in range(batch):
        xi = x[i] if f64 else x[i].astype(np.float32).astype(np.float64)
        W = po.cwt(xi, DT, dj, -1, -1, po.Morlet(6))[0]
        ratio, where = oa.averages_gate(g[i], b[i], W, sj, band, factor, tol, resolved)
        assert ratio <= 1.0, f"series {i}: {ratio:.3g} of the bound at {where}"
        del W
    P, _ = shim.cwt(x, DT, dj, -1, -1, 0, 6.0, f64=f64)
    P = P.astype(np.float64)
    lo, hi = band
    ref_g = P.mean(axis=2)
    ref_b = factor * (P[:, lo:hi + 1] * (1.0 / sj[lo:hi + 1])[None, :, None]).sum(axis=1)
    del P
    for got, ref in ((g, ref_g), (b, ref_b)):
        if f64:
            assert (np.abs(got - ref) / np.abs(ref)).max() <= 1e-13
        else:
            ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
            assert (np.abs(got.astype(np.float64) - ref) / ulp).max() <= 1.0


def test_averages_one_chunk_per_series_past_1_gib(shim):
    n0, dj, batch = 1 << 20, 1 / 12, 2
    x = _inputs("white", batch, n0, seed=16)
    _, sj, _, _ = shim.cwt_axes_mother(n0, DT, dj, -1, -1, 0, 6.0)
    S = sj.size
    assert 8 * S * n0 > 1 << 30 and cl.averages_chunk_rows(batch, S, n0, True) == 1
    before = shim.kernel_launches()
    g, _ = shim.cwt_averages(x, DT, dj, -1, -1, 0, 6.0, f64=True)
    assert shim.kernel_launches() - before == batch * (cl.launches(n0, True, 1, S) + 1)
    g1, _ = shim.cwt_averages(x[1], DT, dj, -1, -1, 0, 6.0, f64=True)
    assert np.array_equal(g1, g[1]) and np.all(g > 0)


# ---- façade --------------------------------------------------------------------------------------------
def test_pycwt_compat_cwt_of_10000_samples(shim):
    from wavelet_transformer_b200 import pycwt_compat as pc
    x = _inputs("ar1_0.989", 1, 10000, seed=17)[0]
    W, sj, freqs, coi, fft, fftfreqs = pc.cwt(x, 1.0, 1 / 12, -1, -1, "morlet")
    Wr, sjr, fr, coir, fftr, ffr = po.cwt(x, 1.0, 1 / 12, -1, -1, po.Morlet(6))
    assert W.shape == Wr.shape == (sjr.size, 10000)
    ratio, where = cr.row_gate(W, Wr, 1e-10)
    assert ratio <= 1.0, f"{ratio:.3g} of the row bound at {where}"
    assert np.allclose(sj, sjr, rtol=1e-13) and np.allclose(coi, coir, rtol=1e-13)
    xr = pc.icwt(W, sj, 1.0, 1 / 12, "morlet")
    ref = po.icwt(Wr, sjr, 1.0, 1 / 12, po.Morlet(6))
    assert np.abs(xr - ref).max() <= 1e-10 * np.abs(ref).max()
