"""GPU: time- and scale-averaged wavelet power (wtb_cwt_averages).

Each kernel class of the power plane feeds the reduction: the averages are held to the float64 oracle
(po.cwt -> |W|^2 -> mean and band sum) through `averages_gate`, and to a NumPy float64 reduction of the
engine's own power plane of the same call (1 ulp of float32, 1e-13 relative in FP64), which pins the
reduction kernel apart from the transform.  Results are bit-identical across batch sizes, pool sizes and
chunk boundaries; device pointers give the host path's bits; writes stay inside their outputs."""

import ctypes as C
import os

import numpy as np
import pytest
from scipy.signal import lfilter

from oracle import averages as oa
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1 / 12
DJ, S0, J = 1 / 12, 2 * DT, 119
S = J + 1
FACTOR = DJ * DT / 0.776
BANDS = {"narrow": (30, 41), "full": (0, J)}
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


# (kernel, n0, batch, mother, nfft): the kernel classes and shapes of test_gpu_cwt_rows.py
CASES = [
    ("fast1024", 1024, 1, "morlet", None),
    ("fast1024", 1024, 300, "morlet", None),
    ("fast1024", 700, 1, "morlet", None),
    ("fast1024", 700, 300, "morlet", None),
    ("half", 400, 7, "morlet", None),
    ("dif2", 1346, 13, "morlet", None),
    ("dif4", 3351, 5, "morlet", None),
    ("generic", 3351, 3, "morlet", None),
    ("fp64", 1346, 2, "morlet", None),
    ("generic", 1024, 3, "paul4", None),
    ("generic", 1024, 3, "dog2", None),
    ("generic", 700, 3, "morlet", 700),
]
# launches of the transform of one call (forward-FFT kernels + row kernel); the reduction adds one
LAUNCHES = {"fast1024": 1, "half": 1, "dif2": 2, "dif4": 3, "generic": 2, "fp64": 2}
MOTHERS = {"morlet": (0, 6.0, po.Morlet(6)), "paul4": (1, 4.0, po.Paul(4)), "dog2": (2, 2.0, po.DOG(2))}


def _case_id(c):
    return f"{c[0]}-{c[3]}-{c[1]}x{c[2]}" + (f"-nfft{c[4]}" if c[4] else "")


def _averages(shim, x, mother="morlet", band=BANDS["full"], f64=False, nfft=None, generic=False):
    code, param, _ = MOTHERS[mother]
    return shim.cwt_averages(x, DT, DJ, S0, J, code, param, band=band, band_factor=FACTOR, f64=f64, nfft=nfft,
                             generic_only=generic)


@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_averages_against_float64_and_own_plane(shim, case, inp):
    kernel, n0, batch, mother, nfft = case
    f64 = kernel == "fp64"
    generic = kernel in ("generic", "fp64")
    code, param, ref_m = MOTHERS[mother]
    x = _inputs(inp, batch, n0, seed=n0 * 1000 + batch)
    nf = nfft or (1 << (n0 - 1).bit_length())
    resolved = cr.resolved_rows(n0, nf, DT, DJ, S0, J) if mother == "morlet" else np.ones(S, bool)
    _, sj, _, _ = shim.cwt_axes_mother(n0, DT, DJ, S0, J, code, param)
    tol = 1e-10 if f64 else 1e-4
    for name, band in BANDS.items():
        launches = shim.kernel_launches()
        g, b = _averages(shim, x, mother, band, f64=f64, nfft=nfft, generic=generic)
        assert shim.kernel_launches() - launches == LAUNCHES[kernel] + 1, "another kernel served the call"
        assert g.shape == (batch, S) and b.shape == (batch, n0) and g.dtype == (np.float64 if f64 else np.float32)
        worst = 0.0
        for i in sorted({0, batch - 1}):
            W = po.cwt(x[i], DT, DJ, S0, J, ref_m, pad_pow2=nfft is None)[0]
            ratio, where = oa.averages_gate(g[i], b[i], W, sj, band, FACTOR, tol, resolved)
            assert ratio <= 1.0, f"{_case_id(case)} {inp} {name} series {i}: {ratio:.3g} of the bound at {where}"
            worst = max(worst, ratio)
        # the reduction alone: a float64 NumPy reduction of the plane the same call's transform produces
        P, _ = shim.cwt(x, DT, DJ, S0, J, code, param, f64=f64, nfft=nfft, generic_only=generic)
        P = P.astype(np.float64)
        lo, hi = band
        ref_g = P.mean(axis=2)
        ref_b = FACTOR * (P[:, lo:hi + 1] * (1.0 / sj[lo:hi + 1])[None, :, None]).sum(axis=1)
        for got, ref, what in ((g, ref_g, "global"), (b, ref_b, "band")):
            if f64:
                err = np.abs(got - ref) / np.abs(ref)
                assert err.max() <= 1e-13, f"{what}: {err.max():.3g} relative to a float64 reduction"
            else:
                ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
                err = np.abs(got.astype(np.float64) - ref) / ulp
                assert err.max() <= 1.0, f"{what}: {err.max():.3g} ulp from a float64 reduction"
        print(f"AVGGATE {_case_id(case)} {inp} {name}: oracle {worst:.3g}")


# ---- invariance ----------------------------------------------------------------------------------------
def _chunk_rows(shim, batch, n0, elem):
    """The chunk rule of averages.cu: power rows of a chunk within 1 GiB, at least 16 warps per SM, even."""
    import torch
    fill = 16 * torch.cuda.get_device_properties(0).multi_processor_count
    return min(batch, max(fill, (1 << 30) // (elem * S * n0)) & ~1)


def test_averages_do_not_depend_on_the_batch(shim):
    x = _inputs("white", 300, 700, seed=11)
    g300, b300 = _averages(shim, x, band=BANDS["narrow"])
    for n in (1, 11):
        g, b = _averages(shim, x[:n], band=BANDS["narrow"])
        assert np.array_equal(g, g300[:n]) and np.array_equal(b, b300[:n])
    g1, b1 = _averages(shim, x[-1], band=BANDS["narrow"])
    assert g1.shape == (S,) and np.array_equal(g1, g300[-1]) and np.array_equal(b1, b300[-1])


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
def test_averages_split_over_the_pool(shim, pool, f64):
    x = _inputs("ar1_0.989", 37, 700, seed=12)
    g2, b2 = _averages(shim, x, f64=f64, generic=f64)
    shim.init_multi(1)
    g1, b1 = _averages(shim, x, f64=f64, generic=f64)
    assert np.array_equal(g1, g2) and np.array_equal(b1, b2)


def test_averages_across_a_chunk_boundary(shim):
    rows = _chunk_rows(shim, 10 ** 9, 700, 4)
    batch = rows + 7
    x = _inputs("white", batch, 700, seed=13).astype(np.float32)
    launches = shim.kernel_launches()
    g, b = _averages(shim, x, band=BANDS["narrow"])
    assert shim.kernel_launches() - launches == 2 * (LAUNCHES["fast1024"] + 1), "expected two chunks"
    part = slice(rows - 5, rows + 5)
    gp, bp = _averages(shim, x[part], band=BANDS["narrow"])
    assert np.array_equal(g[part], gp) and np.array_equal(b[part], bp)
    gt, bt = _averages(shim, x[-7:], band=BANDS["narrow"])
    assert np.array_equal(g[-7:], gt) and np.array_equal(b[-7:], bt)


# ---- device pointers and guard writes ------------------------------------------------------------------
@pytest.mark.parametrize("n0,batch,f64", [(1346, 13, False), (700, 300, False), (1346, 3, True)])
def test_resident_equals_host(shim, n0, batch, f64):
    import torch
    from wavelet_transformer_b200 import engine
    x = _inputs("ar1_0.989", batch, n0, seed=14)
    g, b = _averages(shim, x, band=BANDS["narrow"], f64=f64)
    dtype = torch.float64 if f64 else torch.float32
    xd = torch.as_tensor(x, dtype=dtype, device="cuda").contiguous()
    gd = torch.empty((batch, S), dtype=dtype, device="cuda")
    bd = torch.empty((batch, n0), dtype=dtype, device="cuda")
    engine.cwt_averages_resident(xd, gd, bd, DT, DJ, S0, J, band=BANDS["narrow"], band_factor=FACTOR)
    assert np.array_equal(gd.cpu().numpy(), g) and np.array_equal(bd.cpu().numpy(), b)
    # one output alone
    g_only = torch.empty_like(gd)
    engine.cwt_averages_resident(xd, g_only, None, DT, DJ, S0, J)
    b_only = torch.empty_like(bd)
    engine.cwt_averages_resident(xd, None, b_only, DT, DJ, S0, J, band=BANDS["narrow"], band_factor=FACTOR)
    assert torch.equal(g_only, gd) and torch.equal(b_only, bd)


GUARD = 4096


def _guarded(torch, shape, dtype):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * GUARD,), -7.0e33, dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n].view(*shape)


def _intact(buf, n):
    return bool((buf[:GUARD] == -7.0e33).all()) and bool((buf[GUARD + n:] == -7.0e33).all())


@pytest.mark.parametrize("n0,batch,J_,dj,f64", [(777, 5, 100, 1 / 12, False), (1346, 13, 84, 1 / 12, False),
                                                (400, 7, 91, 1 / 12, False), (3351, 3, 65, 1 / 8, False),
                                                (100, 3, 20, 1 / 4, False), (1025, 2, 84, 1 / 12, True)])
def test_averages_stay_inside_their_outputs(shim, n0, batch, J_, dj, f64):
    import torch
    from wavelet_transformer_b200 import engine
    dtype = torch.float64 if f64 else torch.float32
    x = torch.randn(batch, n0, dtype=dtype, device="cuda")
    gbuf, g = _guarded(torch, (batch, J_ + 1), dtype)
    bbuf, b = _guarded(torch, (batch, n0), dtype)
    engine.cwt_averages_resident(x, g, b, DT, dj, 2 * DT, J_, band=(1, J_ - 1), band_factor=0.5)
    torch.cuda.synchronize()
    assert _intact(gbuf, g.numel()) and _intact(bbuf, b.numel())
    assert bool(torch.isfinite(g).all()) and bool(torch.isfinite(b).all()) and bool((g > 0).all())


# ---- façade --------------------------------------------------------------------------------------------
def test_run_cwt_averages_matches_the_pycwt_sample(shim, series):
    """The averages section of the pycwt sample composed from the oracle, for the inflation series."""
    from wavelet_transformer_b200.api import cwt as api
    y = series["inflation_value"]
    n0 = y.size
    t = np.arange(n0).astype("datetime64[M]").astype("datetime64[D]")
    data = api.DataForCWT(t, y, api.MOTHER, api.DT, api.DJ, api.S0, api.LEVELS)
    other = api.DataForCWT(t, y[::-1].copy() * 3.0, api.MOTHER, api.DT, api.DJ, api.S0, api.LEVELS)
    res = api.run_cwt_averages([data, other])
    for r, yy in zip(res, (y, y[::-1] * 3.0)):
        W, sj, freqs, _, _, _ = po.cwt(yy, api.DT, api.DJ, api.S0, int(api.J), po.Morlet(6))
        power = np.abs(W) ** 2
        period = 1 / freqs
        var, alpha = yy.var(), po.ar1(yy)[0]
        glbl_signif, _ = oa.significance(var, api.DT, sj, 1, alpha, dof=n0 - sj)
        sel = np.nonzero((period >= 2) & (period < 8))[0]
        scale_avg = api.DJ * api.DT / 0.776 * (power / sj[:, None])[sel].sum(axis=0)
        avg_signif, _ = oa.significance(var, api.DT, sj, 2, alpha, dof=[sj[sel[0]], sj[sel[-1]]])
        assert np.allclose(r.period, period, rtol=1e-13)
        assert np.abs(r.glbl_power - power.mean(axis=1)).max() <= 1e-10 * power.mean(axis=1).max()
        assert np.allclose(r.glbl_signif, glbl_signif, rtol=1e-12)
        assert np.abs(r.scale_avg - scale_avg).max() <= 1e-10 * scale_avg.max()
        assert r.scale_avg_signif == pytest.approx(avg_signif, rel=1e-12)
    with pytest.raises(ValueError):
        api.run_cwt_averages([data], period_band=(2.0, 2.01))
    with pytest.raises(Warning):
        bad = series["pair_inflation"]
        api.run_cwt_averages([api.DataForCWT(t[:bad.size], bad, api.MOTHER, api.DT, api.DJ, api.S0, api.LEVELS)])


# ---- refusals ------------------------------------------------------------------------------------------
def test_refusals_return_einval(shim):
    lib = shim.lib()
    x = np.random.default_rng(3).standard_normal((2, 64))
    glob, band = np.zeros((2, 9)), np.zeros((2, 64))
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)

    def call(lo=0, hi=8, factor=1.0, flags=shim.F64, g=glob, b=band, batch=2):
        return lib.wtb_cwt_averages(p(x), batch, 64, 64, DT, 0.25, 2 * DT, 8, 0, 6.0, lo, hi, factor, flags, p(g),
                                    p(b), None)

    launches = shim.kernel_launches()
    for kwargs in ({"g": None, "b": None}, {"lo": -1}, {"lo": 5, "hi": 4}, {"hi": 9}, {"factor": float("nan")},
                   {"factor": float("inf")}, {"flags": shim.F64 | shim.COI_MASK}):
        assert call(**kwargs) == -1, kwargs
        assert lib.wtb_last_error()
    assert call(lo=-1, b=None) == 0                    # no band output: the band is not read
    assert call(batch=0) == 0
    assert shim.kernel_launches() - launches == LAUNCHES["generic"] + 1
    assert call() == 0
    W = po.cwt(x[1], DT, 0.25, 2 * DT, 8)[0]
    assert np.allclose(glob[1], (np.abs(W) ** 2).mean(axis=1), rtol=1e-10)
