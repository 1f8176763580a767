"""Per-scale-row parity of the FP32 Morlet CWT, XWT and WCT kernels (oracle/cwt_rows.py).

Every scale row of an FP32 transform is its own pruned inverse transform, so its error is
relative to that row, not to the plane maximum.  Each FP32 kernel is held row by row to
`row_gate` at 1e-4 on the resolved rows (the others keep the plane gate): against the float64
oracle on sampled series, and against the FP64 generic kernel on every series of the batch.
The shapes reach every row class of each kernel's pruned transforms (the host row rules are
replicated in oracle/cwt_rows.py).  The inputs are zero-mean and cover the spectra the project
is for: white, AR(1) 0.7 (cfg4), AR(1) 0.989 (cfg5), a random walk, and a unit sine with a 1e-3
sine at a 3-sample period (rows down to 1e-10 of the plane maximum)."""

import numpy as np
import pytest
from scipy.signal import lfilter

from conftest import normwise_close
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1 / 12
DJ, S0, J = 1 / 12, 2 * DT, 119          # 120 rows: s/dt from 2 to 1956, every row class of every kernel

INPUTS = ["white", "ar1_0.7", "ar1_0.989", "walk", "two_tone"]


def _inputs(kind, batch, n0, seed):
    rng = np.random.default_rng(seed)
    if kind == "white":
        x = rng.standard_normal((batch, n0))
    elif kind.startswith("ar1_"):
        g = float(kind[4:])
        burn = 2000
        x = lfilter([1.0], [1.0, -g], rng.standard_normal((batch, n0 + burn)), axis=1)[:, burn:]
    elif kind == "walk":
        x = rng.standard_normal((batch, n0)).cumsum(axis=1)
    elif kind == "two_tone":
        t = np.arange(n0)
        period = rng.uniform(20.0, 60.0, size=(batch, 1))
        ph = rng.uniform(0, 2 * np.pi, size=(batch, 2))
        x = np.sin(2 * np.pi * t / period + ph[:, :1]) + 1e-3 * np.sin(2 * np.pi * t / 3.0 + ph[:, 1:])
    else:
        raise ValueError(kind)
    return x - x.mean(axis=1, keepdims=True)


# (kernel, n0, batch, output, env): the batch sizes give the 1024 kernel row splits of 16 and 7,
# odd batches leave the two-series kernels (HALF, register rows) with a half-empty last item
CASES = [
    ("fast1024", 1024, 1, "power", None),
    ("fast1024", 1024, 300, "power", None),
    ("fast1024", 700, 1, "power", None),
    ("fast1024", 700, 300, "power", None),
    ("half", 400, 7, "power", None),
    ("half", 512, 5, "power", None),
    ("dif2", 1346, 13, "power", None),
    ("dif2", 2048, 13, "power", None),
    ("dif4", 3351, 5, "power", None),
    ("dif4", 4096, 5, "power", None),
    ("rows4096", 3351, 5, "power", "default_min_batch"),
    ("rows4096", 4096, 5, "coef", None),
    ("generic", 1024, 3, "power", None),
    ("generic", 3351, 3, "coef", None),
    ("fp64", 1346, 2, "power", None),
    ("fp64", 4096, 2, "coef", None),
]
# launches of one call: forward-FFT kernels + row kernel
LAUNCHES = {"fast1024": 1, "half": 1, "dif2": 2, "dif4": 3, "rows4096": 2}


def _case_id(c):
    return f"{c[0]}-{c[3]}-{c[1]}x{c[2]}"


def _run(shim, kernel, x, output, f64=False, generic=None):
    generic = kernel in ("generic", "fp64") if generic is None else generic
    p, c = shim.cwt_morlet(x, DT, DJ, S0, J, f64=f64, want_power=output == "power", want_coef=output == "coef",
                           generic_only=generic)
    return p if output == "power" else c


def _nfft(n0):
    return 1 << (n0 - 1).bit_length()


def _check_rows(got, ref, resolved, tol, what):
    """row_gate on the resolved rows, the plane gate on the rest; returns the row-gate ratio."""
    ratio, where = cr.row_gate(got, ref, tol, resolved)
    assert ratio <= 1.0, f"{what}: {ratio:.3g} of the per-row bound at (row, t) = {where}"
    if (~resolved).any():
        a, b = got[~resolved].astype(ref.dtype), ref[~resolved]
        err = np.abs(a - b) - tol * np.abs(b)
        assert err.max() <= tol * np.abs(ref).max(), f"{what}: unresolved rows fail the plane gate"
    return ratio


@pytest.mark.parametrize("inp", INPUTS)
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_cwt_rows_against_float64(shim, monkeypatch, case, inp):
    kernel, n0, batch, output, env = case
    if env == "default_min_batch":
        monkeypatch.delenv("WTB_CWT_MIN_BATCH")        # 5 series: below the DIF kernel's four per SM
    x = _inputs(inp, batch, n0, seed=n0 * 1000 + batch)
    nfft = _nfft(n0)
    resolved = cr.resolved_rows(n0, nfft, DT, DJ, S0, J)
    assert resolved.sum() >= 90
    f64 = kernel == "fp64"
    if kernel in LAUNCHES:
        classes = cr.row_classes(kernel, DT, DJ, S0, J)
        assert set(classes) == cr.ROW_CLASSES[cr.class_family(kernel)], "the shape misses a row class"
    launches = shim.kernel_launches()
    got = _run(shim, kernel, x, output, f64=f64)
    if kernel in LAUNCHES:
        assert shim.kernel_launches() - launches == LAUNCHES[kernel], "another kernel served the call"
        gen32 = _run(shim, kernel, x[:2], output, generic=True)
        assert not np.array_equal(got[:2], gen32), "the FP32 generic kernel served the call"
    tol = 1e-10 if f64 else 1e-4
    tag = f"{_case_id(case)} {inp}"
    worst_oracle = 0.0
    for b in sorted({0, batch - 1}):
        W = po.cwt(x[b], DT, DJ, S0, J, po.Morlet(6))[0]
        ref = W if output == "coef" else np.abs(W) ** 2
        worst_oracle = max(worst_oracle, _check_rows(got[b], ref, resolved, tol, f"{tag} series {b} vs oracle"))
    worst_f64 = 0.0
    if not f64:
        ref64 = _run(shim, "fp64", x, output, f64=True)
        for b in range(batch):
            worst_f64 = max(worst_f64, _check_rows(got[b], ref64[b], resolved, tol, f"{tag} series {b} vs FP64"))
    print(f"ROWGATE {tag}: oracle {worst_oracle:.3g}, fp64-generic {worst_f64:.3g}")


# ---- amplitude equivariance: bit-exact ------------------------------------------------------
EQ_CASES = [
    ("fast1024", 1024, 4, "power", None),
    ("fast1024", 700, 3, "power", None),
    ("half", 400, 7, "power", None),
    ("dif2", 1346, 13, "power", None),
    ("dif4", 3351, 5, "power", None),
    ("rows4096", 3351, 5, "power", "default_min_batch"),
    ("rows4096", 4096, 5, "coef", None),
    ("generic", 1024, 3, "power", None),
    ("generic", 3351, 3, "coef", None),
    ("fp64", 1346, 2, "power", None),
    ("fp64", 4096, 2, "coef", None),
]
TINY = 2.0 ** -100


@pytest.mark.parametrize("case", EQ_CASES, ids=_case_id)
def test_cwt_amplitude_equivariance_is_exact(shim, monkeypatch, case):
    """Scaling the even-indexed series of a batch by 2^k scales their power by exactly 4^k (their
    coefficients by 2^k) and leaves the odd series bit-unchanged: the daughter does not depend on
    the data, HALF renormalises each series by an exact power of two, and the two series that share
    a warp (HALF) or the two FFMA2 lanes of a CTA (register rows) must not leak into each other.
    Checked on every element whose unscaled and scaled magnitudes are both >= 2^-100 (no
    subnormals).  Also catches flush-to-zero or an amplitude-dependent path at 1e+-12."""
    kernel, n0, batch, output, env = case
    if env == "default_min_batch":
        monkeypatch.delenv("WTB_CWT_MIN_BATCH")
    f64 = kernel == "fp64"
    rt = np.float64 if f64 else np.float32
    x = _inputs("walk", batch, n0, seed=7 + n0).astype(rt)
    base = _run(shim, kernel, x, output, f64=f64)
    even = np.arange(batch) % 2 == 0
    for k in (16, -16, 40, -40):
        xs = x.copy()
        xs[even] *= rt(2.0 ** k)
        got = _run(shim, kernel, xs, output, f64=f64)
        gain = 4.0 ** k if output == "power" else 2.0 ** k
        parts = (lambda v: (v,)) if output == "power" else (lambda v: (v.real, v.imag))
        for b in range(batch):
            for u, s in zip(parts(base[b]), parts(got[b])):
                want = u * rt(gain) if even[b] else u
                mask = (np.abs(u) >= TINY) & (np.abs(s) >= TINY) & (np.abs(want) >= TINY)
                bad = mask & (s != want)
                assert not bad.any(), (f"{_case_id(case)} k={k} series {b}: {int(bad.sum())} elements not exactly "
                                       f"{'scaled' if even[b] else 'unchanged'}, first at {np.argwhere(bad)[0]}")
                print(f"EQUIV {_case_id(case)} k={k} series {b}: {mask.mean():.4f} of the plane compared")


# ---- XWT / WCT in FP32 ---------------------------------------------------------------------
def _pair(kind, n0, seed):
    rng = np.random.default_rng(seed)
    if kind == "ar1_0.989_0.966":
        y1, y2 = po.rednoise(n0, 0.989, 1, rng), po.rednoise(n0, 0.966, 1, rng)
    elif kind == "walk_pair":
        a, b = rng.standard_normal((2, n0)).cumsum(axis=1)
        y1, y2 = a, 0.6 * a + 0.8 * b
    else:
        raise ValueError(kind)
    return (y1 - y1.mean()) / y1.std(), (y2 - y2.mean()) / y2.std()


# (n0, nfft or None = next power of two, generic_only): nfft 4096 fast and generic kernels, the
# generic kernels at nfft 1024 and 2048, and an un-padded (Bluestein) length
XWT_SHAPES = [(3351, None, False), (3351, None, True), (1000, None, False), (1346, None, False), (700, 700, False)]


def _xwt_case(shim, y1, y2, n0, nfft, generic, dj, Jx, tag, check_wct=True):
    pad = nfft is None
    nf = _nfft(n0) if pad else nfft
    wct, phase, w12 = shim.xwt_wct(y1, y2, DT, dj, S0, Jx, f64=False, want_w12=True, nfft=nfft,
                                   generic_only=generic)
    W1 = po.cwt(y1, DT, dj, S0, Jx, po.Morlet(6), pad_pow2=pad)[0]
    W2 = po.cwt(y2, DT, dj, S0, Jx, po.Morlet(6), pad_pow2=pad)[0]
    ref12 = W1 * W2.conj()
    resolved = cr.resolved_rows(n0, nf, DT, dj, S0, Jx)
    r_w12 = _check_rows(w12, ref12, resolved, 1e-4, f"{tag} w12")
    # the phase as the phasor |W12| e^{i phase}: the circle distance weighted by the magnitude, so
    # the phase of a near-zero cross spectrum does not count
    r_ph = _check_rows(np.abs(ref12) * np.exp(1j * phase.astype(np.float64)), ref12, resolved, 1e-4, f"{tag} phase")
    err = float("nan")
    if check_wct:
        WCT = po.wct(y1, y2, DT, dj=dj, s0=S0, J=Jx, sig=False, normalize=False, pad_pow2=pad)[0]
        ok, err = normwise_close(wct, WCT, 1e-4)
        assert ok, f"{tag} wct: {err:.3e}"
    print(f"ROWGATE xwt {tag}: w12 {r_w12:.3g}, phase {r_ph:.3g}, wct plane {err:.3g}")


@pytest.mark.parametrize("n0,nfft,generic", XWT_SHAPES)
@pytest.mark.parametrize("pair", ["ar1_0.989_0.966", "walk_pair"])
def test_xwt_wct_fp32_rows(shim, pair, n0, nfft, generic):
    y1, y2 = _pair(pair, n0, seed=n0)
    jx = int(np.floor(np.log2(n0 / 2.0) / (1 / 8)))
    _xwt_case(shim, y1, y2, n0, nfft, generic, 1 / 8, jx, f"{pair} n0={n0} nfft={nfft} generic={generic}")


@pytest.mark.parametrize("nfft", [None, 565])
def test_xwt_wct_fp32_rows_cfg3_pair(shim, series, nfft):
    """BASELINE cfg3's real pair (inflation, expectation; n0 = 565, dj = 1/8, 66 scales)."""
    y1, y2 = series["pair_inflation"], series["pair_expectation"]
    y1, y2 = (y1 - y1.mean()) / y1.std(), (y2 - y2.mean()) / y2.std()
    _xwt_case(shim, y1, y2, 565, nfft, False, 1 / 8, 65, f"cfg3 nfft={nfft}")


# ---- a strong line just past a 256-bin block of the register rows' band -----------------------
def _edge_lines(n0, seed):
    """A line of amplitude 30 at bin 1024 of 4096 (period 4 samples) and a unit line at the peak of
    row 21 (dj = 1/12, s0 = 2 dt: s/dt = 6.73, peak bin 581).  Row 21's band ends at k_hi = 1095,
    so its register-row transform must read the block of bins 1024 .. 2047, where the daughter is
    3e-5 of its peak (z = 4.57) but the line is 30 times stronger: the row sits at 2e-3 of the
    plane maximum and a band cut short of k_hi errs by about 10 times the per-row bound there."""
    rng = np.random.default_rng(seed)
    t = np.arange(n0)
    a = (6.0 / (2 * 2.0 ** (21 / 12) * 2 * np.pi / 4096))
    ph = rng.uniform(0, 2 * np.pi, 2)
    x = 30 * np.cos(2 * np.pi * t / 4 + ph[0]) + np.cos(2 * np.pi * t * a / 4096 + ph[1])
    return x - x.mean()


@pytest.mark.parametrize("case", [("rows4096", 4096, 3, "power", "default_min_batch"), ("rows4096", 4096, 3, "coef", None),
                                  ("dif4", 4096, 3, "power", None), ("generic", 4096, 3, "power", None)], ids=_case_id)
def test_cwt_rows_band_edge_lines(shim, monkeypatch, case):
    kernel, n0, batch, output, env = case
    if env == "default_min_batch":
        monkeypatch.delenv("WTB_CWT_MIN_BATCH")
    x = np.stack([_edge_lines(n0, b) for b in range(batch)])
    resolved = cr.resolved_rows(n0, 4096, DT, DJ, S0, J)
    got = _run(shim, kernel, x, output)
    worst = 0.0
    for b in range(batch):
        W = po.cwt(x[b], DT, DJ, S0, J, po.Morlet(6))[0]
        ref = W if output == "coef" else np.abs(W) ** 2
        assert 1e-3 < ref[21].max() / ref.max() < 1e-2 or output == "coef"
        worst = max(worst, _check_rows(got[b], ref, resolved, 1e-4, f"{_case_id(case)} series {b}"))
    print(f"ROWGATE {_case_id(case)} edge_lines: oracle {worst:.3g}")


def test_xwt_rows_band_edge_lines(shim):
    """The same lines through the nfft = 4096 cross-spectrum kernel (k_wct_spec_4096, same row rules).
    Cross spectrum and phase only: far from both lines the smoothed spectra of two pure lines
    underflow, and even the float64 oracle's coherence is 0 / 0 there."""
    y1, y2 = _edge_lines(4096, 1), _edge_lines(4096, 2)
    y1, y2 = y1 / y1.std(), y2 / y2.std()
    _xwt_case(shim, y1, y2, 4096, None, False, DJ, J, "edge_lines n0=4096", check_wct=False)


# ---- FP32 inverse transform ----------------------------------------------------------------
@pytest.mark.parametrize("mother", ["morlet", "dog2"])
def test_icwt_fp32(shim, mother):
    """wtb_icwt in FP32 on the FP32 coefficients of a Morlet and a DOG transform against the
    oracle's icwt of the same coefficients, norm-wise at 1e-4."""
    x = _inputs("ar1_0.7", 1, 1345, seed=3)[0]
    x /= x.std()
    if mother == "morlet":
        code, param, ref_m, psi0 = shim.MORLET, 6.0, po.Morlet(6), np.pi ** -0.25
    else:
        code, param, ref_m = shim.DOG, 2, po.DOG(2)
        psi0 = ref_m.psi0()
    _, coef = shim.cwt(x, DT, 1 / 12, S0, -1, code, param, f64=False, want_power=False, want_coef=True)
    _, sj, _, _ = shim.cwt_axes_mother(x.size, DT, 1 / 12, S0, -1, code, param)
    factor = (1 / 12) * np.sqrt(DT) / (ref_m.cdelta * psi0)
    rec = shim.icwt(coef, sj, factor, f64=False)
    ref = po.icwt(coef.astype(np.complex128), sj, DT, 1 / 12, ref_m)
    assert rec.dtype == np.float32 and rec.shape == ref.shape
    ok, err = normwise_close(rec, ref, 1e-4)
    assert ok, f"{mother}: {err:.3e}"
    # and the transform round trip itself is the oracle's to the same gate
    W = po.cwt(x, DT, 1 / 12, S0, -1, ref_m)[0]
    ok, err = normwise_close(rec, po.icwt(W, sj, DT, 1 / 12, ref_m), 1e-4)
    assert ok, f"{mother} round trip: {err:.3e}"
