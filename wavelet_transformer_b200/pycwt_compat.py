"""pycwt-shaped facade over the B200 engine.

The reference reaches its CWT/XWT/WCT numerics through ``import pycwt as
wavelet`` (src/cwt.py:19, src/wct.py:14, src/xwt.py:12,
constants/results_configs.py:4).  Swapping that line for
``from wavelet_transformer_b200 import pycwt_compat as wavelet`` keeps every
call site unchanged: same function names, argument order, return tuples, and
the ``Warning`` that ``ar1`` raises for an unbounded AR(1) estimate (caught at
src/wavelet_plots.py:684).

Heavy arithmetic (transforms, smoothing, Monte Carlo) runs in
libwavelet_sm100a.so; only O(n) closed forms (``ar1``, ``significance``, axes)
stay on the host.  Outputs are float64 / complex128 like pycwt's.
"""

from __future__ import annotations

import math
import os
from pathlib import Path

import numpy as np

from . import _shim

__all__ = ["Morlet", "Paul", "DOG", "MexicanHat", "ar1", "ar1_spectrum", "significance", "cwt", "icwt", "xwt",
           "wct", "wct_significance", "rednoise", "rect"]


class Morlet:
    """Morlet mother wavelet, pycwt.mothers.Morlet attribute-compatible."""

    name = "morlet"

    def __init__(self, f0: float = 6):
        self.f0 = f0
        self.dofmin = 2
        if f0 == 6:
            self.cdelta, self.gamma, self.deltaj0 = 0.776, 2.32, 0.60
        else:
            self.cdelta = self.gamma = self.deltaj0 = -1

    def psi_ft(self, f):
        return np.pi ** -0.25 * np.exp(-0.5 * (np.asarray(f) - self.f0) ** 2)

    def psi(self, t):
        t = np.asarray(t)
        return np.pi ** -0.25 * np.exp(1j * self.f0 * t - t ** 2 / 2)

    def flambda(self):
        return 4 * np.pi / (self.f0 + np.sqrt(2 + self.f0 ** 2))

    def coi(self):
        return 1.0 / np.sqrt(2)

    def sup(self):
        return 1.0 / self.coi()


class _NoSmooth:
    """pycwt implements ``smooth`` (hence ``wct``) for Morlet only; Paul and DOG raise."""

    def smooth(self, *_a, **_k):
        raise NotImplementedError(f"{type(self).__name__}.smooth: pycwt only smooths with the Morlet wavelet")


class Paul(_NoSmooth):
    """Paul wavelet of order m (pycwt.mothers.Paul; Torrence & Compo table 1)."""

    name = "paul"

    def __init__(self, m: int = 4):
        self.m = m
        self.dofmin = 2
        if m == 4:
            self.cdelta, self.gamma, self.deltaj0 = 1.132, 1.17, 1.50
        else:
            self.cdelta = self.gamma = self.deltaj0 = -1

    def psi_ft(self, f):
        f = np.asarray(f, dtype=float)
        c = 2 ** self.m / np.sqrt(self.m * math.factorial(2 * self.m - 1))
        return c * np.where(f > 0, f, 0.0) ** self.m * np.exp(-np.where(f > 0, f, 0.0)) * (f > 0)

    def psi(self, t):
        t = np.asarray(t, dtype=float)
        c = 2 ** self.m * 1j ** self.m * math.factorial(self.m) / np.sqrt(np.pi * math.factorial(2 * self.m))
        return c * (1 - 1j * t) ** (-(self.m + 1))

    def flambda(self):
        return 4 * np.pi / (2 * self.m + 1)

    def coi(self):
        return np.sqrt(2)

    def sup(self):
        return 1.0 / self.coi()


class DOG(_NoSmooth):
    """Derivative-of-Gaussian wavelet of order m (m = 2: Mexican hat)."""

    name = "dog"

    def __init__(self, m: int = 2):
        self.m = m
        self.dofmin = 1
        if m == 2:
            self.cdelta, self.gamma, self.deltaj0 = 3.541, 1.43, 1.40
        elif m == 6:
            self.cdelta, self.gamma, self.deltaj0 = 1.966, 1.37, 0.97
        else:
            self.cdelta = self.gamma = self.deltaj0 = -1

    def psi_ft(self, f):
        f = np.asarray(f, dtype=float)
        return -(1j ** self.m) / np.sqrt(math.gamma(self.m + 0.5)) * f ** self.m * np.exp(-0.5 * f ** 2)

    def psi(self, t):
        from numpy.polynomial.hermite_e import hermeval
        t = np.asarray(t, dtype=float)
        he = hermeval(t, [0] * self.m + [1])
        return (-1) ** (self.m + 1) * he * np.exp(-t ** 2 / 2) / np.sqrt(math.gamma(self.m + 0.5))

    def flambda(self):
        return 2 * np.pi / np.sqrt(self.m + 0.5)

    def coi(self):
        return 1.0 / np.sqrt(2)

    def sup(self):
        return 1.0 / self.coi()


class MexicanHat(DOG):
    name = "mexicanhat"

    def __init__(self):
        super().__init__(m=2)


_MOTHERS = {"morlet": Morlet, "paul": Paul, "dog": DOG, "mexicanhat": MexicanHat, "mexican hat": MexicanHat}


def _as_mother(wavelet):
    """pycwt._check_parameter_wavelet: a mother object or its name."""
    if isinstance(wavelet, str):
        try:
            return _MOTHERS[wavelet.lower()]()
        except KeyError:
            raise ValueError(f"Unknown wavelet '{wavelet}'") from None
    return wavelet


def _mother_code(wavelet):
    if isinstance(wavelet, Paul):
        return _shim.PAUL, float(wavelet.m)
    if isinstance(wavelet, DOG):
        return _shim.DOG, float(wavelet.m)
    if isinstance(wavelet, Morlet) or getattr(wavelet, "name", None) == "morlet":
        return _shim.MORLET, float(wavelet.f0)
    raise NotImplementedError(f"mother wavelet {wavelet!r} is not implemented on the B200 engine")


def _as_morlet(wavelet) -> Morlet:
    """XWT / WCT / significance run with Morlet only (pycwt smooths with Morlet only; the
    reference never selects another mother, constants/results_configs.py:26)."""
    wavelet = _as_mother(wavelet)
    if isinstance(wavelet, Morlet) or getattr(wavelet, "name", None) == "morlet":
        return wavelet
    raise NotImplementedError("cross-wavelet, coherence and significance use the Morlet wavelet only")


def rect(n, normalize=False):
    w = np.ones(int(n))
    w[0] = w[-1] = 0.5
    return w / w.sum() if normalize else w


def ar1(x):
    """Allen & Smith (1996) lag-1 autocorrelation.  Raises ``Warning`` (an
    Exception subclass, as pycwt does) when no upper bound can be placed."""
    x = np.asarray(x, dtype=float)
    N = x.size
    d = x - x.mean()
    c0 = float(d @ d) / N
    c1 = float(d[:-1] @ d[1:]) / (N - 1)
    A = c0 * N ** 2
    B = -c1 * N - c0 * N ** 2 - 2 * c0 + 2 * c1 - c1 * N ** 2 + c0 * N
    Cq = N * (c0 + c1 * N - c1)
    disc = B ** 2 - 4 * A * Cq
    if not disc > 0:
        raise Warning("Cannot place an upperbound on the unbiased AR(1). "
                      "Series is too short or trend is to large.")
    g = (-B - disc ** 0.5) / (2 * A)
    mu2 = -1 / N + (2 / N ** 2) * ((N - g ** N) / (1 - g) - g * (1 - g ** (N - 1)) / (1 - g) ** 2)
    a = ((1 - g ** 2) * c0 / (1 - mu2)) ** 0.5
    return g, a, mu2


def ar1_spectrum(freqs, ar1=0.0):
    freqs = np.asarray(freqs)
    return (1 - ar1 ** 2) / np.abs(1 - ar1 * np.exp(-2j * np.pi * freqs)) ** 2


def _chi2_ppf(level, dof):
    if dof == 2:
        return -2.0 * math.log1p(-level)
    from scipy.stats import chi2
    return chi2.ppf(level, dof)


def significance(signal, dt, scales, sigma_test=0, alpha=None, significance_level=0.95, dof=-1,
                 wavelet="morlet"):
    """Red-noise significance levels (Torrence & Compo 1998 sec. 4); returns
    ``(signif, fft_theor)``.  sigma_test 0 (no smoothing), 1 (time average) and 2 (scale average over
    ``dof = [s1, s2]``, eqs. 25-28: returns the scale-averaged ``fft_theor``).  Any mother wavelet:
    flambda, dofmin and gamma enter, and for sigma_test 2 cdelta and deltaj0 as well."""
    wavelet = _as_mother(wavelet)
    try:
        n0 = len(signal)
    except TypeError:
        n0 = 1
    scales = np.asarray(scales, dtype=float)
    variance = signal if n0 == 1 else np.asarray(signal).std() ** 2
    if alpha is None:
        alpha, _, _ = ar1(signal)
    freq = dt / (scales * wavelet.flambda())
    fft_theor = variance * (1 - alpha ** 2) / (1 + alpha ** 2 - 2 * alpha * np.cos(2 * np.pi * freq))
    dofmin = wavelet.dofmin
    if sigma_test == 0:
        signif = fft_theor * _chi2_ppf(significance_level, dofmin) / dofmin
    elif sigma_test == 1:
        from scipy.stats import chi2
        dofv = np.full(scales.shape, float(dof)) if np.ndim(dof) == 0 else np.asarray(dof, dtype=float)
        dofv = np.maximum(dofv, 1.0)
        dofv = dofmin * np.sqrt(1 + (dofv * dt / wavelet.gamma / scales) ** 2)
        dofv = np.maximum(dofv, dofmin)
        signif = fft_theor * chi2.ppf(significance_level, dofv) / dofv
    elif sigma_test == 2:
        from scipy.stats import chi2
        if np.ndim(dof) != 1 or len(dof) != 2:
            raise Exception("DOF must be set to [s1, s2], the range of scale-averages")
        if wavelet.cdelta == -1:
            raise ValueError(f"Cdelta and dj0 not defined for {wavelet.name} with these parameters")
        s1, s2 = float(dof[0]), float(dof[1])
        sel = (scales >= s1) & (scales <= s2)
        navg = int(sel.sum())
        if navg == 0:
            raise ValueError(f"No valid scales between {s1} and {s2}.")
        dj = np.log2(scales[1] / scales[0])
        savg = 1 / np.sum(1 / scales[sel])                                         # eq. 25
        smid = np.exp((np.log(s1) + np.log(s2)) / 2)
        dofv = dofmin * navg * savg / smid * np.sqrt(1 + (navg * dj / wavelet.deltaj0) ** 2)   # eq. 28
        fft_theor = savg * np.sum(fft_theor[sel] / scales[sel])                    # eq. 27
        signif = dj * dt / (wavelet.cdelta * savg) * fft_theor * chi2.ppf(significance_level, dofv) / dofv  # eq. 26
    else:
        raise NotImplementedError("significance: sigma_test must be 0, 1 or 2")
    return signif, fft_theor


def _resolve_s0_J(n0, dt, dj, s0, J, wavelet):
    kind, param = _mother_code(wavelet)
    return _shim.cwt_axes_mother(n0, dt, dj, s0, int(J) if J != -1 else -1, kind, param)


def cwt(signal, dt, dj=1 / 12, s0=-1, J=-1, wavelet="morlet", freqs=None):
    """Continuous wavelet transform.  Returns ``(W, sj, freqs, coi, fft, fftfreqs)``
    with ``W`` complex128 of shape [J+1, n0]."""
    wavelet = _as_mother(wavelet)
    if freqs is not None:
        raise NotImplementedError("custom `freqs` are not supported; use dj/s0/J")
    x = np.ascontiguousarray(signal, dtype=float)
    n0 = x.size
    Jr, sj, fr, coi = _resolve_s0_J(n0, dt, dj, s0, J, wavelet)
    kind, param = _mother_code(wavelet)
    _, W = _shim.cwt(x, dt, dj, s0, Jr if J != -1 else -1, kind, param, want_power=False, want_coef=True)
    W = np.asarray(W, dtype=np.complex128)
    # Side outputs pycwt also returns and the reference discards (src/cwt.py:109):
    # one O(N log N) host FFT, outside the hot path.
    N = _shim.default_nfft(n0)
    sft = np.fft.fft(x, N)
    ftfreqs = 2 * np.pi * np.fft.fftfreq(N, dt)
    return W, sj, fr, coi, sft[1:N // 2] / N ** 0.5, ftfreqs[1:N // 2] / (2 * np.pi)


def icwt(W, sj, dt, dj=1 / 12, wavelet="morlet"):
    """Inverse continuous wavelet transform (Torrence & Compo 1998, eq. 11):
    ``dj sqrt(dt) / (C_delta psi_0(0)) * sum_j Re(W_j) / sqrt(s_j)``; the sum over scales runs
    on the device.  ``W`` is [S, n0] (or its transpose, as pycwt accepts)."""
    wavelet = _as_mother(wavelet)
    W = np.asarray(W)
    sj = np.asarray(sj, dtype=float)
    a, b = W.shape
    if a != sj.size:
        if b != sj.size:
            raise Warning("Input array dimensions do not match.")
        W = W.T
    factor = dj * np.sqrt(dt) / (wavelet.cdelta * np.real(wavelet.psi(0)))
    return np.asarray(_shim.icwt(W, sj, factor, f64=True), dtype=float)


def _normalised(y, normalize):
    y = np.asarray(y, dtype=float)
    return (y - y.mean()) / y.std() if normalize else y


def xwt(y1, y2, dt, dj=1 / 12, s0=-1, J=-1, significance_level=0.95, wavelet="morlet", normalize=True):
    """Cross wavelet transform.  Returns ``(W12, coi, freq, signif)``.  Any mother wavelet
    (pycwt.xwt needs no smoothing): Morlet takes the fused pair kernel, Paul / DOG two CWTs."""
    wavelet = _as_mother(wavelet)
    y1 = np.asarray(y1, dtype=float)
    y2 = np.asarray(y2, dtype=float)
    std1, std2 = y1.std(), y2.std()
    a, b = _normalised(y1, normalize), _normalised(y2, normalize)
    Jr, sj, freq, coi = _resolve_s0_J(y1.size, dt, dj, s0, J, wavelet)
    if isinstance(wavelet, Morlet):
        _, _, W12 = _shim.xwt_wct(a, b, dt, dj, s0, Jr, wavelet.f0, want_wct=False, want_phase=False,
                                  want_w12=True)
    else:
        kind, param = _mother_code(wavelet)
        _, W = _shim.cwt(np.stack([a, b]), dt, dj, s0, Jr, kind, param, want_power=False, want_coef=True)
        W12 = W[0] * np.conj(W[1])
    if normalize:
        std1 = std2 = 1.0
    a1, a2 = ar1(y1)[0], ar1(y2)[0]
    Pk1, Pk2 = ar1_spectrum(freq * dt, a1), ar1_spectrum(freq * dt, a2)
    dof = wavelet.dofmin
    signif = std1 * std2 * (Pk1 * Pk2) ** 0.5 * _chi2_ppf(significance_level, dof) / dof
    return np.asarray(W12, dtype=np.complex128), coi, freq, signif


def wct(y1, y2, dt, dj=1 / 12, s0=-1, J=-1, sig=True, significance_level=0.95, wavelet="morlet",
        normalize=True, **kwargs):
    """Wavelet coherence.  Returns ``(WCT, aWCT, coi, freq, sig)``.  Unknown
    keyword arguments are swallowed when ``sig=False`` (the reference relies on
    that at src/xwt.py:126) and forwarded to ``wct_significance`` otherwise."""
    wavelet = _as_morlet(wavelet)
    y1 = np.asarray(y1, dtype=float)
    y2 = np.asarray(y2, dtype=float)
    if s0 == -1:
        s0 = 2 * dt / wavelet.flambda()
    if J == -1:
        J = int(np.round(np.log2(y1.size * dt / s0) / dj))
    a, b = _normalised(y1, normalize), _normalised(y2, normalize)
    _, _, freq, coi = _resolve_s0_J(y1.size, dt, dj, s0, J, wavelet)
    WCT, aWCT, _ = _shim.xwt_wct(a, b, dt, dj, s0, J, wavelet.f0, want_wct=True, want_phase=True)
    if sig:
        a1, a2 = ar1(y1)[0], ar1(y2)[0]
        sig = wct_significance(a1, a2, dt=dt, dj=dj, s0=s0, J=J, significance_level=significance_level,
                               wavelet=wavelet, **kwargs)
    else:
        sig = np.asarray([0])
    return np.asarray(WCT, dtype=float), np.asarray(aWCT, dtype=float), coi, freq, sig


def _cache_file(al1, al2, dt, dj, s0, J, level, mc_count, seed, white, wavelet, prec=None) -> Path:
    root = Path(os.environ.get("WTB_CACHE_DIR", Path.home() / ".cache" / "wavelet_b200"))
    key = (f"wct_sig_{al1:.10f}_{al2:.10f}_{dj:.6f}_{s0 / dt:.6f}_{J:d}_{level:.4f}_{mc_count:d}_{seed:d}_"
           f"{'white' if white else 'ar1'}_{wavelet.name}_{prec or _shim.get_precision()}")
    return root / f"{key}.gz"


_PYCWT_NAMES = {"morlet": "Morlet", "paul": "Paul", "dog": "DOG", "mexicanhat": "Mexican Hat"}


def pycwt_cache_file(al1, al2, dt, dj, s0, J, wavelet="morlet") -> Path:
    """The file pycwt 0.4.0b0's ``wct_significance`` itself would use under ``~/.cache/pycwt``
    (SURVEY A.7): ``wct_sig_{aa0:.5f}_{aa1:.5f}_{dj:.5f}_{s0/dt:.5f}_{J}_{name}.gz`` with
    ``aa = round(arctanh([al1, al2] * 4))`` -- pycwt's own expression, which is NaN for any
    coefficient above 0.25, so distinct AR(1) pairs share one file.  That collision is why this
    cache is only consulted on request (``WTB_PYCWT_CACHE=read`` or ``readwrite``)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        aa = np.round(np.arctanh(np.array([al1, al2], dtype=float) * 4.0))
    aa = np.abs(aa) + 0.5 * (aa < 0)
    name = _PYCWT_NAMES.get(getattr(_as_mother(wavelet), "name", "morlet"), "Morlet")
    root = Path(os.environ.get("WTB_PYCWT_CACHE_DIR", Path.home() / ".cache" / "pycwt"))
    return root / f"wct_sig_{aa[0]:0.5f}_{aa[1]:0.5f}_{dj:0.5f}_{s0 / dt:0.5f}_{int(J):d}_{name}.gz"


def wct_significance(al1, al2, dt, dj, s0, J, significance_level=0.95, wavelet="morlet", mc_count=300,
                     progress=True, cache=True, seed=0, white=False, surrogates=None, n_gpus=None,
                     precision=None):
    """Monte Carlo coherence significance (one value per scale).

    Runs entirely on the GPU: Philox AR(1) surrogates -> CWT -> smoothing ->
    coherence -> per-scale histograms.  ``cache=True`` stores the result on disk
    keyed on the exact arguments (pycwt keeps a similar cache under
    ~/.cache/pycwt).  ``surrogates`` ([mc_count, 2, N]) injects ready-made noise.

    The realisations are spread over every GPU the library drives (``n_gpus`` here, or
    ``_shim.init_multi`` / ``WTB_GPUS`` beforehand); the Philox streams are keyed by the global
    realisation index, so the thresholds do not depend on the number of GPUs.

    ``precision``: "fp32" | "fp64" | None.  None keeps the global precision when surrogates
    are injected (the per-realisation parity mode) and uses the FP32 register-FFT kernels with
    the device RNG: the thresholds are Monte Carlo estimates with errors of order 1e-2, seven
    orders above FP32 round-off (WTB_MC_PRECISION=fp64 restores the global setting)."""
    wavelet = _as_morlet(wavelet)
    J = int(J)
    if precision is None and surrogates is None and os.environ.get("WTB_MC_PRECISION", "fp32").lower() != "fp64":
        precision = "fp32"
    f64 = None if precision is None else {"fp32": False, "fp64": True}[precision.lower()]
    path = _cache_file(al1, al2, dt, dj, s0, J, significance_level, mc_count, seed, white, wavelet,
                       None if precision is None else precision.lower())
    pycwt_mode = os.environ.get("WTB_PYCWT_CACHE", "").lower()
    pycwt_path = pycwt_cache_file(al1, al2, dt, dj, s0, J, wavelet)
    if cache and surrogates is None:
        for candidate in ([pycwt_path] if pycwt_mode in ("read", "readwrite") else []) + [path]:
            try:
                return np.loadtxt(candidate, unpack=True)
            except OSError:
                pass
    if n_gpus is not None and int(n_gpus) != _shim.gpu_count():
        _shim.init_multi(int(n_gpus))
    sig95 = _shim.wct_significance(al1, al2, dt, dj, s0, J, wavelet.f0, level=significance_level,
                                   mc_count=mc_count, seed=seed, surrogates=surrogates, white=white, f64=f64)
    if cache and surrogates is None:
        for target in [path] + ([pycwt_path] if pycwt_mode == "readwrite" else []):
            try:
                target.parent.mkdir(parents=True, exist_ok=True)
                np.savetxt(target, sig95)   # one float per line, gzip by suffix: pycwt's format
            except OSError:
                pass
    return sig95


def rednoise(N, g, a=1.0, seed=0):
    """AR(1) red noise of length N generated on the GPU (Philox, Box-Muller)."""
    out = _shim.rednoise(g, g, int(N), 0, 1, seed, f64=True)
    return out[0, 0] * a
