"""ctypes binding of include/wtb.h (libwavelet_sm100a.so).

Thin by design: NumPy buffers (or raw device addresses) in, NumPy buffers out.
There is NO CPU fallback -- a missing library or a missing B200 raises.
"""

from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

import numpy as np

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libwavelet_sm100a.so"

F64 = 1 << 0
DEVICE_PTRS = 1 << 1
COI_MASK = 1 << 2
NOISE_WHITE = 1 << 3
GENERIC_ONLY = 1 << 4
PLANE_COMPLEX = 1 << 5
FFT_NO_PAD = 1 << 6
NBINS = 1000

_lock = threading.Lock()
_lib = None
_precision = os.environ.get("WTB_PRECISION", "fp64").lower()


class WaveletEngineError(RuntimeError):
    """Raised for every non-zero status returned by the C ABI."""


def set_precision(name: str) -> None:
    """'fp64' (default for the drop-in entry points) or 'fp32'."""
    global _precision
    if name not in ("fp32", "fp64"):
        raise ValueError("precision must be 'fp32' or 'fp64'")
    _precision = name


def get_precision() -> str:
    return _precision


_fft_pad = os.environ.get("WTB_FFT_PAD", "pow2").lower()


def set_fft_padding(mode: str) -> None:
    """'pow2' (default): every transform is zero-padded to the next power of two, as pycwt does
    on top of scipy.fftpack -- the reference's pip / uv install.  'none': transforms run at the
    series' own length, as pycwt does when mkl_fft is importable -- the reference's conda
    install (environment.yml:126).  The two give different numbers near the edges."""
    global _fft_pad
    if mode not in ("pow2", "none"):
        raise ValueError("fft padding must be 'pow2' or 'none'")
    _fft_pad = mode


def get_fft_padding() -> str:
    return _fft_pad


def default_nfft(n0: int) -> int:
    return next_pow2(n0) if _fft_pad == "pow2" else max(int(n0), 2)


def _dtype(f64):
    return np.float64 if f64 else np.float32


def _resolve_f64(f64):
    return (_precision == "fp64") if f64 is None else bool(f64)


_vp, _i64, _i32, _f64, _u64 = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_uint64
_pd, _pi = C.POINTER(C.c_double), C.POINTER(C.c_int)

_SIGNATURES = {
    "wtb_version": ([], _i32),
    "wtb_device_count": ([], _i32),
    "wtb_init": ([_i32], _i32),
    "wtb_init_multi": ([_i32], _i32),
    "wtb_gpu_count": ([], _i32),
    "wtb_scratch_bytes": ([], C.c_uint64),
    "wtb_shutdown": ([], None),
    "wtb_last_error": ([], C.c_char_p),
    "wtb_kernel_launches": ([], C.c_uint64),
    "wtb_cwt_axes": ([_i32, _f64, _f64, _f64, _i32, _f64, _pi, _pd, _pd, _pd], _i32),
    "wtb_cwt_axes_mother": ([_i32, _f64, _f64, _f64, _i32, _i32, _f64, _pi, _pd, _pd, _pd], _i32),
    "wtb_cwt": ([_vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _i32, _f64, _i32, _vp, _vp, _vp], _i32),
    "wtb_icwt": ([_vp, _i64, _i32, _i32, _pd, _f64, _i32, _vp, _vp], _i32),
    "wtb_cwt_averages": ([_vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _i32, _f64, _i32, _i32, _f64, _i32, _vp, _vp,
                          _vp], _i32),
    "wtb_cwt_morlet": ([_vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _f64, _i32, _vp, _vp, _vp], _i32),
    "wtb_series_prep": ([_vp, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _pd, _vp], _i32),
    "wtb_ratio_planes": ([_vp, _i64, _i32, _i32, _vp, _i64, _i32, _vp, _vp, _vp], _i32),
    "wtb_phase_arrows": ([_vp, _i64, _i32, _vp, _vp, _vp], _i32),
    "wtb_xwt_wct": ([_vp, _vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _f64, _i32, _vp, _vp, _vp, _vp], _i32),
    "wtb_partial_wct": ([_vp, _vp, _vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _f64, _i32, _vp, _vp, _vp, _vp],
                        _i32),
    "wtb_wct_mc_geometry": ([_f64, _f64, _f64, _i32, _f64, _pi, _pi], _i32),
    "wtb_wct_mc_hist": ([_f64, _f64, _f64, _f64, _f64, _i32, _f64, _i64, _i64, _u64, _vp, _i32, _vp, _vp], _i32),
    "wtb_wct_sig_from_hist": ([_vp, _i32, _i32, _f64, _vp, _pd], _i32),
    "wtb_wct_sig_from_hist_device": ([_vp, _i32, _i32, _f64, _vp, _vp, _vp], _i32),
    "wtb_wct_significance": ([_f64, _f64, _f64, _f64, _f64, _i32, _f64, _f64, _i64, _u64, _vp, _i32, _pd, _vp], _i32),
    "wtb_rednoise": ([_f64, _f64, _i32, _i64, _i64, _u64, _i32, _vp, _vp], _i32),
    "wtb_rednoise_triples": ([_f64, _f64, _f64, _i32, _i64, _i64, _u64, _i32, _vp, _vp], _i32),
    "wtb_partial_wct_mc_hist": ([_f64, _f64, _f64, _f64, _f64, _f64, _i32, _f64, _i64, _i64, _u64, _vp, _i32, _vp,
                                 _vp], _i32),
    "wtb_partial_wct_significance": ([_f64, _f64, _f64, _f64, _f64, _f64, _i32, _f64, _f64, _i64, _u64, _vp, _i32,
                                      _pd, _pd, _vp], _i32),
    "wtb_modwt": ([_vp, _i64, _i32, _pd, _pd, _i32, _i32, _i32, _vp, _vp], _i32),
    "wtb_imodwt": ([_vp, _i64, _i32, _pd, _pd, _i32, _i32, _i32, _vp, _vp], _i32),
    "wtb_modwtmra": ([_vp, _i64, _i32, _pd, _i32, _i32, _vp, _vp], _i32),
    "wtb_modwtmra_taps": ([_vp, _i64, _i32, _pd, _pd, _i32, _i32, _i32, _vp, _vp], _i32),
    "wtb_modwt_wavelet_stats": ([_vp, _vp, _i64, _i32, _pd, _pd, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp], _i32),
    "wtb_dwt_coeff_lens": ([_i32, _i32, _i32, _pi], _i32),
    "wtb_dwt_max_level": ([_i32, _i32], _i32),
    "wtb_rowwise_ols": ([_vp, _i64, _vp, _i64, _i32, _i32, _i32, _pd, _vp], _i32),
    "wtb_wavedec": ([_vp, _i64, _i32, _pd, _pd, _i32, _i32, _i32, _vp, _vp], _i32),
    "wtb_waverec_len": ([_pi, _i32, _i32], _i32),
    "wtb_waverec": ([_vp, _i64, _pi, _i32, _pd, _pd, _i32, _i32, _vp, _vp], _i32),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    """Load libwavelet_sm100a.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not _LIB_PATH.exists():
                    raise WaveletEngineError(
                        f"{_LIB_PATH} is missing: build it with "
                        "`python -m wavelet_transformer_b200._build` (needs nvcc). "
                        "There is no CPU fallback.")
                handle = C.CDLL(str(_LIB_PATH))
                for name, (argtypes, restype) in _SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.argtypes = argtypes
                    fn.restype = restype
                _lib = handle
                if os.environ.get("WTB_GPUS"):      # one process, several GPUs (SURVEY 8e)
                    rc = handle.wtb_init_multi(int(os.environ["WTB_GPUS"]))
                    if rc != 0:
                        raise WaveletEngineError("wtb_init_multi(WTB_GPUS) failed: "
                                                 + handle.wtb_last_error().decode("utf-8", "replace"))
    return _lib


def lib_path() -> Path:
    return _LIB_PATH


def _check(rc: int, what: str):
    if rc != 0:
        msg = lib().wtb_last_error().decode("utf-8", "replace")
        exc = ValueError if rc == -1 else WaveletEngineError
        raise exc(f"{what} failed (status {rc}): {msg}")


def init(device: int = 0) -> None:
    _check(lib().wtb_init(int(device)), "wtb_init")


def init_multi(n_gpus: int = 0) -> int:
    """One process, several GPUs: host-buffer batches and Monte Carlo realisations are split over
    devices 0 .. n_gpus-1 (0: WTB_GPUS, else every visible device).  Returns the device count in use."""
    _check(lib().wtb_init_multi(int(n_gpus)), "wtb_init_multi")
    return gpu_count()


def gpu_count() -> int:
    """Devices one call is spread over (1 unless init_multi made a pool)."""
    return int(lib().wtb_gpu_count())


def scratch_bytes() -> int:
    """Bytes of device scratch the library holds right now (all threads)."""
    return int(lib().wtb_scratch_bytes())


def shutdown() -> None:
    if _lib is not None:
        _lib.wtb_shutdown()


def kernel_launches() -> int:
    """Kernels launched by the library so far in this process."""
    return int(lib().wtb_kernel_launches())


def device_count() -> int:
    return int(lib().wtb_device_count())


def _ptr(a):
    """numpy array -> void*, int device address -> void*, None -> NULL."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return a.ctypes.data_as(C.c_void_p)


def _dp(a):
    return a.ctypes.data_as(_pd)


def next_pow2(n: int) -> int:
    return 1 << max(int(n) - 1, 0).bit_length() if n > 1 else 2


# ---------------------------------------------------------------- CWT
def cwt_axes(n0, dt, dj, s0=-1, J=-1, f0=6.0):
    """(J, scales[S], freqs[S], coi[n0]) as pycwt.cwt forms them."""
    Jout = C.c_int(0)
    _check(lib().wtb_cwt_axes(n0, dt, dj, s0, int(J), f0, C.byref(Jout), None, None, None), "wtb_cwt_axes")
    S = Jout.value + 1
    scales, freqs, coi = np.empty(S), np.empty(S), np.empty(n0)
    _check(lib().wtb_cwt_axes(n0, dt, dj, s0, int(J), f0, C.byref(Jout), _dp(scales), _dp(freqs), _dp(coi)),
           "wtb_cwt_axes")
    return Jout.value, scales, freqs, coi


MORLET, PAUL, DOG = 0, 1, 2  # WTB_MORLET / WTB_PAUL / WTB_DOG


def cwt_axes_mother(n0, dt, dj, s0=-1, J=-1, mother=MORLET, param=6.0):
    """cwt_axes for any mother wavelet (param = f0 for Morlet, the order m otherwise)."""
    Jout = C.c_int(0)
    _check(lib().wtb_cwt_axes_mother(n0, dt, dj, s0, int(J), int(mother), float(param), C.byref(Jout), None, None,
                                     None), "wtb_cwt_axes_mother")
    S = Jout.value + 1
    scales, freqs, coi = np.empty(S), np.empty(S), np.empty(n0)
    _check(lib().wtb_cwt_axes_mother(n0, dt, dj, s0, int(J), int(mother), float(param), C.byref(Jout), _dp(scales),
                                     _dp(freqs), _dp(coi)), "wtb_cwt_axes_mother")
    return Jout.value, scales, freqs, coi


def cwt(x, dt, dj, s0, J, mother=MORLET, param=6.0, *, nfft=None, f64=None, want_power=True, want_coef=False,
        coi_mask=False, generic_only=False):
    """Batched CWT of host data with any mother wavelet (wtb_cwt); see cwt_morlet."""
    f64 = _resolve_f64(f64)
    rt = _dtype(f64)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=rt)
    batch, n0 = x2.shape
    Jr, _, _, _ = cwt_axes_mother(n0, dt, dj, s0, J, mother, param)
    S = Jr + 1
    nfft = int(nfft) if nfft else default_nfft(n0)
    flags = (F64 if f64 else 0) | (COI_MASK if coi_mask else 0) | (GENERIC_ONLY if generic_only else 0)
    power = np.empty((batch, S, n0), dtype=rt) if want_power else None
    coef = np.empty((batch, S, n0), dtype=np.complex128 if f64 else np.complex64) if want_coef else None
    _check(lib().wtb_cwt(_ptr(x2), batch, n0, nfft, dt, dj, s0, int(J), int(mother), float(param), flags,
                         _ptr(power), _ptr(coef), None), "wtb_cwt")
    if np.ndim(x) == 1:
        power = power[0] if power is not None else None
        coef = coef[0] if coef is not None else None
    return power, coef


def _averages_args(band, band_factor, want_global, S):
    """Validates the arguments of wtb_cwt_averages before any transform runs; returns (band_lo, band_hi)."""
    if band is None:
        if not want_global:
            raise ValueError("cwt_averages: no output requested (band=None and want_global=False)")
        return 0, 0
    if len(band) != 2 or any(isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)) for v in band):
        raise ValueError(f"cwt_averages: band must be two scale indices (lo, hi), got {band!r}")
    lo, hi = int(band[0]), int(band[1])
    if not 0 <= lo <= hi < S:
        raise ValueError(f"cwt_averages: band ({lo}, {hi}) must satisfy 0 <= lo <= hi < S = {S}")
    if not np.isfinite(band_factor):
        raise ValueError("cwt_averages: band_factor must be finite")
    return lo, hi


def cwt_averages(x, dt, dj, s0, J, mother=MORLET, param=6.0, *, band=None, band_factor=1.0, want_global=True,
                 nfft=None, f64=None, generic_only=False):
    """Time- and scale-averaged wavelet power of host data (wtb_cwt_averages, Torrence & Compo 1998 eqs. 22
    and 24) without the power plane leaving the device.  x: [n0] or [batch, n0].
    band = (lo, hi): scale indices, inclusive.  Returns (global [batch, S] or None, band [batch, n0] or None)
    with global = mean_t |W|^2 and band = band_factor * sum_{s=lo..hi} |W_s|^2 / scales[s]; the batch axis
    is dropped for 1-D input."""
    f64 = _resolve_f64(f64)
    rt = _dtype(f64)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=rt)
    batch, n0 = x2.shape
    Jr, _, _, _ = cwt_axes_mother(n0, dt, dj, s0, J, mother, param)      # host arithmetic only
    S = Jr + 1
    lo, hi = _averages_args(band, band_factor, want_global, S)
    nfft = int(nfft) if nfft else default_nfft(n0)
    flags = (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    glob = np.empty((batch, S), dtype=rt) if want_global else None
    bnd = np.empty((batch, n0), dtype=rt) if band is not None else None
    _check(lib().wtb_cwt_averages(_ptr(x2), batch, n0, nfft, dt, dj, s0, int(J), int(mother), float(param), lo, hi,
                                  float(band_factor), flags, _ptr(glob), _ptr(bnd), None), "wtb_cwt_averages")
    if np.ndim(x) == 1:
        glob = glob[0] if glob is not None else None
        bnd = bnd[0] if bnd is not None else None
    return glob, bnd


def cwt_averages_device(x_ptr, batch, n0, dt, dj, s0, J, mother, param, global_ptr, band_ptr, *, band=None,
                        band_factor=1.0, nfft=None, f64=False, stream=0):
    """Device-resident wtb_cwt_averages: raw device addresses (global_ptr / band_ptr may be 0 for "not
    wanted"), asynchronous on `stream`."""
    if bool(band_ptr) != (band is not None):
        raise ValueError("cwt_averages_device: band_ptr and band are given together")
    Jr, _, _, _ = cwt_axes_mother(n0, dt, dj, s0, J, mother, param)
    lo, hi = _averages_args(band, band_factor, bool(global_ptr), Jr + 1)
    nfft = int(nfft) if nfft else default_nfft(n0)
    _check(lib().wtb_cwt_averages(_ptr(int(x_ptr)), int(batch), int(n0), nfft, dt, dj, s0, int(J), int(mother),
                                  float(param), lo, hi, float(band_factor), DEVICE_PTRS | (F64 if f64 else 0),
                                  _ptr(int(global_ptr)) if global_ptr else None,
                                  _ptr(int(band_ptr)) if band_ptr else None, C.c_void_p(int(stream))),
           "wtb_cwt_averages")


def icwt(W, scales, factor, *, f64=None):
    """factor * sum_s Re(W[s, t]) / sqrt(scales[s]) for W [S, n0] or [batch, S, n0] (wtb_icwt)."""
    f64 = _resolve_f64(f64)
    W = np.asarray(W)
    w3 = np.ascontiguousarray(W[None] if W.ndim == 2 else W, dtype=np.complex128 if f64 else np.complex64)
    batch, S, n0 = w3.shape
    scales = np.ascontiguousarray(scales, dtype=np.float64)
    if scales.shape != (S,):
        raise ValueError("Input array dimensions do not match.")
    out = np.empty((batch, n0), dtype=_dtype(f64))
    _check(lib().wtb_icwt(_ptr(w3), batch, S, n0, _dp(scales), float(factor), F64 if f64 else 0, _ptr(out), None),
           "wtb_icwt")
    return out[0] if W.ndim == 2 else out


def cwt_morlet(x, dt, dj, s0, J, f0=6.0, *, nfft=None, f64=None, want_power=True, want_coef=False,
               coi_mask=False, generic_only=False):
    """Batched Morlet CWT of host data (wtb_cwt_morlet: one-CTA transform lengths; `cwt` takes longer series).
    x: [n0] or [batch, n0].  Returns (power or None, coef or None) with shapes [batch, S, n0] (batch axis
    dropped for 1-D input); dtype float32/complex64 or float64/complex128."""
    f64 = _resolve_f64(f64)
    rt = _dtype(f64)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=rt)
    batch, n0 = x2.shape
    Jr, _, _, _ = cwt_axes(n0, dt, dj, s0, J, f0)
    S = Jr + 1
    nfft = int(nfft) if nfft else default_nfft(n0)
    flags = (F64 if f64 else 0) | (COI_MASK if coi_mask else 0) | (GENERIC_ONLY if generic_only else 0)
    power = np.empty((batch, S, n0), dtype=rt) if want_power else None
    coef = np.empty((batch, S, n0), dtype=np.complex128 if f64 else np.complex64) if want_coef else None
    _check(lib().wtb_cwt_morlet(_ptr(x2), batch, n0, nfft, dt, dj, s0, int(J), f0, flags,
                                _ptr(power), _ptr(coef), None), "wtb_cwt_morlet")
    if np.ndim(x) == 1:
        power = power[0] if power is not None else None
        coef = coef[0] if coef is not None else None
    return power, coef


def cwt_power_device(x_ptr, batch, n0, dt, dj, s0, J, f0, power_ptr, *, nfft=None, f64=False,
                     stream=0, generic_only=False):
    """Device-resident Morlet CWT power (wtb_cwt, every transform length it takes): raw device addresses,
    asynchronous on `stream`."""
    nfft = int(nfft) if nfft else default_nfft(n0)
    flags = DEVICE_PTRS | (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    _check(lib().wtb_cwt(_ptr(int(x_ptr)), batch, n0, nfft, dt, dj, s0, int(J), MORLET, float(f0), flags,
                         _ptr(int(power_ptr)), None, C.c_void_p(int(stream))), "wtb_cwt")


def series_prep(x, *, detrend=True, remove_mean=False, standardize=True, f64=None, want_y=True, want_ar1=True):
    """Batched standardize_series + pycwt.ar1 of host data.  x: [n] or [batch, n].
    Returns (y or None, ar1 or None); ar1 is NaN where the estimate cannot be bounded."""
    f64 = _resolve_f64(f64)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=_dtype(f64))
    batch, n = x2.shape
    y = np.empty_like(x2) if want_y else None
    a = np.empty(batch) if want_ar1 else None
    _check(lib().wtb_series_prep(_ptr(x2), batch, n, int(detrend), int(remove_mean), int(standardize),
                                 F64 if f64 else 0, _ptr(y), None if a is None else _dp(a), None),
           "wtb_series_prep")
    if np.ndim(x) == 1:
        y = None if y is None else y[0]
        a = None if a is None else a[0]
    return y, a


def series_prep_device(x_ptr, batch, n, y_ptr, ar1_ptr, *, detrend=True, remove_mean=False, standardize=True,
                       f64=False, stream=0):
    """Device-resident variant (y_ptr / ar1_ptr may be 0 for "not wanted")."""
    _check(lib().wtb_series_prep(_ptr(int(x_ptr)), batch, n, int(detrend), int(remove_mean), int(standardize),
                                 DEVICE_PTRS | (F64 if f64 else 0), C.c_void_p(int(y_ptr)) if y_ptr else None,
                                 C.cast(C.c_void_p(int(ar1_ptr)), _pd) if ar1_ptr else None,
                                 C.c_void_p(int(stream))), "wtb_series_prep")


def rowwise_ols(x, y, *, add_constant=True, f64=None):
    """One simple regression per row (wtb_rowwise_ols).  x, y: [rows, n] or [n] (a single row is
    broadcast against the other argument's rows).  Returns [rows, 8] float64 stats:
    nobs, intercept, slope, ssr, tss, sxx, mean_x, mean_y."""
    f64 = _resolve_f64(f64)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=_dtype(f64))
    y2 = np.ascontiguousarray(np.atleast_2d(np.asarray(y)), dtype=_dtype(f64))
    if x2.shape[1] != y2.shape[1]:
        raise ValueError(f"x and y must have the same number of observations ({x2.shape[1]} != {y2.shape[1]})")
    rows = max(x2.shape[0], y2.shape[0])
    stats = np.empty((rows, 8))
    _check(lib().wtb_rowwise_ols(_ptr(x2), x2.shape[0], _ptr(y2), y2.shape[0], x2.shape[1], int(bool(add_constant)),
                                 F64 if f64 else 0, _dp(stats), None), "wtb_rowwise_ols")
    return stats


# ---------------------------------------------------------------- post-processing
def ratio_planes(plane, signif, *, f64=None, want_power=False):
    """ratio = |plane| / signif[..., None] for real planes [S, n0] or [batch, S, n0]; for complex
    planes power = |z|**2 and ratio = power / signif (wtb_ratio_planes).  signif: [S] or [batch, S].
    Returns ratio, or (power, ratio) with want_power."""
    f64 = _resolve_f64(f64)
    plane = np.asarray(plane)
    cx = np.iscomplexobj(plane)
    p3 = np.ascontiguousarray(plane[None] if plane.ndim == 2 else plane,
                              dtype=(np.complex128 if f64 else np.complex64) if cx else _dtype(f64))
    batch, S, n0 = p3.shape
    sig = np.ascontiguousarray(np.atleast_2d(np.asarray(signif, dtype=np.float64)))
    if sig.shape not in ((1, S), (batch, S)):
        raise ValueError(f"signif must have shape ({S},) or ({batch}, {S})")
    if want_power and not cx:
        raise ValueError("want_power needs a complex plane")
    ratio = np.empty((batch, S, n0), dtype=_dtype(f64))
    power = np.empty((batch, S, n0), dtype=_dtype(f64)) if want_power else None
    _check(lib().wtb_ratio_planes(_ptr(p3), batch, S, n0, _ptr(sig), sig.shape[0],
                                  (F64 if f64 else 0) | (PLANE_COMPLEX if cx else 0), _ptr(power), _ptr(ratio), None),
           "wtb_ratio_planes")
    if plane.ndim == 2:
        ratio, power = ratio[0], (None if power is None else power[0])
    return (power, ratio) if want_power else ratio


def ratio_planes_device(plane_ptr, batch, S, n0, signif_ptr, sig_rows, ratio_ptr, *, power_ptr=0, complex_plane=False,
                        f64=False, stream=0):
    """Device-resident wtb_ratio_planes (signif is a device float64 buffer [sig_rows, S])."""
    flags = DEVICE_PTRS | (F64 if f64 else 0) | (PLANE_COMPLEX if complex_plane else 0)
    _check(lib().wtb_ratio_planes(_ptr(int(plane_ptr)), int(batch), int(S), int(n0), _ptr(int(signif_ptr)), int(sig_rows),
                                  flags, _ptr(int(power_ptr)) if power_ptr else None,
                                  _ptr(int(ratio_ptr)) if ratio_ptr else None, C.c_void_p(int(stream))), "wtb_ratio_planes")


def phase_arrows(phase, *, f64=None):
    """(u, v) = (cos(pi/2 - phase), sin(pi/2 - phase)), any shape (wtb_phase_arrows)."""
    f64 = _resolve_f64(f64)
    ph = np.ascontiguousarray(phase, dtype=_dtype(f64))
    u, v = np.empty_like(ph), np.empty_like(ph)
    _check(lib().wtb_phase_arrows(_ptr(ph), ph.size, F64 if f64 else 0, _ptr(u), _ptr(v), None), "wtb_phase_arrows")
    return u, v


def phase_arrows_device(phase_ptr, count, u_ptr, v_ptr, *, f64=False, stream=0):
    _check(lib().wtb_phase_arrows(_ptr(int(phase_ptr)), int(count), DEVICE_PTRS | (F64 if f64 else 0),
                                  _ptr(int(u_ptr)) if u_ptr else None, _ptr(int(v_ptr)) if v_ptr else None,
                                  C.c_void_p(int(stream))), "wtb_phase_arrows")


# ---------------------------------------------------------------- XWT / WCT
def xwt_wct(y1, y2, dt, dj, s0, J, f0=6.0, *, nfft=None, f64=None, want_wct=True, want_phase=True,
            want_w12=False, generic_only=False):
    """Batched cross-wavelet / coherence of already-normalised host series.
    Returns (wct, phase, w12), each [batch, S, n0] or None."""
    f64 = _resolve_f64(f64)
    rt = _dtype(f64)
    a = np.ascontiguousarray(np.atleast_2d(np.asarray(y1)), dtype=rt)
    b = np.ascontiguousarray(np.atleast_2d(np.asarray(y2)), dtype=rt)
    if a.shape != b.shape:
        raise ValueError("y1 and y2 must have the same shape")
    batch, n0 = a.shape
    Jr, _, _, _ = cwt_axes(n0, dt, dj, s0, J, f0)
    S = Jr + 1
    nfft = int(nfft) if nfft else default_nfft(n0)
    wct = np.empty((batch, S, n0), dtype=rt) if want_wct else None
    phase = np.empty((batch, S, n0), dtype=rt) if want_phase else None
    w12 = np.empty((batch, S, n0), dtype=np.complex128 if f64 else np.complex64) if want_w12 else None
    flags = (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    _check(lib().wtb_xwt_wct(_ptr(a), _ptr(b), batch, n0, nfft, dt, dj, s0, int(J), f0, flags,
                             _ptr(wct), _ptr(phase), _ptr(w12), None), "wtb_xwt_wct")
    if np.ndim(y1) == 1:
        wct, phase, w12 = (None if v is None else v[0] for v in (wct, phase, w12))
    return wct, phase, w12


def partial_wct(y, x1, x2, dt, dj, s0, J, f0=6.0, *, nfft=None, f64=None, want_pwc=True, want_phase=True,
                want_mwc=True, generic_only=False):
    """Batched partial and multiple wavelet coherence of already-normalised host series (wtb_partial_wct):
    the partial coherence of y and x1 given x2, its phase, and the multiple coherence of y on x1 and x2.
    Returns (pwc, phase, mwc), each [batch, S, n0] or None (batch axis dropped for 1-D input)."""
    f64 = _resolve_f64(f64)
    rt = _dtype(f64)
    a, b, c = (np.ascontiguousarray(np.atleast_2d(np.asarray(v)), dtype=rt) for v in (y, x1, x2))
    if not a.shape == b.shape == c.shape:
        raise ValueError("y, x1 and x2 must have the same shape")
    batch, n0 = a.shape
    Jr, _, _, _ = cwt_axes(n0, dt, dj, s0, J, f0)
    S = Jr + 1
    nfft = int(nfft) if nfft else default_nfft(n0)
    pwc, phase, mwc = (np.empty((batch, S, n0), dtype=rt) if w else None for w in (want_pwc, want_phase, want_mwc))
    flags = (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    _check(lib().wtb_partial_wct(_ptr(a), _ptr(b), _ptr(c), batch, n0, nfft, dt, dj, s0, int(J), f0, flags,
                                 _ptr(pwc), _ptr(phase), _ptr(mwc), None), "wtb_partial_wct")
    if np.ndim(y) == 1:
        pwc, phase, mwc = (None if v is None else v[0] for v in (pwc, phase, mwc))
    return pwc, phase, mwc


# ---------------------------------------------------------------- Monte Carlo significance
def wct_mc_geometry(dt, dj, s0, J, f0=6.0):
    """(nsurr, maxscale) of pycwt.wct_significance."""
    n, m = C.c_int(0), C.c_int(0)
    _check(lib().wtb_wct_mc_geometry(dt, dj, s0, int(J), f0, C.byref(n), C.byref(m)), "wtb_wct_mc_geometry")
    return n.value, m.value


def wct_mc_hist(a1, a2, dt, dj, s0, J, f0=6.0, *, mc_first=0, mc_count=300, seed=0, surrogates=None,
                f64=None, white=False, hist=None, generic_only=False):
    """Per-scale coherence histogram [S, 1000] (uint64) of `mc_count` realisations.
    `surrogates` ([mc_count, 2, nsurr] host array) switches to injected-noise mode."""
    f64 = _resolve_f64(f64)
    S = int(J) + 1
    if hist is None:
        hist = np.zeros((S, NBINS), dtype=np.uint64)
    sur = None
    if surrogates is not None:
        nsurr, _ = wct_mc_geometry(dt, dj, s0, J, f0)
        sur = np.ascontiguousarray(surrogates, dtype=_dtype(f64))
        if sur.shape != (mc_count, 2, nsurr):
            raise ValueError(f"surrogates must have shape ({mc_count}, 2, {nsurr}), got {sur.shape}")
    flags = ((F64 if f64 else 0) | (NOISE_WHITE if white else 0) | (GENERIC_ONLY if generic_only else 0)
             | (FFT_NO_PAD if _fft_pad == "none" else 0))
    _check(lib().wtb_wct_mc_hist(a1, a2, dt, dj, s0, int(J), f0, int(mc_first), int(mc_count),
                                 C.c_uint64(int(seed)), _ptr(sur), flags, _ptr(hist), None), "wtb_wct_mc_hist")
    return hist


def wct_mc_hist_device(a1, a2, dt, dj, s0, J, f0, mc_first, mc_count, seed, hist_ptr, *, f64=False,
                       white=False, stream=0):
    """Device-resident variant: hist_ptr is a device uint64 [S,1000] buffer (added to)."""
    flags = DEVICE_PTRS | (F64 if f64 else 0) | (NOISE_WHITE if white else 0)
    _check(lib().wtb_wct_mc_hist(a1, a2, dt, dj, s0, int(J), f0, int(mc_first), int(mc_count),
                                 C.c_uint64(int(seed)), None, flags, _ptr(int(hist_ptr)),
                                 C.c_void_p(int(stream))), "wtb_wct_mc_hist")


def row_has_points(dt, dj, s0, J, f0=6.0):
    """Boolean [S]: scales with at least one sample inside the reliable region."""
    nsurr, _ = wct_mc_geometry(dt, dj, s0, J, f0)
    _, _, freqs, coi = cwt_axes(nsurr, dt, dj, s0, J, f0)
    return (1.0 / freqs) <= coi.max()


def wct_sig_from_hist(hist, maxscale, level, has_points=None):
    hist = np.ascontiguousarray(hist, dtype=np.uint64)
    S = hist.shape[0]
    sig = np.empty(S)
    hp = None if has_points is None else np.ascontiguousarray(has_points, dtype=np.uint8)
    _check(lib().wtb_wct_sig_from_hist(_ptr(hist), S, int(maxscale), float(level), _ptr(hp), _dp(sig)),
           "wtb_wct_sig_from_hist")
    return sig


def wct_significance(a1, a2, dt, dj, s0, J, f0=6.0, *, level=0.95, mc_count=300, seed=0, surrogates=None,
                     f64=None, white=False, generic_only=False, return_hist=False):
    """pycwt.wct_significance in one call (wtb_wct_significance): every device of init_multi()
    takes a block of realisations, device 0 sums the histograms over NVLink, percentile step.
    Returns sig95 [J+1] (and the summed histogram [J+1, 1000] with return_hist)."""
    f64 = _resolve_f64(f64)
    S = int(J) + 1
    sur = None
    if surrogates is not None:
        nsurr, _ = wct_mc_geometry(dt, dj, s0, J, f0)
        sur = np.ascontiguousarray(surrogates, dtype=_dtype(f64))
        if sur.shape != (mc_count, 2, nsurr):
            raise ValueError(f"surrogates must have shape ({mc_count}, 2, {nsurr}), got {sur.shape}")
    flags = ((F64 if f64 else 0) | (NOISE_WHITE if white else 0) | (GENERIC_ONLY if generic_only else 0)
             | (FFT_NO_PAD if _fft_pad == "none" else 0))
    sig = np.empty(S)
    hist = np.zeros((S, NBINS), dtype=np.uint64) if return_hist else None
    _check(lib().wtb_wct_significance(a1, a2, dt, dj, s0, int(J), f0, float(level), int(mc_count),
                                      C.c_uint64(int(seed)), _ptr(sur), flags, _dp(sig), _ptr(hist)),
           "wtb_wct_significance")
    return (sig, hist) if return_hist else sig


def wct_sig_from_hist_device(hist_ptr, S, maxscale, level, has_points, sig_ptr, *, stream=0):
    """Device-resident percentile step: hist_ptr / sig_ptr are device addresses of uint64 [S, 1000]
    and float64 [S]; has_points is a host array (or None).  Asynchronous on `stream`."""
    hp = None if has_points is None else np.ascontiguousarray(has_points, dtype=np.uint8)
    _check(lib().wtb_wct_sig_from_hist_device(_ptr(int(hist_ptr)), int(S), int(maxscale), float(level), _ptr(hp),
                                              _ptr(int(sig_ptr)), C.c_void_p(int(stream))),
           "wtb_wct_sig_from_hist_device")


def rednoise(a1, a2, nsurr, first, count, seed, *, f64=False, white=False):
    out = np.empty((count, 2, nsurr), dtype=_dtype(f64))
    flags = (F64 if f64 else 0) | (NOISE_WHITE if white else 0)
    _check(lib().wtb_rednoise(a1, a2, nsurr, int(first), int(count), C.c_uint64(int(seed)), flags,
                              _ptr(out), None), "wtb_rednoise")
    return out


def _mc_flags(f64, white, generic_only):
    return ((F64 if f64 else 0) | (NOISE_WHITE if white else 0) | (GENERIC_ONLY if generic_only else 0)
            | (FFT_NO_PAD if _fft_pad == "none" else 0))


def _triples(surrogates, mc_count, dt, dj, s0, J, f0, f64):
    if surrogates is None:
        return None
    nsurr, _ = wct_mc_geometry(dt, dj, s0, J, f0)
    sur = np.ascontiguousarray(surrogates, dtype=_dtype(f64))
    if sur.shape != (mc_count, 3, nsurr):
        raise ValueError(f"surrogates must have shape ({mc_count}, 3, {nsurr}), got {sur.shape}")
    return sur


def partial_wct_mc_hist(ay, a1, a2, dt, dj, s0, J, f0=6.0, *, mc_first=0, mc_count=300, seed=0, surrogates=None,
                        f64=None, white=False, hist=None, generic_only=False):
    """Per-scale histograms [2, S, 1000] (uint64; PWC rows, then MWC rows) of the partial and multiple coherence
    of `mc_count` AR(1) surrogate triples (y, x1, x2) with coefficients (ay, a1, a2).  `surrogates`
    ([mc_count, 3, nsurr] host array) switches to injected-noise mode."""
    f64 = _resolve_f64(f64)
    S = int(J) + 1
    if hist is None:
        hist = np.zeros((2, S, NBINS), dtype=np.uint64)
    sur = _triples(surrogates, mc_count, dt, dj, s0, J, f0, f64)
    _check(lib().wtb_partial_wct_mc_hist(ay, a1, a2, dt, dj, s0, int(J), f0, int(mc_first), int(mc_count),
                                         C.c_uint64(int(seed)), _ptr(sur), _mc_flags(f64, white, generic_only),
                                         _ptr(hist), None), "wtb_partial_wct_mc_hist")
    return hist


def partial_wct_significance(ay, a1, a2, dt, dj, s0, J, f0=6.0, *, level=0.95, mc_count=300, seed=0,
                             surrogates=None, f64=None, white=False, generic_only=False, return_hist=False):
    """Monte-Carlo significance of partial and multiple coherence in one call (wtb_partial_wct_significance):
    every device of init_multi() takes a block of realisations.  Returns (sig_pwc, sig_mwc), each [J+1] (and the
    summed histogram [2, J+1, 1000] with return_hist)."""
    f64 = _resolve_f64(f64)
    S = int(J) + 1
    sur = _triples(surrogates, mc_count, dt, dj, s0, J, f0, f64)
    sig_pwc, sig_mwc = np.empty(S), np.empty(S)
    hist = np.zeros((2, S, NBINS), dtype=np.uint64) if return_hist else None
    _check(lib().wtb_partial_wct_significance(ay, a1, a2, dt, dj, s0, int(J), f0, float(level), int(mc_count),
                                              C.c_uint64(int(seed)), _ptr(sur), _mc_flags(f64, white, generic_only),
                                              _dp(sig_pwc), _dp(sig_mwc), _ptr(hist)),
           "wtb_partial_wct_significance")
    return (sig_pwc, sig_mwc, hist) if return_hist else (sig_pwc, sig_mwc)


def rednoise_triples(ay, a1, a2, nsurr, first, count, seed, *, f64=False, white=False):
    """The device surrogate triples of partial_wct_mc_hist: [count, 3, nsurr]."""
    out = np.empty((count, 3, nsurr), dtype=_dtype(f64))
    flags = (F64 if f64 else 0) | (NOISE_WHITE if white else 0)
    _check(lib().wtb_rednoise_triples(ay, a1, a2, nsurr, int(first), int(count), C.c_uint64(int(seed)), flags,
                                      _ptr(out), None), "wtb_rednoise_triples")
    return out


def rednoise_device(a1, a2, nsurr, first, count, seed, out_ptr, *, f64=False, white=False, stream=0):
    """Device-resident variant of `rednoise`: out_ptr is a device [count, 2, nsurr] buffer."""
    flags = DEVICE_PTRS | (F64 if f64 else 0) | (NOISE_WHITE if white else 0)
    _check(lib().wtb_rednoise(a1, a2, nsurr, int(first), int(count), C.c_uint64(int(seed)), flags,
                              _ptr(int(out_ptr)), C.c_void_p(int(stream))), "wtb_rednoise")


# ---------------------------------------------------------------- MODWT / DWT
def _taps(lo, hi):
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    if lo.shape != hi.shape or lo.ndim != 1:
        raise ValueError("filter banks must be 1-D and of equal length")
    return lo, hi


def modwt(x, g, h, J, *, f64=None, generic_only=False):
    f64 = _resolve_f64(f64)
    g, h = _taps(g, h)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=_dtype(f64))
    batch, n = x2.shape
    out = np.empty((batch, J + 1, n), dtype=x2.dtype)
    _check(lib().wtb_modwt(_ptr(x2), batch, n, _dp(g), _dp(h), g.size, int(J),
                           (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0), _ptr(out), None), "wtb_modwt")
    return out[0] if np.ndim(x) == 1 else out


def modwt_device(x_ptr, batch, n, g, h, J, out_ptr, *, f64=False, stream=0):
    """Device-resident MODWT: x [batch, n] -> out [batch, J+1, n], asynchronous on `stream`."""
    g, h = _taps(g, h)
    _check(lib().wtb_modwt(_ptr(int(x_ptr)), batch, n, _dp(g), _dp(h), g.size, int(J),
                           DEVICE_PTRS | (F64 if f64 else 0), _ptr(int(out_ptr)), C.c_void_p(int(stream))),
           "wtb_modwt")


def imodwt_device(w_ptr, batch, n, g, h, J, out_ptr, *, f64=False, stream=0):
    g, h = _taps(g, h)
    _check(lib().wtb_imodwt(_ptr(int(w_ptr)), batch, n, _dp(g), _dp(h), g.size, int(J),
                            DEVICE_PTRS | (F64 if f64 else 0), _ptr(int(out_ptr)), C.c_void_p(int(stream))),
           "wtb_imodwt")


def wavedec_device(x_ptr, batch, n, dec_lo, dec_hi, level, out_ptr, *, f64=False, stream=0):
    lo, hi = _taps(dec_lo, dec_hi)
    _check(lib().wtb_wavedec(_ptr(int(x_ptr)), batch, n, _dp(lo), _dp(hi), lo.size, int(level),
                             DEVICE_PTRS | (F64 if f64 else 0), _ptr(int(out_ptr)), C.c_void_p(int(stream))),
           "wtb_wavedec")


def imodwt(w, g, h, *, f64=None, generic_only=False):
    f64 = _resolve_f64(f64)
    g, h = _taps(g, h)
    w = np.asarray(w)
    w3 = np.ascontiguousarray(w[None] if w.ndim == 2 else w, dtype=_dtype(f64))
    batch, rows, n = w3.shape
    out = np.empty((batch, n), dtype=w3.dtype)
    _check(lib().wtb_imodwt(_ptr(w3), batch, n, _dp(g), _dp(h), g.size, rows - 1,
                            (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0), _ptr(out), None), "wtb_imodwt")
    return out[0] if w.ndim == 2 else out


def modwtmra(w, filt, *, f64=None):
    f64 = _resolve_f64(f64)
    w = np.asarray(w)
    w3 = np.ascontiguousarray(w[None] if w.ndim == 2 else w, dtype=_dtype(f64))
    batch, rows, n = w3.shape
    filt = np.ascontiguousarray(filt, dtype=np.float64)
    if filt.shape != (rows, n):
        raise ValueError(f"filt must have shape ({rows}, {n})")
    out = np.empty_like(w3)
    _check(lib().wtb_modwtmra(_ptr(w3), batch, n, _dp(filt), rows - 1, F64 if f64 else 0, _ptr(out), None),
           "wtb_modwtmra")
    return out[0] if w.ndim == 2 else out


def modwtmra_taps(w, g, h, *, f64=None, generic_only=False):
    """MRA rows D_1..D_J, S_J from the wavelet taps (synthesis cascade, wtb_modwtmra_taps)."""
    f64 = _resolve_f64(f64)
    w = np.asarray(w)
    w3 = np.ascontiguousarray(w[None] if w.ndim == 2 else w, dtype=_dtype(f64))
    batch, rows, n = w3.shape
    g, h = _taps(g, h)
    out = np.empty_like(w3)
    _check(lib().wtb_modwtmra_taps(_ptr(w3), batch, n, _dp(g), _dp(h), g.size, rows - 1,
                                   (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0), _ptr(out), None),
           "wtb_modwtmra_taps")
    return out[0] if w.ndim == 2 else out


def modwt_wavelet_stats(x, y, g, h, J, max_lag=0, f64=None, generic_only=False):
    """MODWT wavelet variance and cross-covariance by level over the coefficients free of the circular wrap
    (wtb_modwt_wavelet_stats).  x, y: [n] or [batch, n] (y None: the variance of x alone).  Returns
    (var_x [batch, J], var_y [batch, J] or None, xcov [batch, J, 2 max_lag + 1] or None), float64, lags
    -max_lag..max_lag; NaN where a level has no such coefficients or a lag reaches past them.  The batch axis is
    dropped for 1-D input."""
    f64 = _resolve_f64(f64)
    g, h = _taps(g, h)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=_dtype(f64))
    y2 = None if y is None else np.ascontiguousarray(np.atleast_2d(np.asarray(y)), dtype=_dtype(f64))
    if y2 is not None and y2.shape != x2.shape:
        raise ValueError("x and y must have the same shape")
    batch, n = x2.shape
    J, K = int(J), int(max_lag)
    var_x = np.empty((batch, max(J, 0)))
    var_y = None if y2 is None else np.empty((batch, max(J, 0)))
    xcov = None if y2 is None else np.empty((batch, max(J, 0), 2 * max(K, 0) + 1))
    flags = (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    _check(lib().wtb_modwt_wavelet_stats(_ptr(x2), _ptr(y2), batch, n, _dp(g), _dp(h), g.size, J, K, flags,
                                         _ptr(var_x), _ptr(var_y), _ptr(xcov), None), "wtb_modwt_wavelet_stats")
    if np.ndim(x) == 1:
        var_x, var_y, xcov = (None if v is None else v[0] for v in (var_x, var_y, xcov))
    return var_x, var_y, xcov


def modwt_wavelet_stats_device(x_ptr, y_ptr, batch, n, g, h, J, max_lag, var_x_ptr, var_y_ptr, xcov_ptr, *,
                               f64=False, generic_only=False, stream=0):
    """Device-resident wtb_modwt_wavelet_stats: raw device addresses (y_ptr and any output may be 0 for "none"),
    float64 outputs, asynchronous on `stream`."""
    g, h = _taps(g, h)
    dp = lambda v: _ptr(int(v)) if v else None
    flags = DEVICE_PTRS | (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0)
    _check(lib().wtb_modwt_wavelet_stats(dp(x_ptr), dp(y_ptr), int(batch), int(n), _dp(g), _dp(h), g.size, int(J),
                                         int(max_lag), flags, dp(var_x_ptr), dp(var_y_ptr), dp(xcov_ptr),
                                         C.c_void_p(int(stream))), "wtb_modwt_wavelet_stats")


def waverec_len(lens, L):
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    nout = lib().wtb_waverec_len(lens.ctypes.data_as(_pi), lens.size - 1, int(L))
    if nout < 0:
        _check(nout, "wtb_waverec_len")
    return int(nout)


def waverec_device(coeffs_ptr, batch, lens, rec_lo, rec_hi, out_ptr, *, f64=False, stream=0):
    lo, hi = _taps(rec_lo, rec_hi)
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    _check(lib().wtb_waverec(_ptr(int(coeffs_ptr)), batch, lens.ctypes.data_as(_pi), lens.size - 1, _dp(lo), _dp(hi),
                             lo.size, DEVICE_PTRS | (F64 if f64 else 0), _ptr(int(out_ptr)), C.c_void_p(int(stream))),
           "wtb_waverec")


def modwtmra_taps_device(w_ptr, batch, n, g, h, J, out_ptr, *, f64=False, stream=0):
    g, h = _taps(g, h)
    _check(lib().wtb_modwtmra_taps(_ptr(int(w_ptr)), batch, n, _dp(g), _dp(h), g.size, int(J),
                                   DEVICE_PTRS | (F64 if f64 else 0), _ptr(int(out_ptr)), C.c_void_p(int(stream))),
           "wtb_modwtmra_taps")


def dwt_max_level(n, L):
    return int(lib().wtb_dwt_max_level(int(n), int(L)))


def dwt_coeff_lens(n, L, level):
    lens = np.zeros(level + 1, dtype=np.int32)
    _check(lib().wtb_dwt_coeff_lens(int(n), int(L), int(level), lens.ctypes.data_as(_pi)), "wtb_dwt_coeff_lens")
    return lens


def wavedec(x, dec_lo, dec_hi, level, *, f64=None, generic_only=False):
    """Packed coefficients [batch, sum(lens)] + lens (cA_L, cD_L, ..., cD_1)."""
    f64 = _resolve_f64(f64)
    lo, hi = _taps(dec_lo, dec_hi)
    x2 = np.ascontiguousarray(np.atleast_2d(np.asarray(x)), dtype=_dtype(f64))
    batch, n = x2.shape
    lens = dwt_coeff_lens(n, lo.size, level)
    out = np.empty((batch, int(lens.sum())), dtype=x2.dtype)
    _check(lib().wtb_wavedec(_ptr(x2), batch, n, _dp(lo), _dp(hi), lo.size, int(level),
                             (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0), _ptr(out), None), "wtb_wavedec")
    return (out[0] if np.ndim(x) == 1 else out), lens


def waverec(packed, lens, rec_lo, rec_hi, *, f64=None, generic_only=False):
    f64 = _resolve_f64(f64)
    lo, hi = _taps(rec_lo, rec_hi)
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    level = lens.size - 1
    p = np.asarray(packed)
    p2 = np.ascontiguousarray(np.atleast_2d(p), dtype=_dtype(f64))
    if p2.shape[1] != int(lens.sum()):
        raise ValueError("packed coefficient row does not match lens")
    nout = lib().wtb_waverec_len(lens.ctypes.data_as(_pi), level, lo.size)
    if nout < 0:
        _check(nout, "wtb_waverec_len")
    out = np.empty((p2.shape[0], nout), dtype=p2.dtype)
    _check(lib().wtb_waverec(_ptr(p2), p2.shape[0], lens.ctypes.data_as(_pi), level, _dp(lo), _dp(hi),
                             lo.size, (F64 if f64 else 0) | (GENERIC_ONLY if generic_only else 0), _ptr(out), None),
           "wtb_waverec")
    return out[0] if p.ndim == 1 else out
