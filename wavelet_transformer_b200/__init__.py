"""wavelet_transformer_b200 -- B200-native (sm_100a) wavelet engine.

Drop-in for the numerics behind o-nate/wavelet-transformer's ``src/cwt.py``,
``src/wct.py``, ``src/xwt.py``, ``src/dwt.py`` and ``src/modwt.py``.  All
arithmetic on the hot path runs in ``lib/libwavelet_sm100a.so`` (hand-written
CUDA, reached through the C ABI of ``include/wtb.h`` via ctypes); there is no
CPU fallback.

Layout
    _shim.py          ctypes binding (NumPy buffers <-> C ABI)
    _build.py         nvcc recipe for the shared library
    csrc/             CUDA kernels + C ABI
    pycwt_compat.py   pycwt-shaped facade   (``import ... as wavelet``)
    pywt_compat.py    PyWavelets-shaped facade (``import ... as pywt``)
    api/              re-authored reference entry points (same names/signatures)
    engine.py         batched / multi-GPU entry points (series and Monte Carlo shards)
    partial_coherence.py  partial and multiple wavelet coherence of three series (``partial_wct``) and their
                      Monte-Carlo significance (``partial_wct_significance``)
    wavelet_stats.py  MODWT wavelet variance, covariance and cross-correlation by level with confidence
                      intervals (``wavelet_variance``, ``wavelet_correlation``)
"""

from ._shim import (WaveletEngineError, device_count, get_fft_padding, get_precision, gpu_count, init,  # noqa: F401
                    init_multi, lib_path, set_fft_padding, set_precision, shutdown)
from .partial_coherence import partial_wct, partial_wct_significance  # noqa: F401
from .wavelet_stats import wavelet_correlation, wavelet_variance  # noqa: F401

__version__ = "0.1.0"
