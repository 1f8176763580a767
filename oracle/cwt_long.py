"""Long-series CWT (cwt_long.cu) -- TEST INFRASTRUCTURE ONLY.

* ``cwt_rows``: chosen scale rows of pycwt's CWT in float64.  One forward FFT of the padded series and one
  inverse FFT per chosen row, so a test at nfft = 2^22 never holds the whole [S, n0] plane;
* a replica of the host rules of the long path: which transforms it takes (``route``), the wave rule
  (``wave_rows``), the launch count of one ``cwt_device`` call (``launches``) and the chunk rule of
  ``wtb_cwt_averages`` at those lengths (``averages_chunk_rows``).
"""

import numpy as np

from oracle import pycwt_oracle as po

MAX_NFFT = 1 << 22
SMEM_LIMIT = 227 * 1024
WAVE_BYTES = 64 << 20
AVG_BUDGET = 1 << 30


def cwt_rows(signal, dt, dj, s0, J, wavelet, rows, nfft=None):
    """W[rows, :n0] (complex128) of ``po.cwt(signal, dt, dj, s0, J, wavelet)``; nfft defaults to pycwt's
    padding to the next power of two."""
    x = np.asarray(signal, dtype=float)
    n0 = x.size
    sj, _, _ = po.cwt_axes(n0, dt, dj, s0, J, wavelet)
    N = nfft or po._pow2(n0)
    xf = np.fft.fft(x, n=N)
    ftfreqs = 2 * np.pi * np.fft.fftfreq(N, dt)
    out = np.empty((len(rows), n0), dtype=np.complex128)
    for i, s in enumerate(rows):
        psi_bar = (sj[s] * ftfreqs[1] * N) ** 0.5 * np.conjugate(wavelet.psi_ft(sj[s] * ftfreqs))
        out[i] = np.fft.ifft(xf * psi_bar)[:n0]
    return out


def _elem(f64):
    return 8 if f64 else 4


def long_takes(nfft, f64):
    """cwt_long_takes: a power of two whose two shared-memory buffers (2 nfft complex) exceed 227 KB."""
    return nfft > 0 and nfft & (nfft - 1) == 0 and 2 * 2 * _elem(f64) * nfft > SMEM_LIMIT


def route(nfft, f64):
    """'long', 'refused' (a power of two past 2^22) or 'generic' (everything cwt_device did before)."""
    if long_takes(nfft, f64):
        return "long" if nfft <= MAX_NFFT else "refused"
    return "generic"


def wave_rows(nfft, f64, rows):
    """long_wave_rows: rows whose intermediate (nfft complex each) fit 64 MiB, at least 1, at most ``rows``."""
    return min(rows, max(1, WAVE_BYTES // (2 * _elem(f64) * nfft)))


def waves(nfft, f64, batch, S):
    """(forward waves, row waves) of one call."""
    wf, wi = wave_rows(nfft, f64, batch), wave_rows(nfft, f64, batch * S)
    return -(-batch // wf), -(-(batch * S) // wi)


def launches(nfft, f64, batch, S):
    """Kernel launches of one long-path cwt_device call: two passes per wave, forward and inverse."""
    fw, iw = waves(nfft, f64, batch, S)
    return 2 * fw + 2 * iw


def averages_chunk_rows(batch, S, n0, f64):
    """averages_chunk_rows at the lengths the long path serves: series within 1 GiB of power rows, at least 1."""
    return min(batch, max(1, AVG_BUDGET // (_elem(f64) * S * n0)))
