"""float64 references for the filterbanks of long series, and a replica of the long path's route and wave rules.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  ``pywt_oracle.dwt`` loops in Python over every output and
``modwt_oracle.modwtmra`` correlates with dense [J+1, N] periodised filters (O(N^2)); both are the pinned
definitions at short lengths, and tests/test_oracle_filterbank_long.py holds these vectorised forms to them:

* ``dwt`` / ``idwt`` -- one symmetric-mode analysis step as L strided gathers of the half-sample symmetric
  extension, and the synthesis step as L/2 strided taps per output parity; ``wavedec`` / ``waverec`` chain them
  as pywt does.
* ``modwtmra`` -- the synthesis cascade D_j = G_1' .. G_{j-1}' H_j' w_j, S_J = G_1' .. G_J' v_J with
  X_k' v[t] = sum_l x[l] / sqrt(2) v[(t + 2^(k-1) l) mod N]: the same rows as the equivalent-filter correlation at
  sum_j j L gathers per sample.
* ``modwt`` / ``imodwt`` are modwt_oracle's, which already gather one tap at a time.

The replica mirrors filterbank.cu's ``fb_plan`` and filterbank_long.cu: ``route`` says whether a call takes the long
path, ``launches`` how many kernels it runs there.
"""

from __future__ import annotations

import numpy as np

from . import modwt_oracle
from .pywt_oracle import _as_wavelet, _sym_ext, dwt_coeff_len, dwt_max_level

modwt = modwt_oracle.modwt
imodwt = modwt_oracle.imodwt

SMEM_LIMIT = 227 * 1024
WAVE_BYTES = 64 << 20
CHUNK_BYTES = 1 << 30


# ---- references -------------------------------------------------------------------------------------------------
def dwt(x, wavelet):
    """cA[i] = sum_j lo[j] xe[2i+1-j], cD with hi (pywt mode='symmetric')."""
    w = _as_wavelet(wavelet)
    x = np.asarray(x, dtype=float)
    L = w.dec_len
    xe = _sym_ext(x, L - 1)                      # xe[p] == x_ext[p - (L-1)]
    nout = dwt_coeff_len(x.size, L)
    base = 2 * np.arange(nout) + L               # 2i + 1 + (L-1)
    cA, cD = np.zeros(nout), np.zeros(nout)
    for j, (lo, hi) in enumerate(zip(w.dec_lo, w.dec_hi)):
        seg = xe[base - j]
        cA += lo * seg
        cD += hi * seg
    return cA, cD


def idwt(cA, cD, wavelet):
    """full[p] = sum_k rec_lo[p-2k] cA[k] + rec_hi[p-2k] cD[k], kept p in [L-2, L-2 + 2m-L+2)."""
    w = _as_wavelet(wavelet)
    cA, cD = np.asarray(cA, dtype=float), np.asarray(cD, dtype=float)
    L, m = w.dec_len, cA.size
    nout = 2 * m - L + 2
    p = np.arange(nout) + L - 2
    out = np.zeros(nout)
    for e in range(L):                           # tap e meets k = (p - e) / 2 where p - e is even and in range
        k = p - e
        ok = (k % 2 == 0) & (k >= 0) & (k < 2 * m)
        kk = k[ok] // 2
        out[ok] += w.rec_lo[e] * cA[kk] + w.rec_hi[e] * cD[kk]
    return out


def wavedec(data, wavelet, level=None):
    """[cA_L, cD_L, ..., cD_1]."""
    w = _as_wavelet(wavelet)
    a = np.asarray(data, dtype=float)
    if level is None:
        level = dwt_max_level(a.size, w.dec_len)
    out = []
    for _ in range(level):
        a, d = dwt(a, w)
        out.append(d)
    out.append(a)
    return out[::-1]


def waverec(coeffs, wavelet):
    w = _as_wavelet(wavelet)
    a = np.asarray(coeffs[0], dtype=float)
    for d in coeffs[1:]:
        d = np.asarray(d, dtype=float)
        if a.size == d.size + 1:
            a = a[:-1]
        a = idwt(a, d, w)
    return a


def _synth(v, taps, k):
    """X_k' v: sum_l taps[l] v[(t + 2^(k-1) l) mod N]."""
    return modwt_oracle._circ_gather(v, taps, 2 ** (k - 1), +1)


def modwtmra(w, filters):
    """Details D_1..D_J and smooth S_J of MODWT rows w [J+1, N], stacked as (J+1, N)."""
    h, g = modwt_oracle._taps(filters)
    h_t, g_t = h / np.sqrt(2), g / np.sqrt(2)
    w = np.asarray(w, dtype=float)
    J = w.shape[0] - 1
    rows = []
    for j in range(1, J + 1):
        a = _synth(w[j - 1], h_t, j)
        for k in range(j - 1, 0, -1):
            a = _synth(a, g_t, k)
        rows.append(a)
    a = w[J]
    for k in range(J, 0, -1):
        a = _synth(a, g_t, k)
    rows.append(a)
    return np.vstack(rows)


# ---- replica of the route and wave rules ------------------------------------------------------------------------
def _elem(f64):
    return 8 if f64 else 4


def _ceil4(n):
    return (n + 3) & ~3


def _chain_threads(n, L, J, R):
    """filterbank_fast.cu chain_threads != 0."""
    if J > 10 or ((((L - 1) << (J - 1)) + 3) & ~3) > n:
        return False
    most = max(-(-n // ((1 << (j - 1)) * R)) * (1 << (j - 1)) for j in range(1, J + 1))
    return most <= 512


def mra_fast_covers(n, L, J, f64):
    """filterbank_fast.cu blk_shape(FbOp::kMraTaps, ...).threads != 0: the MRA cascade kernel k_mra_blk serves the
    shape."""
    def fits(R):
        return _chain_threads(n, L, J, R) and _elem(f64) * _ceil4(n + (R + L - 2) * (1 << (J - 1)) + 4) <= SMEM_LIMIT
    return L in (2, 4, 6, 8) and ((n >= 2048 and fits(17)) or fits(9))


def coeff_lens(n, L, level):
    """wtb_dwt_coeff_lens: [cA_L, cD_L, ..., cD_1]."""
    lens, cur = [0] * (level + 1), n
    for l in range(level):
        cur = (cur + L - 1) // 2
        lens[level - l] = cur
    lens[0] = cur
    return lens


def waverec_len(lens, L):
    a = lens[0]
    for d in lens[1:]:
        a = 2 * d - L + 2
    return a


# Static shared memory of the generic one-CTA kernels (ptxas: tap tables and mbarrier, padded to 16 B), FP32 / FP64.
# It counts against the 227 KB with the dynamic buffers: fits_one_cta, called by fb_plan in filterbank.cu.
STATIC_SMEM = {"modwt": (400, 656), "imodwt": (400, 656), "modwtmra": (16, 16), "modwtmra_taps": (16, 16),
               "wavedec": (16, 16), "waverec": (0, 0)}


def route(entry, n, f64, L=8, J=1, level=None, generic_only=False):
    """'long' or 'one-cta' for a call of wtb_<entry> on series of n samples (for waverec: the n whose wavedec
    coefficients it reconstructs)."""
    E = _elem(f64)
    static = STATIC_SMEM[entry][bool(f64)]
    if entry in ("modwt", "modwtmra", "wavedec"):
        takes = E * 2 * _ceil4(n) + static > SMEM_LIMIT
    elif entry == "imodwt":
        takes = E * 3 * _ceil4(n) + static > SMEM_LIMIT
    elif entry == "modwtmra_taps":
        fast = not generic_only and mra_fast_covers(n, L, J, f64)
        takes = not fast and E * 2 * _ceil4(n) + static > SMEM_LIMIT
    elif entry == "waverec":
        lens = coeff_lens(n, L, level)
        longest = max([waverec_len(lens, L)] + lens)
        takes = E * 2 * _ceil4(longest + L) + static > SMEM_LIMIT
    else:
        raise ValueError(entry)
    return "long" if takes else "one-cta"


def first_long_n(entry, f64, L=8, J=1, level=1):
    """The shortest series that route() sends to the long path (n grows: every rule is monotone in n)."""
    lo, hi = 1, 1 << 20
    while lo < hi:
        mid = (lo + hi) // 2
        if route(entry, mid, f64, L, J, level) == "long":
            hi = mid
        else:
            lo = mid + 1
    return lo


def _rows(entry, n, L, J, level):
    """(in_row, out_row, per-series intermediate, launches per wave) in elements."""
    if entry == "modwt":
        return n, (J + 1) * n, 2 * n, J
    if entry == "imodwt":
        return (J + 1) * n, n, 2 * n, J
    if entry == "modwtmra_taps":
        return (J + 1) * n, (J + 1) * n, 2 * (J + 1) * n, J
    if entry == "modwtmra":
        return (J + 1) * n, (J + 1) * n, 2 * (J + 1) * n, 1
    lens = coeff_lens(n, L, level)
    if entry == "wavedec":
        return n, sum(lens), 2 * n, level
    if entry == "waverec":
        nout = waverec_len(lens, L)
        return sum(lens), nout, 2 * nout, level
    raise ValueError(entry)


def wave_rows(per_series_bytes, rows):
    """Series per wave: those whose intermediates fit 64 MiB, at least one, at most ``rows``."""
    return min(rows, max(1, WAVE_BYTES // per_series_bytes))


def launches(entry, n, f64, batch, L=8, J=1, level=1, device_ptrs=False):
    """Kernel launches of one long-path call: per host chunk of stage_rows (1 GiB of input and output rows,
    the whole batch with device pointers), waves of wave_rows series, each with its launches per wave."""
    E = _elem(f64)
    in_row, out_row, inter, per_wave = _rows(entry, n, L, J, level)
    chunk = batch if device_ptrs else max(1, min(batch, CHUNK_BYTES // (E * (in_row + out_row))))
    cap = wave_rows(E * inter, batch)
    total = 0
    for b0 in range(0, batch, chunk):
        nb = min(chunk, batch - b0)
        total += -(-nb // min(cap, nb)) * per_wave
    return total
