"""Per-scale-row view of the FP32 Morlet CWT kernels -- TEST INFRASTRUCTURE ONLY.

The FP32 error of the fused CWT kernels is per scale row: every row is its own inverse transform
of X^ * daughter_s, pruned to the daughter's band, and takes its own branch of the pruned
transform.  A gate relative to the plane maximum (``conftest.normwise_close``) sees the
high-power rows only; for red-noise inputs the small-scale rows hold 1e-3 .. 1e-4 of the plane
maximum and are barely checked by it.  This module holds

* ``row_gate``: ``|a - b| <= tol * (|b| + scale_row)`` on chosen rows, with
  ``scale_row = max(max_t |b_row|, 1e-5 * max |b_plane|)``.  The floor admits the forward
  transform's round-off of the whole series, which reaches every row;
* ``resolved_rows``: the rows whose daughter band holds at least two bins below the Nyquist
  frequency and whose peak lies below it.  The other rows hold only the daughter's tail, which
  the kernels' one-sided band cut drops by design (DESIGN section 2), so they keep the plane gate;
* a replica of the host row rules of ``row_params`` in ``cwt_fast.cu`` (nfft 1024 and the two-series
  nfft 512, nfft 2048 / 4096) and ``fill_rows`` (``k_cwt_rows_4096`` and the coherence
  kernels), so that tests can prove which branches of the pruned transforms their shapes reach.
"""

import math

import numpy as np

ZCUT_F32 = float(np.float32(5.3))    # kZCut of cwt_paths.cuh (a float constant, widened to double)
ZCUT_F64 = 5.3                       # fill_rows of wct_fast.cu (a double literal)
ROW_FLOOR = 1e-5


def row_gate(got, ref, tol, rows=None):
    """Worst ratio of |got - ref| to tol * (|ref| + scale_row) over ``rows`` (bool mask or indices
    of the first axis; None: every row) of [S, n0] planes, and where it sits as (row, t).  The gate
    passes when the ratio is <= 1.  scale_row = max(max_t |ref_row|, 1e-5 * max |ref_plane|)."""
    a = np.asarray(got)
    b = np.asarray(ref)
    assert a.shape == b.shape and b.ndim == 2, (a.shape, b.shape)
    if a.dtype.kind == "c" or b.dtype.kind == "c":
        a, b = a.astype(np.complex128), b.astype(np.complex128)
    else:
        a, b = a.astype(np.float64), b.astype(np.float64)
    mag = np.abs(b)
    scale_row = np.maximum(mag.max(axis=1), ROW_FLOOR * mag.max())
    idx = np.arange(b.shape[0]) if rows is None else np.arange(b.shape[0])[rows]
    if idx.size == 0:
        return 0.0, None
    ratio = np.abs(a[idx] - b[idx]) / (tol * (mag[idx] + scale_row[idx, None]) + 1e-300)
    r, t = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    return float(ratio[r, t]), (int(idx[r]), int(t))


def scales(dt, dj, s0, J):
    """The scale axis as the host forms it (runtime.cu: s0 * pow(2, j * dj))."""
    return s0 * 2.0 ** (np.arange(J + 1) * dj)


def _a(sc, dt, n):
    return sc / dt * 2.0 * math.pi / n


def resolved_rows(n0, nfft, dt, dj, s0, J, f0=6.0):
    """Rows with floor((f0 + 5.3) nfft dt / (2 pi s)) >= 2 (two bins of daughter support) and
    s / dt >= f0 / pi (the daughter peaks below the Nyquist frequency)."""
    del n0                                   # the rule depends on the transform length only
    sc = scales(dt, dj, s0, J)
    khi = np.floor((f0 + 5.3) * nfft * dt / (2.0 * math.pi * sc))
    return (khi >= 2) & (sc / dt >= f0 / math.pi)


def _ilog2(n):
    """common.cuh ilog2: smallest l with 2^l >= n."""
    l = 0
    while (1 << l) < n:
        l += 1
    return l


def fast_rows(nfft, dt, dj, s0, J, f0=6.0):
    """(multi, L) per row as row_params fills RowParam for k_cwt_fast_1024 (nfft 1024) and its
    two-series HALF variant (nfft 512: 1024-point a and band edge, one bin further out)."""
    assert nfft in (512, 1024)
    half = nfft == 512
    out = []
    for sc in scales(dt, dj, s0, J):
        khi = int(math.floor((f0 + ZCUT_F32) / _a(sc, dt, 1024))) + (1 if half else 0)
        khi = max(1, min(khi, 511))
        if khi >= 32:
            out.append((1, max(1, min(4, _ilog2(khi // 32 + 1)))))
        else:
            out.append((0, _ilog2(khi + 1)))
    return out


def dif_rows(nfft, dt, dj, s0, J, f0=6.0):
    """(multi, L) per row as row_params fills RowParam for k_cwt_dif<D>, D = nfft / 1024: a warp
    transforms the bins of one residue mod D, j = k / D <= jhi.  L == 1 rows (either pass kind)
    take the two-input DFT."""
    assert nfft in (2048, 4096)
    D = nfft // 1024
    out = []
    for sc in scales(dt, dj, s0, J):
        khi = int(math.floor((f0 + ZCUT_F32) / _a(sc, dt, nfft)))
        khi = max(1, min(khi, nfft // 2 - 1))
        jhi = khi // D
        if jhi >= 32:
            out.append((1, max(1, min(4, _ilog2(jhi // 32 + 1)))))
        else:
            out.append((0, max(1, _ilog2(jhi + 1))))
    return out


def wrow_rows(dt, dj, s0, J, f0=6.0):
    """(R1, L1) per row as fill_rows fills WRow (k_cwt_rows_4096, k_wct_spec_4096): R1 = 2^L1
    blocks of 256 bins hold the daughter's support."""
    out = []
    for sc in scales(dt, dj, s0, J):
        khi = int(math.floor((f0 + ZCUT_F64) / _a(sc, dt, 4096)))
        khi = max(1, min(khi, 2047))
        L1 = _ilog2(khi // 256 + 1)
        out.append((1 << L1, L1))
    return out


# Every row class each kernel has a branch for.
ROW_CLASSES = {
    "fast": {(0, L) for L in range(1, 6)} | {(1, L) for L in range(1, 5)},
    "dif": {(0, L) for L in range(1, 6)} | {(1, L) for L in range(1, 5)},
    "wrow": {(1 << L1, L1) for L1 in range(4)},
}


def row_classes(kernel, dt, dj, s0, J, f0=6.0):
    """Row classes of one call: kernel in 'fast1024', 'half', 'dif2', 'dif4', 'rows4096'."""
    if kernel == "fast1024":
        return fast_rows(1024, dt, dj, s0, J, f0)
    if kernel == "half":
        return fast_rows(512, dt, dj, s0, J, f0)
    if kernel in ("dif2", "dif4"):
        return dif_rows(1024 * int(kernel[-1]), dt, dj, s0, J, f0)
    if kernel == "rows4096":
        return wrow_rows(dt, dj, s0, J, f0)
    raise ValueError(kernel)


def class_family(kernel):
    return {"fast1024": "fast", "half": "fast", "dif2": "dif", "dif4": "dif", "rows4096": "wrow"}[kernel]
