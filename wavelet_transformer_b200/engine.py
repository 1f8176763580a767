"""Batched and multi-GPU entry points.

One process per GPU (``torch.distributed``); the two shardable units of the hot
path are independent *series* (fused CWT+power) and independent Monte Carlo
*realisations* (coherence significance).  Series need no collective at all;
realisations need exactly one: an integer all-reduce of the per-scale
histograms, after which every rank holds the same thresholds.

PyTorch is used here only as plumbing (device buffers, streams, NCCL); every
kernel is in libwavelet_sm100a.so.
"""

from __future__ import annotations

import numpy as np

from . import _shim


def shard_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [start, stop) of `total` units owned by `rank`; the first
    ``total % world`` ranks get one extra unit."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("need 0 <= rank < world")
    base, extra = divmod(int(total), world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def cwt_power_resident(x, power, dt, dj, s0, J, f0=6.0, generic_only=False):
    """Fused CWT+power of a device-resident batch.

    x: torch CUDA float32/float64 tensor [batch, n0]; power: preallocated
    [batch, J+1, n0] tensor of the same dtype.  Runs on the device that owns x
    (the library reads it off the pointer), enqueued on torch's current stream
    of that device; nothing is copied or synchronised."""
    import torch
    if not (x.is_cuda and power.is_cuda and x.is_contiguous() and power.is_contiguous()):
        raise ValueError("x and power must be contiguous CUDA tensors")
    if x.device != power.device:
        raise ValueError("x and power must live on the same device")
    if x.dtype != power.dtype or x.dtype not in (torch.float32, torch.float64):
        raise ValueError("x and power must both be float32 or both float64")
    batch, n0 = x.shape
    if tuple(power.shape) != (batch, int(J) + 1, n0):
        raise ValueError(f"power must have shape {(batch, int(J) + 1, n0)}")
    _shim.cwt_power_device(x.data_ptr(), batch, n0, dt, dj, s0, int(J), f0, power.data_ptr(),
                           f64=x.dtype == torch.float64,
                           stream=torch.cuda.current_stream(x.device).cuda_stream, generic_only=generic_only)
    return power


def cwt_averages_resident(x, global_out, band_out, dt, dj, s0, J, mother=_shim.MORLET, param=6.0, band=None,
                          band_factor=1.0, nfft=None):
    """Time- and scale-averaged wavelet power of a device-resident batch (wtb_cwt_averages).

    x: torch CUDA float32/float64 tensor [batch, n0].  global_out: preallocated [batch, J+1] tensor of the same
    dtype, or None; band_out: [batch, n0] or None, given together with ``band = (lo, hi)`` (scale indices,
    inclusive).  global = mean_t |W|^2, band = band_factor * sum_{s=lo..hi} |W_s|^2 / scales[s].  Runs on the
    device that owns x, enqueued on torch's current stream of that device; the power plane never exists
    outside the library's scratch.  Returns (global_out, band_out)."""
    import torch
    outs = [t for t in (global_out, band_out) if t is not None]
    if not (x.is_cuda and x.is_contiguous() and all(t.is_cuda and t.is_contiguous() for t in outs)):
        raise ValueError("x and the outputs must be contiguous CUDA tensors")
    if any(t.device != x.device for t in outs):
        raise ValueError("x and the outputs must live on the same device")
    if x.dtype not in (torch.float32, torch.float64) or any(t.dtype != x.dtype for t in outs):
        raise ValueError("x and the outputs must all be float32 or all float64")
    batch, n0 = x.shape
    if global_out is not None and tuple(global_out.shape) != (batch, int(J) + 1):
        raise ValueError(f"global_out must have shape {(batch, int(J) + 1)}")
    if band_out is not None and tuple(band_out.shape) != (batch, n0):
        raise ValueError(f"band_out must have shape {(batch, n0)}")
    _shim.cwt_averages_device(x.data_ptr(), batch, n0, dt, dj, s0, int(J), mother, param,
                              0 if global_out is None else global_out.data_ptr(),
                              0 if band_out is None else band_out.data_ptr(), band=band, band_factor=band_factor,
                              nfft=nfft, f64=x.dtype == torch.float64,
                              stream=torch.cuda.current_stream(x.device).cuda_stream)
    return global_out, band_out


def cwt_batch_resident(x, dt, dj, s0, J, f0=6.0, detrend=True, remove_mean=False, standardize=True,
                       significance_level=None):
    """Device-resident batch version of the reference's CWT request (src/wavelet_plots.py:32
    -> src/cwt.py:85): standardize_series -> ar1 -> cwt -> |W|^2 [-> power / significance].

    x: torch CUDA tensor [batch, n0] (float32 or float64).  Returns a dict of device tensors:
    ``power`` [batch, J+1, n0], ``ar1`` [batch] (NaN where pycwt.ar1 would raise), and, when
    ``significance_level`` is given, ``signif`` [batch, J+1] with ``power / signif[..., None]``
    being the ratio run_cwt returns.  Nothing leaves the GPU."""
    import torch
    if not (x.is_cuda and x.is_contiguous() and x.dtype in (torch.float32, torch.float64)):
        raise ValueError("x must be a contiguous CUDA float32/float64 tensor")
    batch, n0 = x.shape
    f64 = x.dtype == torch.float64
    stream = torch.cuda.current_stream(x.device).cuda_stream
    y = torch.empty_like(x)
    ar1 = torch.empty(batch, dtype=torch.float64, device=x.device)
    _shim.series_prep_device(x.data_ptr(), batch, n0, y.data_ptr(), ar1.data_ptr(), detrend=detrend,
                             remove_mean=remove_mean, standardize=standardize, f64=f64, stream=stream)
    Jr, scales, freqs, coi = _shim.cwt_axes(n0, dt, dj, s0, J, f0)
    power = torch.empty((batch, Jr + 1, n0), dtype=x.dtype, device=x.device)
    cwt_power_resident(y, power, dt, dj, s0, Jr, f0)
    out = {"power": power, "ar1": ar1, "scales": scales, "period": 1.0 / freqs, "coi": coi}
    if significance_level is not None:
        # pycwt.significance(1.0, dt, scales, 0, alpha): red-noise spectrum x chi2(2)/2, per series
        fl = 4 * np.pi / (f0 + np.sqrt(2 + f0 ** 2))
        freq = torch.as_tensor(dt / (scales * fl), device=x.device)[None, :]
        a = ar1[:, None]
        theor = (1 - a ** 2) / (1 + a ** 2 - 2 * a * torch.cos(2 * np.pi * freq))
        out["signif"] = (theor * (-np.log1p(-significance_level))).contiguous()
        # run_cwt's `power / signif[:, None]` plane (src/cwt.py:118-133), one streaming kernel
        out["ratio"] = ratio_planes_resident(power, out["signif"])
    return out


def ratio_planes_resident(plane, signif, want_power=False):
    """Device-resident ratio planes (wtb_ratio_planes): ``|plane| / signif[..., None]`` for a real
    CUDA tensor [batch, S, n0]; for a complex tensor ``power = |z|**2`` and ``power / signif``
    (normalize_xwt_results, src/utils/wavelet_helpers.py:60-78).  signif: float64 CUDA tensor [S]
    or [batch, S].  Returns ratio, or (power, ratio) with want_power."""
    import torch
    if not (plane.is_cuda and plane.is_contiguous() and plane.dim() == 3):
        raise ValueError("plane must be a contiguous CUDA tensor [batch, S, n0]")
    cx = plane.is_complex()
    real_dtype = {torch.float32: torch.float32, torch.float64: torch.float64, torch.complex64: torch.float32,
                  torch.complex128: torch.float64}[plane.dtype]
    batch, S, n0 = plane.shape
    sig = signif.reshape(-1, S).to(device=plane.device, dtype=torch.float64).contiguous()
    if sig.shape[0] not in (1, batch):
        raise ValueError(f"signif must have shape ({S},) or ({batch}, {S})")
    ratio = torch.empty((batch, S, n0), dtype=real_dtype, device=plane.device)
    power = torch.empty_like(ratio) if (want_power and cx) else None
    src = torch.view_as_real(plane) if cx else plane
    _shim.ratio_planes_device(src.data_ptr(), batch, S, n0, sig.data_ptr(), sig.shape[0], ratio.data_ptr(),
                              power_ptr=power.data_ptr() if power is not None else 0, complex_plane=cx,
                              f64=real_dtype == torch.float64, stream=torch.cuda.current_stream(plane.device).cuda_stream)
    return (power, ratio) if want_power else ratio


def phase_arrows_resident(phase):
    """Device-resident ``calculate_phase_difference`` (src/wct.py:143-158): (u, v) CUDA tensors."""
    import torch
    if not (phase.is_cuda and phase.is_contiguous() and phase.dtype in (torch.float32, torch.float64)):
        raise ValueError("phase must be a contiguous CUDA float32/float64 tensor")
    u, v = torch.empty_like(phase), torch.empty_like(phase)
    _shim.phase_arrows_device(phase.data_ptr(), phase.numel(), u.data_ptr(), v.data_ptr(),
                              f64=phase.dtype == torch.float64,
                              stream=torch.cuda.current_stream(phase.device).cuda_stream)
    return u, v


def wct_batch_resident(y1, y2, dt, dj, s0, J, f0=6.0, signif=None):
    """Device-resident batch version of the reference's WCT request (src/wct.py:96-140 without the
    Monte Carlo): coherence, phase arrows and -- when the thresholds ``signif`` [S] (or [batch, S])
    are given -- the ``|coherence| / signif[:, None]`` plane.  y1, y2: CUDA tensors [batch, n0],
    already normalised.  Returns a dict of device tensors; nothing leaves the GPU."""
    import torch
    if not (y1.is_cuda and y2.is_cuda and y1.is_contiguous() and y2.is_contiguous() and y1.shape == y2.shape
            and y1.dtype == y2.dtype and y1.dtype in (torch.float32, torch.float64)):
        raise ValueError("y1 and y2 must be contiguous CUDA tensors of one shape and dtype")
    batch, n0 = y1.shape
    Jr, scales, freqs, coi = _shim.cwt_axes(n0, dt, dj, s0, J, f0)
    S = Jr + 1
    wct = torch.empty((batch, S, n0), dtype=y1.dtype, device=y1.device)
    phase = torch.empty_like(wct)
    f64 = y1.dtype == torch.float64
    flags = _shim.DEVICE_PTRS | (_shim.F64 if f64 else 0)
    stream = torch.cuda.current_stream(y1.device).cuda_stream
    import ctypes as C
    _shim._check(_shim.lib().wtb_xwt_wct(C.c_void_p(y1.data_ptr()), C.c_void_p(y2.data_ptr()), batch, n0,
                                         _shim.default_nfft(n0), dt, dj, s0, Jr, f0, flags, C.c_void_p(wct.data_ptr()),
                                         C.c_void_p(phase.data_ptr()), None, C.c_void_p(stream)), "wtb_xwt_wct")
    u, v = phase_arrows_resident(phase)
    out = {"coherence": wct, "phase": phase, "phase_diff_u": u, "phase_diff_v": v, "period": 1.0 / freqs, "coi": coi,
           "scales": scales}
    if signif is not None:
        out["ratio"] = ratio_planes_resident(wct, torch.as_tensor(signif, dtype=torch.float64, device=y1.device))
    return out


def wct_hist_resident(hist, a1, a2, dt, dj, s0, J, f0, mc_first, mc_count, seed, f64=False, white=False):
    """Add the coherence histograms of realisations [mc_first, mc_first+mc_count)
    to the device int64 tensor `hist` [J+1, 1000] (bit-identical to uint64)."""
    import torch
    if not (hist.is_cuda and hist.dtype == torch.int64 and hist.is_contiguous()):
        raise ValueError("hist must be a contiguous CUDA int64 tensor")
    if tuple(hist.shape) != (int(J) + 1, _shim.NBINS):
        raise ValueError(f"hist must have shape {(int(J) + 1, _shim.NBINS)}")
    _shim.wct_mc_hist_device(a1, a2, dt, dj, s0, int(J), f0, mc_first, mc_count, seed, hist.data_ptr(),
                             f64=f64, white=white, stream=torch.cuda.current_stream(hist.device).cuda_stream)
    return hist


def reduce_histogram(hist, group=None):
    """Sum the per-rank histograms in place over the process group (the only
    collective of the whole hot path).  `hist` is a torch int64 tensor (CUDA for
    NCCL, CPU for gloo).  No-op without an initialised process group."""
    dist = _dist()
    if dist is not None and dist.get_world_size(group) > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
    return hist


def wct_significance_sharded(a1, a2, dt, dj, s0, J, significance_level=0.95, mc_count=300, seed=0,
                             f0=6.0, f64=False, white=False, group=None, hist_fn=None, device=None):
    """Monte Carlo coherence significance with realisations sharded over ranks.

    Every rank computes the histogram of its contiguous block of realisations
    (Philox streams are keyed by the GLOBAL realisation index, so the sum does
    not depend on the partition), the histograms are all-reduced, and every rank
    returns the same ``(sig95[J+1], hist[J+1,1000])``.

    ``hist_fn(first, count) -> int64 array [J+1, 1000]`` replaces the GPU kernel
    (used by the CPU gloo tests of the sharding / reduction logic)."""
    import torch
    dist = _dist()
    rank = dist.get_rank(group) if dist else 0
    world = dist.get_world_size(group) if dist else 1
    first, stop = shard_range(mc_count, rank, world)
    S = int(J) + 1
    if hist_fn is not None:
        local = np.asarray(hist_fn(first, stop - first), dtype=np.int64)
        hist = torch.from_numpy(np.ascontiguousarray(local))
        if device is not None:
            hist = hist.to(device)
    else:
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        hist = torch.zeros((S, _shim.NBINS), dtype=torch.int64, device=dev)
        if stop > first:
            wct_hist_resident(hist, a1, a2, dt, dj, s0, J, f0, first, stop - first, seed, f64=f64, white=white)
    reduce_histogram(hist, group)
    total = hist.cpu().numpy().astype(np.uint64)
    sig = significance_from_histogram(total, dt, dj, s0, J, significance_level, f0)
    return sig, total


def significance_from_histogram(hist, dt, dj, s0, J, significance_level=0.95, f0=6.0):
    """Percentile step of pycwt.wct_significance on an accumulated histogram."""
    _, maxscale = _shim.wct_mc_geometry(dt, dj, s0, int(J), f0)
    has = _shim.row_has_points(dt, dj, s0, int(J), f0)
    return _shim.wct_sig_from_hist(hist, maxscale, significance_level, has)
