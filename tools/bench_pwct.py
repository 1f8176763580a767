"""Partial and multiple wavelet coherence (wtb_partial_wct): device time per triple, and the float64 NumPy route.

    python tools/bench_pwct.py [--out profiles/r4_pwct.json]

Shapes, each in FP32 and FP64, device-resident (WTB_DEVICE_PTRS), CUDA events around repeated calls after a
warm-up of the same shape:
  * cfg3: one triple of 565 samples, dj = 1/8 (dt = 1/12, s0 = 2 dt: 67 scales), padded to 1024;
  * batch: 1000 triples x 1346 samples x 85 scales (dj = 1/12, J = 84), padded to 2048.  Its intermediates
    (about 9.3 GB in FP32) are far past the 126 MB L2.
Each shape is also timed with only the coherence kernels' inputs in place, i.e. the CWT of the 3 x batch
series alone (wtb_cwt with a coefficient output), so that the share of the smoothing and scale passes shows.
The float64 NumPy version of one cfg3 triple (three CWTs, six smoothed spectra, the closed forms; the same
operations as the reference) is timed on one CPU core (OMP/MKL/OpenBLAS threads set to 1 before NumPy loads).
The card's name and power limit are read in the same run.  Prints one JSON line and writes it to --out.
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from pathlib import Path

for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
    os.environ[_v] = "1"

import numpy as np  # noqa: E402

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DT = 1 / 12
S0 = 2 * DT
# name, triples, n0, dj, J
SHAPES = [("cfg3", 1, 565, 1 / 8, -1), ("batch_1346", 1000, 1346, 1 / 12, 84)]


def _card():
    import torch
    rec = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        rec["nvidia_smi"] = out
    except (OSError, subprocess.SubprocessError) as e:
        rec["nvidia_smi"] = f"unavailable: {e}"
    return rec


def _events(torch, fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3


def _numpy_triple(y, x1, x2, dj, J):
    """float64 NumPy, one triple: pycwt's CWT and Morlet.smooth, then the closed forms."""
    from scipy import fft
    from scipy.signal import convolve2d
    n0 = y.size
    N = 1 << (n0 - 1).bit_length()
    sj = S0 * 2 ** (np.arange(J + 1) * dj)
    w = 2 * np.pi * fft.fftfreq(N, DT)
    daughter = (sj[:, None] * w[1] * N) ** 0.5 * np.pi ** -0.25 * np.exp(-0.5 * (sj[:, None] * w - 6) ** 2)
    W = [fft.ifft(fft.fft(v, N) * daughter, axis=1)[:, :n0] for v in (y, x1, x2)]
    k = 2 * np.pi * fft.fftfreq(N)
    gauss = np.exp(-0.5 * (sj / DT)[:, None] ** 2 * k ** 2)
    K = int(np.round(0.6 / dj * 2))
    win = np.ones(K)
    win[0] = win[-1] = 0.5
    win /= win.sum()

    def smooth(a):
        T = fft.ifft(gauss * fft.fft(a / sj[:, None], n=N, axis=1), axis=1)[:, :n0]
        return convolve2d(T, win[:, None], "same")

    Syy, S11, S22 = (smooth(np.abs(v) ** 2).real for v in W)
    Sy1, Sy2, S12 = smooth(W[0] * W[1].conj()), smooth(W[0] * W[2].conj()), smooth(W[1] * W[2].conj())
    num = Sy1 * S22 - Sy2 * S12.conj()
    d12 = S11 * S22 - np.abs(S12) ** 2
    pwc = np.abs(num) ** 2 / ((Syy * S22 - np.abs(Sy2) ** 2) * d12)
    mwc = (np.abs(Sy1) ** 2 * S22 + np.abs(Sy2) ** 2 * S11 - 2 * np.real(Sy1 * Sy2.conj() * S12)) / (Syy * d12)
    return pwc, np.angle(num), mwc


def run_shape(shim, torch, name, triples, n0, dj, J, f64, iters):
    Jr, _, _, _ = shim.cwt_axes(n0, DT, dj, S0, J)
    S = Jr + 1
    nfft = shim.next_pow2(n0)
    dtype = torch.float64 if f64 else torch.float32
    g = torch.Generator("cuda").manual_seed(n0)
    ys = [torch.randn(triples, n0, dtype=dtype, device="cuda", generator=g) for _ in range(3)]
    outs = [torch.empty(triples, S, n0, dtype=dtype, device="cuda") for _ in range(3)]
    stacked = torch.stack(ys, dim=1).reshape(3 * triples, n0).contiguous()
    coef = torch.empty(3 * triples, S, n0, dtype=torch.complex128 if f64 else torch.complex64, device="cuda")
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib = shim.lib()

    def pwct():
        rc = lib.wtb_partial_wct(*(ptr(v) for v in ys), triples, n0, nfft, DT, dj, S0, Jr, 6.0, flags,
                                 *(ptr(o) for o in outs), stream)
        assert rc == 0, lib.wtb_last_error()

    def cwt_only():
        rc = lib.wtb_cwt(ptr(stacked), 3 * triples, n0, nfft, DT, dj, S0, Jr, shim.MORLET, 6.0, flags, None,
                         ptr(coef), stream)
        assert rc == 0, lib.wtb_last_error()

    before = shim.kernel_launches()
    pwct()
    torch.cuda.synchronize()
    launches = shim.kernel_launches() - before
    # alternate the two, twice, and keep the faster of each
    t_p = t_c = float("inf")
    for _ in range(2):
        t_p = min(t_p, _events(torch, pwct, iters))
        t_c = min(t_c, _events(torch, cwt_only, iters))
    rec = {"shape": name, "precision": "fp64" if f64 else "fp32", "triples": triples, "n0": n0, "S": S, "nfft": nfft,
           "launches_per_call": launches, "call_ms": t_p * 1e3, "per_triple_us": t_p / triples * 1e6,
           "cwt_of_the_3_series_ms": t_c * 1e3, "smooth_and_scale_share": (t_p - t_c) / t_p,
           "points_per_s": triples * S * n0 / t_p}
    if triples > 1:
        rec.update(_kernel_times(torch, pwct, triples * S * n0, 8 if f64 else 4))
    del ys, outs, stacked, coef
    torch.cuda.empty_cache()
    return rec


def _kernel_times(torch, fn, points, elem):
    """Per-kernel device time of one call (torch.profiler, a separate run from the timed one), and the
    bandwidth the scale pass reaches: it reads the nine smoothed planes (each row again for every boxcar tap,
    counted once here) and writes three.  Near the HBM rate, its double-precision arithmetic is not what
    bounds it."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("wtb::", "")
            per[name] = per.get(name, 0.0) + e.device_time_total * 1e-3
    scale_ms = sum(v for k, v in per.items() if "k_pwct_scale" in k)
    return {"kernel_ms": per, "scale_pass_min_bytes": 12 * elem * points,
            "scale_pass_GB_per_s": 12 * elem * points / (scale_ms * 1e-3) / 1e9 if scale_ms else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_pwct.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_pwct needs a GPU: nothing is measured on the CPU")
    from wavelet_transformer_b200 import _shim
    _shim.init(0)
    out = {"card": _card(), "shapes": []}
    for name, triples, n0, dj, J in SHAPES:
        for f64 in (False, True):
            out["shapes"].append(run_shape(_shim, torch, name, triples, n0, dj, J, f64,
                                           args.iters if triples == 1 else max(3, args.iters // 4)))
    rng = np.random.default_rng(0)
    y, x1, x2 = rng.standard_normal((3, 565))
    Jr, _, _, _ = _shim.cwt_axes(565, DT, 1 / 8, S0, -1)
    _numpy_triple(y, x1, x2, 1 / 8, Jr)
    best = float("inf")
    for _ in range(5):
        t0 = time.perf_counter()
        _numpy_triple(y, x1, x2, 1 / 8, Jr)
        best = min(best, time.perf_counter() - t0)
    out["numpy_fp64_cfg3_one_core_ms"] = best * 1e3
    cfg3 = [r for r in out["shapes"] if r["shape"] == "cfg3"]
    out["cfg3_speedup_over_numpy"] = {r["precision"]: best / (r["call_ms"] * 1e-3) for r in cfg3}
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
