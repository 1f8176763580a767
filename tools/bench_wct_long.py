"""Cross spectra, coherence and Monte-Carlo significance of long series (wct_long.cu): rates, kernel shares and the
continuity with the one-CTA kernels.

    python tools/bench_wct_long.py [--out profiles/r3_wct_long.json]

* Device-resident wtb_xwt_wct (coherence + phase), FP32 and FP64, at 64 x 16 384 and 4 x 2^20 samples, dt = 1,
  dj = 1/12, default s0 and J (CUDA events): coherence values per second.
* Continuity, in the same process: the long path at FP32 nfft 16384 / FP64 8192 against the one-CTA generic
  kernels at FP32 8192 / FP64 4096, with the batch sized for about 0.5 G coherence values per call.
* wtb_wct_mc_hist with the FP32 device RNG at run_wct's geometry (dt 1/12, dj 1/8, s0 2 dt) for 2000 and 10 000
  samples (12 288- and 58 452-sample surrogates): realisations per second (CUDA events), and each kernel's share
  of the device time from torch.profiler in a separate run, k_wct_scale<T,1> (one global atomic per sample)
  named on its own.
* pycwt_compat.wct(sig=True, mc_count=300, cache=False) of 2000- and 10 000-sample pairs, end to end.

The card's name and power limit are read in the same run.  Prints one JSON line and writes it to --out.
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from collections import defaultdict
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DT, DJ = 1.0, 1 / 12
SHAPES = [(64, 16384), (4, 1 << 20)]
MC_DT, MC_DJ = 1 / 12, 1 / 8
MC_CASES = [(2000, 200), (10_000, 40)]        # (series length run_wct sees, realisations per timed call)


def _card():
    import torch
    rec = {"device": torch.cuda.get_device_name(0)}
    try:
        rec["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                                           timeout=60).stdout.strip()
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


def _wct_rate(shim, torch, batch, n0, f64, iters, generic_only=False):
    J = shim.cwt_axes(n0, DT, DJ, -1, -1)[0]
    S = J + 1
    dtype = torch.float64 if f64 else torch.float32
    g = torch.Generator("cuda").manual_seed(0)
    y1 = torch.randn(batch, n0, dtype=dtype, device="cuda", generator=g)
    y2 = torch.randn(batch, n0, dtype=dtype, device="cuda", generator=g)
    wct = torch.empty((batch, S, n0), dtype=dtype, device="cuda")
    phase = torch.empty_like(wct)
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0) | (shim.GENERIC_ONLY if generic_only else 0)
    stream = torch.cuda.current_stream().cuda_stream
    nfft = 1 << (n0 - 1).bit_length()

    def call():
        rc = shim.lib().wtb_xwt_wct(C.c_void_p(y1.data_ptr()), C.c_void_p(y2.data_ptr()), batch, n0, nfft, DT, DJ,
                                    -1.0, J, 6.0, flags, C.c_void_p(wct.data_ptr()), C.c_void_p(phase.data_ptr()),
                                    None, C.c_void_p(stream))
        assert rc == 0, shim.lib().wtb_last_error()

    launches = shim.kernel_launches()
    call()
    torch.cuda.synchronize()
    rec = {"batch": batch, "n0": n0, "nfft": nfft, "S": S, "precision": "fp64" if f64 else "fp32",
           "launches_per_call": shim.kernel_launches() - launches}
    t = _events(torch, call, iters)
    rec.update(time_ms=t * 1e3, values_per_s=batch * S * n0 / t)
    del y1, y2, wct, phase
    torch.cuda.empty_cache()
    return rec


def _mc_geometry(shim, n0):
    s0 = 2 * MC_DT
    J = int(np.round(np.log2(n0 * MC_DT / s0) / MC_DJ))
    nsurr, maxscale = shim.wct_mc_geometry(MC_DT, MC_DJ, s0, J)
    return s0, J, nsurr


def _mc_rate(shim, torch, n0, count, iters):
    s0, J, nsurr = _mc_geometry(shim, n0)
    hist = torch.zeros((J + 1, shim.NBINS), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    call = lambda: shim.wct_mc_hist_device(0.72, 0.55, MC_DT, MC_DJ, s0, J, 6.0, 0, count, 7, hist.data_ptr(),
                                           f64=False, stream=stream)
    t = _events(torch, call, iters)
    rec = {"n0": n0, "nsurr": nsurr, "nfft": 1 << (nsurr - 1).bit_length(), "S": J + 1, "realisations": count,
           "time_ms": t * 1e3, "realisations_per_s": count / t}
    # kernel shares, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    dev = defaultdict(float)
    for e in prof.key_averages():
        d = getattr(e, "device_time_total", None)
        if d is None:
            d = getattr(e, "cuda_time_total", 0.0)
        if d and e.key not in ("Memset (Device)",) and not e.key.startswith("Memcpy"):
            dev[e.key] += d
    total = sum(dev.values()) or 1.0
    shares = {k: v / total for k, v in sorted(dev.items(), key=lambda kv: -kv[1])}
    rec["kernel_shares"] = shares
    rec["k_wct_scale_hist_share"] = sum(v for k, v in shares.items() if "k_wct_scale" in k)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_wct_long.json"))
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_wct_long needs a GPU: nothing is measured on the CPU")
    from wavelet_transformer_b200 import _shim, pycwt_compat
    _shim.init(0)
    out = {"card": _card(), "dt": DT, "dj": DJ, "shapes": [], "continuity": [], "mc": [], "e2e": []}
    for f64 in (False, True):
        for batch, n0 in SHAPES:
            rec = _wct_rate(_shim, torch, batch, n0, f64, args.iters)
            out["shapes"].append(rec)
            print(json.dumps(rec), flush=True)

    for f64, n_gen, n_long in ((False, 8192, 16384), (True, 4096, 8192)):
        for n0, path in ((n_gen, "generic"), (n_long, "long")):
            S = _shim.cwt_axes(n0, DT, DJ, -1, -1)[0] + 1
            batch = max(1, int(0.5e9 // (S * n0)) // (2 if f64 else 1))
            rec = _wct_rate(_shim, torch, batch, n0, f64, args.iters, generic_only=path == "generic")
            rec["path"] = path
            out["continuity"].append(rec)
            print(json.dumps(rec), flush=True)
    for f64 in (False, True):
        g, l = [r for r in out["continuity"] if (r["precision"] == "fp64") == f64]
        out[f"continuity_ratio_{'fp64' if f64 else 'fp32'}"] = l["values_per_s"] / g["values_per_s"]

    for n0, count in MC_CASES:
        rec = _mc_rate(_shim, torch, n0, count, max(2, args.iters // 2))
        out["mc"].append(rec)
        print(json.dumps({k: v for k, v in rec.items() if k != "kernel_shares"}), flush=True)

    rng = np.random.default_rng(1)
    for n0 in (2000, 10_000):
        y1 = np.cumsum(rng.standard_normal(n0)) * 0.05 + rng.standard_normal(n0)
        y2 = 0.5 * y1 + rng.standard_normal(n0)
        pycwt_compat.wct(y1, y2, 1 / 12, 1 / 8, 2 / 12, -1, sig=True, mc_count=300, cache=False, progress=False)
        best = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            pycwt_compat.wct(y1, y2, 1 / 12, 1 / 8, 2 / 12, -1, sig=True, mc_count=300, cache=False, progress=False)
            best = min(best, time.perf_counter() - t0)
        rec = {"n0": n0, "mc_count": 300, "seconds": best}
        out["e2e"].append(rec)
        print(json.dumps(rec), flush=True)
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
