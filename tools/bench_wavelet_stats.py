"""MODWT wavelet variance and cross-covariance (wtb_modwt_wavelet_stats): device time per call and per kernel, the
share of the HBM bound, and the float64 NumPy route.

    python tools/bench_wavelet_stats.py [--out profiles/r6_wavelet_stats.json]

Shapes, each in FP32 and FP64, sym4:
  * cfg: one pair of 1333 samples, J = 6, K = 36, end to end from host buffers (host clock around the synchronous
    call, best of many);
  * batch: 10 000 pairs x 1333 samples, J = 6, K = 36, device-resident (WTB_DEVICE_PTRS), CUDA events;
  * long: one pair of 2^22 samples, J = 10, K = 256, device-resident, CUDA events.
Per-kernel device time comes from torch.profiler in a separate run of one call.  The HBM bound counts the bytes the
two passes must move per pair: the MODWT reads x and y and writes 2 (J+1) n samples, the reduction reads the 2 J
detail rows once; against 7.7 TB/s (the HGX B200 data sheet figure for one GPU).  The float64 oracle
(oracle/wavelet_stats_oracle.py) of the cfg pair is timed on one CPU core.  The card's name and power limit are
read in the same run.  Prints one JSON line and writes it to --out.
"""

from __future__ import annotations

import argparse
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

HBM_BYTES_PER_S = 7.7e12
# name, pairs, n, J, K, host buffers
SHAPES = [("cfg", 1, 1333, 6, 36, True), ("batch", 10000, 1333, 6, 36, False), ("long", 1, 1 << 22, 10, 256, False)]


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


def _kernel_ms(torch, fn):
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
    return per


def run_shape(shim, torch, name, pairs, n, J, K, host, f64, iters):
    from wavelet_transformer_b200 import pywt_compat as pywt
    w = pywt.Wavelet("sym4")
    elem = 8 if f64 else 4
    dtype = torch.float64 if f64 else torch.float32
    gen = torch.Generator("cuda").manual_seed(n)
    x, y = (torch.randn(pairs, n, dtype=dtype, device="cuda", generator=gen).cumsum(1) * 0.01 +
            torch.randn(pairs, n, dtype=dtype, device="cuda", generator=gen) for _ in range(2))
    outs = [torch.empty(pairs, J, dtype=torch.float64, device="cuda") for _ in range(2)]
    outs.append(torch.empty(pairs, J, 2 * K + 1, dtype=torch.float64, device="cuda"))
    stream = torch.cuda.current_stream().cuda_stream

    def device_call():
        shim.modwt_wavelet_stats_device(x.data_ptr(), y.data_ptr(), pairs, n, w.dec_lo, w.dec_hi, J, K,
                                        *(o.data_ptr() for o in outs), f64=f64, stream=stream)

    xh, yh = x.cpu().numpy(), y.cpu().numpy()

    def host_call():
        shim.modwt_wavelet_stats(xh, yh, w.dec_lo, w.dec_hi, J, K, f64=f64)

    before = shim.kernel_launches()
    device_call()
    torch.cuda.synchronize()
    launches = shim.kernel_launches() - before
    rec = {"shape": name, "precision": "fp64" if f64 else "fp32", "pairs": pairs, "n": n, "J": J, "K": K,
           "launches_per_call": launches}
    t_dev = min(_events(torch, device_call, iters) for _ in range(3))
    rec["device_call_ms"] = t_dev * 1e3
    if host:
        host_call()
        best = float("inf")
        for _ in range(200):
            t0 = time.perf_counter()
            host_call()
            best = min(best, time.perf_counter() - t0)
        rec["host_buffers_call_ms"] = best * 1e3
    per = _kernel_ms(torch, device_call)
    modwt_ms = sum(v for k, v in per.items() if "modwt" in k)
    red_ms = sum(v for k, v in per.items() if k.startswith("k_wstats"))
    rec["kernel_ms"] = per
    rec["modwt_pass_ms"], rec["reduction_pass_ms"] = modwt_ms, red_ms
    b_modwt = pairs * 2 * (n + (J + 1) * n) * elem
    b_red = pairs * 2 * J * n * elem
    rec["min_bytes_modwt_pass"], rec["min_bytes_reduction_pass"] = b_modwt, b_red
    rec["hbm_bound_share_call"] = (b_modwt + b_red) / HBM_BYTES_PER_S / t_dev
    if modwt_ms:
        rec["hbm_bound_share_modwt_pass"] = b_modwt / HBM_BYTES_PER_S / (modwt_ms * 1e-3)
    if red_ms:
        rec["hbm_bound_share_reduction_pass"] = b_red / HBM_BYTES_PER_S / (red_ms * 1e-3)
        rec["reduction_dfma_per_s"] = pairs * J * n * (2 * K + 3) / (red_ms * 1e-3)
    del x, y, outs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r6_wavelet_stats.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_wavelet_stats needs a GPU: nothing is measured on the CPU")
    from wavelet_transformer_b200 import _shim
    _shim.init(0)
    out = {"card": _card(), "hbm_bytes_per_s_assumed": HBM_BYTES_PER_S, "shapes": []}
    for name, pairs, n, J, K, host in SHAPES:
        for f64 in (False, True):
            out["shapes"].append(run_shape(_shim, torch, name, pairs, n, J, K, host, f64,
                                           args.iters if pairs * n < 10 ** 6 else max(3, args.iters // 4)))
    from oracle import wavelet_stats_oracle as wo
    rng = np.random.default_rng(0)
    x, y = rng.standard_normal((2, 1333))
    wo.stats(x, y, "sym4", 6, 36)
    best = float("inf")
    for _ in range(5):
        t0 = time.perf_counter()
        wo.stats(x, y, "sym4", 6, 36)
        best = min(best, time.perf_counter() - t0)
    out["oracle_fp64_cfg_one_core_ms"] = best * 1e3
    cfg = [r for r in out["shapes"] if r["shape"] == "cfg"]
    out["cfg_host_call_speedup_over_oracle"] = {r["precision"]: best / (r["host_buffers_call_ms"] * 1e-3) for r in cfg}
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
