"""The CWT of long series (cwt_long.cu): rates, bounds and the continuity with the one-CTA kernels.

    python tools/bench_cwt_long.py [--out profiles/r3_cwt_long.json]

* FP32 device-resident power (engine.cwt_power_resident, CUDA events) at 256 x 16 384, 16 x 2^20 and
  2 x 2^22 samples, dt = 1, dj = 1/12, default s0 and J.  For each: coeff/s; the share of the FP32-flop bound
  (BASELINE's convention: 5 N log2 N (1 + S) flop per series at the nominal 74.4 TFLOP/s) and of the HBM bound
  (4 n0 (1 + S) bytes per series at 6.5 TB/s); and the HBM bytes this design moves, from the shapes (below).
* The drop-in FP64 pycwt_compat.cwt of one 10 000-sample series, end to end, against the float64 oracle
  (NumPy's FFT on one CPU core, oracle/pycwt_oracle.py).
* Continuity, in the same process: coeff/s of the long path at FP32 nfft 16384 / FP64 8192 against the one-CTA
  generic kernel at FP32 8192 / FP64 4096, with the batch sized for about 2.5 G coefficients per call.

Traffic this design moves per series (bytes, E = sizeof(complex)): forward: x read (4 n0), X^ written (E N); per
scale row: X^ read by pass 1 (E N), power written by pass 2 (4 n0).  The intermediate of a wave stays in L2 by
construction (64 MiB of 126 MB), so it is not counted; where an X^ row (E N) stays in L2 across its S rows the
real figure is lower.  The card's name and power limit are read in the same run.  Prints one JSON line and
writes it to --out.
"""

from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DT, DJ = 1.0, 1 / 12
FP32_PEAK = 148 * 128 * 2 * 1.965e9          # BASELINE.md: nominal non-tensor FP32 peak
HBM_PEAK = 6547e9                             # BASELINE.md: measured HBM rate
SHAPES = [(256, 16384), (16, 1 << 20), (2, 1 << 22)]


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


def _power_rate(shim, engine, torch, batch, n0, f64, iters, generic_only=False):
    J = shim.cwt_axes(n0, DT, DJ, -1, -1)[0]
    S = J + 1
    dtype = torch.float64 if f64 else torch.float32
    x = torch.randn(batch, n0, dtype=dtype, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    power = torch.empty((batch, S, n0), dtype=dtype, device="cuda")
    launches = shim.kernel_launches()
    engine.cwt_power_resident(x, power, DT, DJ, -1, J, generic_only=generic_only)
    torch.cuda.synchronize()
    rec = {"batch": batch, "n0": n0, "nfft": 1 << (n0 - 1).bit_length(), "S": S, "precision": "fp64" if f64 else "fp32",
           "launches_per_call": shim.kernel_launches() - launches}
    t = _events(torch, lambda: engine.cwt_power_resident(x, power, DT, DJ, -1, J, generic_only=generic_only), iters)
    coeffs = batch * S * n0
    rec.update(time_ms=t * 1e3, coeff_per_s=coeffs / t)
    del x, power
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_cwt_long.json"))
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cwt_long needs a GPU: nothing is measured on the CPU")
    from oracle import pycwt_oracle as po
    from wavelet_transformer_b200 import _shim, engine, pycwt_compat
    _shim.init(0)
    out = {"card": _card(), "dt": DT, "dj": DJ, "fp32_peak_flops": FP32_PEAK, "hbm_peak_bytes_per_s": HBM_PEAK,
           "shapes": [], "continuity": []}
    for batch, n0 in SHAPES:
        rec = _power_rate(_shim, engine, torch, batch, n0, False, args.iters)
        N, S = rec["nfft"], rec["S"]
        flop = batch * 5 * N * math.log2(N) * (1 + S)
        hbm_min = batch * 4 * n0 * (1 + S)
        moved = batch * ((4 * n0 + 8 * N) + S * (8 * N + 4 * n0))
        t = rec["time_ms"] * 1e-3
        rec.update(flop_bound_share=flop / FP32_PEAK / t, hbm_bound_share=hbm_min / HBM_PEAK / t,
                   hbm_bytes_min=hbm_min, hbm_bytes_design=moved, design_bytes_at_hbm_peak_share=moved / HBM_PEAK / t)
        out["shapes"].append(rec)
        print(json.dumps(rec), flush=True)

    # continuity: long path just past the one-CTA limit against the generic kernel at the limit
    for f64, n_gen, n_long in ((False, 8192, 16384), (True, 4096, 8192)):
        for n0, path in ((n_gen, "generic"), (n_long, "long")):
            S = _shim.cwt_axes(n0, DT, DJ, -1, -1)[0] + 1
            batch = max(1, int(2.5e9 // (S * n0)) // (2 if f64 else 1))
            rec = _power_rate(_shim, engine, torch, batch, n0, f64, args.iters, generic_only=path == "generic")
            rec["path"] = path
            out["continuity"].append(rec)
            print(json.dumps(rec), flush=True)
    for f64 in (False, True):
        pair = [r for r in out["continuity"] if (r["precision"] == "fp64") == f64]
        g, l = (pair[0], pair[1])
        out[f"continuity_ratio_{'fp64' if f64 else 'fp32'}"] = l["coeff_per_s"] / g["coeff_per_s"]

    # drop-in FP64 pycwt_compat.cwt of one 10 000-sample series against the float64 oracle on one CPU core
    x = np.random.default_rng(1).standard_normal(10000)
    pycwt_compat.cwt(x, 1.0, 1 / 12, -1, -1, "morlet")
    best_e = best_o = float("inf")
    for _ in range(5):
        t0 = time.perf_counter()
        W = pycwt_compat.cwt(x, 1.0, 1 / 12, -1, -1, "morlet")[0]
        best_e = min(best_e, time.perf_counter() - t0)
        t0 = time.perf_counter()
        Wr = po.cwt(x, 1.0, 1 / 12, -1, -1, po.Morlet(6))[0]
        best_o = min(best_o, time.perf_counter() - t0)
    out["pycwt_compat_fp64_10000"] = {"S": int(W.shape[0]), "engine_s": best_e, "oracle_numpy_s": best_o,
                                      "speedup": best_o / best_e,
                                      "max_abs_diff_over_max": float(np.abs(W - Wr).max() / np.abs(Wr).max())}
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
