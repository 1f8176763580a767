"""Time- and scale-averaged wavelet power (wtb_cwt_averages) against the routes a user has without it.

    python tools/bench_cwt_averages.py [--out profiles/r3_cwt_averages.json]

Two shapes, FP32: 16 384 series x 1024 samples x 120 scales (the nfft-1024 warp kernel) and 4096 series of
cfg1's 1346 samples x 85 scales (nfft 2048).  The band is the pycwt sample's 2-8 year periods (dt = 1/12).
For each shape:
  * host buffers, end to end: wtb_cwt_averages against wtb_cwt_morlet's power plane copied to the host
    plus a NumPy float64 reduction (the plane is 8 GB / 2 GB, far past the 126 MB L2 and any host cache);
  * device only, CUDA events: engine.cwt_averages_resident against engine.cwt_power_resident alone, the
    difference being the cost of the second pass over the plane.
Rates are power coefficients (batch x S x n0) per second.  The card's name and power limit are read in the
same run and written beside the numbers.  Prints one JSON line and writes it to --out.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DT = 1 / 12
SHAPES = [("fast1024", 16384, 1024, 1 / 12, 119), ("cfg1_1346", 4096, 1346, 1 / 12, 84)]


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


def _band(shim, n0, dj, J):
    _, sj, freqs, _ = shim.cwt_axes(n0, DT, dj, 2 * DT, J)
    period = 1 / freqs
    sel = np.nonzero((period >= 2) & (period < 8))[0]
    return (int(sel[0]), int(sel[-1])), sj


def _wall(fn, reps):
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


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


def run_shape(shim, engine, torch, name, batch, n0, dj, J, reps, iters):
    S = J + 1
    band, sj = _band(shim, n0, dj, J)
    lo, hi = band
    factor = dj * DT / 0.776
    x = np.random.default_rng(0).standard_normal((batch, n0)).astype(np.float32)
    coeffs = batch * S * n0
    rec = {"shape": name, "batch": batch, "n0": n0, "S": S, "band": band, "coeffs": coeffs}

    # host buffers, end to end (warm-up on a small batch of the same shape: modules, tables, scratch)
    shim.cwt_averages(x[:64], DT, dj, 2 * DT, J, band=band, band_factor=factor, f64=False)
    shim.cwt_morlet(x[:64], DT, dj, 2 * DT, J, f64=False)
    t_avg = _wall(lambda: shim.cwt_averages(x, DT, dj, 2 * DT, J, band=band, band_factor=factor, f64=False), reps)
    holder = {}

    def plane():
        holder["p"], _ = shim.cwt_morlet(x, DT, dj, 2 * DT, J, f64=False)

    def reduce():
        p = holder["p"]
        g = p.mean(axis=2, dtype=np.float64)
        b = factor * np.einsum("bst,s->bt", p[:, lo:hi + 1].astype(np.float64), 1.0 / sj[lo:hi + 1])
        return g, b

    t_plane = _wall(plane, reps)
    t_red = _wall(reduce, reps)
    g_host, b_host = reduce()
    g_dev, b_dev = shim.cwt_averages(x[:8], DT, dj, 2 * DT, J, band=band, band_factor=factor, f64=False)
    rec["host_max_rel_diff_first8"] = float(max(np.abs(g_dev - g_host[:8]).max() / np.abs(g_host[:8]).max(),
                                                np.abs(b_dev - b_host[:8]).max() / np.abs(b_host[:8]).max()))
    holder.clear()
    rec["host_averages_s"] = t_avg
    rec["host_plane_s"] = t_plane
    rec["host_numpy_reduce_s"] = t_red
    rec["host_averages_coeff_per_s"] = coeffs / t_avg
    rec["host_plane_plus_numpy_coeff_per_s"] = coeffs / (t_plane + t_red)
    rec["host_speedup"] = (t_plane + t_red) / t_avg

    # device only
    xd = torch.as_tensor(x, device="cuda")
    power = torch.empty((batch, S, n0), dtype=torch.float32, device="cuda")
    gd = torch.empty((batch, S), dtype=torch.float32, device="cuda")
    bd = torch.empty((batch, n0), dtype=torch.float32, device="cuda")
    t_pow = _events(torch, lambda: engine.cwt_power_resident(xd, power, DT, dj, 2 * DT, J), iters)
    t_both = _events(torch, lambda: engine.cwt_averages_resident(xd, gd, bd, DT, dj, 2 * DT, J, band=band,
                                                                 band_factor=factor), iters)
    rec["device_power_ms"] = t_pow * 1e3
    rec["device_averages_ms"] = t_both * 1e3
    rec["device_second_pass_ms"] = (t_both - t_pow) * 1e3
    rec["device_second_pass_share"] = (t_both - t_pow) / t_pow
    rec["device_averages_coeff_per_s"] = coeffs / t_both
    rec["plane_bytes"] = 4 * coeffs
    del power, xd, gd, bd
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_cwt_averages.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cwt_averages needs a GPU: nothing is measured on the CPU")
    from wavelet_transformer_b200 import _shim, engine
    _shim.init(0)
    out = {"card": _card(), "precision": "fp32", "shapes": []}
    for shape in SHAPES:
        out["shapes"].append(run_shape(_shim, engine, torch, *shape, args.reps, args.iters))
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
