"""Monte-Carlo significance of partial and multiple coherence (wtb_partial_wct_mc_hist): device time of a
300-realisation job, and the float64 NumPy route.

    python tools/bench_pwct_mc.py [--out profiles/r5_pwct_mc.json]

cfg3 geometry (dt = 1/12, dj = 1/8, s0 = 2 dt, J = 65: 3351-sample surrogate triples, padded to 4096, 66 scales),
300 realisations, device RNG, in FP32 and FP64:
  * device time of one job, histogram in device memory (WTB_DEVICE_PTRS), CUDA events around repeated calls after
    a warm-up of the same call;
  * the one-call entry (wtb_partial_wct_significance: host histogram, percentile step), host wall clock;
  * the device time per kernel of one job (torch.profiler, a separate run from the timed one).
The float64 oracle (oracle/pwct_mc_oracle.py: pycwt's CWT and Morlet.smooth, the closed forms, the reliable-region
samples) is timed on a few realisations on one CPU core and extrapolated to 300 (labelled as such).  The card's
name and power limit are read in the same run.  Prints one JSON line and writes it to --out.
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
DJ, S0, J = 1 / 8, 2 * DT, 65
COEFS = (0.72, 0.65, 0.58)
MC = 300
SEED = 2024


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


def _kernel_times(torch, fn):
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


def run(shim, torch, f64, iters):
    S = J + 1
    hist = torch.zeros(2 * S * shim.NBINS, dtype=torch.int64, device="cuda")
    flags = shim.DEVICE_PTRS | (shim.F64 if f64 else 0)
    lib = shim.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def job():
        rc = lib.wtb_partial_wct_mc_hist(*COEFS, DT, DJ, S0, J, 6.0, 0, MC, SEED, None, flags,
                                         C.c_void_p(hist.data_ptr()), stream)
        assert rc == 0, lib.wtb_last_error()

    before = shim.kernel_launches()
    job()
    torch.cuda.synchronize()
    launches = shim.kernel_launches() - before
    t_dev = min(_events(torch, job, iters) for _ in range(2))
    hist.zero_()
    job()
    host = shim.partial_wct_mc_hist(*COEFS, DT, DJ, S0, J, mc_count=MC, seed=SEED, f64=f64)
    same = bool(np.array_equal(hist.cpu().numpy().astype(np.uint64).reshape(host.shape), host))
    shim.partial_wct_significance(*COEFS, DT, DJ, S0, J, mc_count=MC, seed=SEED, f64=f64)
    walls = []
    for _ in range(5):
        t0 = time.perf_counter()
        shim.partial_wct_significance(*COEFS, DT, DJ, S0, J, mc_count=MC, seed=SEED, f64=f64)
        walls.append(time.perf_counter() - t0)
    return {"precision": "fp64" if f64 else "fp32", "realisations": MC, "launches_per_job": launches,
            "device_ms_per_job": t_dev * 1e3, "us_per_realisation": t_dev / MC * 1e6,
            "one_call_significance_wall_ms_min": min(walls) * 1e3,
            "device_histogram_equals_host_call": same, "hist_total": int(host.sum()),
            "kernel_ms_one_job": _kernel_times(torch, job)}


def oracle_time(shim, count):
    from oracle import pwct_mc_oracle as pmo
    from oracle import pycwt_oracle as po
    N, *_ = po.mc_geometry(DT, DJ, S0, J, po.Morlet())
    sur = pmo.device_surrogate_triples(*COEFS, N, 0, count + 1, SEED)
    pmo.partial_coherence_samples(*sur[0], DT, DJ, S0, J)
    t0 = time.perf_counter()
    for t in sur[1:]:
        pmo.partial_coherence_samples(*t, DT, DJ, S0, J)
    per = (time.perf_counter() - t0) / count
    return {"realisations_timed": count, "s_per_realisation": per,
            "extrapolated_s_for_300": per * MC,
            "note": "float64 NumPy on one core (threads set to 1), timed on the realisations above and "
                    "extrapolated linearly to 300: not measured at 300"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r5_pwct_mc.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--oracle-realisations", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_pwct_mc needs a GPU: nothing is measured on the CPU")
    from wavelet_transformer_b200 import _shim
    _shim.init(0)
    nsurr, maxscale = _shim.wct_mc_geometry(DT, DJ, S0, J)
    out = {"card": _card(),
           "geometry": {"dt": DT, "dj": DJ, "s0": S0, "J": J, "nsurr": nsurr, "nfft": _shim.next_pow2(nsurr),
                        "maxscale": maxscale, "coefficients": COEFS, "seed": SEED},
           "runs": [run(_shim, torch, f64, args.iters) for f64 in (False, True)],
           "oracle": oracle_time(_shim, args.oracle_realisations)}
    fp32 = out["runs"][0]["device_ms_per_job"] * 1e-3
    out["speedup_fp32_over_extrapolated_oracle"] = out["oracle"]["extrapolated_s_for_300"] / fp32
    print(json.dumps(out))
    path = Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
