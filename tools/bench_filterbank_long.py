"""MODWT, inverse MODWT, MRA and DWT of long series (filterbank_long.cu): device rates against the HBM bound, the
continuity with the one-CTA kernels and the end-to-end façades.

    python tools/bench_filterbank_long.py [--out profiles/r3_filterbank_long.json]

* Device-resident calls (CUDA events), FP32 and FP64, db4, at 64 x 2^20 samples and 4 x 2^22 samples with J = 10
  (wavedec / waverec: level 10): wtb_modwt, wtb_imodwt, wtb_modwtmra_taps, wtb_wavedec, wtb_waverec.  Each rate
  is also given as a fraction of the HBM bound at 6.5 TB/s (BASELINE's convention) with algorithmic bytes: what
  the call must read and write once, e.g. E (n + (J+1) n) per series for the MODWT.
* Continuity, in one process and run alternately: the one-CTA generic kernel at the last length it serves against
  the long path at the next length, same wavelet (db4), J = 6 and batch.
* api.modwt.smooth_signal (db4, J = 8, 4 levels) and src.dwt.run_dwt (db4, full depth) of a 100 000-sample
  series, end to end, against the float64 oracle on one CPU core.

The card's name and power limit are read in the same run.  Prints one JSON line and writes it to --out.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

os.environ.setdefault("OMP_NUM_THREADS", "1")      # the oracle's baseline is one CPU core

import numpy as np  # noqa: E402

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

HBM = 6.5e12
SHAPES = [(64, 1 << 20), (4, 1 << 22)]
J = 10


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
    return a.elapsed_time(b) / 1e3 / iters


def _device_calls(shim, torch, batch, n, f64, wavelet="db4", J=J):
    """name -> (call, algorithmic bytes) of device-resident calls on one shape."""
    from oracle.pywt_oracle import Wavelet
    w = Wavelet(wavelet)
    lo, hi, rlo, rhi = map(np.asarray, (w.dec_lo, w.dec_hi, w.rec_lo, w.rec_hi))
    dt = torch.float64 if f64 else torch.float32
    E = 8 if f64 else 4
    s = torch.cuda.current_stream().cuda_stream
    x = torch.randn(batch, n, dtype=dt, device="cuda")
    wd = torch.empty(batch, J + 1, n, dtype=dt, device="cuda")
    xr = torch.empty(batch, n, dtype=dt, device="cuda")
    md = torch.empty_like(wd)
    lens = shim.dwt_coeff_lens(n, lo.size, J)
    total = int(lens.sum())
    pd = torch.empty(batch, total, dtype=dt, device="cuda")
    nout = shim.waverec_len(lens, lo.size)
    rd = torch.empty(batch, nout, dtype=dt, device="cuda")
    shim.modwt_device(x.data_ptr(), batch, n, lo, hi, J, wd.data_ptr(), f64=f64, stream=s)
    shim.wavedec_device(x.data_ptr(), batch, n, lo, hi, J, pd.data_ptr(), f64=f64, stream=s)
    return {
        "modwt": (lambda: shim.modwt_device(x.data_ptr(), batch, n, lo, hi, J, wd.data_ptr(), f64=f64, stream=s),
                  E * batch * (n + (J + 1) * n)),
        "imodwt": (lambda: shim.imodwt_device(wd.data_ptr(), batch, n, lo, hi, J, xr.data_ptr(), f64=f64, stream=s),
                   E * batch * ((J + 1) * n + n)),
        "modwtmra_taps": (lambda: shim.modwtmra_taps_device(wd.data_ptr(), batch, n, lo, hi, J, md.data_ptr(),
                                                            f64=f64, stream=s), E * batch * 2 * (J + 1) * n),
        "wavedec": (lambda: shim.wavedec_device(x.data_ptr(), batch, n, lo, hi, J, pd.data_ptr(), f64=f64, stream=s),
                    E * batch * (n + total)),
        "waverec": (lambda: shim.waverec_device(pd.data_ptr(), batch, lens, rlo, rhi, rd.data_ptr(), f64=f64,
                                                stream=s), E * batch * (total + nout)),
    }


def rates(shim, torch):
    out = []
    for f64 in (False, True):
        for batch, n in SHAPES:
            calls = _device_calls(shim, torch, batch, n, f64)
            for name, (fn, nbytes) in calls.items():
                sec = _events(torch, fn, 5)
                out.append({"entry": name, "precision": "fp64" if f64 else "fp32", "batch": batch, "n": n, "J": J,
                            "seconds": sec, "samples_per_s": batch * n / sec, "alg_bytes": nbytes,
                            "GB_per_s": nbytes / sec / 1e9, "frac_hbm_6p5": nbytes / sec / HBM})
            del calls
            torch.cuda.empty_cache()
    return out


def continuity(shim, torch):
    from oracle import filterbank_long as fl
    out = []
    for f64 in (False, True):
        for entry in ("modwt", "imodwt", "wavedec", "waverec"):
            n1 = fl.first_long_n(entry, f64, L=8, J=6, level=6)
            batch = 1024
            a = _device_calls(shim, torch, batch, n1 - 1, f64, J=6)[entry]
            b = _device_calls(shim, torch, batch, n1, f64, J=6)[entry]
            ta, tb = [], []
            for _ in range(5):
                ta.append(_events(torch, a[0], 3))
                tb.append(_events(torch, b[0], 3))
            ra, rb = batch * (n1 - 1) / np.median(ta), batch * n1 / np.median(tb)
            out.append({"entry": entry, "precision": "fp64" if f64 else "fp32", "batch": batch, "J": 6,
                        "one_cta": {"n": n1 - 1, "samples_per_s": ra, "frac_hbm_6p5": a[1] / np.median(ta) / HBM},
                        "long": {"n": n1, "samples_per_s": rb, "frac_hbm_6p5": b[1] / np.median(tb) / HBM},
                        "long_over_one_cta": rb / ra})
            del a, b
            torch.cuda.empty_cache()
    return out


def end_to_end():
    from oracle import filterbank_long as fl
    from oracle import modwt_oracle as mo
    from src import dwt as sdwt
    from wavelet_transformer_b200 import pywt_compat as pywt
    from wavelet_transformer_b200.api import modwt as api
    x = np.random.default_rng(5).standard_normal(100_000).cumsum()
    coeffs = api.modwt(x, "db4", 8)
    res = {}

    def best(fn, reps=3):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts)

    res["smooth_signal_100k"] = {"b200_s": best(lambda: api.smooth_signal(coeffs, "db4", 4)),
                                 "oracle_1core_s": best(lambda: mo.smooth_signal(coeffs, "db4", 4), 1)}
    w = pywt.Wavelet("db4")
    res["run_dwt_100k"] = {"b200_s": best(lambda: sdwt.run_dwt(sdwt.DataForDWT(x, w, None))),
                           "oracle_1core_s": best(lambda: fl.wavedec(x, "db4"), 1),
                           "note": "oracle: the vectorised float64 wavedec of oracle/filterbank_long.py"}
    for v in res.values():
        if "oracle_1core_s" in v:
            v["speedup"] = v["oracle_1core_s"] / v["b200_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_filterbank_long.json"))
    args = ap.parse_args()
    import torch
    from wavelet_transformer_b200 import _shim as shim
    shim.init(0)
    rec = {"tool": "tools/bench_filterbank_long.py", "card": _card(), "wavelet": "db4",
           "hbm_bound_bytes_per_s": HBM, "rates": rates(shim, torch), "continuity": continuity(shim, torch),
           "end_to_end": end_to_end()}
    line = json.dumps(rec)
    print(line)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
