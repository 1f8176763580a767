"""Host-buffer wtb_xwt_wct over several staging chunks: wall time per call, and a digest of the outputs.

    python tools/bench_xwt_host.py [--pairs 1000] [--n0 4096] [--reps 7] [--out FILE]

FP32 coherence + phase of `pairs` white-noise pairs of n0 samples (dt = 1, dj = 1/8, default s0 and J), from
NumPy arrays in pageable host memory, as pycwt_compat passes them.  At the default shape a call streams its pairs
through nine 1 GiB staging chunks (89 scales; each chunk: rows up, transforms, spectra, coherence; 2.9 GB of
planes back in all), so the time is the library's host staging loop end to end, not a kernel rate.  One warm-up
call, then `reps` timed calls (host wall clock; the call returns after its last chunk's copies, with the stream
synchronised).  The sha256 of the last call's coherence and phase planes lets two builds be compared bit for bit.

The card's name and power limit are read in the same run.  Prints one JSON line, also written to --out.
"""

from __future__ import annotations

import argparse
import hashlib
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DT, DJ = 1.0, 1 / 8


def _card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--pairs", type=int, default=1000)
    ap.add_argument("--n0", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from wavelet_transformer_b200 import _shim

    rng = np.random.default_rng(11)
    y1 = rng.standard_normal((args.pairs, args.n0)).astype(np.float32)
    y2 = rng.standard_normal((args.pairs, args.n0)).astype(np.float32)

    def call():
        return _shim.xwt_wct(y1, y2, DT, DJ, -1, -1, f64=False)

    wct, phase, _ = call()
    times = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        wct, phase, _ = call()
        times.append(time.perf_counter() - t0)
    digest = hashlib.sha256(wct.tobytes() + phase.tobytes()).hexdigest()
    line = {"card": _card(), "lib": str(_shim.lib_path()), "pairs": args.pairs, "n0": args.n0,
            "scales": int(wct.shape[1]), "fp32": True, "reps": args.reps,
            "seconds": [round(t, 4) for t in times], "median_s": round(statistics.median(times), 4),
            "min_s": round(min(times), 4), "sha256": digest}
    print(json.dumps(line))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
