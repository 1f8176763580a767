"""GPU: bench.py --dump-outputs writes the last timed step's outputs, and two runs with the same
arguments write the same numbers (every input comes from a fixed seed)."""

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]


@pytest.mark.parametrize("workload,shapes", [("wct_mc", {"sig95": (65,), "hist": (66, 1000)}),
                                             ("cwt", {"power_sample": (64, 120, 1024)})])
def test_dump_outputs_repeat_across_runs(tmp_path, workload, shapes):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--workload", workload, "--steps", "2", "--warmup", "1",
           "--realisations", "3000", "--series", "1000", "--e2e-series", "64", "--e2e-steps", "1",
           "--no-cpu", "--no-secondary", "--no-injected"]
    runs = []
    for i in range(2):
        out = tmp_path / str(i)
        proc = subprocess.run(cmd + ["--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert proc.returncode == 0, proc.stderr[-2000:]
        assert json.loads(proc.stdout)["steps"] == 2
        assert sorted(p.name for p in out.iterdir()) == sorted(f"{n}.npy" for n in shapes)
        assert sum(p.stat().st_size for p in out.iterdir()) <= 64 << 20
        runs.append({n: np.load(out / f"{n}.npy") for n in shapes})
    for name, shape in shapes.items():
        a, b = runs[0][name], runs[1][name]
        assert a.shape == shape and a.dtype in (np.float32, np.float64), (name, a.shape, a.dtype)
        assert np.isfinite(a).all() and np.array_equal(a, b), name
    if workload == "wct_mc":
        assert runs[0]["hist"].sum() > 0
