"""CPU: the parts of bench.py's contract that need no GPU -- the reference arm prints one JSON
line with the keys the driver parses, and the host helpers of the shim behave."""

import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.mark.parametrize("workload,metric,unit", [("wct_mc", "wct_mc_surrogates_per_sec", "surrogates/s"),
                                                  ("cwt", "cwt_coeffs_per_sec", "coeff/s")])
def test_reference_arm_prints_one_contract_line(workload, metric, unit):
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", workload,
                           "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == metric and line["unit"] == unit
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                           "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert proc.returncode == 0 and proc.stdout.strip() == ""


@pytest.mark.parametrize("extra,message", [(["--steps", "0"], "--steps"),
                                           (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs")])
def test_bad_arguments_are_refused(extra, message):
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                          cwd=ROOT)
    assert proc.returncode == 2 and message in proc.stderr and proc.stdout == ""


def test_fft_padding_rule_and_shard_ranges():
    from wavelet_transformer_b200 import _shim, engine
    assert _shim.get_fft_padding() == "pow2"
    assert [_shim.default_nfft(n) for n in (1, 2, 565, 1024, 1346, 4096)] == [2, 2, 1024, 1024, 2048, 4096]
    _shim.set_fft_padding("none")
    try:
        assert [_shim.default_nfft(n) for n in (1, 565, 1024, 3351)] == [2, 565, 1024, 3351]
    finally:
        _shim.set_fft_padding("pow2")
    with pytest.raises(ValueError):
        _shim.set_fft_padding("reflect")
    # strong scaling of bench.py: contiguous blocks that tile the job exactly
    for world in (1, 2, 3, 4, 8):
        parts = [engine.shard_range(100_000, r, world) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == 100_000
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
        assert max(b - a for a, b in parts) - min(b - a for a, b in parts) <= 1
