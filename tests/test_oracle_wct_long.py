"""CPU: the per-row float64 reference and the host-rule replica of the long-series coherence (oracle/wct_long.py)."""

import numpy as np
import pytest

from oracle import pycwt_oracle as po
from oracle import wct_long as wl


def _pair(n0, seed):
    rng = np.random.default_rng(seed)
    a = np.cumsum(rng.standard_normal(n0)) * 0.1 + rng.standard_normal(n0)
    b = 0.6 * a + rng.standard_normal(n0)
    return a, b


@pytest.mark.parametrize("n0,dt,dj", [(3000, 1.0, 1 / 4), (2100, 1 / 12, 1 / 8)])
@pytest.mark.parametrize("which", ["ends", "middle", "every_fifth"])
def test_wct_rows_against_the_full_plane(n0, dt, dj, which):
    y1, y2 = _pair(n0, seed=n0)
    WCT, aWCT, _, _, _ = po.wct(y1, y2, dt, dj=dj, s0=-1, J=-1, sig=False)
    W12 = po.xwt(y1, y2, dt, dj=dj, s0=-1, J=-1)[0]
    S = WCT.shape[0]
    rows = {"ends": [0, 1, S - 2, S - 1], "middle": [S // 3, S // 2, S // 2 + 1],
            "every_fifth": list(range(0, S, 5)) + [S - 1]}[which]
    wct, phase, w12 = wl.wct_rows(y1, y2, dt, dj, -1, -1, rows)
    assert wct.shape == (len(rows), n0)
    assert np.abs(wct - WCT[rows]).max() <= 1e-13
    scale = np.abs(W12[rows]).max(axis=1, keepdims=True)
    assert (np.abs(w12 - W12[rows]) / scale).max() <= 1e-13
    # the phase as the phasor |W12| e^{i phi}: no wrap-around at +-pi
    got = np.abs(w12) * np.exp(1j * phase)
    ref = np.abs(W12[rows]) * np.exp(1j * aWCT[rows])
    assert (np.abs(got - ref) / scale).max() <= 1e-13


def test_boxcar_of_the_reference_scale_step():
    w, up = wl.boxcar(1 / 8)
    assert w.size == 10 and up == 4 and abs(w.sum() - 1) < 1e-15 and w[0] == w[-1] == 0.5 * w[1]


# ---- host rules -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("nfft,f64,route", [
    (8192, False, "generic"), (16384, False, "long"), (4096, True, "generic"), (8192, True, "long"),
    (1 << 22, False, "long"), (1 << 22, True, "long"), (1 << 23, False, "refused"), (1 << 23, True, "refused"),
    (12288, True, "generic"), (5000, False, "generic")])
def test_route(nfft, f64, route):
    assert wl.route(nfft, f64) == route


def test_wave_rule_at_hand_checked_shapes():
    # 64 MiB / (4 fields x 8 B x 16384) = 128 rows; 256 without smoothing; FP64 half of each
    assert wl.wave_rows(16384, False, 1000) == 128 and wl.wave_rows(16384, False, 1000, smooth=False) == 256
    assert wl.wave_rows(16384, True, 1000) == 64 and wl.wave_rows(16384, False, 50) == 50
    # one row is past 64 MiB at 2^22: still one row per wave
    assert wl.wave_rows(1 << 22, False, 17) == 1 and wl.wave_rows(1 << 21, False, 17) == 1
    assert wl.wave_rows(1 << 20, False, 164) == 2 and wl.wave_rows(1 << 20, True, 164) == 1


def test_launches_at_hand_checked_shapes():
    # one pair, 9 scales at 16384: one forward wave (2 passes), one row wave (5 or 2), the scale kernel
    assert wl.launches(16384, False, 1, 9, "plane") == 8
    assert wl.launches(16384, False, 1, 9, "hist") == 8
    assert wl.launches(16384, False, 1, 9, "w12") == 4
    # 4 pairs x 41 scales at 2^20 FP32: 8 series in one forward wave; 164 rows, 2 per wave
    assert wl.launches(1 << 20, False, 4, 41, "plane") == 2 + 5 * 82 + 1
    assert wl.launches(1 << 20, False, 4, 41, "w12") == 2 + 2 * 41
    # FP64 2^20: 4 series per forward wave, one row per wave
    assert wl.launches(1 << 20, True, 4, 41, "plane") == 2 * 2 + 5 * 164 + 1


def test_xwt_chunks_at_hand_checked_shapes():
    # 2^22 FP64 with 17 scales: one pair is past 1 GiB of intermediates, so it is a chunk of its own
    assert wl.pair_bytes(3_000_000, 1 << 22, 17, True) > 1 << 30
    assert wl.xwt_chunk_rows(3, 3_000_000, 1 << 22, 17, True) == 1
    assert wl.xwt_launches(3, 3_000_000, 1 << 22, 17, True) == 3 * wl.launches(1 << 22, True, 1, 17, "plane")
    # 64 pairs x 16384 FP32, 81 scales: 4 B x 16384 x 164 staged + 21 495 808 B of intermediates per pair,
    # 33 pairs in 1 GiB -> chunks of 33 and 31
    assert wl.xwt_chunk_rows(64, 16384, 16384, 81, False) == 33
    assert wl.xwt_launches(64, 16384, 16384, 81, False) == wl.launches(16384, False, 33, 81, "plane") + \
        wl.launches(16384, False, 31, 81, "plane")


# run_wct (dt 1/12, dj 1/8, s0 2 dt) and pycwt's defaults (dj 1/12, s0 2 dt / flambda): surrogate length and FFT
GEOMETRIES = [
    (565, 3351, 4096, 3338, 4096), (1346, 7968, 8192, 7939, 8192), (1400, 8689, 16384, 8411, 16384),
    (2000, 12288, 16384, 11895, 16384), (10_000, 58452, 65536, 59947, 65536),
    (100_000, 606_422, 1 << 20, 604_226, 1 << 20)]


def _nsurr(n0, dj, s0):
    dt = 1 / 12
    J = int(np.round(np.log2(n0 * dt / s0) / dj))
    return po.mc_geometry(dt, dj, s0, J, po.Morlet())[0]


@pytest.mark.parametrize("g", GEOMETRIES, ids=lambda g: str(g[0]))
def test_monte_carlo_geometries(g):
    n0, ns_run, nfft_run, ns_py, nfft_py = g
    dt = 1 / 12
    assert _nsurr(n0, 1 / 8, 2 * dt) == ns_run and wl.mc_nfft(ns_run) == nfft_run
    assert _nsurr(n0, 1 / 12, 2 * dt / po.Morlet().flambda()) == ns_py and wl.mc_nfft(ns_py) == nfft_py
    for ns, nfft in ((ns_run, nfft_run), (ns_py, nfft_py)):
        assert wl.route(nfft, False) == ("long" if nfft >= 16384 else "generic")
        assert wl.route(nfft, True) == ("long" if nfft >= 8192 else "generic")


def test_long_route_starts_past_the_one_cta_lengths():
    assert wl.route(wl.mc_nfft(8192), False) == "generic" and wl.route(wl.mc_nfft(8193), False) == "long"
    assert wl.route(wl.mc_nfft(4096), True) == "generic" and wl.route(wl.mc_nfft(4097), True) == "long"
