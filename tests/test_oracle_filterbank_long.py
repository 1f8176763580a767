"""CPU: the vectorised float64 references of oracle/filterbank_long.py against the pinned per-output ones, and the
replica of the long filterbank path's route and wave rules."""

import numpy as np
import pytest

from oracle import filterbank_long as fl
from oracle import modwt_oracle as mo
from oracle import pywt_oracle as po

WAVELETS = ["haar", "db2", "db4", "sym4", "db5"]


@pytest.mark.parametrize("wavelet", WAVELETS)
@pytest.mark.parametrize("n", [1, 2, 7, 64, 257, 1001])
def test_dwt_pair_equals_pywt_oracle(wavelet, n):
    x = np.random.default_rng(n).standard_normal(n)
    top = po.dwt_max_level(n, po.Wavelet(wavelet).dec_len)
    for level in sorted({0, 1, top, top + 2}):
        ref, got = po.wavedec(x, wavelet, level=level), fl.wavedec(x, wavelet, level=level)
        assert [r.size for r in ref] == [g.size for g in got]
        assert max(np.abs(r - g).max() for r, g in zip(ref, got)) <= 1e-13
        assert np.abs(po.waverec(ref, wavelet) - fl.waverec(ref, wavelet)).max() <= 1e-13


@pytest.mark.parametrize("wavelet", WAVELETS)
@pytest.mark.parametrize("n,J", [(20, 6), (64, 3), (257, 5), (1000, 7)])
def test_mra_cascade_equals_equivalent_filters(wavelet, n, J):
    w = mo.modwt(np.random.default_rng(J).standard_normal(n), wavelet, J)
    ref, got = mo.modwtmra(w, wavelet), fl.modwtmra(w, wavelet)
    assert np.abs(ref - got).max() <= 1e-13 * max(1.0, np.abs(ref).max())


# ---- route ------------------------------------------------------------------------------------------------------
FIRST_LONG = {  # (entry, f64, L, J or level) -> first n on the long path
    ("modwt", True, 8, 6): 14485, ("modwt", False, 8, 6): 29005,
    ("modwtmra", True, 8, 6): 14525, ("modwtmra", False, 8, 6): 29053,
    ("wavedec", True, 8, 5): 14525, ("wavedec", False, 8, 5): 29053,
    ("imodwt", True, 8, 6): 9657, ("imodwt", False, 8, 6): 19337,
    ("modwtmra_taps", True, 2, 1): 14525, ("modwtmra_taps", True, 8, 10): 14525,
    ("modwtmra_taps", True, 10, 4): 14525, ("modwtmra_taps", False, 8, 10): 29053,
    ("waverec", True, 2, 1): 14527, ("waverec", True, 8, 5): 14521, ("waverec", True, 10, 5): 14519,
    ("waverec", False, 2, 1): 29055, ("waverec", False, 8, 5): 29049, ("waverec", False, 10, 5): 29047,
}


@pytest.mark.parametrize("key", list(FIRST_LONG), ids=lambda k: "-".join(map(str, k)))
def test_first_long_lengths(key):
    entry, f64, L, J = key
    n = FIRST_LONG[key]
    kw = dict(L=L, J=J, level=J)
    assert fl.first_long_n(entry, f64, **kw) == n
    assert fl.route(entry, n - 1, f64, **kw) == "one-cta"
    assert all(fl.route(entry, m, f64, **kw) == "long" for m in (n, n + 1, n + 2, n + 3, 2 * n, 3_000_000))


def test_mra_cascade_kernel_never_reaches_the_long_lengths():
    """blk_shape covers no MRA length past the generic kernel's limit, so the long MRA starts where that limit is."""
    for f64 in (False, True):
        for L in (2, 4, 6, 8):
            for J in range(1, 11):
                assert not any(fl.mra_fast_covers(n, L, J, f64) for n in range(8705, 30000, 7))
                assert fl.route("modwtmra_taps", 14525, True, L=L, J=J) == "long"
                assert fl.mra_fast_covers(1024, L, 1, f64)


# ---- waves and launches -----------------------------------------------------------------------------------------
def test_wave_rows():
    assert fl.wave_rows(2 * 8 * (1 << 20), 64) == 4            # FP64 MODWT, 2^20 samples: 4 series per wave
    assert fl.wave_rows(2 * 4 * (1 << 20), 64) == 8
    assert fl.wave_rows(2 * 8 * 11 * (1 << 20), 64) == 1       # FP64 MRA with J = 10: one series per wave
    assert fl.wave_rows(2 * 4 * 29057, 3) == 3


@pytest.mark.parametrize("entry,per_wave", [("modwt", "J"), ("imodwt", "J"), ("modwtmra_taps", "J"),
                                            ("modwtmra", 1), ("wavedec", "level"), ("waverec", "level")])
def test_launches_per_wave(entry, per_wave):
    J = level = 6
    count = {"J": J, "level": level}.get(per_wave, per_wave)
    assert fl.launches(entry, 20001, True, 1, J=J, level=level) == count
    # 1 << 20 samples in FP64: 4 series per wave, 1 for the MRAs' J + 1 rows
    n, batch = 1 << 20, 7
    E = 8
    inter = {"modwtmra_taps": 2 * (J + 1) * n, "modwtmra": 2 * (J + 1) * n}.get(entry, 2 * n)
    if entry == "waverec":
        inter = 2 * fl.waverec_len(fl.coeff_lens(n, 8, level), 8)
    cap = fl.wave_rows(E * inter, batch)
    got = fl.launches(entry, n, True, batch, J=J, level=level, device_ptrs=True)
    assert got == -(-batch // cap) * count


def test_host_chunks_split_the_waves():
    """64 series of 2^20 samples, FP64, J = 6: 16 series per 1 GiB host chunk, 4 series per wave."""
    n, J = 1 << 20, 6
    chunk = (1 << 30) // (8 * (n + (J + 1) * n))
    assert chunk == 16
    assert fl.launches("modwt", n, True, 64, J=J) == 4 * (4 * J)
    assert fl.launches("modwt", n, True, 64, J=J, device_ptrs=True) == 16 * J
    assert fl.launches("modwt", n, True, 17, J=J) == (4 + 1) * J
    assert fl.launches("wavedec", n, True, 5, level=0) == 0
