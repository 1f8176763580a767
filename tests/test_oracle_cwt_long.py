"""CPU: the per-row float64 reference and the host-rule replica of the long-series CWT (oracle/cwt_long.py)."""

import numpy as np
import pytest

from oracle import cwt_long as cl
from oracle import pycwt_oracle as po

MOTHERS = {"morlet": po.Morlet(6), "paul4": po.Paul(4), "dog2": po.DOG(2), "dog6": po.DOG(6)}


@pytest.mark.parametrize("n0", [100, 1346, 3351, 4096])
@pytest.mark.parametrize("mother", list(MOTHERS))
def test_rows_match_the_whole_plane(n0, mother):
    rng = np.random.default_rng(n0)
    x = rng.standard_normal(n0)
    wl = MOTHERS[mother]
    W = po.cwt(x, 1.0, 1 / 8, -1, -1, wl)[0]
    rows = sorted({0, 3, W.shape[0] // 2, W.shape[0] - 1})
    got = cl.cwt_rows(x, 1.0, 1 / 8, -1, -1, wl, rows)
    assert np.abs(got - W[rows]).max() <= 1e-13 * np.abs(W).max()
    # the un-padded transform too
    Wn = po.cwt(x, 1.0, 1 / 8, -1, -1, wl, pad_pow2=False)[0]
    gotn = cl.cwt_rows(x, 1.0, 1 / 8, -1, -1, wl, rows, nfft=n0)
    assert np.abs(gotn - Wn[rows]).max() <= 1e-13 * np.abs(Wn).max()


def test_dispatch_boundaries():
    assert cl.route(8192, f64=False) == "generic" and cl.route(16384, f64=False) == "long"
    assert cl.route(4096, f64=True) == "generic" and cl.route(8192, f64=True) == "long"
    assert cl.route(1 << 22, f64=False) == "long" and cl.route(1 << 22, f64=True) == "long"
    assert cl.route(1 << 23, f64=False) == "refused" and cl.route(1 << 23, f64=True) == "refused"
    # un-padded lengths keep the Bluestein path (and its refusal past 4096 / 2048)
    for n in (5000, 8193, 3 * 2 ** 20):
        assert cl.route(n, f64=False) == "generic" and cl.route(n, f64=True) == "generic"


# (nfft, f64, batch, S) -> (forward waves, row waves) at the shapes tests/test_gpu_cwt_long.py uses
@pytest.mark.parametrize("shape,expected", [
    ((16384, False, 1, 49), (1, 1)),          # FP32 n0 = 8193: 512 rows per wave
    ((8192, True, 1, 45), (1, 1)),            # FP64 n0 = 4097: 512 rows per wave
    ((1 << 17, False, 1, 33), (1, 1)),        # 64 rows per wave
    ((1 << 17, True, 1, 33), (1, 2)),         # 32 rows per wave
    ((1 << 20, False, 1, 39), (1, 5)),        # 8 rows per wave
    ((1 << 20, True, 1, 39), (1, 10)),        # 4 rows per wave
    ((1 << 22, False, 1, 17), (1, 9)),        # two rows (32 MiB each) per wave
    ((1 << 22, True, 1, 17), (1, 17)),        # one row (64 MiB) per wave
    ((1 << 19, False, 7, 37), (1, 17)),       # invariance: 16 rows per wave, 259 rows
    ((1 << 19, False, 3, 37), (1, 7)),
    ((1 << 18, True, 7, 35), (1, 16)),        # 16 rows per wave, 245 rows
    ((1 << 18, True, 3, 35), (1, 7)),
])
def test_wave_counts(shape, expected):
    nfft, f64, batch, S = shape
    assert cl.waves(nfft, f64, batch, S) == expected
    assert cl.launches(nfft, f64, batch, S) == 2 * sum(expected)


def test_wave_rule():
    assert cl.wave_rows(1 << 22, False, 100) == 2 and cl.wave_rows(1 << 22, True, 100) == 1
    assert cl.wave_rows(16384, False, 10 ** 6) == 512 and cl.wave_rows(16384, False, 7) == 7
    # the forward transform of a large batch runs in waves of series too
    assert cl.waves(16384, False, 1300, 1) == (3, 3)


def test_averages_chunk_rule_at_long_lengths():
    # 1 GiB of power rows, no floor: one series per chunk once its plane passes 1 GiB
    assert cl.averages_chunk_rows(4, 230, 1 << 20, f64=True) == 1
    assert cl.averages_chunk_rows(4, 39, 1 << 20, f64=False) == 4
    assert cl.averages_chunk_rows(100, 39, 1 << 20, f64=False) == 6
    assert cl.averages_chunk_rows(3, 61, 20000, f64=False) == 3
