"""CPU checks of oracle/cwt_rows.py: the replica of the host row rules is pinned to the counts
DESIGN.md states and to the benchmarked shapes, and the per-row gate accepts round-off while it
rejects errors the plane gate lets through."""

from collections import Counter

import numpy as np
from scipy.signal import lfilter

from conftest import normwise_close
from oracle import cwt_rows as cr
from oracle import pycwt_oracle as po

DT = 1 / 12


def test_cfg1_rows_of_the_nfft2048_kernel():
    """DESIGN section 4, k_cwt_dif<2> on cfg1 (1345 / 1346 samples, dj = 1/12, J = 84): a row is
    single-pass while k_hi < 64 (31 % of the 85 rows) and 12 rows take the two-input DFT."""
    rows = cr.dif_rows(2048, DT, 1 / 12, 2 * DT, 84)
    assert len(rows) == 85
    single = sum(1 for multi, _ in rows if not multi)
    assert single == 26 and round(100 * single / 85) == 31
    assert sum(1 for _, L in rows if L == 1) == 12
    assert Counter(rows) == {(1, 4): 23, (1, 3): 12, (1, 2): 12, (1, 1): 12, (0, 5): 12, (0, 4): 12, (0, 3): 2}


def test_cfg4_rows_of_the_nfft1024_kernel():
    """cfg4 (n0 = 1024, dj = 1/12, J = 119): every branch of k_cwt_fast_1024 is taken."""
    rows = cr.fast_rows(1024, DT, 1 / 12, 2 * DT, 119)
    assert Counter(rows) == {(0, 1): 13, (0, 2): 12, (0, 3): 12, (0, 4): 12, (0, 5): 12,
                             (1, 1): 12, (1, 2): 12, (1, 3): 12, (1, 4): 23}
    assert set(rows) == cr.ROW_CLASSES["fast"]
    # the two-series variant has its band edge one bin further out
    half = cr.fast_rows(512, DT, 1 / 12, 2 * DT, 119)
    assert Counter(half)[(0, 1)] == 1 and set(half) == cr.ROW_CLASSES["fast"]
    assert cr.resolved_rows(1024, 1024, DT, 1 / 12, 2 * DT, 119).sum() == 107


def test_cfg5_rows_of_the_nfft4096_kernels():
    """cfg5 (3351 samples padded to 4096, dj = 1/8, J = 65): the register rows (and the coherence
    kernels, same fill_rows) and the four-warps-per-row kernel."""
    w = cr.wrow_rows(DT, 1 / 8, 2 * DT, 65)
    assert Counter(w) == {(1, 0): 35, (2, 1): 8, (4, 2): 8, (8, 3): 15}
    d = cr.dif_rows(4096, DT, 1 / 8, 2 * DT, 65)
    assert Counter(d) == {(0, 2): 3, (0, 3): 8, (0, 4): 8, (0, 5): 8, (1, 1): 8, (1, 2): 8, (1, 3): 8, (1, 4): 15}
    assert cr.resolved_rows(3351, 4096, DT, 1 / 8, 2 * DT, 65).all()


def test_resolved_rows_rule():
    # s0 = dt: with f0 = 6 the first rows peak beyond the Nyquist frequency (s/dt < 6/pi)
    sc = cr.scales(1.0, 1 / 4, 1.0, 40)
    res = cr.resolved_rows(1024, 1024, 1.0, 1 / 4, 1.0, 40)
    assert not res[sc < 6 / np.pi].any() and res[(sc >= 6 / np.pi) & (sc < 100)].all()
    # the largest scales keep fewer than two bins of daughter support
    khi = np.floor(11.3 * 1024 / (2 * np.pi * sc))
    assert np.array_equal(res, (khi >= 2) & (sc >= 6 / np.pi)) and (khi < 2).any()


def _ar1_plane(n0=3351, g=0.989, seed=5):
    rng = np.random.default_rng(seed)
    x = lfilter([1.0], [1.0, -g], rng.standard_normal(n0 + 3000))[3000:]
    x -= x.mean()
    return np.abs(po.cwt(x, DT, 1 / 8, 2 * DT, 65)[0]) ** 2


def test_row_gate_accepts_round_off():
    ref = _ar1_plane()
    rng = np.random.default_rng(1)
    eps = 2.0 ** -24
    rowmax = ref.max(axis=1, keepdims=True)
    noisy = ref * (1 + 4 * eps * rng.standard_normal(ref.shape)) + 4 * eps * rowmax * rng.standard_normal(ref.shape)
    ratio, _ = cr.row_gate(noisy, ref, 1e-4)
    assert ratio < 0.05          # 4 ulp of noise: a few hundredths of the 1e-4 bound
    assert cr.row_gate(ref, ref, 1e-4)[0] == 0.0


def test_row_gate_rejects_what_the_plane_gate_accepts():
    """A 3e-4 gain on a row at 1e-3 of the plane maximum: the plane gate passes it, the row gate
    does not."""
    ref = _ar1_plane()
    share = ref.max(axis=1) / ref.max()
    s = int(np.argmin(np.abs(np.log(share / 1e-3))))
    assert 5e-4 < share[s] < 2e-3
    bad = ref.copy()
    bad[s] *= 1 + 3e-4
    assert normwise_close(bad, ref, 1e-4)[0]
    ratio, where = cr.row_gate(bad, ref, 1e-4)
    assert ratio > 1.0 and where[0] == s
    # and on complex coefficients: the same gain on W is caught the same way
    W = np.sqrt(ref) * np.exp(1j * np.linspace(0, 50, ref.shape[1]))
    Wb = W.copy()
    Wb[s] *= 1 + 3e-4
    assert cr.row_gate(Wb, W, 1e-4)[0] > 1.0
    # the floor: a row at 1e-10 of the plane is held to 1e-5 of the plane maximum, not to itself
    tiny = ref.copy()
    tiny[0] = ref[0] / ref[0].max() * 1e-10 * ref.max()
    off = tiny.copy()
    off[0] += 1e-10 * ref.max()
    assert cr.row_gate(off, tiny, 1e-4)[0] <= 0.1 + 1e-9
