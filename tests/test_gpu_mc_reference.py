"""GPU: the Monte-Carlo coherence chain checked one realisation at a time against float64
references -- device surrogates against the Philox restatement of noise.cu, histograms of
device-RNG and injected runs against the oracle's per-row samples (exact row totals, bin edges
within a rounding band), chunked runs, and the coherence plane of the direct large-scale kernel."""

import numpy as np
import pytest

from conftest import normwise_close
from oracle import mc_oracle as mo
from oracle import pycwt_oracle as po

pytestmark = pytest.mark.gpu

DT = 1 / 12
CFG5 = (0.989, 0.966, 1 / 8, 65)          # a1, a2, dj, J: 3351-sample surrogates, nfft 4096
SEED = 0x9E3779B9_00C0FFEE                 # non-zero high word: both key words matter
DELTA32 = 2e-4                             # BASELINE.md FP32 gate 1e-4 (|v| + max v) at v <= 1
DELTA64 = 1e-10                            # FP64 gate
FIRST = 99_994                             # realisations near the end of a 100 000-pair job


def _norm(y):
    return (y - y.mean()) / y.std()


def _geometry(dj, J):
    N, _, _, outside, maxscale = po.mc_geometry(DT, dj, 2 * DT, J, po.Morlet())
    return N, maxscale, outside.any(axis=1)


# ---------------------------------------------------------------- surrogates
@pytest.mark.parametrize("a1,a2", [(0.989, 0.966), (-0.5, 0.3), (0.0, 0.9)])
@pytest.mark.parametrize("white", [False, True], ids=["red", "white"])
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_rednoise_is_the_philox_stream(shim, a1, a2, white, f64):
    """wtb_rednoise reproduces the Philox4x32-10 restatement sample by sample.  nsurr 1 and 5 leave
    all but one thread idle and end inside a block of four normals; 3351 is the cfg5 length;
    first = 2^32 - 2 with four realisations crosses the counter's high word."""
    for nsurr, first, count in [(1, 0, 3), (5, 99_996, 4), (3351, 99_996, 4), (20_000, 0, 2),
                                (3351, 2**32 - 2, 4)]:
        dev = shim.rednoise(a1, a2, nsurr, first, count, SEED, f64=f64, white=white).astype(np.float64)
        ref = mo.device_surrogates(a1, a2, nsurr, first, count, SEED, white=white)
        err = np.abs(dev - ref)
        if white:
            bound = 1e-6 * (1 + np.abs(ref))
        else:
            bound = 1e-5 * np.abs(ref).max(axis=-1, keepdims=True)
        if not f64:
            bound = bound + np.abs(ref) * 2.0 ** -24
        bad = np.argwhere(err > bound)
        assert bad.size == 0, (nsurr, first, count, bad[:4].tolist(), float(err.max()))


# ---------------------------------------------------------------- device-RNG chain
@pytest.fixture(scope="module")
def cfg5_ref():
    """Oracle samples of realisations FIRST .. FIRST + 5 of the cfg5 job, from the Philox restatement."""
    a1, a2, dj, J = CFG5
    N, _, _ = _geometry(dj, J)
    return mo.mc_samples(mo.device_surrogates(a1, a2, N, FIRST, 6, SEED), DT, dj, 2 * DT, J)


@pytest.mark.parametrize("generic_only", [False, True], ids=["default", "generic"])
def test_mc_device_rng_cfg5_fp32(shim, cfg5_ref, generic_only):
    """The bench's chain at cfg5 in FP32.  The default dispatch takes the nfft-4096 kernels with the
    28 largest scales on the direct kernel; generic_only the shared-memory kernels."""
    a1, a2, dj, J = CFG5
    assert mo.direct_split(DT, dj, 2 * DT, J) == 38
    hist = shim.wct_mc_hist(a1, a2, DT, dj, 2 * DT, J, mc_first=FIRST, mc_count=6, seed=SEED, f64=False,
                            generic_only=generic_only)
    mo.assert_hist_matches(hist, cfg5_ref, DELTA32)


def test_mc_device_rng_cfg5_fp64(shim):
    """FP64: the oracle gets the device's own FP64 surrogates (its float32 Box-Muller normals differ
    from the float64 restatement by ~1e-7, far above the 1e-10 band; the surrogates themselves are
    held to the restatement above)."""
    a1, a2, dj, J = CFG5
    N, _, _ = _geometry(dj, J)
    sur = shim.rednoise(a1, a2, N, FIRST, 4, SEED, f64=True)
    assert np.abs(sur - mo.device_surrogates(a1, a2, N, FIRST, 4, SEED)).max() <= 1e-3
    hist = shim.wct_mc_hist(a1, a2, DT, dj, 2 * DT, J, mc_first=FIRST, mc_count=4, seed=SEED, f64=True)
    mo.assert_hist_matches(hist, mo.mc_samples(sur, DT, dj, 2 * DT, J), DELTA64)


@pytest.mark.parametrize("dj,J,pad", [(1 / 4, 24, "pow2"), (1 / 8, 50, "none")], ids=["nfft1024", "nopad914"])
@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_mc_device_rng_generic_shapes(shim, dj, J, pad, f64):
    """Generic kernels: 768 samples padded to 1024, and 914 samples transformed at their own length
    (set_fft_padding('none'), pycwt with mkl_fft)."""
    a1, a2, first, mc = 0.8, 0.6, 12_345, 8
    N, _, _ = _geometry(dj, J)
    assert N == {24: 768, 50: 914}[J]
    old = shim.get_fft_padding()
    shim.set_fft_padding(pad)
    try:
        hist = shim.wct_mc_hist(a1, a2, DT, dj, 2 * DT, J, mc_first=first, mc_count=mc, seed=SEED, f64=f64)
    finally:
        shim.set_fft_padding(old)
    if f64:
        sur = shim.rednoise(a1, a2, N, first, mc, SEED, f64=True)
    else:
        sur = mo.device_surrogates(a1, a2, N, first, mc, SEED)
    ref = mo.mc_samples(sur, DT, dj, 2 * DT, J, pad_pow2=pad == "pow2")
    mo.assert_hist_matches(hist, ref, DELTA64 if f64 else DELTA32)


def test_mc_significance_one_call_cfg5(shim):
    """wtb_wct_significance (device RNG, histogram, percentile step in one call) at cfg5."""
    a1, a2, dj, J = CFG5
    N, maxscale, rows_any = _geometry(dj, J)
    sig, hist = shim.wct_significance(a1, a2, DT, dj, 2 * DT, J, mc_count=4, seed=SEED, f64=False,
                                      return_hist=True)
    ref = mo.mc_samples(mo.device_surrogates(a1, a2, N, 0, 4, SEED), DT, dj, 2 * DT, J)
    mo.assert_hist_matches(hist, ref, DELTA32)
    sig_ref = po.sig_from_histogram(mo.samples_histogram(ref), maxscale, 0.95, rows_any)
    assert np.array_equal(np.isnan(sig), np.isnan(sig_ref))
    assert np.abs(sig[:maxscale] - sig_ref[:maxscale]).max() <= 2e-3
    assert np.array_equal(np.nan_to_num(sig[maxscale:], nan=-1), np.nan_to_num(sig_ref[maxscale:], nan=-1))


# ---------------------------------------------------------------- chunked runs
# cfg5 costs 4 417 720 B of scratch per pair in FP32 and 8 835 440 B in FP64 (wct.cu, per_pair):
# 9 MB / 17 MB budgets hold two pairs, so seven realisations run as chunks of 2, 2, 2 and 1.
CHUNK_MB = {False: "9", True: "17"}
CHUNK_FIRST, CHUNK_MC = 4242, 7


@pytest.fixture(scope="module")
def chunk_sur():
    a1, a2, dj, J = CFG5
    N, _, _ = _geometry(dj, J)
    sur = mo.device_surrogates(a1, a2, N, CHUNK_FIRST, CHUNK_MC, SEED)
    return sur, mo.mc_samples(sur, DT, dj, 2 * DT, J)


def _chunked(shim, monkeypatch, f64, **kw):
    """(unchunked, chunked) histograms of the same call, and the launch counts of each."""
    a1, a2, dj, J = CFG5
    args = (a1, a2, DT, dj, 2 * DT, J)
    n0 = shim.kernel_launches()
    whole = shim.wct_mc_hist(*args, mc_count=CHUNK_MC, f64=f64, **kw)
    n1 = shim.kernel_launches()
    monkeypatch.setenv("WTB_MC_CHUNK_MB", CHUNK_MB[f64])
    chunked = shim.wct_mc_hist(*args, mc_count=CHUNK_MC, f64=f64, **kw)
    n2 = shim.kernel_launches()
    monkeypatch.delenv("WTB_MC_CHUNK_MB")
    return whole, chunked, n1 - n0, n2 - n1


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_mc_chunked_device_rng(shim, monkeypatch, chunk_sur, f64):
    """Chunk k draws realisations mc_first + m0 .. : the histogram is the unchunked one, bit for bit."""
    whole, chunked, l_whole, l_chunked = _chunked(shim, monkeypatch, f64, mc_first=CHUNK_FIRST, seed=SEED)
    assert l_chunked == 4 * l_whole, (l_whole, l_chunked)      # four chunks, the same kernels each
    assert np.array_equal(chunked, whole)
    if f64:
        a1, a2, dj, J = CFG5
        sur = shim.rednoise(a1, a2, chunk_sur[0].shape[2], CHUNK_FIRST, CHUNK_MC, SEED, f64=True)
        mo.assert_hist_matches(chunked, mo.mc_samples(sur, DT, dj, 2 * DT, J), DELTA64)
    else:
        mo.assert_hist_matches(chunked, chunk_sur[1], DELTA32)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
def test_mc_chunked_injected(shim, monkeypatch, chunk_sur, f64):
    """Host-injected surrogates over several chunks take the two-buffer pipeline (the copy of chunk
    k + 1 overlaps the kernels of chunk k)."""
    sur, ref = chunk_sur
    whole, chunked, l_whole, l_chunked = _chunked(shim, monkeypatch, f64, surrogates=sur)
    assert l_chunked == 4 * l_whole, (l_whole, l_chunked)
    assert np.array_equal(chunked, whole)
    mo.assert_hist_matches(chunked, ref, DELTA64 if f64 else DELTA32)


# ---------------------------------------------------------------- direct kernel as a plane
@pytest.fixture(scope="module")
def cfg5_pairs():
    a1, a2, dj, J = CFG5
    N, _, _ = _geometry(dj, J)
    sur = mo.device_surrogates(a1, a2, N, 0, 2, SEED)
    y1 = np.stack([_norm(p[0]) for p in sur])
    y2 = np.stack([_norm(p[1]) for p in sur])
    ref = np.stack([po.wct(y1[b], y2[b], DT, dj=dj, s0=2 * DT, J=J, sig=False, normalize=False)[0]
                    for b in range(2)])
    return y1, y2, ref


def _plane_gate(got, ref, rows, tag):
    for b in range(got.shape[0]):
        ok, worst = normwise_close(got[b], ref[b], 1e-4)
        assert ok, (tag, b, worst)
        assert np.abs(got[b] - ref[b]).mean() <= 2e-6, (tag, b)
        ok, worst = normwise_close(got[b, rows], ref[b, rows], 1e-4)
        assert ok, (tag, "direct rows", b, worst)
        assert np.abs(got[b, rows] - ref[b, rows]).mean() <= 2e-6, (tag, "direct rows", b)


def test_direct_rows_plane_cfg5(shim, monkeypatch, cfg5_pairs):
    """Without phase or cross spectrum the FP32 nfft-4096 plane takes its 28 largest scales from the
    direct band-limited kernel.  Oracle gate on the whole plane and on those rows alone, for every
    split point WTB_MC_DIRECT_B gives (0 = off; values above the kernel's 128 bins are clamped)."""
    y1, y2, ref = cfg5_pairs
    _, _, dj, J = CFG5
    s_split = mo.direct_split(DT, dj, 2 * DT, J)
    assert s_split == 38
    rows = slice(s_split, J + 1)

    def run():
        n = shim.kernel_launches()
        wct = shim.xwt_wct(y1, y2, DT, dj, 2 * DT, J, f64=False, want_phase=False)[0]
        return wct, shim.kernel_launches() - n

    default, n_default = run()
    _plane_gate(default, ref, rows, "default")
    out, launches = {}, {}
    for bmax in (0, 1, 16, 64, 128, 1000):
        monkeypatch.setenv("WTB_MC_DIRECT_B", str(bmax))
        out[bmax], launches[bmax] = run()
        _plane_gate(out[bmax], ref, rows, f"WTB_MC_DIRECT_B={bmax}")
    monkeypatch.delenv("WTB_MC_DIRECT_B")
    assert n_default - launches[0] == 1                       # the direct kernel ran by default
    assert np.array_equal(out[128], default)
    assert np.array_equal(out[1000], out[128])
    for bmax in (1, 16, 64):
        assert launches[bmax] == launches[0] + (mo.direct_split(DT, dj, 2 * DT, J, bmax=bmax) <= J)


def test_direct_rows_fuzz(shim):
    """Random and edge shapes through the direct kernel (plane without phase), against the FP64
    generic kernels: n0 = 2049 (the longest zero tail of a 4096-point transform), n0 = 4096 with
    dj 1/8, J 88 (last rows one bin wide, no Gaussian bins but 0), f0 = 5.3 (bands from bin 0)."""
    rng = np.random.default_rng(2049)
    cases = [(2049, DT, 1 / 8, 2 * DT, 80, 6.0), (4096, DT, 1 / 8, 2 * DT, 88, 6.0), (3000, 0.5, 1 / 10, 0.5, 100, 5.3)]
    for _ in range(3):
        n0 = int(rng.integers(2049, 4097))
        dt = float(rng.choice([1 / 12, 0.5, 2.0]))
        dj = float(rng.choice([1 / 4, 1 / 8, 1 / 10, 1 / 12]))
        s0 = dt * float(rng.choice([1.0, 2.0, 4.0]))
        f0 = float(rng.choice([6.0, 7.5, 10.0]))
        jmax = int(np.floor(np.log2(n0 * dt / s0) / dj))
        cases.append((n0, dt, dj, s0, int(rng.integers(jmax // 2, min(jmax, 110) + 1)), f0))
    seen = set()
    for n0, dt, dj, s0, J, f0 in cases:
        assert J <= int(np.floor(np.log2(n0 * dt / s0) / dj))
        s_split = mo.direct_split(dt, dj, s0, J, f0)
        for l0, B, kc in mo.row_bands(dt, dj, s0, J, f0)[s_split:]:
            seen |= {"B1kc0"} if (B, kc) == (1, 0) else set()
            seen |= {"l0=0"} if l0 == 0 else set()
            seen |= {"B120..128"} if 120 <= B <= 128 else set()
        y1 = _norm(po.rednoise(n0, 0.8, 1, rng))
        y2 = _norm(0.5 * y1 + po.rednoise(n0, 0.5, 1, rng))
        wct = shim.xwt_wct(y1, y2, dt, dj, s0, J, f0, f64=False, want_phase=False)[0]
        ref = shim.xwt_wct(y1, y2, dt, dj, s0, J, f0, f64=True, want_phase=False, generic_only=True)[0]
        tag = f"n0={n0} dt={dt} dj={dj:.4f} s0={s0} f0={f0} J={J} split={s_split}"
        # rows whose daughter peaks beyond Nyquist see only the wavelet's tail (test_gpu_wct's fuzz)
        sj = s0 * 2.0 ** (np.arange(J + 1) * dj)
        resolvable = sj / dt >= f0 / np.pi
        ok, worst = normwise_close(wct[resolvable], ref[resolvable], 1e-4)
        assert ok, (tag, worst)
        assert np.abs(wct - ref).max() <= 2e-3, tag
        assert np.abs(wct[resolvable] - ref[resolvable]).mean() <= 5e-6, tag
        if s_split <= J:
            ok, worst = normwise_close(wct[s_split:], ref[s_split:], 1e-4)
            assert ok, (tag, "direct rows", worst)
    assert seen == {"B1kc0", "l0=0", "B120..128"}, seen
