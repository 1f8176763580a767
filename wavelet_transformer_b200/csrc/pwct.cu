// Partial and multiple wavelet coherence of three series (Aguiar-Conraria & Soares 2014; Ng & Chan 2012), built
// from pycwt's Morlet CWT and Morlet.smooth exactly as pycwt.wct forms S1, S2 and S12.
//
// Per chunk of triples (y, x1, x2), the series interleaved as [triple, 3, n0]:
//   cwt_device           W [triple, 3, S, n0] complex                 (cwt.cu: wtb_cwt's own coefficients)
//   k_pwct_smooth (b, s) five packed fields of one scale row, each time-smoothed as Morlet.smooth does:
//                          (|Wy|^2 + i |W1|^2)/s, |W2|^2/s, Wy conj(W1)/s, Wy conj(W2)/s, W1 conj(W2)/s
//                        -> sm [triple, S, 9, n0]: Syy, S11, S22, Re/Im Sy1, Re/Im Sy2, Re/Im S12
//   k_pwct_scale  (b, t) boxcar over scales (convolve2d 'same', zero fill), then
//                          PWC   = |Sy1 S22 - Sy2 conj(S12)|^2 / ((Syy S22 - |Sy2|^2)(S11 S22 - |S12|^2))
//                          phase = angle(Sy1 S22 - Sy2 conj(S12))
//                          MWC   = (|Sy1|^2 S22 + |Sy2|^2 S11 - 2 Re(Sy1 conj(Sy2) S12)) / (Syy (S11 S22 - |S12|^2))
//                        -> output planes, or (HIST) PWC and MWC binned into per-scale histograms
//
// The Monte-Carlo significance (wtb_partial_wct_mc_hist) runs the same three passes on AR(1) surrogate triples
// (noise.cu, K = 3) and bins the reliable region of rows s < maxscale as k_wct_scale's MODE 1 bins R^2.
// The Gaussian is real and even, so the packed real fields come back in the real and imaginary parts of one
// transform, as in k_wct_rows.  sm keeps each of the nine smoothed reals of a (triple, scale) row as its own
// n0-sample plane: the scale pass, one thread per (triple, t), then reads every field of a row as one coalesced
// run of consecutive t across a warp.
#include "cwt_paths.cuh"
#include "spectral.cuh"

namespace wtb {

constexpr int kPwctFields = 9;

// One CTA = one (triple, scale).  smem: 2 * plan.M complex, the same as k_cwt_rows, so the lengths this takes are
// those of the generic CWT.  W: [triple, 3, S, n0].  sm: [triple, S, 9, n0].
template <typename T>
__global__ void k_pwct_smooth(const cplx<T> *__restrict__ W, int n0, FftPlan<T> plan, int S,
                              const double *__restrict__ scales, double dt, T *__restrict__ sm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T> *const buf0 = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *const buf1 = buf0 + plan.M;
  const int N = plan.n;
  const int64_t tri = blockIdx.x / S;
  const int s = blockIdx.x % S;
  const int64_t plane = (int64_t)S * n0;
  const cplx<T> *wy = W + tri * 3 * plane + (int64_t)s * n0;
  const cplx<T> *w1 = wy + plane;
  const cplx<T> *w2 = w1 + plane;
  const double sc = scales[s];
  const T s_over_dt = T(sc / dt);
  const T inv_s = T(1.0 / sc);
  const T invN = T(1.0 / N);
  T *out = sm + (tri * S + s) * (int64_t)kPwctFields * n0;
  for (int f = 0; f < 5; ++f) {
    // pycwt truncates W to n0 samples before it smooths: the row is zero past n0
    for (int t = threadIdx.x; t < N; t += blockDim.x) {
      cplx<T> v = mk<T>(T(0), T(0));
      if (t < n0) {
        if (f == 0) {
          const cplx<T> a = wy[t], b = w1[t];
          v = mk<T>((a.x * a.x + a.y * a.y) * inv_s, (b.x * b.x + b.y * b.y) * inv_s);
        } else if (f == 1) {
          const cplx<T> a = w2[t];
          v = mk<T>((a.x * a.x + a.y * a.y) * inv_s, T(0));
        } else {
          const cplx<T> x = f == 2 ? cmulc(wy[t], w1[t]) : (f == 3 ? cmulc(wy[t], w2[t]) : cmulc(w1[t], w2[t]));
          v = mk<T>(x.x * inv_s, x.y * inv_s);
        }
      }
      buf0[t] = v;
    }
    __syncthreads();
    cplx<T> *r = plan_fft<T, -1>(buf0, buf1, plan);
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
      const T g = smooth_gauss<T>(k, N, s_over_dt, invN);
      const cplx<T> v = r[k];
      r[k] = mk<T>(v.x * g, v.y * g);
    }
    __syncthreads();
    r = plan_fft<T, +1>(r, r == buf0 ? buf1 : buf0, plan);
    // field f -> planes: 0 -> Syy, S11; 1 -> S22; 2 -> Sy1; 3 -> Sy2; 4 -> S12
    T *o = out + (int64_t)(f == 0 ? 0 : (f == 1 ? 2 : 2 * f - 1)) * n0;
    for (int t = threadIdx.x; t < n0; t += blockDim.x) {
      const cplx<T> v = r[t];
      o[t] = v.x;
      if (f != 1) o[n0 + t] = v.y;
    }
    __syncthreads();  // the next field overwrites both buffers
  }
}

// bin = min(floor(v * WTB_NBINS), WTB_NBINS - 1) as k_wct_scale forms it; NaN and negative values are skipped.  The
// minimum is taken in double, so +inf (a zero denominator under a non-zero numerator) lands in the last bin.
__device__ __forceinline__ void hist_add(unsigned long long *row, double v) {
  if (!(v >= 0.0)) return;
  atomicAdd(&row[(int)fmin(floor(v * WTB_NBINS), WTB_NBINS - 1.0)], 1ULL);
}

// One thread = one (triple, t) column; walks the scales.  The boxcar sums and the closed forms run in double in
// both precisions: S11 S22 - |S12|^2 cancels when x1 and x2 are coherent.  0/0 gives NaN, as pycwt's WCT does.
// HIST: rows s < maxscale only, t in [tlo[s], thi[s]] only; PWC adds to hist[0, s, bin], MWC to hist[1, s, bin]
// (hist: [2, S, WTB_NBINS]), from the double values; no planes, no phase.
template <typename T, bool HIST>
__global__ void k_pwct_scale(const T *__restrict__ sm, int64_t triples, int n0, int S, ScaleWin win,
                             T *__restrict__ pwc, T *__restrict__ pphase, T *__restrict__ mwc,
                             unsigned long long *__restrict__ hist, const int *__restrict__ tlo,
                             const int *__restrict__ thi, int maxscale) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= triples * n0) return;
  const int64_t tri = gid / n0;
  const int t = (int)(gid % n0);
  const T *col = sm + tri * S * (int64_t)kPwctFields * n0 + t;
  const int s_end = HIST ? maxscale : S;
  for (int s = 0; s < s_end; ++s) {
    if (HIST && (t < tlo[s] || t > thi[s])) continue;
    double a[kPwctFields];
#pragma unroll
    for (int f = 0; f < kPwctFields; ++f) a[f] = 0.0;
    for (int k = 0; k < win.K; ++k) {
      const int row = s + win.up - k;
      if (row < 0 || row >= S) continue;
      const T *v = col + (int64_t)row * kPwctFields * n0;
      const double w = win.w[k];
#pragma unroll
      for (int f = 0; f < kPwctFields; ++f) a[f] += w * (double)v[(int64_t)f * n0];
    }
    const double syy = a[0], s11 = a[1], s22 = a[2];
    const double y1r = a[3], y1i = a[4], y2r = a[5], y2i = a[6], c12r = a[7], c12i = a[8];
    const int64_t o = (tri * S + s) * (int64_t)n0 + t;
    // Sy1 S22 - Sy2 conj(S12)
    const double nr = y1r * s22 - (y2r * c12r + y2i * c12i);
    const double ni = y1i * s22 - (y2i * c12r - y2r * c12i);
    const double d12 = s11 * s22 - (c12r * c12r + c12i * c12i);
    if (HIST || pwc) {
      const double dy2 = syy * s22 - (y2r * y2r + y2i * y2i);
      const double v = (nr * nr + ni * ni) / (dy2 * d12);
      if (HIST) hist_add(hist + (size_t)s * WTB_NBINS, v);
      else pwc[o] = T(v);
    }
    if (!HIST && pphase) pphase[o] = T(atan2(ni, nr));
    if (HIST || mwc) {
      // Re(Sy1 conj(Sy2) S12)
      const double pr = y1r * y2r + y1i * y2i, pi = y1i * y2r - y1r * y2i;
      const double cross = pr * c12r - pi * c12i;
      const double num = (y1r * y1r + y1i * y1i) * s22 + (y2r * y2r + y2i * y2i) * s11 - 2.0 * cross;
      const double v = num / (syy * d12);
      if (HIST) hist_add(hist + ((size_t)S + s) * WTB_NBINS, v);
      else mwc[o] = T(v);
    }
  }
}

// bytes of staging one triple costs: interleaved series, coefficients, smoothed fields
template <typename T> static size_t triple_bytes(int n0, int S) {
  return sizeof(T) * 3 * (size_t)n0 + sizeof(cplx<T>) * 3 * (size_t)S * n0 + sizeof(T) * kPwctFields * (size_t)S * n0;
}

// d_hist (device, [2, S, WTB_NBINS]): bin rows s < maxscale over the host ranges h_tlo / h_thi instead of writing
// the planes.
template <typename T>
static int pwct_device(const T *d_y, int64_t nb, int n0, int N, double dt, const Axes &ax, double f0,
                       const ScaleWin &win, int flags, cplx<T> *d_W, T *d_sm, T *d_pwc, T *d_phase, T *d_mwc,
                       cudaStream_t st, unsigned long long *d_hist = nullptr, const int *h_tlo = nullptr,
                       const int *h_thi = nullptr, int maxscale = 0) {
  const int S = ax.J + 1;
  Mother mo;
  mo.kind = WTB_MORLET;
  mo.param = f0;
  WTB_TRY(cwt_device<T>(d_y, 3 * nb, n0, N, dt, ax, mo, flags, nullptr, d_W, st));
  FftPlan<T> plan;
  WTB_TRY(make_plan<T>(N, &plan));
  const size_t smem = 2 * sizeof(cplx<T>) * (size_t)plan.M;
  // cwt_device keeps its scales and spectra in the arena; this copy of the same scales is ordered behind its kernels
  void *scratch = nullptr;
  const size_t b_sc = align256(sizeof(double) * S), b_rng = align256(sizeof(int) * S);
  WTB_TRY(arena_reserve(b_sc + (d_hist ? 2 * b_rng : 0), &scratch));
  double *d_scales = (double *)scratch;
  int *d_tlo = (int *)((char *)scratch + b_sc), *d_thi = (int *)((char *)scratch + b_sc + b_rng);
  WTB_CUDA(cudaMemcpyAsync(d_scales, ax.scales.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  if (d_hist) {
    WTB_CUDA(cudaMemcpyAsync(d_tlo, h_tlo, sizeof(int) * S, cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync(d_thi, h_thi, sizeof(int) * S, cudaMemcpyHostToDevice, st));
  }
  const int threads = plan_threads(plan.M);
  WTB_CUDA(cudaFuncSetAttribute(k_pwct_smooth<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_pwct_smooth<T><<<(unsigned)(nb * S), threads, smem, st>>>(d_W, n0, plan, S, d_scales, dt, d_sm);
  WTB_LAUNCH_CHECK();
  const int64_t cols = nb * n0;
  const unsigned blocks = (unsigned)((cols + 255) / 256);
  if (d_hist)
    k_pwct_scale<T, true><<<blocks, 256, 0, st>>>(d_sm, nb, n0, S, win, nullptr, nullptr, nullptr, d_hist, d_tlo,
                                                  d_thi, maxscale);
  else
    k_pwct_scale<T, false><<<blocks, 256, 0, st>>>(d_sm, nb, n0, S, win, d_pwc, d_phase, d_mwc, nullptr, nullptr,
                                                   nullptr, 0);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

template <typename T>
static int pwct_entry(const void *y, const void *x1, const void *x2, int64_t batch, int n0, int N, double dt,
                      const Axes &ax, double f0, const ScaleWin &win, int flags, void *pwc_out, void *phase_out,
                      void *mwc_out, cudaStream_t st) {
  const int S = ax.J + 1;
  const size_t plane = (size_t)S * n0, row = sizeof(T) * n0;
  const InRows a{y, row}, b{x1, row}, c{x2, row};
  const OutRows pw{pwc_out, sizeof(T) * plane}, ph{phase_out, sizeof(T) * plane}, mw{mwc_out, sizeof(T) * plane};
  // triples per chunk: their staged rows and their intermediates within 1 GiB, with host and device pointers alike
  const size_t per_triple = sizeof(T) * (3 * (size_t)n0 + (pwc_out ? plane : 0) + (phase_out ? plane : 0) +
                                         (mwc_out ? plane : 0)) + triple_bytes<T>(n0, S);
  return shard_host_rows(batch, flags, st, [&](int64_t first, int64_t count, cudaStream_t s) {
    const int64_t rows = std::max<int64_t>(1, std::min<int64_t>(count, (int64_t)((size_t(1) << 30) / per_triple)));
    WTB_REQUIRE(rows * S < (1LL << 31), WTB_EUNSUPPORTED, "wtb_partial_wct: %d scales are too many for one launch", S);
    const size_t b_y = align256(3 * row * rows), b_W = align256(sizeof(cplx<T>) * 3 * plane * rows);
    const size_t b_sm = sizeof(T) * kPwctFields * plane * rows;
    return stage_rows(count, rows, flags, s, {a.at(first), b.at(first), c.at(first)},
                      {pw.at(first), ph.at(first), mw.at(first)}, b_y + b_W + b_sm,
                      [&](const void *const *in, void *const *out, void *extra, int64_t, int64_t nb) {
                        // interleave the triples' rows as [triple, 3, n0]: dst pitch 3 n0, src pitch n0
                        T *d_y = (T *)extra;
                        for (int i = 0; i < 3; ++i)
                          WTB_CUDA(cudaMemcpy2DAsync(d_y + i * n0, 3 * row, in[i], row, row, nb,
                                                     cudaMemcpyDeviceToDevice, s));
                        cplx<T> *d_W = (cplx<T> *)((char *)extra + b_y);
                        T *d_sm = (T *)((char *)extra + b_y + b_W);
                        return pwct_device<T>(d_y, nb, n0, N, dt, ax, f0, win, flags, d_W, d_sm, (T *)out[0],
                                              (T *)out[1], (T *)out[2], s);
                      });
  });
}

// implemented in noise.cu
template <typename T>
int rednoise_triples_device(double ay, double a1, double a2, int nsurr, int64_t first, int64_t count,
                            uint64_t seed, bool white, T *d_out, cudaStream_t st);

// Realisations mc_first .. mc_first + mc_count - 1, one chunk at a time: surrogate triples [chunk, 3, nsurr] (device
// Philox, or the caller's), then pwct_device in histogram mode.  Chunks are bounded as pwct_entry's (1 GiB of
// staged series and intermediates, WTB_MC_CHUNK_MB overrides); the histogram is a sum of integer counts, so its
// bits do not depend on the chunking.
template <typename T>
static int pwct_mc_entry(double ay, double a1, double a2, double dt, const Axes &ax, double f0, const ScaleWin &win,
                         int nsurr, int N, int maxscale, int64_t mc_first, int64_t mc_count, uint64_t seed,
                         const void *surrogates, int flags, uint64_t *hist, cudaStream_t st) {
  const int S = ax.J + 1;
  std::vector<int> tlo, thi;
  std::vector<uint8_t> any;
  coi_ranges(nsurr, dt, ax, f0, &tlo, &thi, &any);
  const bool dev = flags & WTB_DEVICE_PTRS;
  const size_t per_triple = sizeof(T) * 3 * (size_t)nsurr + triple_bytes<T>(nsurr, S);
  size_t budget = size_t(1) << 30;
  if (const char *e = std::getenv("WTB_MC_CHUNK_MB")) budget = (size_t)std::max(1, std::atoi(e)) << 20;
  const int64_t rows = std::max<int64_t>(1, std::min<int64_t>(mc_count, (int64_t)(budget / per_triple)));
  WTB_REQUIRE(rows * S < (1LL << 31), WTB_EUNSUPPORTED, "wtb_partial_wct_mc_hist: %d scales are too many", S);
  const size_t plane = (size_t)S * nsurr;
  const size_t b_y = align256(sizeof(T) * 3 * nsurr * rows), b_W = align256(sizeof(cplx<T>) * 3 * plane * rows);
  const size_t b_sm = align256(sizeof(T) * kPwctFields * plane * rows);
  const size_t cells = 2 * (size_t)S * WTB_NBINS;
  char *stage = nullptr;
  WTB_TRY(staging_reserve(b_y + b_W + b_sm + (dev ? 0 : align256(sizeof(uint64_t) * cells)), (void **)&stage));
  T *d_y = (T *)stage;
  cplx<T> *d_W = (cplx<T> *)(stage + b_y);
  T *d_sm = (T *)(stage + b_y + b_W);
  unsigned long long *d_hist = dev ? (unsigned long long *)hist : (unsigned long long *)(stage + b_y + b_W + b_sm);
  if (!dev) WTB_CUDA(cudaMemsetAsync(d_hist, 0, sizeof(uint64_t) * cells, st));
  for (int64_t m0 = 0; m0 < mc_count; m0 += rows) {
    const int64_t nb = std::min(rows, mc_count - m0);
    const T *src = d_y;
    if (!surrogates)
      WTB_TRY(rednoise_triples_device<T>(ay, a1, a2, nsurr, mc_first + m0, nb, seed, flags & WTB_NOISE_WHITE, d_y, st));
    else if (dev)
      src = (const T *)surrogates + m0 * 3 * nsurr;
    else
      WTB_CUDA(cudaMemcpyAsync(d_y, (const T *)surrogates + m0 * 3 * nsurr, sizeof(T) * 3 * nsurr * nb,
                               cudaMemcpyHostToDevice, st));
    WTB_TRY(pwct_device<T>(src, nb, nsurr, N, dt, ax, f0, win, flags, d_W, d_sm, nullptr, nullptr, nullptr, st,
                           d_hist, tlo.data(), thi.data(), maxscale));
  }
  if (!dev) {
    void *pin = nullptr;
    WTB_TRY(pinned_reserve(sizeof(uint64_t) * cells, &pin));
    WTB_CUDA(cudaMemcpyAsync(pin, d_hist, sizeof(uint64_t) * cells, cudaMemcpyDeviceToHost, st));
    WTB_CUDA(cudaStreamSynchronize(st));
    const uint64_t *h = (const uint64_t *)pin;
    for (size_t i = 0; i < cells; ++i) hist[i] += h[i];
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_partial_wct(const void *y, const void *x1, const void *x2, int64_t batch, int n0, int nfft,
                               double dt, double dj, double s0, int J, double f0, int flags, void *pwc_out,
                               void *pphase_out, void *mwc_out, void *stream) {
  WTB_REQUIRE(y && x1 && x2 && batch >= 0 && n0 > 0, WTB_EINVAL, "wtb_partial_wct: bad inputs");
  WTB_REQUIRE(pwc_out || pphase_out || mwc_out, WTB_EINVAL, "wtb_partial_wct: no output requested");
  WTB_REQUIRE(nfft >= n0 && nfft >= 2, WTB_EINVAL, "nfft=%d must be >= n0=%d", nfft, n0);
  const bool f64 = flags & WTB_F64;
  const size_t elem = f64 ? sizeof(double) : sizeof(float);
  WTB_REQUIRE(route_of(nfft, elem) == Route::kOneCta, WTB_EUNSUPPORTED,   // partial coherence has no long kernels
              "wtb_partial_wct: nfft=%d is past one CTA per transform: a power of two up to %d, any other length up "
              "to %d for %s", nfft, cta_max_work(elem), cta_max_work(elem) / 2, f64 ? "double" : "float");
  WTB_ENTER(flags, y, stream);
  Axes ax;
  WTB_TRY(resolve_axes(n0, dt, dj, s0, J, f0, &ax));
  ScaleWin win;
  WTB_TRY(make_win(dj, &win));
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (f64)
    return pwct_entry<double>(y, x1, x2, batch, n0, nfft, dt, ax, f0, win, flags, pwc_out, pphase_out, mwc_out, st);
  return pwct_entry<float>(y, x1, x2, batch, n0, nfft, dt, ax, f0, win, flags, pwc_out, pphase_out, mwc_out, st);
}

extern "C" int wtb_partial_wct_mc_hist(double ay, double a1, double a2, double dt, double dj, double s0, int J,
                                       double f0, int64_t mc_first, int64_t mc_count, uint64_t seed,
                                       const void *surrogates, int flags, uint64_t *hist, void *stream) {
  WTB_REQUIRE(hist && mc_count >= 0 && mc_first >= 0, WTB_EINVAL, "wtb_partial_wct_mc_hist: bad arguments");
  WTB_REQUIRE(J >= 0, WTB_EINVAL, "wtb_partial_wct_mc_hist needs a resolved J");
  WTB_REQUIRE(fabs(ay) < 1 && fabs(a1) < 1 && fabs(a2) < 1, WTB_EINVAL, "AR(1) coefficients must lie in (-1, 1)");
  int nsurr = 0, maxscale = 0;
  WTB_TRY(wtb_wct_mc_geometry(dt, dj, s0, J, f0, &nsurr, &maxscale));
  const int N = (flags & WTB_FFT_NO_PAD) ? nsurr : (1 << ilog2(nsurr));   // pycwt with / without mkl_fft
  const bool f64 = flags & WTB_F64;
  const size_t elem = f64 ? sizeof(double) : sizeof(float);
  WTB_REQUIRE(route_of(N, elem) == Route::kOneCta, WTB_EUNSUPPORTED,   // partial coherence has no long kernels
              "wtb_partial_wct_mc_hist: %d-sample surrogates transform at nfft=%d, past one CTA per transform: a "
              "power of two up to %d, any other length up to %d for %s", nsurr, N, cta_max_work(elem),
              cta_max_work(elem) / 2, f64 ? "double" : "float");
  WTB_ENTER(flags, hist, stream);
  Axes ax;
  WTB_TRY(resolve_axes(nsurr, dt, dj, s0, J, f0, &ax));
  ScaleWin win;
  WTB_TRY(make_win(dj, &win));
  if (mc_count == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (f64)
    return pwct_mc_entry<double>(ay, a1, a2, dt, ax, f0, win, nsurr, N, maxscale, mc_first, mc_count, seed,
                                 surrogates, flags, hist, st);
  return pwct_mc_entry<float>(ay, a1, a2, dt, ax, f0, win, nsurr, N, maxscale, mc_first, mc_count, seed, surrogates,
                              flags, hist, st);
}
