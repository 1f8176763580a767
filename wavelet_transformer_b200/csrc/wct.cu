// Cross-wavelet / wavelet-coherence pipeline (pycwt.xwt, pycwt.wct,
// pycwt.wct_significance; reference call sites src/wct.py:106, src/xwt.py:93,122).
//
//   k_fwd_fft            X1, X2 = fft(y1), fft(y2)                     (cwt.cu)
//   k_wct_rows  (b, s)   W1, W2 = ifft(X * daughter_s)
//                        P  = (|W1|^2 + i |W2|^2) / s       two real fields packed in one FFT
//                        C  = W1 conj(W2) / s
//                        T  = ifft(gauss_s * fft(.))        time smoothing (Morlet.smooth)
//                        -> tsm[b, s, t] = (T1, T2, Re T12, Im T12)
//   k_wct_scale (b, t)   boxcar over scales (convolve2d 'same', zero fill), then
//                        WCT = |S12|^2 / (S1 S2)  -> output plane, or -> histogram bins
//
// The Gaussian filter is real and even, so filtering the packed field P gives
// smooth(|W1|^2) in its real part and smooth(|W2|^2) in its imaginary part.
#include "cwt_paths.cuh"
#include "spectral.cuh"

#include <type_traits>

namespace wtb {

// One CTA = one (pair, scale).  smem: 3 * N complex (U, V, tmp).
// xhat: [pairs, 2, N].  tsm: [pairs, S, n0] vec4.  phase/w12 optional [pairs,S,n0].
template <typename T>
__global__ void k_wct_rows(const cplx<T> *__restrict__ xhat, int n0, FftPlan<T> plan, int S,
                           const double *__restrict__ scales, double dt, double f0,
                           vec4<T> *__restrict__ tsm,
                           T *__restrict__ phase, cplx<T> *__restrict__ w12, int smooth) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T> *U = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *V = U + plan.M;
  cplx<T> *Tm = V + plan.M;
  const int N = plan.n;
  const int64_t pair = blockIdx.x / S;
  const int s = blockIdx.x % S;
  const cplx<T> *x1 = xhat + (pair * 2) * (int64_t)N;
  const cplx<T> *x2 = x1 + N;
  const double sc = scales[s];
  const T s_over_dt = T(sc / dt);
  const T norm = T(sqrt(2.0 * kPi * sc / dt) * kPiM14 / double(N));
  for (int k = threadIdx.x; k < N; k += blockDim.x) {
    const T d = morlet_daughter<T>(k, N, s_over_dt, norm, T(f0));
    const cplx<T> a = x1[k], b = x2[k];
    U[k] = mk<T>(a.x * d, a.y * d);
    V[k] = mk<T>(b.x * d, b.y * d);
  }
  __syncthreads();
  cplx<T> *r;
  r = plan_fft<T, +1>(U, Tm, plan);
  if (r != U) { Tm = U; U = r; }
  r = plan_fft<T, +1>(V, Tm, plan);
  if (r != V) { Tm = V; V = r; }
  // U = W1 row, V = W2 row (valid for t < n0; pycwt truncates before smoothing)
  const int64_t obase = (pair * S + s) * (int64_t)n0;
  const T inv_s = T(1.0 / sc);
  for (int t = threadIdx.x; t < N; t += blockDim.x) {
    cplx<T> p = mk<T>(T(0), T(0)), c = p;
    if (t < n0) {
      const cplx<T> a = U[t], b = V[t];
      const cplx<T> x = cmulc(a, b);  // W1 * conj(W2)
      if (w12) w12[obase + t] = x;
      if (phase) phase[obase + t] = dev_atan2<T>(x.y, x.x);
      p = mk<T>((a.x * a.x + a.y * a.y) * inv_s, (b.x * b.x + b.y * b.y) * inv_s);
      c = mk<T>(x.x * inv_s, x.y * inv_s);
    }
    U[t] = p;
    V[t] = c;
  }
  if (!smooth) return;
  __syncthreads();
  r = plan_fft<T, -1>(U, Tm, plan);
  if (r != U) { Tm = U; U = r; }
  r = plan_fft<T, -1>(V, Tm, plan);
  if (r != V) { Tm = V; V = r; }
  // Gaussian in the Fourier domain: exp(-0.5 (s/dt)^2 k^2), k = 2*pi*fftfreq(N)
  const T invN = T(1.0 / N);
  for (int k = threadIdx.x; k < N; k += blockDim.x) {
    const int kk = (k < (N + 1) / 2) ? k : k - N;
    const T w = T(2.0 * kPi) * T(kk) / T(N) * s_over_dt;
    const T g = dev_exp<T>(T(-0.5) * w * w) * invN;
    cplx<T> p = U[k], c = V[k];
    U[k] = mk<T>(p.x * g, p.y * g);
    V[k] = mk<T>(c.x * g, c.y * g);
  }
  __syncthreads();
  r = plan_fft<T, +1>(U, Tm, plan);
  if (r != U) { Tm = U; U = r; }
  r = plan_fft<T, +1>(V, Tm, plan);
  if (r != V) { Tm = V; V = r; }
  for (int t = threadIdx.x; t < n0; t += blockDim.x) {
    const cplx<T> p = U[t], c = V[t];
    vec4<T> o;
    o.x = p.x; o.y = p.y; o.z = c.x; o.w = c.y;
    tsm[obase + t] = o;
  }
}

// One thread = one (pair, t) column; walks the scales.  MODE 0: write WCT plane;
// MODE 1: add to the per-scale histogram for t inside [tlo[s], thi[s]] and s < maxscale.
template <typename T, int MODE>
__global__ void k_wct_scale(const vec4<T> *__restrict__ tsm, int64_t pairs, int n0, int S,
                            ScaleWin win, T *__restrict__ wct,
                            unsigned long long *__restrict__ hist, const int *__restrict__ tlo,
                            const int *__restrict__ thi, int maxscale) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= pairs * n0) return;
  const int64_t pair = gid / n0;
  const int t = (int)(gid % n0);
  const vec4<T> *col = tsm + pair * (int64_t)S * n0 + t;
  const int s_end = MODE == 1 ? maxscale : S;
  for (int s = 0; s < s_end; ++s) {
    if (MODE == 1 && (t < tlo[s] || t > thi[s])) continue;
    T s1 = 0, s2 = 0, cr = 0, ci = 0;
    for (int k = 0; k < win.K; ++k) {
      const int row = s + win.up - k;
      if (row < 0 || row >= S) continue;
      const vec4<T> v = col[(int64_t)row * n0];
      const T w = T(win.w[k]);
      s1 += w * v.x; s2 += w * v.y; cr += w * v.z; ci += w * v.w;
    }
    const T r2 = (cr * cr + ci * ci) / (s1 * s2);
    if (MODE == 0) {
      wct[(pair * S + s) * (int64_t)n0 + t] = r2;
    } else {
      if (r2 >= T(0)) {  // NaN (0/0) is skipped
        int bin = (int)floor(r2 * T(WTB_NBINS));
        bin = min(bin, WTB_NBINS - 1);
        atomicAdd(&hist[(size_t)s * WTB_NBINS + bin], 1ULL);
      }
    }
  }
}

static int make_win(double dj, ScaleWin *win) {
  // Morlet.smooth: rect(int(round(deltaj0/dj*2)), normalize=True), deltaj0 = 0.6
  const int K = (int)std::nearbyint(0.6 / dj * 2);
  WTB_REQUIRE(K >= 1 && K <= kMaxWin, WTB_EUNSUPPORTED, "scale window of %d taps (dj=%g) unsupported", K, dj);
  win->K = K;
  win->up = (K - 1) / 2;
  double sum = 0;
  for (int k = 0; k < K; ++k) {
    win->w[k] = (k == 0 || k == K - 1) ? 0.5 : 1.0;
    sum += win->w[k];
  }
  for (int k = 0; k < K; ++k) win->w[k] /= sum;
  return WTB_OK;
}

// Scale boxcar and coherence of tsm [pairs, S, n0]: the plane, or the histogram when d_hist.
template <typename T>
static int wct_scale_pass(const vec4<T> *d_tsm, int64_t pairs, int n0, int S, const ScaleWin &win, T *d_wct,
                          unsigned long long *d_hist, const int *d_tlo, const int *d_thi, int maxscale,
                          cudaStream_t st) {
  const int64_t cols = pairs * n0;
  const unsigned blocks = (unsigned)((cols + 255) / 256);
  if (d_hist)
    k_wct_scale<T, 1><<<blocks, 256, 0, st>>>(d_tsm, pairs, n0, S, win, nullptr, d_hist, d_tlo, d_thi, maxscale);
  else
    k_wct_scale<T, 0><<<blocks, 256, 0, st>>>(d_tsm, pairs, n0, S, win, d_wct, nullptr, nullptr, nullptr, 0);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

// Shared device pipeline.  d_y: [pairs, 2, n0] (series interleaved per pair).  generic: the generic kernels at
// every shape (WTB_GENERIC_ONLY).
template <typename T>
static int wct_device(const T *d_y, int64_t pairs, int n0, int N, double dt, double dj,
                      const Axes &ax, double f0, bool generic, T *d_wct, T *d_phase, cplx<T> *d_w12,
                      unsigned long long *d_hist, const int *h_tlo, const int *h_thi, int maxscale,
                      cudaStream_t st) {
  const int S = ax.J + 1;
  const bool smooth = d_wct || d_hist;
  if (cwt_long_takes(N, sizeof(T))) {
    // powers of two past one CTA's shared memory, up to 2^22: the four-step rows of wct_long.cu, then the same
    // scale boxcar and coherence kernels (WTB_GENERIC_ONLY has no other kernels for these lengths)
    ScaleWin win;
    WTB_TRY(make_win(dj, &win));
    WTB_REQUIRE(pairs * S < (1LL << 31) && pairs * 2 < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
    WctLongOut<T> o;
    WTB_TRY(wct_long<T>(d_y, pairs, n0, N, dt, ax, f0, smooth, d_phase, d_w12, d_hist ? h_tlo : nullptr,
                        d_hist ? h_thi : nullptr, &o, st));
    if (smooth) WTB_TRY(wct_scale_pass<T>(o.tsm, pairs, n0, S, win, d_wct, d_hist, o.tlo, o.thi, maxscale, st));
    return WTB_OK;
  }
  FftPlan<T> plan;
  WTB_TRY(make_plan<T>(N, &plan));
  const size_t smem_fwd = 2 * sizeof(cplx<T>) * (size_t)plan.M;
  const size_t smem_rows = 3 * sizeof(cplx<T>) * (size_t)plan.M;
  WTB_REQUIRE(smem_rows <= 227 * 1024, WTB_EUNSUPPORTED,
              "nfft=%d needs %zu B of shared memory per CTA (limit 227 KB): a power of two up to %d, any other "
              "length up to %d for %s", N, smem_rows, sizeof(T) == 4 ? 8192 : 4096, sizeof(T) == 4 ? 4096 : 2048,
              sizeof(T) == 4 ? "float" : "double");
  ScaleWin win;
  WTB_TRY(make_win(dj, &win));
  // FP32, nfft = 4096: the radix-16 forward kernel, and the register-FFT pipeline of wct_fast.cu where its one-sided
  // daughters hold (f0 >= kMinF0), its shared-memory rows and its boxcar ring fit
  const bool fast_fwd = std::is_same<T, float>::value && !generic && N == 4096;
  const bool fast = fast_fwd && f0 >= kMinF0 && S <= kMaxRowsC && win.K <= 32;
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t b_sc = al(sizeof(double) * S);
  const size_t b_rng = al(sizeof(int) * S);
  const size_t b_xh = al(sizeof(cplx<T>) * (size_t)pairs * 2 * N);
  const size_t b_ts = smooth ? al(sizeof(vec4<T>) * (size_t)pairs * S * N) : 0;  // N >= n0: also fits the fast path's spectra
  void *scratch = nullptr;
  const size_t b_rows = al(32 * (size_t)S);   // the fast path's row parameters (WRow)
  WTB_TRY(arena_reserve(b_sc + 2 * b_rng + b_rows + b_xh + b_ts, &scratch));
  char *p = (char *)scratch;
  void *d_rows_scratch = p; p += b_rows;
  double *d_scales = (double *)p; p += b_sc;
  int *d_tlo = (int *)p; p += b_rng;
  int *d_thi = (int *)p; p += b_rng;
  cplx<T> *d_xhat = (cplx<T> *)p; p += b_xh;
  vec4<T> *d_tsm = (vec4<T> *)p;
  WTB_CUDA(cudaMemcpyAsync(d_scales, ax.scales.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  if (d_hist) {
    WTB_CUDA(cudaMemcpyAsync(d_tlo, h_tlo, sizeof(int) * S, cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync(d_thi, h_thi, sizeof(int) * S, cudaMemcpyHostToDevice, st));
  }
  const int threads = plan.M >= 1024 ? 256 : (plan.M >= 256 ? 128 : 64);
  WTB_CUDA(cudaFuncSetAttribute(k_fwd_fft<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fwd));
  WTB_CUDA(cudaFuncSetAttribute(k_wct_rows<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_rows));
  WTB_REQUIRE(pairs * S < (1LL << 31) && pairs * 2 < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
  WTB_TRACE_POINT(st, "wct: scratch + small copies");
  if (fast_fwd) {
    WTB_TRY(fwd_fft_4096((const float *)d_y, pairs * 2, n0, (float2 *)d_xhat, st));
  } else {
    k_fwd_fft<T><<<(unsigned)(pairs * 2), threads, smem_fwd, st>>>(d_y, n0, plan, d_xhat);
    WTB_LAUNCH_CHECK();
  }
  WTB_TRACE_POINT(st, "wct: forward transforms");
  if (fast)
    return wct_fast((const float2 *)d_xhat, pairs, n0, dt, ax, f0, d_rows_scratch, (float4 *)d_tsm, win,
                    (float *)d_wct, (float *)d_phase, (float2 *)d_w12, d_hist, d_tlo, d_thi, maxscale, st);
  k_wct_rows<T><<<(unsigned)(pairs * S), threads, smem_rows, st>>>(
      d_xhat, n0, plan, S, d_scales, dt, f0, d_tsm, d_phase, d_w12, smooth ? 1 : 0);
  WTB_LAUNCH_CHECK();
  if (smooth) WTB_TRY(wct_scale_pass<T>(d_tsm, pairs, n0, S, win, d_wct, d_hist, d_tlo, d_thi, maxscale, st));
  return WTB_OK;
}

// bytes of arena + staging one pair costs (for batching decisions)
template <typename T> static size_t pair_bytes(int n0, int N, int S) {
  return sizeof(cplx<T>) * 2 * (size_t)N + sizeof(vec4<T>) * (size_t)S * N;
}

static thread_local bool g_in_shard = false;   // set on a pool worker while it runs its block

template <typename T>
static int xwt_wct_entry(const void *y1, const void *y2, int64_t batch, int n0, int N, double dt,
                         double dj, const Axes &ax, double f0, int flags, void *wct_out,
                         void *phase_out, void *w12_out, cudaStream_t st) {
  const int S = ax.J + 1;
  const size_t plane = (size_t)S * n0;
  // host buffers, several GPUs (wtb_init_multi): contiguous blocks of pairs, one per device
  if (!(flags & WTB_DEVICE_PTRS) && pool_size() > 1 && batch >= 2 * pool_size() && !g_in_shard) {
    return run_sharded_fn(batch, 2, st, [&](int, int64_t first, int64_t count, cudaStream_t s) {
      g_in_shard = true;
      const int rc = xwt_wct_entry<T>((const T *)y1 + first * n0, (const T *)y2 + first * n0, count, n0, N, dt, dj, ax,
                                      f0, flags, wct_out ? (T *)wct_out + first * plane : nullptr,
                                      phase_out ? (T *)phase_out + first * plane : nullptr,
                                      w12_out ? (cplx<T> *)w12_out + first * plane : nullptr, s);
      g_in_shard = false;
      return rc;
    });
  }
  // stage inputs interleaved [pair, 2, n0] and outputs per chunk
  const size_t per_pair = sizeof(T) * (2 * (size_t)n0 + (wct_out ? plane : 0) + (phase_out ? plane : 0) +
                                       (w12_out ? 2 * plane : 0));
  const size_t budget = size_t(1) << 30;
  const int64_t rows = std::max<int64_t>(
      1, std::min<int64_t>(batch, (int64_t)(budget / (per_pair + pair_bytes<T>(n0, N, S)))));
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  void *stage = nullptr;
  WTB_TRY(staging_reserve(al(sizeof(T) * rows * 2 * n0) + al(sizeof(T) * rows * plane) * 4 + 1024, &stage));
  char *p = (char *)stage;
  T *d_y = (T *)p; p += al(sizeof(T) * rows * 2 * n0);
  T *d_wct = nullptr, *d_phase = nullptr;
  cplx<T> *d_w12 = nullptr;
  const bool dev = flags & WTB_DEVICE_PTRS;
  if (wct_out) { d_wct = (T *)p; p += al(sizeof(T) * rows * plane); }
  if (phase_out) { d_phase = (T *)p; p += al(sizeof(T) * rows * plane); }
  if (w12_out) { d_w12 = (cplx<T> *)p; }
  const cudaMemcpyKind in_kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  for (int64_t b0 = 0; b0 < batch; b0 += rows) {
    const int64_t nb = std::min(rows, batch - b0);
    // interleave y1/y2 rows: dst pitch 2*n0, src pitch n0
    WTB_CUDA(cudaMemcpy2DAsync(d_y, sizeof(T) * 2 * n0, (const T *)y1 + b0 * n0, sizeof(T) * n0,
                               sizeof(T) * n0, nb, in_kind, st));
    WTB_CUDA(cudaMemcpy2DAsync(d_y + n0, sizeof(T) * 2 * n0, (const T *)y2 + b0 * n0, sizeof(T) * n0,
                               sizeof(T) * n0, nb, in_kind, st));
    T *o_wct = dev && wct_out ? (T *)wct_out + b0 * plane : d_wct;
    T *o_phase = dev && phase_out ? (T *)phase_out + b0 * plane : d_phase;
    cplx<T> *o_w12 = dev && w12_out ? (cplx<T> *)w12_out + b0 * plane : d_w12;
    WTB_TRY(wct_device<T>(d_y, nb, n0, N, dt, dj, ax, f0, flags & WTB_GENERIC_ONLY, o_wct, o_phase, o_w12, nullptr,
                          nullptr, nullptr, 0, st));
    if (!dev) {
      if (wct_out)
        WTB_TRY(copy_to_host((T *)wct_out + b0 * plane, d_wct, sizeof(T) * nb * plane, st));
      if (phase_out)
        WTB_TRY(copy_to_host((T *)phase_out + b0 * plane, d_phase, sizeof(T) * nb * plane, st));
      if (w12_out)
        WTB_TRY(copy_to_host((cplx<T> *)w12_out + b0 * plane, d_w12, sizeof(cplx<T>) * nb * plane, st));
      WTB_CUDA(cudaStreamSynchronize(st));
    }  // device buffers: chunks reuse the arena without a host sync (all work is ordered on `st`)
  }
  return WTB_OK;
}

// implemented in noise.cu
template <typename T>
int rednoise_device(double a1, double a2, int nsurr, int64_t first, int64_t count, uint64_t seed,
                    bool white, T *d_out, cudaStream_t st);

// Reliable-region column range per scale, evaluated in double exactly as pycwt does.
static void coi_ranges(int nsurr, double dt, const Axes &ax, double f0, std::vector<int> *tlo,
                       std::vector<int> *thi, std::vector<uint8_t> *any) {
  const int S = ax.J + 1;
  const double c = morlet_flambda(f0) / std::sqrt(2.0) * dt;
  tlo->assign(S, 1);
  thi->assign(S, 0);
  any->assign(S, 0);
  // pycwt's predicate, period <= coi[t], with coi[t] = c (N/2 - |t - (N-1)/2|) in the same double
  // operations.  |t - (N-1)/2| and N/2 - that are exact, and multiplying by c > 0 is monotone,
  // so the predicate is monotone on either side of the centre: two binary searches per scale
  // give the same interval a scan over t would (a scan costs S x N evaluations per call --
  // 0.3 ms at the cfg5 shape, comparable to a 300-realisation run).
  auto coi_at = [&](int t) { return c * (nsurr / 2.0 - std::fabs(t - (nsurr - 1) / 2.0)); };
  const int mid_lo = (nsurr - 1) / 2, mid_hi = nsurr / 2;   // the one or two samples next to the centre
  for (int s = 0; s < S; ++s) {
    const double period = 1.0 / ax.freqs[s];
    if (!(period <= coi_at(mid_lo)) && !(period <= coi_at(mid_hi))) continue;
    int a = 0, b = mid_lo;                   // first t in [0, mid_lo] inside (mid_lo is: coi is symmetric)
    while (a < b) {
      const int m = (a + b) / 2;
      if (period <= coi_at(m)) b = m; else a = m + 1;
    }
    int lo = a;
    a = mid_hi; b = nsurr - 1;               // last t in [mid_hi, N-1] inside
    while (a < b) {
      const int m = (a + b + 1) / 2;
      if (period <= coi_at(m)) a = m; else b = m - 1;
    }
    (*tlo)[s] = lo; (*thi)[s] = a; (*any)[s] = 1;
  }
}

void mc_row_has_points(int nsurr, double dt, const Axes &ax, double f0, std::vector<uint8_t> *any) {
  std::vector<int> tlo, thi;
  coi_ranges(nsurr, dt, ax, f0, &tlo, &thi, any);
}

// Percentile step on the device, one thread per scale row, the SAME double operations in the same
// order as wtb_wct_sig_from_hist (runtime.cu) -- explicit _rn intrinsics so that no multiply-add
// is contracted: bit-identical thresholds, and the whole Monte-Carlo step stays on one stream.
__global__ void k_sig_from_hist(const unsigned long long *__restrict__ hist, int S, int maxscale, double level,
                                const uint8_t *__restrict__ has_points, double *__restrict__ sig95) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const int nb = WTB_NBINS;
  if (s >= maxscale) {
    sig95[s] = (has_points && has_points[s]) ? __longlong_as_double(0x7ff8000000000000LL) : 0.0;
    return;
  }
  const unsigned long long *h = hist + (size_t)s * nb;
  unsigned long long tot_i = 0;
  int b_first = -1, b_last = -1;
  for (int b = 0; b < nb; ++b)
    if (h[b]) { tot_i += h[b]; if (b_first < 0) b_first = b; b_last = b; }
  if (b_first < 0) { sig95[s] = __longlong_as_double(0x7ff8000000000000LL); return; }
  // the host loop accumulates the counts in double: sums of integers below 2^53 are exact
  const double tot = (double)tot_i;
  auto Pof = [&](double cum) { return __ddiv_rn(__dsub_rn(cum, 0.5), tot); };
  auto Yof = [&](int b) { return __ddiv_rn(__dadd_rn((double)b, 0.5), (double)nb); };
  const double P_front = Pof((double)h[b_first]), P_back = Pof(tot);
  double v;
  if (level <= P_front) v = Yof(b_first);
  else if (level >= P_back) v = Yof(b_last);
  else {
    // interval [i-1, i] over the non-empty bins with P[i-1] <= level < P[i]
    double cum = (double)h[b_first];
    double p_prev = P_front, p_cur = P_front;
    int y_prev = b_first, y_cur = b_first;
    for (int b = b_first + 1; b <= b_last; ++b) {
      if (!h[b]) continue;
      cum = __dadd_rn(cum, (double)h[b]);
      p_prev = p_cur; y_prev = y_cur;
      p_cur = Pof(cum); y_cur = b;
      if (p_cur > level) break;
    }
    const double slope = __ddiv_rn(__dsub_rn(Yof(y_cur), Yof(y_prev)), __dsub_rn(p_cur, p_prev));
    v = __dadd_rn(__dmul_rn(slope, __dsub_rn(level, p_prev)), Yof(y_prev));
  }
  sig95[s] = v;
}

template <typename T>
static int mc_hist_entry(double a1, double a2, double dt, double dj, const Axes &ax, double f0,
                         int nsurr, int maxscale, int64_t mc_first, int64_t mc_count, uint64_t seed,
                         const void *surrogates, int flags, uint64_t *hist, cudaStream_t st) {
  const int S = ax.J + 1;
  const int N = (flags & WTB_FFT_NO_PAD) ? nsurr : (1 << ilog2(nsurr));   // pycwt with / without mkl_fft
  std::vector<int> tlo, thi;
  std::vector<uint8_t> any;
  WTB_TRACE_POINT(st, "mc: entry");
  coi_ranges(nsurr, dt, ax, f0, &tlo, &thi, &any);
  WTB_TRACE_POINT(st, "mc: coi ranges");
  const bool dev = flags & WTB_DEVICE_PTRS;
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t per_pair = sizeof(T) * 2 * (size_t)nsurr + pair_bytes<T>(nsurr, N, S);
  // Intermediates per chunk.  Launch tails are what chunking costs (1.5 GiB chunks: 253 k pairs/s,
  // one 18 GB chunk: 263 k at 2048 pairs), so the default spends a tenth of the 180 GB HBM3e;
  // chunks are balanced so that no short tail chunk is left over.
  size_t budget = size_t(20) << 30;
  if (const char *e = std::getenv("WTB_MC_CHUNK_MB")) {
    budget = (size_t)std::max(1, std::atoi(e)) << 20;
  } else if (per_pair * (size_t)mc_count > (size_t(4) << 30)) {
    // never ask for more than half of what is free right now.  cudaMemGetInfo costs 1.6 - 8 ms of
    // host time on this driver (WTB_TRACE), more than a whole 300-realisation run: only jobs
    // that want more than 4 GiB of scratch pay for the question.
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
      budget = std::max(size_t(3) << 29, std::min(budget, free_b / 2));
  }
  const int64_t rows_max = std::max<int64_t>(1, (int64_t)(budget / per_pair));
  const int64_t n_chunks = (mc_count + rows_max - 1) / rows_max;
  const int64_t rows = std::max<int64_t>(1, (mc_count + n_chunks - 1) / std::max<int64_t>(1, n_chunks));
  void *stage = nullptr;
  const size_t b_hist = al(sizeof(uint64_t) * S * WTB_NBINS);
  const size_t b_y = al(sizeof(T) * rows * 2 * nsurr);
  // Host-injected surrogates in several chunks: two staging buffers, the copy of chunk k + 1 runs
  // on a copy stream while the kernels of chunk k run (2.7 GB of H2D for 100 000 realisations is
  // 49 ms next to 290 ms of kernels when they are serial).
  const bool pipelined = surrogates && !dev && n_chunks >= 2;
  WTB_TRY(staging_reserve((pipelined ? 2 : 1) * b_y + b_hist, &stage));
  T *d_ybuf[2] = {(T *)stage, (T *)((char *)stage + (pipelined ? b_y : 0))};
  unsigned long long *d_hist = (unsigned long long *)((char *)stage + (pipelined ? 2 : 1) * b_y);
  unsigned long long *hist_dev = dev ? (unsigned long long *)hist : d_hist;
  if (!dev) WTB_CUDA(cudaMemsetAsync(d_hist, 0, sizeof(uint64_t) * S * WTB_NBINS, st));
  WTB_TRACE_POINT(st, "mc: budget, staging, memset");
  cudaStream_t cs = st;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // copied[2], consumed[2], entry
  struct EvGuard {
    cudaEvent_t *e;
    ~EvGuard() { for (int i = 0; i < 5; ++i) if (e[i]) cudaEventDestroy(e[i]); }
  } guard{ev};
  auto copy_chunk = [&](int64_t m0, int buf) -> int {
    const int64_t nb = std::min(rows, mc_count - m0);
    WTB_CUDA(cudaMemcpyAsync(d_ybuf[buf], (const T *)surrogates + m0 * 2 * nsurr, sizeof(T) * nb * 2 * nsurr,
                             cudaMemcpyHostToDevice, cs));
    if (pipelined) WTB_CUDA(cudaEventRecord(ev[buf], cs));
    return WTB_OK;
  };
  if (pipelined) {
    WTB_TRY(copy_stream(&cs));
    for (int i = 0; i < 5; ++i) WTB_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    WTB_CUDA(cudaEventRecord(ev[4], st));              // the staging buffers may still feed the previous call
    WTB_CUDA(cudaStreamWaitEvent(cs, ev[4], 0));
    WTB_TRY(copy_chunk(0, 0));
  }
  int64_t chunk = 0;
  for (int64_t m0 = 0; m0 < mc_count; m0 += rows, ++chunk) {
    const int64_t nb = std::min(rows, mc_count - m0);
    const int buf = pipelined ? (int)(chunk & 1) : 0;
    const T *src = d_ybuf[buf];
    if (surrogates) {
      if (dev) {
        src = (const T *)surrogates + m0 * 2 * nsurr;
      } else if (pipelined) {
        if (m0 + rows < mc_count) {                    // start the next chunk's copy before this chunk's kernels
          if (chunk >= 1) WTB_CUDA(cudaStreamWaitEvent(cs, ev[2 + (buf ^ 1)], 0));
          WTB_TRY(copy_chunk(m0 + rows, buf ^ 1));
        }
        WTB_CUDA(cudaStreamWaitEvent(st, ev[buf], 0));
      } else {
        WTB_TRY(copy_chunk(m0, 0));
      }
    } else {
      WTB_TRY(rednoise_device<T>(a1, a2, nsurr, mc_first + m0, nb, seed, flags & WTB_NOISE_WHITE, d_ybuf[0], st));
    }
    WTB_TRACE_POINT(st, "mc: surrogates");
    WTB_TRY(wct_device<T>(src, nb, nsurr, N, dt, dj, ax, f0, flags & WTB_GENERIC_ONLY, nullptr, nullptr, nullptr,
                          hist_dev, tlo.data(), thi.data(), maxscale, st));
    if (pipelined) WTB_CUDA(cudaEventRecord(ev[2 + buf], st));
    // chunks reuse the arena without a host sync: every kernel and copy is ordered on `st`
    WTB_TRACE_POINT(st, "mc: pipeline (fft, A, C, B)");
  }
  if (!dev) {
    // through a pinned bounce buffer: a pageable 528 KB copy costs 0.2 - 0.3 ms, this one 30 us
    const size_t cells = (size_t)S * WTB_NBINS;
    void *pin = nullptr;
    WTB_TRY(pinned_reserve(sizeof(uint64_t) * cells, &pin));
    const uint64_t *h = (const uint64_t *)pin;
    WTB_CUDA(cudaMemcpyAsync(pin, d_hist, sizeof(uint64_t) * cells, cudaMemcpyDeviceToHost, st));
    WTB_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < cells; ++i) hist[i] += h[i];
    WTB_TRACE_POINT(st, "mc: histogram to host");
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_xwt_wct(const void *y1, const void *y2, int64_t batch, int n0, int nfft, double dt,
                           double dj, double s0, int J, double f0, int flags, void *wct_out,
                           void *phase_out, void *w12_out, void *stream) {
  WTB_REQUIRE(y1 && y2 && batch >= 0 && n0 > 0, WTB_EINVAL, "wtb_xwt_wct: bad inputs");
  WTB_REQUIRE(wct_out || phase_out || w12_out, WTB_EINVAL, "wtb_xwt_wct: no output requested");
  WTB_REQUIRE(nfft >= n0 && nfft >= 2, WTB_EINVAL, "nfft=%d must be >= n0=%d", nfft, n0);
  WTB_ENTER(flags, y1, stream);
  Axes ax;
  WTB_TRY(resolve_axes(n0, dt, dj, s0, J, f0, &ax));
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64)
    return xwt_wct_entry<double>(y1, y2, batch, n0, nfft, dt, dj, ax, f0, flags, wct_out, phase_out, w12_out, st);
  return xwt_wct_entry<float>(y1, y2, batch, n0, nfft, dt, dj, ax, f0, flags, wct_out, phase_out, w12_out, st);
}

extern "C" int wtb_wct_mc_hist(double a1, double a2, double dt, double dj, double s0, int J, double f0,
                               int64_t mc_first, int64_t mc_count, uint64_t seed, const void *surrogates,
                               int flags, uint64_t *hist, void *stream) {
  WTB_REQUIRE(hist && mc_count >= 0 && mc_first >= 0, WTB_EINVAL, "wtb_wct_mc_hist: bad arguments");
  WTB_REQUIRE(J >= 0, WTB_EINVAL, "wtb_wct_mc_hist needs a resolved J");
  WTB_REQUIRE(fabs(a1) < 1 && fabs(a2) < 1, WTB_EINVAL, "AR(1) coefficients must lie in (-1, 1)");
  WTB_ENTER(flags, hist, stream);
  int nsurr = 0, maxscale = 0;
  WTB_TRY(wtb_wct_mc_geometry(dt, dj, s0, J, f0, &nsurr, &maxscale));
  Axes ax;
  WTB_TRY(resolve_axes(nsurr, dt, dj, s0, J, f0, &ax));
  if (mc_count == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64)
    return mc_hist_entry<double>(a1, a2, dt, dj, ax, f0, nsurr, maxscale, mc_first, mc_count, seed,
                                 surrogates, flags, hist, st);
  return mc_hist_entry<float>(a1, a2, dt, dj, ax, f0, nsurr, maxscale, mc_first, mc_count, seed,
                              surrogates, flags, hist, st);
}

// Device-resident percentile step: hist and sig95 are device buffers, has_points (may be NULL) is a
// HOST array of S flags; everything is enqueued on `stream`.
extern "C" int wtb_wct_sig_from_hist_device(const uint64_t *hist, int S, int maxscale, double level,
                                            const uint8_t *row_has_points, double *sig95, void *stream) {
  WTB_REQUIRE(hist && sig95 && S > 0 && S <= 4096, WTB_EINVAL, "wtb_wct_sig_from_hist_device: bad arguments");
  WTB_REQUIRE(maxscale >= 0 && maxscale <= S, WTB_EINVAL, "maxscale out of range");
  WTB_ENTER(WTB_DEVICE_PTRS, hist, stream);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t *d_flags = nullptr;
  if (row_has_points) {
    void *prm = nullptr;
    WTB_TRY(params_reserve(4096, &prm));
    d_flags = (uint8_t *)prm;
    WTB_CUDA(cudaMemcpyAsync(d_flags, row_has_points, S, cudaMemcpyHostToDevice, st));
  }
  k_sig_from_hist<<<(S + 63) / 64, 64, 0, st>>>((const unsigned long long *)hist, S, maxscale, level, d_flags, sig95);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}
