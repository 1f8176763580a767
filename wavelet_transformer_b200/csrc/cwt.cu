// Batched CWT (pycwt.cwt, src/cwt.py:110-114 of the reference), Morlet unless stated:
//   X = fft(x, nfft);  W[s,:] = ifft(X * sqrt(2*pi*s/dt) * pi^-1/4 * exp(-(s*w-f0)^2/2));
//   power = |W|^2, truncated to the first n0 samples.
// Generic kernels (any pow2 nfft, float/double) live here; cwt_plan picks them or one of
// the FP32 fast paths (cwt_fast.cu, wct_fast.cu) or the long transforms (cwt_long.cu).
#include "cwt_paths.cuh"
#include "spectral.cuh"

namespace wtb {

// One CTA = one (series, chunk of scales).  smem: 2 * N complex.
template <typename T>
__global__ void k_cwt_rows(const cplx<T> *__restrict__ xhat, int n0, FftPlan<T> plan, int S,
                           int chunk, const double *__restrict__ scales, double dt, double f0,
                           T *__restrict__ power,
                           cplx<T> *__restrict__ coef, int coi_mask, double coi_c, double flambda,
                           int mother, int order, T pre_re, T pre_im) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T> *a = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *b = a + plan.M;
  const int N = plan.n;
  const int nchunks = (S + chunk - 1) / chunk;
  const int64_t row = blockIdx.x / nchunks;
  const int c = blockIdx.x % nchunks;
  const cplx<T> *xh = xhat + row * N;
  const int s_end = min(S, (c + 1) * chunk);
  for (int s = c * chunk; s < s_end; ++s) {
    const double sc = scales[s];
    const T s_over_dt = T(sc / dt);
    // (s * ftfreqs[1] * N)^0.5 * pi^-0.25, times 1/N of the inverse transform
    const T norm = T(sqrt(2.0 * kPi * sc / dt) * kPiM14 / double(N));
    const T nrm = T(sqrt(2.0 * kPi * sc / dt) / double(N));
    for (int k = threadIdx.x; k < N; k += blockDim.x)
      a[k] = daughter_mul<T>(xh[k], k, N, mother, order, s_over_dt, norm, nrm, T(f0), pre_re, pre_im);
    __syncthreads();
    cplx<T> *r = plan_fft<T, +1>(a, b, plan);
    const int64_t obase = (row * S + s) * (int64_t)n0;
    const double period = 1.0 / (1.0 / (flambda * sc));
    for (int t = threadIdx.x; t < n0; t += blockDim.x) {
      const cplx<T> w = r[t];
      if (coef) coef[obase + t] = w;
      if (power) {
        T p = w.x * w.x + w.y * w.y;
        if (coi_mask) {
          const double coi = coi_c * (n0 / 2.0 - fabs(t - (n0 - 1) / 2.0));
          if (period > coi) p = T(NAN);
        }
        power[obase + t] = p;
      }
    }
    __syncthreads();  // r may alias a; next iteration overwrites it
  }
}

// smallest batch a fast kernel takes: WTB_CWT_MIN_BATCH overrides the default (the tests set 1); read on every call
static int64_t min_fast_batch(int64_t dflt) {
  const char *e = std::getenv("WTB_CWT_MIN_BATCH");
  return e ? std::atoll(e) : dflt;
}

CwtPlan cwt_plan(int64_t batch, int n0, int N, int S, double f0, int mother, size_t elem, int flags, bool power,
                 bool coef) {
  const bool fast = elem == sizeof(float) && mother == WTB_MORLET && !(flags & WTB_GENERIC_ONLY);
  const bool power_only = power && !coef;
  // With the rows of a series split over warps, k_cwt_fast_1024 is ahead of the generic kernel at every batch size
  // for nfft = 1024 (0.017 ms for one series against 0.018); two series per warp (nfft = 512) pays off from about
  // 20 series (0.021 ms flat against 0.017 + 0.4 us per series).
  if (fast && power_only && (N == 1024 || N == 512) && f0 >= kZCut && S <= kMaxRows &&
      batch >= min_fast_batch(N == 512 ? 20 : 1))
    return {Fwd::kInKernel, N == 512 ? Rows::kFast512Pairs : Rows::kFast1024};
  if (cwt_long_takes(N, elem)) return {Fwd::kInKernel, Rows::kLong};
  if (!fast) return {Fwd::kGeneric, Rows::kGeneric};
  // k_cwt_dif stores the first half of a row unconditionally (n0 > nfft / 2).  The rows of a series are split over
  // CTAs when the batch is small, but this path also pays for the separate forward-FFT launch: 0.040 ms for 12
  // series of 1346 samples against 0.021 ms + 1.7 us per series for the generic kernel (nfft = 2048 starts at 12
  // series).  nfft = 4096: the register rows of wct_fast.cu (one CTA per two series and scale: finer work items)
  // are faster or equal up to a few series per SM -- 0.037 / 0.064 / 0.110 / 0.185 / 0.286 ms for 12 / 64 / 148 /
  // 300 / 500 series against 0.061 / 0.075 / 0.107 / 0.194 / 0.281 ms for k_cwt_dif<4>; 1000 series: 0.532 against
  // 0.505 ms, 4000: 2.04 against 1.87.
  if (power_only && (N == 2048 || N == 4096) && f0 >= kZCut && S <= kMaxRowsF && n0 > N / 2 &&
      batch >= min_fast_batch(N == 2048 ? kMinBatchF : 4 * (int64_t)sm_count()))
    return N == 2048 ? CwtPlan{Fwd::kPair2048, Rows::kDif2048} : CwtPlan{Fwd::kRadix16Layout4096, Rows::kDif4096};
  if (N == 4096) {
    if (f0 >= kMinF0 && S <= kMaxRowsC) return {Fwd::kRadix16_4096, Rows::kRows4096};
    // no fast row kernel takes this f0 or this many scales, but k_cwt_rows reads the radix-16 kernel's spectra
    return {Fwd::kRadix16_4096, Rows::kGeneric};
  }
  return {Fwd::kGeneric, Rows::kGeneric};
}

// also the first pass of wtb_cwt_averages (averages.cu)
template <typename T>
int cwt_device(const T *d_x, int64_t batch, int n0, int N, double dt, const Axes &ax,
               const Mother &mo, int flags, T *d_power, cplx<T> *d_coef, cudaStream_t st) {
  const int S = ax.J + 1;
  const double f0 = mo.kind == WTB_MORLET ? mo.param : 0.0;
  const CwtPlan pl = cwt_plan(batch, n0, N, S, f0, mo.kind, sizeof(T), flags, d_power != nullptr, d_coef != nullptr);
  switch (pl.rows) {
    case Rows::kFast1024:
    case Rows::kFast512Pairs:
      return cwt_fast_1024(pl, (const float *)d_x, batch, n0, dt, ax, f0, flags, (float *)d_power, st);
    case Rows::kLong:
      return cwt_long<T>(d_x, batch, n0, N, dt, ax, mo, flags, d_power, d_coef, st);
    default:
      break;
  }
  // the other row kernels read the forward spectra from the arena
  FftPlan<T> plan;
  WTB_TRY(make_plan<T>(N, &plan));
  const size_t smem = 2 * sizeof(cplx<T>) * (size_t)plan.M;
  WTB_REQUIRE(smem <= 227 * 1024, WTB_EUNSUPPORTED,
              "nfft=%d needs %zu B of shared memory per CTA (limit 227 KB): a power of two up to %d, any other "
              "length up to %d for %s", N, smem, sizeof(T) == 4 ? 8192 : 4096, sizeof(T) == 4 ? 4096 : 2048,
              sizeof(T) == 4 ? "float" : "double");
  void *scratch = nullptr;
  const size_t sc_bytes = ((sizeof(double) * S + 255) / 256) * 256;
  WTB_TRY(arena_reserve(sc_bytes + sizeof(cplx<T>) * (size_t)batch * N, &scratch));
  double *d_scales = (double *)scratch;
  cplx<T> *d_xhat = (cplx<T> *)((char *)scratch + sc_bytes);
  WTB_CUDA(cudaMemcpyAsync(d_scales, ax.scales.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  const int threads = plan.M >= 1024 ? 256 : (plan.M >= 256 ? 128 : 64);
  WTB_CUDA(cudaFuncSetAttribute(k_fwd_fft<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  WTB_CUDA(cudaFuncSetAttribute(k_cwt_rows<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (pl.rows == Rows::kDif2048 || pl.rows == Rows::kDif4096)   // with its own forward transforms (group layout)
    return cwt_dif(pl, (const float *)d_x, (float2 *)d_xhat, batch, n0, dt, ax, f0, flags, (float *)d_power, st);
  if (pl.fwd == Fwd::kRadix16_4096) {
    WTB_TRY(fwd_fft_4096((const float *)d_x, batch, n0, (float2 *)d_xhat, st));
  } else {
    k_fwd_fft<T><<<(unsigned)batch, threads, smem, st>>>(d_x, n0, plan, d_xhat);
    WTB_LAUNCH_CHECK();
  }
  if (pl.rows == Rows::kRows4096)
    return cwt_rows_4096((const float2 *)d_xhat, batch, n0, dt, ax, f0, flags, (float *)d_power, (float2 *)d_coef, st);
  // enough CTAs to fill the machine for small batches, few forward-FFT re-reads for large ones
  int chunk = S;
  const int64_t want = 4LL * sm_count();
  if (batch < want) chunk = (int)std::max<int64_t>(1, (int64_t)S * batch / want);
  chunk = std::max(1, std::min(chunk, 16));
  const int nchunks = (S + chunk - 1) / chunk;
  WTB_REQUIRE(batch * nchunks < (1LL << 31), WTB_EUNSUPPORTED, "batch too large for one launch");
  double pre_re, pre_im;
  mother_prefactor(mo, &pre_re, &pre_im);
  k_cwt_rows<T><<<(unsigned)(batch * nchunks), threads, smem, st>>>(
      d_xhat, n0, plan, S, chunk, d_scales, dt, f0, d_power, d_coef,
      (flags & WTB_COI_MASK) ? 1 : 0, mother_flambda(mo) * mother_coi(mo) * dt, mother_flambda(mo), mo.kind,
      (int)mo.param, T(pre_re), T(pre_im));
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}
template int cwt_device<float>(const float *, int64_t, int, int, double, const Axes &, const Mother &, int, float *,
                               float2 *, cudaStream_t);
template int cwt_device<double>(const double *, int64_t, int, int, double, const Axes &, const Mother &, int, double *,
                                double2 *, cudaStream_t);

static thread_local bool g_in_shard = false;   // set on a pool worker while it runs its block

template <typename T>
static int cwt_entry(const void *x, int64_t batch, int n0, int N, double dt, const Axes &ax,
                     const Mother &f0, int flags, void *power_out, void *coef_out, cudaStream_t st) {
  const int S = ax.J + 1;
  if (flags & WTB_DEVICE_PTRS)
    return cwt_device<T>((const T *)x, batch, n0, N, dt, ax, f0, flags, (T *)power_out,
                         (cplx<T> *)coef_out, st);
  // host buffers, several GPUs (wtb_init_multi): contiguous blocks of series, one per device
  if (pool_size() > 1 && batch >= 2 * pool_size() && !g_in_shard) {
    return run_sharded_fn(batch, 2, st, [&](int, int64_t first, int64_t count, cudaStream_t s) {
      g_in_shard = true;
      const int rc = cwt_entry<T>((const T *)x + first * n0, count, n0, N, dt, ax, f0, flags,
                                  power_out ? (T *)power_out + first * S * n0 : nullptr,
                                  coef_out ? (cplx<T> *)coef_out + first * S * n0 : nullptr, s);
      g_in_shard = false;
      return rc;
    });
  }
  // host buffers: stream the batch through a bounded staging arena
  const size_t per_row = sizeof(T) * ((size_t)n0 + (power_out ? (size_t)S * n0 : 0) +
                                      (coef_out ? 2 * (size_t)S * n0 : 0));
  const size_t budget = size_t(1) << 30;
  int64_t rows = std::max<int64_t>(1, std::min<int64_t>(batch, (int64_t)(budget / per_row)));
  void *stage = nullptr;
  WTB_TRY(staging_reserve(per_row * rows + 1024, &stage));
  T *d_x = (T *)stage;
  size_t off = (sizeof(T) * (size_t)rows * n0 + 255) / 256 * 256;
  T *d_power = nullptr;
  cplx<T> *d_coef = nullptr;
  if (power_out) { d_power = (T *)((char *)stage + off); off += (sizeof(T) * (size_t)rows * S * n0 + 255) / 256 * 256; }
  if (coef_out) d_coef = (cplx<T> *)((char *)stage + off);
  for (int64_t b0 = 0; b0 < batch; b0 += rows) {
    const int64_t nb = std::min(rows, batch - b0);
    WTB_CUDA(cudaMemcpyAsync(d_x, (const T *)x + b0 * n0, sizeof(T) * nb * n0, cudaMemcpyHostToDevice, st));
    WTB_TRY(cwt_device<T>(d_x, nb, n0, N, dt, ax, f0, flags, d_power, d_coef, st));
    if (power_out)
      WTB_TRY(copy_to_host((T *)power_out + b0 * S * n0, d_power, sizeof(T) * nb * S * n0, st));
    if (coef_out)
      WTB_TRY(copy_to_host((cplx<T> *)coef_out + b0 * S * n0, d_coef, sizeof(cplx<T>) * nb * S * n0, st));
    WTB_CUDA(cudaStreamSynchronize(st));
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_cwt(const void *x, int64_t batch, int n0, int nfft, double dt, double dj, double s0, int J,
                       int mother, double param, int flags, void *power_out, void *coef_out, void *stream) {
  WTB_REQUIRE(x && batch >= 0 && n0 > 0, WTB_EINVAL, "wtb_cwt: bad x/batch/n0");
  WTB_REQUIRE(power_out || coef_out, WTB_EINVAL, "wtb_cwt: no output requested");
  WTB_REQUIRE(nfft >= n0 && nfft >= 2, WTB_EINVAL,
              "nfft=%d must be >= n0=%d (a power of two: pycwt's scipy.fftpack padding rule; n0 itself: "
              "the un-padded mkl_fft rule)", nfft, n0);
  WTB_ENTER(flags, x, stream);
  Mother mo;
  mo.kind = mother;
  mo.param = param;
  Axes ax;
  WTB_TRY(resolve_axes(n0, dt, dj, s0, J, mo, &ax));
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return cwt_entry<double>(x, batch, n0, nfft, dt, ax, mo, flags, power_out, coef_out, st);
  return cwt_entry<float>(x, batch, n0, nfft, dt, ax, mo, flags, power_out, coef_out, st);
}

// The Morlet entry point keeps the transform lengths it has always served: one CTA per transform (powers of two
// up to 8192 in FP32, 4096 in FP64).  Longer series go through wtb_cwt, which takes them up to 2^22.
extern "C" int wtb_cwt_morlet(const void *x, int64_t batch, int n0, int nfft, double dt, double dj,
                              double s0, int J, double f0, int flags, void *power_out,
                              void *coef_out, void *stream) {
  const bool f64 = flags & WTB_F64;
  WTB_REQUIRE(!cwt_long_takes(nfft, f64 ? sizeof(double) : sizeof(float)), WTB_EUNSUPPORTED,
              "wtb_cwt_morlet: nfft=%d is past the one-CTA transform (a power of two up to %d for %s); wtb_cwt with "
              "WTB_MORLET takes powers of two up to 2^22", nfft, f64 ? 4096 : 8192, f64 ? "double" : "float");
  return wtb_cwt(x, batch, n0, nfft, dt, dj, s0, J, WTB_MORLET, f0, flags, power_out, coef_out, stream);
}

// ---- inverse transform (pycwt.icwt): x[t] = factor * sum_s Re(W[s,t]) / sqrt(s_j) ----------
namespace wtb {
template <typename T>
__global__ void k_icwt(const cplx<T> *__restrict__ coef, int S, int n0, const double *__restrict__ scales,
                       double factor, T *__restrict__ out) {
  const int64_t b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n0) return;
  const cplx<T> *w = coef + b * (int64_t)S * n0 + t;
  double acc = 0;
  for (int s = 0; s < S; ++s) acc += (double)w[(int64_t)s * n0].x * rsqrt(scales[s]);
  out[b * (int64_t)n0 + t] = T(factor * acc);
}

template <typename T>
static int icwt_impl(const void *coef, int64_t batch, int S, int n0, const double *scales, double factor, int flags,
                     void *out, cudaStream_t st) {
  const bool dev = flags & WTB_DEVICE_PTRS;
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  void *scratch = nullptr;
  WTB_TRY(arena_reserve(al(sizeof(double) * S), &scratch));
  double *d_scales = (double *)scratch;
  WTB_CUDA(cudaMemcpyAsync(d_scales, scales, sizeof(double) * S, cudaMemcpyHostToDevice, st));
  const size_t in_row = sizeof(cplx<T>) * (size_t)S * n0, out_row = sizeof(T) * (size_t)n0;
  const int64_t rows = dev ? batch : std::max<int64_t>(1, std::min<int64_t>(batch, (int64_t)((size_t(1) << 30) / in_row)));
  const cplx<T> *d_in = (const cplx<T> *)coef;
  T *d_out = (T *)out;
  if (!dev) {
    void *stage = nullptr;
    WTB_TRY(staging_reserve(al(in_row * rows) + al(out_row * rows), &stage));
    d_in = (const cplx<T> *)stage;
    d_out = (T *)((char *)stage + al(in_row * rows));
  }
  for (int64_t b0 = 0; b0 < batch; b0 += rows) {
    const int64_t nb = std::min(rows, batch - b0);
    WTB_REQUIRE(nb < 65536, WTB_EUNSUPPORTED, "wtb_icwt: at most 65535 series per launch");
    if (!dev) WTB_CUDA(cudaMemcpyAsync((void *)d_in, (const char *)coef + b0 * in_row, in_row * nb, cudaMemcpyHostToDevice, st));
    k_icwt<T><<<dim3((n0 + 255) / 256, (unsigned)nb), 256, 0, st>>>(d_in, S, n0, d_scales, factor, d_out);
    WTB_LAUNCH_CHECK();
    if (!dev) {
      WTB_TRY(copy_to_host((char *)out + b0 * out_row, d_out, out_row * nb, st));
      WTB_CUDA(cudaStreamSynchronize(st));
    }
  }
  return WTB_OK;
}
}  // namespace wtb

extern "C" int wtb_icwt(const void *coef, int64_t batch, int S, int n0, const double *scales, double factor,
                        int flags, void *x_out, void *stream) {
  WTB_REQUIRE(coef && x_out && scales && batch >= 0 && S > 0 && n0 > 0, WTB_EINVAL, "wtb_icwt: bad arguments");
  WTB_ENTER(flags, coef, stream);
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return icwt_impl<double>(coef, batch, S, n0, scales, factor, flags, x_out, st);
  return icwt_impl<float>(coef, batch, S, n0, scales, factor, flags, x_out, st);
}
