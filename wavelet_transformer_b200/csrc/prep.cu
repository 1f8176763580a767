// Batched pre-processing on either side of the transforms (SURVEY section 8f rank 2):
//   standardize_series (src/utils/wavelet_helpers.py:22-57): raw mean / population std,
//     optional degree-1 least-squares detrend, optional mean removal, divide by the RAW std;
//   pycwt.ar1 (src/cwt.py:106): Allen & Smith lag-1 autocorrelation of the INPUT series,
//     NaN where the reference raises "Cannot place an upperbound on the unbiased AR(1)".
// One warp per series, statistics accumulated in double whatever the I/O precision.
#include "common.cuh"

namespace wtb {

#define WTB_PREP_DETREND     1
#define WTB_PREP_REMOVE_MEAN 2
#define WTB_PREP_STANDARDIZE 4

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T>
__global__ void k_series_prep(const T *__restrict__ x, int64_t batch, int n, int mode,
                              T *__restrict__ y, double *__restrict__ ar1) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= batch) return;
  const T *xr = x + row * n;
  // pass 1: sums for mean, variance and the degree-1 least-squares fit against t = 0..n-1
  double s1 = 0, st = 0;
  for (int t = lane; t < n; t += 32) {
    const double v = (double)xr[t];
    s1 += v;
    st += v * t;
  }
  s1 = warp_sum(s1);
  st = warp_sum(st);
  const double N = (double)n;
  const double mean = s1 / N;
  // centred sums are better conditioned than the raw normal equations
  const double tbar = 0.5 * (N - 1.0);
  const double stt = N * (N * N - 1.0) / 12.0;              // sum (t - tbar)^2
  const double slope = n > 1 ? (st - tbar * s1) / stt : 0.0; // sum (t - tbar) x / sum (t - tbar)^2
  const double icpt = mean - slope * tbar;
  // pass 2: variance, lag-0 and lag-1 covariances of the mean-removed series
  double c0 = 0, c1 = 0;
  for (int t = lane; t < n; t += 32) {
    const double d = (double)xr[t] - mean;
    c0 += d * d;
    if (t + 1 < n) c1 += d * ((double)xr[t + 1] - mean);
  }
  c0 = warp_sum(c0);
  c1 = warp_sum(c1);
  const double sd = sqrt(c0 / N);                           // numpy .std(): population
  if (y) {
    T *yr = y + row * n;
    for (int t = lane; t < n; t += 32) {
      double v = (double)xr[t];
      if (mode & WTB_PREP_DETREND) v -= icpt + slope * t;
      if (mode & WTB_PREP_REMOVE_MEAN) v -= mean;
      if (mode & WTB_PREP_STANDARDIZE) v /= sd;
      yr[t] = (T)v;
    }
  }
  if (ar1 && lane == 0) {
    // pycwt.helpers.ar1
    const double C0 = c0 / N, C1 = c1 / (N - 1.0);
    const double A = C0 * N * N;
    const double B = -C1 * N - C0 * N * N - 2 * C0 + 2 * C1 - C1 * N * N + C0 * N;
    const double Cq = N * (C0 + C1 * N - C1);
    const double D = B * B - 4 * A * Cq;
    ar1[row] = D > 0 ? (-B - sqrt(D)) / (2 * A) : NAN;
  }
}

template <typename T>
static int prep_impl(const void *x, int64_t batch, int n, int mode, int flags, void *y, double *ar1,
                     cudaStream_t st) {
  // one chunk: the whole batch
  return stage_rows(batch, batch, flags, st, {{x, sizeof(T) * n}}, {{y, sizeof(T) * n}, {ar1, sizeof(double)}}, 0,
                    [&](const void *const *in, void *const *out, void *, int64_t, int64_t nb) {
                      const int warps = 8;
                      const int64_t blocks = (nb + warps - 1) / warps;
                      WTB_REQUIRE(blocks < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
                      k_series_prep<T><<<(unsigned)blocks, warps * 32, 0, st>>>((const T *)in[0], nb, n, mode,
                                                                                (T *)out[0], (double *)out[1]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_series_prep(const void *x, int64_t batch, int n, int detrend, int remove_mean,
                               int standardize, int flags, void *y_out, double *ar1_out, void *stream) {
  WTB_REQUIRE(x && batch >= 0 && n > 1, WTB_EINVAL, "wtb_series_prep: bad x/batch/n");
  WTB_REQUIRE(y_out || ar1_out, WTB_EINVAL, "wtb_series_prep: no output requested");
  WTB_REQUIRE(!(detrend && remove_mean), WTB_EINVAL,
              "Only standardize by either removing secular trend or mean, not both.");
  WTB_ENTER(flags, x, stream);
  if (batch == 0) return WTB_OK;
  const int mode = (detrend ? WTB_PREP_DETREND : 0) | (remove_mean ? WTB_PREP_REMOVE_MEAN : 0) |
                   (standardize ? WTB_PREP_STANDARDIZE : 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return prep_impl<double>(x, batch, n, mode, flags, y_out, ar1_out, st);
  return prep_impl<float>(x, batch, n, mode, flags, y_out, ar1_out, st);
}
