// Per-component simple regressions (SURVEY section 8f rank 1): the reference regresses the
// output series' component vector S_J, D_J, .., D_1 on the input series' one, level by level,
//   sm.OLS(output_j, sm.add_constant(input_j)).fit()     src/regression.py:118-121,
//                                                        src/modwt.py:218-222, regression.py:76-81.
// With one regressor the normal equations are five sums, so one warp owns one (x row, y row)
// pair: pass 1 the means, pass 2 the centred second moments (the second read comes from L1/L2).
// Everything is accumulated in double whatever the I/O precision.
#include "common.cuh"

namespace wtb {

__device__ __forceinline__ double ols_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// stats[row] = { nobs, intercept, slope, ssr, tss, sxx, mean_x, mean_y }
//   add_constant: tss and sxx are centred (statsmodels' centered_tss); otherwise raw sums.
template <typename T>
__global__ void k_rowwise_ols(const T *__restrict__ x, int64_t x_stride, const T *__restrict__ y,
                              int64_t y_stride, int64_t rows, int n, int add_constant,
                              double *__restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const T *xr = x + row * x_stride, *yr = y + row * y_stride;
  double sx = 0, sy = 0;
  for (int t = lane; t < n; t += 32) {
    sx += (double)xr[t];
    sy += (double)yr[t];
  }
  const double N = (double)n;
  const double mean_x = ols_warp_sum(sx) / N, mean_y = ols_warp_sum(sy) / N;
  const double mx = add_constant ? mean_x : 0.0, my = add_constant ? mean_y : 0.0;
  double sxx = 0, sxy = 0, syy = 0;
  for (int t = lane; t < n; t += 32) {
    const double dx = (double)xr[t] - mx, dy = (double)yr[t] - my;
    sxx = fma(dx, dx, sxx);
    sxy = fma(dx, dy, sxy);
    syy = fma(dy, dy, syy);
  }
  sxx = ols_warp_sum(sxx);
  sxy = ols_warp_sum(sxy);
  syy = ols_warp_sum(syy);
  if (lane == 0) {
    const double slope = sxy / sxx;
    double *o = stats + row * 8;
    o[0] = N;
    o[1] = add_constant ? my - slope * mx : 0.0;
    o[2] = slope;
    o[3] = fmax(syy - slope * sxy, 0.0);  // residual sum of squares
    o[4] = syy;
    o[5] = sxx;
    o[6] = mean_x;
    o[7] = mean_y;
  }
}

template <typename T>
static int ols_impl(const void *x, int64_t x_rows, const void *y, int64_t y_rows, int64_t rows, int n,
                    int add_constant, int flags, double *stats, cudaStream_t st) {
  const bool dev = flags & WTB_DEVICE_PTRS;
  const T *d_x = (const T *)x, *d_y = (const T *)y;
  double *d_s = stats;
  if (!dev) {
    const size_t bx = align256(sizeof(T) * (size_t)x_rows * n), by = align256(sizeof(T) * (size_t)y_rows * n);
    void *stage = nullptr;
    WTB_TRY(staging_reserve(bx + by + align256(sizeof(double) * 8 * rows), &stage));
    d_x = (const T *)stage;
    d_y = (const T *)((char *)stage + bx);
    d_s = (double *)((char *)stage + bx + by);
    WTB_CUDA(cudaMemcpyAsync((void *)d_x, x, sizeof(T) * (size_t)x_rows * n, cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync((void *)d_y, y, sizeof(T) * (size_t)y_rows * n, cudaMemcpyHostToDevice, st));
  }
  const int warps = 8;
  const int64_t blocks = (rows + warps - 1) / warps;
  WTB_REQUIRE(blocks < (1LL << 31), WTB_EUNSUPPORTED, "too many rows");
  k_rowwise_ols<T><<<(unsigned)blocks, warps * 32, 0, st>>>(d_x, x_rows == 1 ? 0 : n, d_y, y_rows == 1 ? 0 : n, rows, n,
                                                           add_constant, d_s);
  WTB_LAUNCH_CHECK();
  if (!dev) {
    WTB_TRY(copy_to_host(stats, d_s, sizeof(double) * 8 * rows, st));
    WTB_CUDA(cudaStreamSynchronize(st));
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_rowwise_ols(const void *x, int64_t x_rows, const void *y, int64_t y_rows, int n,
                               int add_constant, int flags, double *stats_out, void *stream) {
  WTB_REQUIRE(x && y && stats_out && x_rows >= 0 && y_rows >= 0, WTB_EINVAL, "wtb_rowwise_ols: bad arguments");
  WTB_REQUIRE(n > (add_constant ? 2 : 1), WTB_EINVAL, "wtb_rowwise_ols: %d observations leave no residual degrees of freedom", n);
  WTB_REQUIRE(x_rows == y_rows || x_rows == 1 || y_rows == 1, WTB_EINVAL,
              "wtb_rowwise_ols: x has %lld rows and y %lld (equal, or one of them 1 to broadcast)",
              (long long)x_rows, (long long)y_rows);
  WTB_ENTER(flags, x, stream);
  const int64_t rows = x_rows > y_rows ? x_rows : y_rows;
  if (x_rows == 0 || y_rows == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return ols_impl<double>(x, x_rows, y, y_rows, rows, n, add_constant, flags, stats_out, st);
  return ols_impl<float>(x, x_rows, y, y_rows, rows, n, add_constant, flags, stats_out, st);
}
