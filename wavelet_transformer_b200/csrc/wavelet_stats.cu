// MODWT wavelet variance, covariance and cross-correlation by level (Percival & Walden 2000, ch. 8; Whitcher,
// Guttorp & Percival 2000) over the coefficients free of the circular wrap:
//   a_j = L_j - 1 = (2^j - 1)(L - 1),  M_j = n - a_j
//   var_x[j]     = (1/M_j) sum_{t=a_j}^{n-1} W_{x,j}[t]^2
//   xcov[j, tau] = (1/M_j) sum_t W_{x,j}[t] W_{y,j}[t+tau] over t, t+tau in [a_j, n-1], |tau| <= K
// NaN where M_j <= 0 and for |tau| >= M_j.
//
// Per chunk of pairs: modwt_device (every kernel and plan rule of wtb_modwt) writes the x and y planes
// [nb, J+1, n] into staging, k_wstats_partial reads each level row once per t-block and writes one partial sum
// per (pair, level, block, slot), and k_wstats_final adds the blocks in ascending order and divides by M_j.
// Only J (2K+3) numbers per pair leave the device.
#include "filterbank_common.cuh"

namespace wtb {

constexpr int kWsTile = 1024;        // samples of W_x staged per step (plus 2K of W_y halo)
constexpr int kWsSpan = 16384;       // samples of one t-block: the block count depends on n alone
constexpr int kWsMaxThreads = 256;
constexpr int kWsMaxLag = 8192;      // window (2 kWsTile + 2K) * 8 B = 144 KB fits one CTA

__host__ __device__ __forceinline__ int64_t ws_first(int j, int L) { return ((int64_t(1) << j) - 1) * (L - 1); }
static int ws_blocks(int n) { return (int)((n + (int64_t)kWsSpan - 1) / kWsSpan); }

// sum_u a[u] b[u], u = 0 .. cnt-1: four interleaved accumulators, combined as (s0 + s1) + (s2 + s3)
__device__ __forceinline__ double ws_dot(const double *a, const double *b, int cnt) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int u = 0;
  for (; u + 4 <= cnt; u += 4) {
    s0 = fma(a[u], b[u], s0);
    s1 = fma(a[u + 1], b[u + 1], s1);
    s2 = fma(a[u + 2], b[u + 2], s2);
    s3 = fma(a[u + 3], b[u + 3], s3);
  }
  for (; u < cnt; ++u) s0 = fma(a[u], b[u], s0);
  return (s0 + s1) + (s2 + s3);
}

// Grid (t-block, level - 1, pair).  Slots: lags tau = s - K for s < 2K+1, then var_x and var_y (pairs); var_x alone
// without y.  Block b covers t in [max(b kWsSpan, a_j), min((b+1) kWsSpan, n)) in tiles of kWsTile: W_x[t0, t0+cnt)
// and W_y[t0-K, t0+kWsTile+K) are staged in shared memory as double (FP32 rows are widened once there, not at every
// product), W_y zero outside [a_j, n-1].  Thread s adds its slot's
// tile sum (W_x[t] a broadcast, W_y[t+tau] consecutive across lanes) to its partial; the order depends on n, L and
// j only.  No atomics.
template <typename T, bool kPair>
__global__ void __launch_bounds__(kWsMaxThreads)
k_wstats_partial(const T *__restrict__ px, const T *__restrict__ py, int n, int J, int L, int K,
                 double *__restrict__ part) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *xs = reinterpret_cast<double *>(smem_raw);
  double *ys = xs + kWsTile;
  const int j = blockIdx.y + 1;
  const int64_t p = blockIdx.z;
  const int lags = kPair ? 2 * K + 1 : 0;
  const int nslots = kPair ? lags + 2 : 1;
  const int64_t a = ws_first(j, L);
  const int64_t row = (p * (J + 1) + (j - 1)) * (int64_t)n;
  const T *x = px + row;
  const T *y = kPair ? py + row : nullptr;
  double *out = part + ((p * J + (j - 1)) * gridDim.x + blockIdx.x) * (int64_t)nslots;
  for (int s = threadIdx.x; s < nslots; s += blockDim.x) out[s] = 0.0;
  const int64_t bs = (int64_t)blockIdx.x * kWsSpan, be = min((int64_t)n, bs + kWsSpan);
  for (int64_t t0 = max(bs, a); t0 < be; t0 += kWsTile) {
    const int cnt = (int)min((int64_t)kWsTile, be - t0);
    __syncthreads();  // the previous tile's readers are done
    for (int u = threadIdx.x; u < cnt; u += blockDim.x) xs[u] = x[t0 + u];
    if (kPair)
      for (int v = threadIdx.x; v < cnt + 2 * K; v += blockDim.x) {
        const int64_t t = t0 - K + v;
        ys[v] = (t >= a && t < n) ? (double)y[t] : 0.0;
      }
    __syncthreads();
    for (int s = threadIdx.x; s < nslots; s += blockDim.x) {
      const double *A = xs, *B = xs;                     // var_x
      if (s < lags) B = ys + s;                          // W_y[t0 + u + (s - K)]
      else if (kPair && s == lags + 1) A = B = ys + K;   // var_y
      out[s] += ws_dot(A, B, cnt);
    }
  }
}

// One CTA per pair: slot s of level j is the sum of its blocks in ascending order, over M_j.
__global__ void __launch_bounds__(kWsMaxThreads)
k_wstats_final(const double *__restrict__ part, int n, int J, int L, int K, int nblk, bool pair,
               double *__restrict__ var_x, double *__restrict__ var_y, double *__restrict__ xcov) {
  const int64_t p = blockIdx.x;
  const int lags = pair ? 2 * K + 1 : 0;
  const int nslots = pair ? lags + 2 : 1;
  for (int i = threadIdx.x; i < J * nslots; i += blockDim.x) {
    const int jj = i / nslots, s = i % nslots;
    const double *src = part + (p * J + jj) * (int64_t)nblk * nslots + s;
    double acc = 0.0;
    for (int b = 0; b < nblk; ++b) acc += src[(int64_t)b * nslots];
    const int64_t M = n - ws_first(jj + 1, L);
    const bool nan = M <= 0 || (s < lags && abs(s - K) >= M);
    const double v = nan ? __longlong_as_double(0x7ff8000000000000LL) : acc / (double)M;
    if (s < lags) {
      if (xcov) xcov[(p * J + jj) * lags + s] = v;
    } else if (s == lags) {
      if (var_x) var_x[p * J + jj] = v;
    } else if (var_y) {
      var_y[p * J + jj] = v;
    }
  }
}

// Pairs per chunk: those whose planes and partial sums fit 1 GiB of staging, at least one (a pair past the budget
// is a chunk of its own), at most the batch and gridDim.z.
static int64_t wstats_chunk_rows(int64_t batch, size_t per_pair) {
  const int64_t by_bytes = (int64_t)((size_t(1) << 30) / per_pair);
  return std::min<int64_t>({batch, std::max<int64_t>(1, by_bytes), 65535});
}

template <typename T>
static int wstats_entry(const void *x, const void *y, int64_t batch, int n, const Taps &taps, int J, int K, int flags,
                        double *var_x, double *var_y, double *xcov, cudaStream_t st) {
  const bool pair = y != nullptr;
  const int lags = pair ? 2 * K + 1 : 0, nslots = pair ? lags + 2 : 1;
  const int nblk = ws_blocks(n);
  const int threads = std::min(kWsMaxThreads, (nslots + 31) / 32 * 32);
  const size_t plane = sizeof(T) * (size_t)(J + 1) * n;
  const size_t part_row = sizeof(double) * (size_t)J * nblk * nslots;
  const size_t smem = sizeof(double) * (kWsTile + (pair ? kWsTile + 2 * (size_t)K : 0));
  auto kern = pair ? k_wstats_partial<T, true> : k_wstats_partial<T, false>;
  const InRows xs{x, sizeof(T) * n}, ys{y, sizeof(T) * n};
  const OutRows vx{var_x, sizeof(double) * J}, vy{var_y, sizeof(double) * J}, xc{xcov, sizeof(double) * J * lags};
  return shard_host_rows(batch, flags, st, [&](int64_t first, int64_t count, cudaStream_t s) {
    WTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // this device
    // the planes and the partial sums live in the staging slot next to the host-path I/O: modwt_device takes no
    // staging, and its long path reserves the arena after these pointers are taken
    const int64_t rows = wstats_chunk_rows(count, (pair ? 2 : 1) * plane + part_row);
    const size_t b_plane = align256(plane * rows);
    return stage_rows(count, rows, flags, s, {xs.at(first), ys.at(first)}, {vx.at(first), vy.at(first), xc.at(first)},
                      (pair ? 2 : 1) * b_plane + part_row * rows,
                      [&](const void *const *in, void *const *out, void *extra, int64_t, int64_t nb) -> int {
                        T *d_px = (T *)extra;
                        T *d_py = pair ? (T *)((char *)extra + b_plane) : nullptr;
                        double *d_part = (double *)((char *)extra + (pair ? 2 : 1) * b_plane);
                        WTB_TRY(modwt_device<T>((const T *)in[0], nb, n, taps, J, flags, d_px, s));
                        if (pair) WTB_TRY(modwt_device<T>((const T *)in[1], nb, n, taps, J, flags, d_py, s));
                        kern<<<dim3((unsigned)nblk, (unsigned)J, (unsigned)nb), threads, smem, s>>>(
                            d_px, d_py, n, J, taps.L, K, d_part);
                        WTB_LAUNCH_CHECK();
                        k_wstats_final<<<(unsigned)nb, kWsMaxThreads, 0, s>>>(d_part, n, J, taps.L, K, nblk, pair,
                                                                              (double *)out[0], (double *)out[1],
                                                                              (double *)out[2]);
                        WTB_LAUNCH_CHECK();
                        return WTB_OK;
                      });
  });
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_modwt_wavelet_stats(const void *x, const void *y, int64_t batch, int n, const double *g,
                                       const double *h, int L, int J, int max_lag, int flags, double *var_x_out,
                                       double *var_y_out, double *xcov_out, void *stream) {
  WTB_REQUIRE(x && batch >= 0 && n > 0, WTB_EINVAL, "wtb_modwt_wavelet_stats: bad x/batch/n");
  WTB_REQUIRE(var_x_out || var_y_out || xcov_out, WTB_EINVAL, "wtb_modwt_wavelet_stats: no output requested");
  WTB_REQUIRE(y || (!var_y_out && !xcov_out), WTB_EINVAL,
              "wtb_modwt_wavelet_stats: var_y_out and xcov_out need y (y == NULL is the variance of x alone)");
  WTB_REQUIRE(J >= 1 && J < 31, WTB_EINVAL, "wtb_modwt_wavelet_stats: J=%d outside [1, 30]", J);
  WTB_REQUIRE(max_lag >= 0 && max_lag <= kWsMaxLag && max_lag < n, WTB_EINVAL,
              "wtb_modwt_wavelet_stats: max_lag=%d must satisfy 0 <= max_lag <= %d and max_lag < n=%d", max_lag,
              kWsMaxLag, n);
  Taps taps;
  WTB_TRY(make_taps(g, h, L, 1.0 / std::sqrt(2.0), &taps));
  WTB_ENTER(flags, x, stream);
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64)
    return wstats_entry<double>(x, y, batch, n, taps, J, max_lag, flags, var_x_out, var_y_out, xcov_out, st);
  return wstats_entry<float>(x, y, batch, n, taps, J, max_lag, flags, var_x_out, var_y_out, xcov_out, st);
}
