// Time- and scale-averaged wavelet power (Torrence & Compo 1998 eqs. 22 and 24), the two reductions the pycwt
// sample computes right after cwt:
//   global[b, s] = (1/n0) sum_{t<n0} |W[b,s,t]|^2
//   band[b, t]   = band_factor * sum_{s=band_lo..band_hi} |W[b,s,t]|^2 / scales[s]
// Two passes per chunk of series: cwt_device (cwt.cu, every kernel and dispatch rule of wtb_cwt) writes the power
// rows into device scratch, then k_cwt_averages reads them once and writes both reductions.  Only S + n0 values per
// series leave the device.
#include "cwt_paths.cuh"
#include "spectral.cuh"

namespace wtb {

constexpr int kAvgThreads = 256;

// Grid (series, part).  global: warp w of part y sums rows 8 (y + Y i) + w, i = 0, 1, ...; each lane adds
// t = lane, lane + 32, ... in ascending order, then a fixed xor-shuffle tree combines the lanes.  band: thread t
// of part y adds rows band_lo .. band_hi in ascending order for t = 256 (y + Y i) + threadIdx.x.  Both read along
// t (coalesced) and accumulate in double; every output is summed by one warp or one thread in an order that
// depends on n0 and S only, never on Y, the batch, the chunk or the device, and there are no atomics.
template <typename T>
__global__ void __launch_bounds__(kAvgThreads)
k_cwt_averages(const T *__restrict__ power, int S, int n0, const double *__restrict__ inv_scales, int band_lo,
               int band_hi, double band_factor, T *__restrict__ global, T *__restrict__ band) {
  const int64_t b = blockIdx.x;
  const T *p = power + b * (int64_t)S * n0;
  if (global) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int s = blockIdx.y * (kAvgThreads / 32) + warp; s < S; s += gridDim.y * (kAvgThreads / 32)) {
      const T *row = p + (int64_t)s * n0;
      double acc = 0.0;
#pragma unroll 4
      for (int t = lane; t < n0; t += 32) acc += (double)row[t];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) global[b * S + s] = T(acc / n0);
    }
  }
  if (band) {
    for (int t = blockIdx.y * kAvgThreads + threadIdx.x; t < n0; t += gridDim.y * kAvgThreads) {
      double acc = 0.0;
      for (int s = band_lo; s <= band_hi; ++s) acc += (double)p[(int64_t)s * n0 + t] * inv_scales[s];
      band[b * (int64_t)n0 + t] = T(band_factor * acc);
    }
  }
}

// Parts per series: one when the batch alone fills the machine (8 CTAs per SM), otherwise enough to, but no
// more than the work has (one row group of 8 rows or one tile of 256 t per part).
static unsigned averages_parts(int64_t nb, int S, int n0) {
  const int64_t work = std::max<int64_t>((S + kAvgThreads / 32 - 1) / (kAvgThreads / 32), (n0 + kAvgThreads - 1) / kAvgThreads);
  const int64_t want = (8LL * sm_count() + nb - 1) / nb;
  return (unsigned)std::max<int64_t>(1, std::min(work, want));
}

// The chunk rule, in one place: series per chunk = the number whose power rows fit a 1 GiB budget (as cwt_entry's
// staging), but at least 16 warps on every SM for the warp-per-series nfft-1024 kernel (148 x 16 = 2368 series on a
// B200), rounded down to an even count so the two-series kernels pair the same neighbours in every chunk.  Lengths
// the long transforms serve (cwt_long.cu) have no such kernel and a plane of up to GBs per series: there the
// budget alone counts, and a series whose plane exceeds it is a chunk of its own.
static int64_t averages_chunk_rows(int64_t batch, int S, int n0, int N, size_t elem) {
  const int64_t by_bytes = (int64_t)((size_t(1) << 30) / (elem * (size_t)S * n0));
  if (cwt_long_takes(N, elem)) return std::min(batch, std::max<int64_t>(1, by_bytes));
  const int64_t fill = 16LL * sm_count();
  return std::min(batch, std::max(fill, by_bytes) & ~int64_t(1));
}

static thread_local bool g_in_shard = false;   // set on a pool worker while it runs its block

template <typename T>
static int averages_entry(const void *x, int64_t batch, int n0, int N, double dt, const Axes &ax, const Mother &mo,
                          int band_lo, int band_hi, double band_factor, int flags, void *global_out, void *band_out,
                          cudaStream_t st) {
  const int S = ax.J + 1;
  const bool dev = flags & WTB_DEVICE_PTRS;
  // host buffers, several GPUs (wtb_init_multi): contiguous blocks of series, one per device, as cwt_entry
  if (!dev && pool_size() > 1 && batch >= 2 * pool_size() && !g_in_shard) {
    return run_sharded_fn(batch, 2, st, [&](int, int64_t first, int64_t count, cudaStream_t s) {
      g_in_shard = true;
      const int rc = averages_entry<T>((const T *)x + first * n0, count, n0, N, dt, ax, mo, band_lo, band_hi,
                                       band_factor, flags, global_out ? (T *)global_out + first * S : nullptr,
                                       band_out ? (T *)band_out + first * n0 : nullptr, s);
      g_in_shard = false;
      return rc;
    });
  }
  // The power chunk lives in the staging slot: cwt_device takes the arena (and its fast paths the parameter
  // buffer), and a slot that grows is moved, so a second user of either in this call would lose its data.
  const int64_t rows = averages_chunk_rows(batch, S, n0, N, sizeof(T));
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t b_inv = al(sizeof(double) * S), b_pow = al(sizeof(T) * (size_t)rows * S * n0);
  const size_t b_x = dev ? 0 : al(sizeof(T) * (size_t)rows * n0);
  const size_t b_g = dev || !global_out ? 0 : al(sizeof(T) * (size_t)rows * S);
  const size_t b_b = dev || !band_out ? 0 : al(sizeof(T) * (size_t)rows * n0);
  void *stage = nullptr;
  WTB_TRY(staging_reserve(b_inv + b_pow + b_x + b_g + b_b, &stage));
  double *d_inv = (double *)stage;
  T *d_pow = (T *)((char *)d_inv + b_inv);
  T *d_x = (T *)((char *)d_pow + b_pow);
  T *d_g = (T *)((char *)d_x + b_x);
  T *d_b = (T *)((char *)d_g + b_g);
  std::vector<double> inv(S);
  for (int s = 0; s < S; ++s) inv[s] = 1.0 / ax.scales[s];
  // inv.data() is pageable: the copy is staged before the call returns
  WTB_CUDA(cudaMemcpyAsync(d_inv, inv.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  for (int64_t b0 = 0; b0 < batch; b0 += rows) {
    const int64_t nb = std::min(rows, batch - b0);
    const T *xin = (const T *)x + b0 * n0;
    T *g = global_out ? (T *)global_out + b0 * S : nullptr;
    T *bo = band_out ? (T *)band_out + b0 * n0 : nullptr;
    if (!dev) {
      WTB_CUDA(cudaMemcpyAsync(d_x, xin, sizeof(T) * nb * n0, cudaMemcpyHostToDevice, st));
      xin = d_x;
      g = global_out ? d_g : nullptr;
      bo = band_out ? d_b : nullptr;
    }
    WTB_TRY(cwt_device<T>(xin, nb, n0, N, dt, ax, mo, flags, d_pow, nullptr, st));
    k_cwt_averages<T><<<dim3((unsigned)nb, averages_parts(nb, S, n0)), kAvgThreads, 0, st>>>(d_pow, S, n0, d_inv, band_lo, band_hi, band_factor, g, bo);
    WTB_LAUNCH_CHECK();
    if (!dev) {
      if (global_out) WTB_TRY(copy_to_host((T *)global_out + b0 * S, d_g, sizeof(T) * nb * S, st));
      if (band_out) WTB_TRY(copy_to_host((T *)band_out + b0 * n0, d_b, sizeof(T) * nb * n0, st));
      WTB_CUDA(cudaStreamSynchronize(st));
    }
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_cwt_averages(const void *x, int64_t batch, int n0, int nfft, double dt, double dj, double s0,
                                int J, int mother, double param, int band_lo, int band_hi, double band_factor,
                                int flags, void *global_out, void *band_out, void *stream) {
  WTB_REQUIRE(x && batch >= 0 && n0 > 0, WTB_EINVAL, "wtb_cwt_averages: bad x/batch/n0");
  WTB_REQUIRE(global_out || band_out, WTB_EINVAL, "wtb_cwt_averages: no output requested");
  WTB_REQUIRE(nfft >= n0 && nfft >= 2, WTB_EINVAL, "wtb_cwt_averages: nfft=%d must be >= n0=%d", nfft, n0);
  WTB_REQUIRE(!(flags & WTB_COI_MASK), WTB_EINVAL,
              "wtb_cwt_averages: WTB_COI_MASK would make every average NaN (COI-restricted averages are not offered)");
  WTB_REQUIRE(std::isfinite(band_factor), WTB_EINVAL, "wtb_cwt_averages: band_factor must be finite");
  Mother mo;
  mo.kind = mother;
  mo.param = param;
  Axes ax;
  WTB_TRY(resolve_axes(n0, dt, dj, s0, J, mo, &ax));
  const int S = ax.J + 1;
  WTB_REQUIRE(!band_out || (0 <= band_lo && band_lo <= band_hi && band_hi < S), WTB_EINVAL,
              "wtb_cwt_averages: band [%d, %d] must satisfy 0 <= band_lo <= band_hi < S = %d", band_lo, band_hi, S);
  WTB_ENTER(flags, x, stream);
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64)
    return averages_entry<double>(x, batch, n0, nfft, dt, ax, mo, band_lo, band_hi, band_factor, flags, global_out,
                                  band_out, st);
  return averages_entry<float>(x, batch, n0, nfft, dt, ax, mo, band_lo, band_hi, band_factor, flags, global_out,
                               band_out, st);
}
