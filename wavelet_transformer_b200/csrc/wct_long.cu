// Cross spectra and coherence of long series: the rows of k_wct_rows (wct.cu) at the power-of-two lengths whose
// shared-memory buffers do not fit one CTA (nfft >= 16384 in FP32, >= 8192 in FP64), up to nfft = 2^22, built
// from the four-step transforms of long_fft.cuh.  wct_device (wct.cu) branches here; its scale boxcar and
// coherence kernels (k_wct_scale) do not depend on the length and read tsm as they do after k_wct_rows.
//
// One call:
//   k_long_pass1<T,false>, k_long_pass2<T,false>   X^ [pairs, 2, N] of the interleaved series (as cwt_long)
// then per wave of (pair, scale) rows, two fields per row (blockIdx.z, or both in one tile):
//   k_wcl_w1   inverse pass 1 of X^_f * daughter_s (Morlet daughter_mul, as k_long_pass1<T,true>)
//   k_wcl_w2   inverse pass 2 of both fields: W1, W2 for t < n0 -> w12 = W1 conj(W2), phase; in place
//              P = (|W1|^2 + i |W2|^2) / s and C = W1 conj(W2) / s, zero for t >= n0 (pycwt truncates first)
//   k_wcl_f1   forward pass 1 of P and C
//   k_wcl_g    per column k2: forward pass 2 -> X[k2 + N2 k1], times exp(-1/2 (s/dt)^2 w_k^2) / N, then the
//              first pass of the inverse with the split roles swapped (N = N2 N1, input index k2 + N2 k1), which
//              runs over the same column: the N1-point transform over k1 -> m, times W_N^{+k2 m}
//   k_wcl_t    per column m: the N2-point transform over k2 -> t = m + N1 j; tsm[pair, s, t] for t < n0
// Without a coherence plane or histogram (Morlet xwt) the row stops after k_wcl_w2.  A row's arithmetic does
// not depend on its wave, so results do not depend on the batch, the host chunk, the pool or the pointers.
#include "long_fft.cuh"

namespace wtb {

// Every length that the generic row kernel served before fits its 3 N complex values in 227 KB: the long path
// starts where cwt_long_takes does, right above them.
static_assert(3 * sizeof(float2) * 8192 <= 227 * 1024 && 2 * 2 * sizeof(float) * 8192 <= 227 * 1024 &&
                  2 * 2 * sizeof(float) * 16384 > 227 * 1024,
              "FP32: nfft 8192 is the last generic length, 16384 the first long one");
static_assert(3 * sizeof(double2) * 4096 <= 227 * 1024 && 2 * 2 * sizeof(double) * 4096 <= 227 * 1024 &&
                  2 * 2 * sizeof(double) * 8192 > 227 * 1024,
              "FP64: nfft 4096 is the last generic length, 8192 the first long one");

// The wave rule: rows per wave = those whose intermediates fit 64 MiB (long_wave_rows), four N-point fields per
// row (two buffers of P and C) when the row is smoothed, two (W1, W2) when it is not.
static int64_t wct_long_wave_rows(int N, size_t cplx_bytes, bool smooth, int64_t rows) {
  return long_wave_rows(N, (smooth ? 4 : 2) * cplx_bytes, rows);
}

// Pass-1 epilogue shared by k_wcl_w1 and k_wcl_f1: twiddle W_N^{SIGN n1 k2}, row n1 of Y (as k_long_pass1).
template <typename T, int SIGN, int C>
__device__ __forceinline__ void wcl_store_pass1(const LongPlan<T> &p, const cplx<T> *tile, int stride, int c0,
                                                cplx<T> *__restrict__ yr) {
  const int N2 = p.N2;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  for (int i = tid; i < C * N2; i += nthr) {
    const int c = i / N2, k2 = i % N2, n1 = c0 + c;
    cplx<T> v = tile[c * stride + k2];
    if (n1 && k2) v = cmul(v, long_twiddle<T, SIGN>(p, n1 * k2));
    yr[(int64_t)n1 * N2 + k2] = v;
  }
}

// Field f = blockIdx.z of row (pair, s) = row0 + blockIdx.y: the inverse pass 1 of X^[pair, f] * daughter_s.
template <typename T>
__global__ void k_wcl_w1(LongPlan<T> p, int64_t row0, const cplx<T> *__restrict__ xhat, int S,
                         const double *__restrict__ scales, double dt, double f0, cplx<T> *__restrict__ y) {
  constexpr int C = long_cols<T>(1);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N2 + long_pad<T>(1);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int f = blockIdx.z, c0 = blockIdx.x * C;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  const cplx<T> *xh = xhat + ((row / S) * 2 + f) * (int64_t)N;
  const double sc = scales[row % S];
  const T s_over_dt = T(sc / dt);
  const T norm = T(sqrt(2.0 * kPi * sc / dt) * kPiM14 / double(N));
  for (int i = tid; i < C * N2; i += nthr) {
    const int c = i % C, n2 = i / C, k = c0 + c + N1 * n2;
    tile[c * stride + n2] = daughter_mul<T>(xh[k], k, N, WTB_MORLET, 0, s_over_dt, norm, T(0), T(f0), T(0), T(0));
  }
  __syncthreads();
  long_columns<T, 1, C>(tile, stride, scratch, N2, p.log2N2, p.tw2);
  wcl_store_pass1<T, 1, C>(p, tile, stride, c0, y + (blockIdx.y * 2 + f) * (int64_t)N);
}

// Both fields of row row0 + blockIdx.y, columns k2 = blockIdx.x * H + c (H of each field): W1, W2 at
// t = k2 + N2 k1.  For t < n0: w12, phase; with smooth, P and C in place of Y (the positions this CTA read).
template <typename T>
__global__ void k_wcl_w2(LongPlan<T> p, int64_t row0, cplx<T> *__restrict__ y, int n0, int S,
                         const double *__restrict__ scales, T *__restrict__ phase, cplx<T> *__restrict__ w12,
                         int smooth) {
  constexpr int C = long_cols<T>(2), H = C / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N1 + long_pad<T>(2);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int c0 = blockIdx.x * H;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  cplx<T> *y0 = y + blockIdx.y * 2 * (int64_t)N, *y1 = y0 + N;
  for (int i = tid; i < C * N1; i += nthr) {
    const int c = i % C, n1 = i / C;
    tile[c * stride + n1] = (c < H ? y0 : y1)[(int64_t)n1 * N2 + c0 + c % H];
  }
  __syncthreads();
  long_columns<T, 1, C>(tile, stride, scratch, N1, p.log2N1, p.tw1);
  const int64_t obase = row * n0;
  const T inv_s = T(1.0 / scales[row % S]);
  for (int i = tid; i < H * N1; i += nthr) {
    const int c = i % H, k1 = i / H, t = c0 + c + N2 * k1;
    cplx<T> pp = mk<T>(T(0), T(0)), cc = pp;
    if (t < n0) {
      const cplx<T> a = tile[c * stride + k1], b = tile[(c + H) * stride + k1];
      const cplx<T> x = cmulc(a, b);  // W1 * conj(W2)
      if (w12) w12[obase + t] = x;
      if (phase) phase[obase + t] = dev_atan2<T>(x.y, x.x);
      pp = mk<T>((a.x * a.x + a.y * a.y) * inv_s, (b.x * b.x + b.y * b.y) * inv_s);
      cc = mk<T>(x.x * inv_s, x.y * inv_s);
    }
    if (smooth) {
      y0[t] = pp;
      y1[t] = cc;
    }
  }
}

// Field f = blockIdx.z of row row0 + blockIdx.y: the forward pass 1 of a (P or C, natural order) into b.
template <typename T>
__global__ void k_wcl_f1(LongPlan<T> p, const cplx<T> *__restrict__ a, cplx<T> *__restrict__ b) {
  constexpr int C = long_cols<T>(1);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N2 + long_pad<T>(1);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int c0 = blockIdx.x * C;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  const int64_t off = (blockIdx.y * 2 + blockIdx.z) * (int64_t)N;
  const cplx<T> *ar = a + off;
  for (int i = tid; i < C * N2; i += nthr) {
    const int c = i % C, n2 = i / C;
    tile[c * stride + n2] = ar[c0 + c + N1 * n2];
  }
  __syncthreads();
  long_columns<T, -1, C>(tile, stride, scratch, N2, p.log2N2, p.tw2);
  wcl_store_pass1<T, -1, C>(p, tile, stride, c0, b + off);
}

// Field f = blockIdx.z of row (pair, s) = row0 + blockIdx.y, columns k2 = blockIdx.x * C + c: forward pass 2,
// the Gaussian of k_wct_rows, and the swapped inverse's first pass; Z[k2 N1 + m] into a.
template <typename T>
__global__ void k_wcl_g(LongPlan<T> p, int64_t row0, int S, const double *__restrict__ scales, double dt,
                        const cplx<T> *__restrict__ b, cplx<T> *__restrict__ a) {
  constexpr int C = long_cols<T>(2);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N1 + long_pad<T>(2);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int c0 = blockIdx.x * C;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  const int64_t off = (blockIdx.y * 2 + blockIdx.z) * (int64_t)N;
  const cplx<T> *br = b + off;
  for (int i = tid; i < C * N1; i += nthr) {
    const int c = i % C, n1 = i / C;
    tile[c * stride + n1] = br[(int64_t)n1 * N2 + c0 + c];
  }
  __syncthreads();
  long_columns<T, -1, C>(tile, stride, scratch, N1, p.log2N1, p.tw1);
  // Gaussian in the Fourier domain: exp(-0.5 (s/dt)^2 k^2), k = 2*pi*fftfreq(N), with k_wct_rows' expression
  const T s_over_dt = T(scales[row % S] / dt);
  const T invN = T(1.0 / N);
  for (int i = tid; i < C * N1; i += nthr) {
    const int c = i % C, k1 = i / C, k = c0 + c + N2 * k1;
    const int kk = (k < (N + 1) / 2) ? k : k - N;
    const T w = T(2.0 * kPi) * T(kk) / T(N) * s_over_dt;
    const T g = dev_exp<T>(T(-0.5) * w * w) * invN;
    const cplx<T> v = tile[c * stride + k1];
    tile[c * stride + k1] = mk<T>(v.x * g, v.y * g);
  }
  __syncthreads();
  long_columns<T, 1, C>(tile, stride, scratch, N1, p.log2N1, p.tw1);
  cplx<T> *ar = a + off;
  for (int i = tid; i < C * N1; i += nthr) {
    const int c = i / N1, m = i % N1, k2 = c0 + c;
    cplx<T> v = tile[c * stride + m];
    if (k2 && m) v = cmul(v, long_twiddle<T, 1>(p, k2 * m));
    ar[(int64_t)k2 * N1 + m] = v;
  }
}

// Both fields of row row0 + blockIdx.y, columns m = blockIdx.x * H + c: the N2-point inverse over k2 (stride N1
// in Z) -> t = m + N1 j; tsm[row, t] = (T1, T2, Re T12, Im T12) for t < n0.
template <typename T>
__global__ void k_wcl_t(LongPlan<T> p, int64_t row0, const cplx<T> *__restrict__ a, int n0,
                        vec4<T> *__restrict__ tsm) {
  constexpr int C = long_cols<T>(2), H = C / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N2 + long_pad<T>(2);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int c0 = blockIdx.x * H;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  const cplx<T> *a0 = a + blockIdx.y * 2 * (int64_t)N, *a1 = a0 + N;
  for (int i = tid; i < C * N2; i += nthr) {
    const int c = i % C, k2 = i / C;
    tile[c * stride + k2] = (c < H ? a0 : a1)[(int64_t)k2 * N1 + c0 + c % H];
  }
  __syncthreads();
  long_columns<T, 1, C>(tile, stride, scratch, N2, p.log2N2, p.tw2);
  const int64_t obase = row * n0;
  for (int i = tid; i < H * N2; i += nthr) {
    const int c = i % H, j = i / H, t = c0 + c + N1 * j;
    if (t >= n0) continue;
    const cplx<T> pp = tile[c * stride + j], cc = tile[(c + H) * stride + j];
    vec4<T> o;
    o.x = pp.x; o.y = pp.y; o.z = cc.x; o.w = cc.y;
    tsm[obase + t] = o;
  }
}

template <typename T>
int wct_long(const T *d_y, int64_t pairs, int n0, int N, double dt, const Axes &ax, double f0, bool smooth,
             T *d_phase, cplx<T> *d_w12, const int *h_tlo, const int *h_thi, WctLongOut<T> *out, cudaStream_t st) {
  LongPlan<T> p;
  WTB_TRY(long_plan<T>(N, st, &p));
  const int S = ax.J + 1;
  const int64_t rows = pairs * S;
  const int64_t wave_fwd = long_wave_rows(N, sizeof(cplx<T>), 2 * pairs);
  const int64_t wave = wct_long_wave_rows(N, sizeof(cplx<T>), smooth, rows);
  // one reservation: scales, COI ranges, X^, tsm (n0 per row, not N) and the wave buffers A, B
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t b_sc = al(sizeof(double) * S), b_rng = al(sizeof(int) * S);
  const size_t b_xh = al(sizeof(cplx<T>) * (size_t)pairs * 2 * N);
  const size_t b_ts = smooth ? al(sizeof(vec4<T>) * (size_t)rows * n0) : 0;
  const size_t half = (size_t)wave * 2 * N;   // complex values of one wave buffer
  const size_t b_wave = sizeof(cplx<T>) * std::max((size_t)wave_fwd * N, (smooth ? 2 : 1) * half);
  void *scratch = nullptr;
  WTB_TRY(arena_reserve(b_sc + 2 * b_rng + b_xh + b_ts + b_wave, &scratch));
  char *q = (char *)scratch;
  double *d_scales = (double *)q; q += b_sc;
  out->tlo = (int *)q; q += b_rng;
  out->thi = (int *)q; q += b_rng;
  cplx<T> *d_xhat = (cplx<T> *)q; q += b_xh;
  out->tsm = (vec4<T> *)q; q += b_ts;
  cplx<T> *d_a = (cplx<T> *)q, *d_b = d_a + half;
  WTB_CUDA(cudaMemcpyAsync(d_scales, ax.scales.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  if (h_tlo) {
    WTB_CUDA(cudaMemcpyAsync(out->tlo, h_tlo, sizeof(int) * S, cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync(out->thi, h_thi, sizeof(int) * S, cudaMemcpyHostToDevice, st));
  }
  const LongLaunch l1 = long_launch<T>(1, p.N2), l2 = long_launch<T>(2, p.N1), lt = long_launch<T>(2, p.N2);
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass1<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass2<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_wcl_w1<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_wcl_w2<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_wcl_f1<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_wcl_g<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_wcl_t<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lt.smem));
  constexpr int C1 = long_cols<T>(1), C2 = long_cols<T>(2);
  const unsigned g1 = p.N1 / C1, g2 = p.N2 / C2;
  for (int64_t r0 = 0; r0 < 2 * pairs; r0 += wave_fwd) {
    const unsigned nw = (unsigned)std::min(wave_fwd, 2 * pairs - r0);
    k_long_pass1<T, false><<<dim3(g1, nw), l1.block, l1.smem, st>>>(p, r0, d_y, n0, nullptr, S, nullptr, dt, 0.0, 0, 0,
                                                                     T(0), T(0), d_a);
    WTB_LAUNCH_CHECK();
    k_long_pass2<T, false><<<dim3(g2, nw), l2.block, l2.smem, st>>>(p, r0, d_a, n0, S, nullptr, d_xhat, nullptr,
                                                                     nullptr, 0, 0.0, 0.0);
    WTB_LAUNCH_CHECK();
  }
  for (int64_t r0 = 0; r0 < rows; r0 += wave) {
    const unsigned nw = (unsigned)std::min(wave, rows - r0);
    k_wcl_w1<T><<<dim3(g1, nw, 2), l1.block, l1.smem, st>>>(p, r0, d_xhat, S, d_scales, dt, f0, d_a);
    WTB_LAUNCH_CHECK();
    k_wcl_w2<T><<<dim3(2 * p.N2 / C2, nw), l2.block, l2.smem, st>>>(p, r0, d_a, n0, S, d_scales, d_phase, d_w12,
                                                                      smooth ? 1 : 0);
    WTB_LAUNCH_CHECK();
    if (!smooth) continue;
    k_wcl_f1<T><<<dim3(g1, nw, 2), l1.block, l1.smem, st>>>(p, d_a, d_b);
    WTB_LAUNCH_CHECK();
    k_wcl_g<T><<<dim3(g2, nw, 2), l2.block, l2.smem, st>>>(p, r0, S, d_scales, dt, d_b, d_a);
    WTB_LAUNCH_CHECK();
    k_wcl_t<T><<<dim3(2 * p.N1 / C2, nw), lt.block, lt.smem, st>>>(p, r0, d_a, n0, out->tsm);
    WTB_LAUNCH_CHECK();
  }
  return WTB_OK;
}
template int wct_long<float>(const float *, int64_t, int, int, double, const Axes &, double, bool, float *, float2 *,
                             const int *, const int *, WctLongOut<float> *, cudaStream_t);
template int wct_long<double>(const double *, int64_t, int, int, double, const Axes &, double, bool, double *,
                              double2 *, const int *, const int *, WctLongOut<double> *, cudaStream_t);

}  // namespace wtb
