// Four-step (Bailey) FFT pieces of the long transforms: powers of two whose shared-memory buffers do not fit one
// CTA, up to nfft = 2^22.  Used by the CWT (cwt_long.cu) and the cross spectra / coherence (wct_long.cu).
//
// N = N1 N2 with N1 = 2^floor(L/2), N2 = 2^ceil(L/2) <= 2048, input index n = n1 + N1 n2 and output index
// k = k2 + N2 k1:
//   X[k2 + N2 k1] = sum_n1 W_N1^{n1 k1} W_N^{n1 k2} sum_n2 x[n1 + N1 n2] W_N2^{n2 k2}.
//   pass 1: per column n1, the N2-point FFT over n2 (input stride N1), times W_N^{n1 k2}; row n1 of Y.
//   pass 2: per column k2, the N1-point FFT over n1 (stride N2 in Y), stored at k2 + N2 k1.
// Both sub-transforms are block_fft (fft_block.cuh).  A CTA takes C adjacent columns so that every strided
// global load and store covers whole 32-byte sectors (C complex values in pass 1, C reals in pass 2), and
// transposes them through a shared-memory tile; G of its columns are transformed at once, one per
// threadIdx.y.  The inter-pass twiddle is the product of two tables built in long double (long_twiddles,
// cwt_long.cu), W_N^m = W_N^{m mod 2048} W_N^{2048 (m / 2048)}.
#pragma once

#include "cwt_paths.cuh"
#include "spectral.cuh"

namespace wtb {

constexpr int kLongMaxN = 1 << 22;
constexpr size_t kWaveBytes = size_t(64) << 20;

// The wave rule: rows per wave = those whose intermediate (N values of cplx_bytes each) fit 64 MiB, at least one,
// at most the rows there are.
inline int64_t long_wave_rows(int N, size_t cplx_bytes, int64_t rows) {
  return std::min(rows, std::max<int64_t>(1, (int64_t)(kWaveBytes / (cplx_bytes * (size_t)N))));
}

template <typename T> struct LongPlan {
  int N, N1, N2, log2N1, log2N2;
  const cplx<T> *tw1, *tw2;  // exp(-2 pi i k / N1), exp(-2 pi i k / N2): block_fft tables of the two passes
  const cplx<T> *tlo, *thi;  // exp(-2 pi i j / N), j < 2048;  exp(-2 pi i 2048 j / N), j < N / 2048
};

// Columns per CTA: C complex values make a 32-byte sector in pass 1, C reals one in pass 2.
template <typename T> __host__ __device__ constexpr int long_cols(int pass) { return pass == 1 ? 32 / (int)sizeof(cplx<T>) : 32 / (int)sizeof(T); }
// Tile column stride L + long_pad: adjacent columns start 128 / C bytes apart, so the transposing accesses
// (column c = thread mod C) of one 128-byte wavefront hit distinct banks.
template <typename T> __host__ __device__ constexpr int long_pad(int pass) { return (128 / (int)sizeof(cplx<T>)) / long_cols<T>(pass); }

template <typename T, int SIGN> __device__ __forceinline__ cplx<T> long_twiddle(const LongPlan<T> &p, int m) {
  cplx<T> w = cmul(p.tlo[m & 2047], p.thi[m >> 11]);
  if (SIGN > 0) w.y = -w.y;
  return w;
}

// The C columns of the tile, G at a time (threadIdx.y), each an L-point block_fft in place in its column.
template <typename T, int SIGN, int C>
__device__ __forceinline__ void long_columns(cplx<T> *tile, int stride, cplx<T> *scratch, int L, int log2L,
                                             const cplx<T> *tw) {
  const int G = blockDim.y;
  cplx<T> *b = scratch + threadIdx.y * L;
  for (int c = threadIdx.y; c < C; c += G) {      // G divides C: every thread runs the same barriers
    cplx<T> *col = tile + c * stride;
    cplx<T> *r = block_fft<T, SIGN>(col, b, L, log2L, tw);
    if (r != col)
      for (int i = threadIdx.x; i < L; i += blockDim.x) col[i] = r[i];
    __syncthreads();
  }
}

// Pass 1 of rows row0 + blockIdx.y, columns n1 = blockIdx.x * C + c.  INV = false: the forward transform of
// series row (x real, zero past n0).  INV = true: the inverse transform of X^[row / S] * daughter(row % S).
template <typename T, bool INV>
__global__ void k_long_pass1(LongPlan<T> p, int64_t row0, const T *__restrict__ x, int n0,
                             const cplx<T> *__restrict__ xhat, int S, const double *__restrict__ scales, double dt,
                             double f0, int mother, int order, T pre_re, T pre_im, cplx<T> *__restrict__ y) {
  constexpr int C = long_cols<T>(1);
  constexpr int SIGN = INV ? 1 : -1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N2 + long_pad<T>(1);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int c0 = blockIdx.x * C;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  if constexpr (INV) {
    const int s = (int)(row % S);
    const cplx<T> *xh = xhat + (row / S) * (int64_t)N;
    const double sc = scales[s];
    const T s_over_dt = T(sc / dt);
    const T norm = T(sqrt(2.0 * kPi * sc / dt) * kPiM14 / double(N));
    const T nrm = T(sqrt(2.0 * kPi * sc / dt) / double(N));
    for (int i = tid; i < C * N2; i += nthr) {
      const int c = i % C, n2 = i / C, k = c0 + c + N1 * n2;
      tile[c * stride + n2] = daughter_mul<T>(xh[k], k, N, mother, order, s_over_dt, norm, nrm, T(f0), pre_re, pre_im);
    }
  } else {
    const T *xr = x + row * n0;
    for (int i = tid; i < C * N2; i += nthr) {
      const int c = i % C, n2 = i / C, n = c0 + c + N1 * n2;
      tile[c * stride + n2] = mk<T>(n < n0 ? xr[n] : T(0), T(0));
    }
  }
  __syncthreads();
  long_columns<T, SIGN, C>(tile, stride, scratch, N2, p.log2N2, p.tw2);
  cplx<T> *yr = y + blockIdx.y * (int64_t)N;
  for (int i = tid; i < C * N2; i += nthr) {
    const int c = i / N2, k2 = i % N2, n1 = c0 + c;
    cplx<T> v = tile[c * stride + k2];
    if (n1 && k2) v = cmul(v, long_twiddle<T, SIGN>(p, n1 * k2));
    yr[(int64_t)n1 * N2 + k2] = v;
  }
}

// Pass 2 of rows row0 + blockIdx.y, columns k2 = blockIdx.x * C + c, output index t = k2 + N2 k1.
// INV = false: X^ of series row, every t.  INV = true: W of row (series, scale) for t < n0 only; power and / or
// coefficients at row * n0 + t, with the WTB_COI_MASK rule of k_cwt_rows.
template <typename T, bool INV>
__global__ void k_long_pass2(LongPlan<T> p, int64_t row0, const cplx<T> *__restrict__ y, int n0, int S,
                             const double *__restrict__ scales, cplx<T> *__restrict__ xhat, T *__restrict__ power,
                             cplx<T> *__restrict__ coef, int coi_mask, double coi_c, double flambda) {
  constexpr int C = long_cols<T>(2);
  constexpr int SIGN = INV ? 1 : -1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.N, N1 = p.N1, N2 = p.N2, stride = N1 + long_pad<T>(2);
  cplx<T> *tile = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *scratch = tile + C * stride;
  const int64_t row = row0 + blockIdx.y;
  const int c0 = blockIdx.x * C;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  const cplx<T> *yr = y + blockIdx.y * (int64_t)N;
  for (int i = tid; i < C * N1; i += nthr) {
    const int c = i % C, n1 = i / C;
    tile[c * stride + n1] = yr[(int64_t)n1 * N2 + c0 + c];
  }
  __syncthreads();
  long_columns<T, SIGN, C>(tile, stride, scratch, N1, p.log2N1, p.tw1);
  if constexpr (INV) {
    const double period = 1.0 / (1.0 / (flambda * scales[row % S]));
    const int64_t obase = row * n0;
    for (int i = tid; i < C * N1; i += nthr) {
      const int c = i % C, k1 = i / C, t = c0 + c + N2 * k1;
      if (t >= n0) continue;
      const cplx<T> w = tile[c * stride + k1];
      if (coef) coef[obase + t] = w;
      if (power) {
        T pw = w.x * w.x + w.y * w.y;
        if (coi_mask) {
          const double coi = coi_c * (n0 / 2.0 - fabs(t - (n0 - 1) / 2.0));
          if (period > coi) pw = T(NAN);
        }
        power[obase + t] = pw;
      }
    }
  } else {
    cplx<T> *o = xhat + row * (int64_t)N;
    for (int i = tid; i < C * N1; i += nthr) {
      const int c = i % C, k1 = i / C;
      o[c0 + c + N2 * k1] = tile[c * stride + k1];
    }
  }
}

// Launch shape of one pass: TX threads per column transform (at most 128, at most L / 4), G columns at once,
// the largest G dividing C whose tile and scratch fit 227 KB with at most 512 threads.
struct LongLaunch {
  dim3 block;
  size_t smem;
};
template <typename T> inline LongLaunch long_launch(int pass, int L) {
  const int C = long_cols<T>(pass);
  const int tx = std::min(L / 4, 128);
  int G = C;
  auto bytes = [&](int g) { return sizeof(cplx<T>) * ((size_t)C * (L + long_pad<T>(pass)) + (size_t)g * L); };
  while (G > 1 && (bytes(G) > 227 * 1024 || tx * G > 512)) G /= 2;
  return {dim3(tx, G), bytes(G)};
}

}  // namespace wtb
