// Device pieces shared by the CWT and WCT translation units.
#pragma once

#include "common.cuh"
#include "fft_block.cuh"

namespace wtb {

template <typename T> __device__ __forceinline__ T dev_exp(T v);
template <> __device__ __forceinline__ float dev_exp<float>(float v) { return expf(v); }
template <> __device__ __forceinline__ double dev_exp<double>(double v) { return exp(v); }
template <typename T> __device__ __forceinline__ T dev_atan2(T y, T x);
template <> __device__ __forceinline__ float dev_atan2<float>(float y, float x) { return atan2f(y, x); }
template <> __device__ __forceinline__ double dev_atan2<double>(double y, double x) { return atan2(y, x); }

constexpr double kPiM14 = 0.75112554446494248286;  // pi^(-1/4)

// Fourier-domain Morlet daughter for bin k of an N-point grid (pycwt.cwt):
// norm * exp(-0.5 (s*w_k - f0)^2), w_k = 2*pi*fftfreq(N, dt)[k]; no Heaviside step.
template <typename T>
__device__ __forceinline__ T morlet_daughter(int k, int N, T s_over_dt, T norm, T f0) {
  const int kk = (k < (N + 1) / 2) ? k : k - N;  // numpy fftfreq layout (N even: N/2 -> -N/2)
  const T w = T(2.0 * kPi) * T(kk) / T(N);       // rad / sample
  const T z = s_over_dt * w - f0;
  return norm * dev_exp<T>(T(-0.5) * z * z);
}

// Time smoothing of Morlet.smooth at bin k of an N-point grid, with the 1/N of the inverse transform folded in:
// exp(-0.5 (s/dt)^2 w_k^2) / N, w_k = 2*pi*fftfreq(N)[k].  Real and even in k, so it filters the real and the
// imaginary part of a packed row independently.
template <typename T>
__device__ __forceinline__ T smooth_gauss(int k, int N, T s_over_dt, T invN) {
  const int kk = (k < (N + 1) / 2) ? k : k - N;
  const T w = T(2.0 * kPi) * T(kk) / T(N) * s_over_dt;
  return dev_exp<T>(T(-0.5) * w * w) * invN;
}

// X^[k] times the conjugated daughter of one scale at bin k of an N-point grid (k_cwt_rows, and the first pass
// of the long transforms in cwt_long.cu).  Morlet: norm = (2 pi s / dt)^0.5 pi^-1/4 / N.  Paul: (sw)^m exp(-sw)
// H(sw); DOG: (sw)^m exp(-(sw)^2/2); both times nrm = (2 pi s / dt)^0.5 / N and conj(prefactor) = pre.
template <typename T>
__device__ __forceinline__ cplx<T> daughter_mul(cplx<T> v, int k, int N, int mother, int order, T s_over_dt, T norm,
                                                T nrm, T f0, T pre_re, T pre_im) {
  if (mother == WTB_MORLET) {
    const T d = morlet_daughter<T>(k, N, s_over_dt, norm, f0);
    return mk<T>(v.x * d, v.y * d);
  }
  const int kk = (k < (N + 1) / 2) ? k : k - N;
  const T z = s_over_dt * (T(2.0 * kPi) * T(kk) / T(N));
  // z^m e^{-z} (Paul) and z^m e^{-z^2/2} (DOG) evaluated as one exponential: z^m alone
  // overflows FP32 for large orders and scales while the product is tiny (inf * 0 = NaN)
  const T az = fabs(z);
  const T lz = T(order) * log(az);                      // -inf at z = 0: the daughter vanishes (m >= 1)
  const T sgn = (z < T(0) && (order & 1)) ? T(-1) : T(1);
  const T g = mother == WTB_PAUL ? (z > T(0) ? dev_exp<T>(lz - z) : T(0))
                                 : (az > T(0) ? sgn * dev_exp<T>(lz - T(0.5) * z * z) : T(0));
  const T dr = nrm * pre_re * g, di = nrm * pre_im * g;
  return mk<T>(v.x * dr - v.y * di, v.x * di + v.y * dr);
}

// Forward FFT of zero-padded real rows: xhat[row, k], k in [0, plan.n).  smem 2 * plan.M complex.
template <typename T>
__global__ void k_fwd_fft(const T *__restrict__ x, int n0, FftPlan<T> plan, cplx<T> *__restrict__ xhat) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T> *a = reinterpret_cast<cplx<T> *>(smem_raw);
  cplx<T> *b = a + plan.M;
  const int N = plan.n;
  const int64_t row = blockIdx.x;
  const T *xr = x + row * n0;
  for (int t = threadIdx.x; t < N; t += blockDim.x) a[t] = mk<T>(t < n0 ? xr[t] : T(0), T(0));
  __syncthreads();
  cplx<T> *r = plan_fft<T, -1>(a, b, plan);
  cplx<T> *o = xhat + row * N;
  for (int k = threadIdx.x; k < N; k += blockDim.x) o[k] = r[k];
}

// Host side: the plan for a one-CTA length nfft (route_of) on the current device (tables are cached).
template <typename T> static int make_plan(int nfft, FftPlan<T> *plan) {
  plan->n = nfft;
  const bool pow2 = is_pow2(nfft);
  plan->M = (int)work_length(nfft);
  plan->log2M = ilog2(plan->M);
  WTB_TRY(twiddles<T>(plan->M, &plan->tw));
  plan->chirp = nullptr;
  plan->chat = nullptr;
  if (!pow2) WTB_TRY(bluestein_tables<T>(nfft, plan->M, &plan->chirp, &plan->chat));
  return WTB_OK;
}
// CTA size of the one-CTA kernels that run a plan (k_fwd_fft, k_cwt_rows, k_wct_rows, k_pwct_smooth)
inline int plan_threads(int M) { return M >= 1024 ? 256 : (M >= 256 ? 128 : 64); }

}  // namespace wtb
