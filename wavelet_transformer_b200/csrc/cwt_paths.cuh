// Which kernels serve a CWT (cwt_plan, cwt.cu), and the host functions the CWT and coherence translation units
// call across files.
#pragma once

#include "wct_common.cuh"

namespace wtb {

// Limits of the FP32 Morlet kernels that the plan reads (each kernel's own transform size kN stays in its file).
constexpr int kMaxRows = 256;    // scale rows k_cwt_fast_1024 stages in shared memory (cwt_fast.cu)
constexpr int kMaxRowsF = 128;   // scale rows k_cwt_dif stages in shared memory (cwt_fast.cu)
constexpr int kMinBatchF = 12;   // smallest batch k_cwt_dif<2> (nfft = 2048) takes by default
constexpr int kMaxRowsC = 512;   // scale rows the register-FFT kernels of wct_fast.cu stage in shared memory
// The one-sided transforms drop the daughter where |s*w - f0| > 5.3 (exp(-14) ~ 8e-7 of its peak).  pycwt's Morlet
// has no Heaviside step: at negative frequencies the daughter is exp(-(f0 + |s*w|)^2 / 2) of its peak, and the
// dropped tail is below the same 8e-7 only for f0 >= 5.3 (f0 = 6, the reference's only value: 1.5e-8); smaller f0
// take the generic kernels.  cwt_fast.cu tests f0 against the float kZCut, wct_fast.cu against the double kMinF0;
// they differ for f0 in [5.3, 5.3f), so each test keeps its own constant.
constexpr float kZCut = 5.3f;
constexpr double kMinF0 = 5.3;

// The forward transform of a CWT: in the row kernel itself, the shared-memory Stockham kernel k_fwd_fft, the
// radix-16 register kernel (FP32, nfft = 4096, natural order), k_fwd_fft_pair2048 (group layout), or the radix-16
// kernel followed by k_dif_layout4096 (group layout).
enum class Fwd { kInKernel, kGeneric, kRadix16_4096, kPair2048, kRadix16Layout4096 };
// The row kernel: k_cwt_fast_1024 (one series per warp, or two for nfft = 512), k_cwt_dif<2> / <4>, k_cwt_rows_4096,
// the four-step transforms of cwt_long.cu, or the generic k_cwt_rows.
enum class Rows { kFast1024, kFast512Pairs, kDif2048, kDif4096, kRows4096, kLong, kGeneric };
struct CwtPlan {
  Fwd fwd;
  Rows rows;
};
CwtPlan cwt_plan(int64_t batch, int n0, int N, int S, double f0, int mother, size_t elem, int flags, bool power,
                 bool coef);

// cwt.cu: the CWT of device-resident series (also the first pass of wtb_cwt_averages)
template <typename T>
int cwt_device(const T *d_x, int64_t batch, int n0, int N, double dt, const Axes &ax, const Mother &mo, int flags,
               T *d_power, cplx<T> *d_coef, cudaStream_t st);

// cwt_fast.cu: Rows::kFast1024 / kFast512Pairs
int cwt_fast_1024(const CwtPlan &pl, const float *d_x, int64_t batch, int n0, double dt, const Axes &ax, double f0,
                  int flags, float *d_power, cudaStream_t st);
// cwt_fast.cu: Rows::kDif2048 / kDif4096, with their forward transforms into d_xhat (batch x nfft complex)
int cwt_dif(const CwtPlan &pl, const float *d_x, float2 *d_xhat, int64_t batch, int n0, double dt, const Axes &ax,
            double f0, int flags, float *d_power, cudaStream_t st);
// cwt_fast.cu: per-row sample interval inside the cone of influence ([1, 0] for none)
void coi_row_ranges(int n0, double dt, const Axes &ax, double f0, std::vector<ushort2> *out);

// wct_fast.cu: forward FFTs of [nseries, n0] real rows into xhat [nseries, 4096] (FP32, natural order)
int fwd_fft_4096(const float *d_y, int64_t nseries, int n0, float2 *d_xhat, cudaStream_t st);
// wct_fast.cu: Rows::kRows4096 from the forward spectra xhat [batch, 4096]
int cwt_rows_4096(const float2 *d_xhat, int64_t batch, int n0, double dt, const Axes &ax, double f0, int flags,
                  float *d_power, float2 *d_coef, cudaStream_t st);
// wct_fast.cu: the FP32 nfft = 4096 coherence pipeline (spectra, boxcar and coherence kernels).  d_rows_scratch:
// 32 bytes per scale; d_spec: [pairs, S, 4096] float4 scratch.
int wct_fast(const float2 *d_xhat, int64_t pairs, int n0, double dt, const Axes &ax, double f0, void *d_rows_scratch,
             float4 *d_spec, const ScaleWin &win, float *d_wct, float *d_phase, float2 *d_w12,
             unsigned long long *d_hist, const int *d_tlo, const int *d_thi, int maxscale, cudaStream_t st);

// cwt_long.cu: four-step transforms for the powers of two past one CTA's shared memory (long_fft.cuh)
bool cwt_long_takes(int N, size_t elem);
template <typename T> struct LongPlan;
template <typename T> int long_plan(int N, cudaStream_t st, LongPlan<T> *p);
template <typename T>
int cwt_long(const T *d_x, int64_t batch, int n0, int N, double dt, const Axes &ax, const Mother &mo, int flags,
             T *d_power, cplx<T> *d_coef, cudaStream_t st);

// wct_long.cu: the smoothed spectra tsm [pairs, S, n0] (when smooth), W12 and its phase of the interleaved
// series d_y [pairs, 2, n0] at a length cwt_long_takes; scales, COI ranges (when h_tlo) and tsm live in its scratch.
template <typename T> struct WctLongOut {
  vec4<T> *tsm;
  int *tlo, *thi;
};
template <typename T>
int wct_long(const T *d_y, int64_t pairs, int n0, int N, double dt, const Axes &ax, double f0, bool smooth,
             T *d_phase, cplx<T> *d_w12, const int *h_tlo, const int *h_thi, WctLongOut<T> *out, cudaStream_t st);

// wct.cu: rows with at least one sample inside the reliable region (multi.cu's percentile step)
void mc_row_has_points(int nsurr, double dt, const Axes &ax, double f0, std::vector<uint8_t> *any);

}  // namespace wtb
