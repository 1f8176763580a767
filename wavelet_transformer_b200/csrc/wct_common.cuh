// Pieces shared by the generic (wct.cu) and fast (wct_fast.cu) coherence kernels.
#pragma once

#include "common.cuh"

namespace wtb {

template <typename T> struct vec4_of;
template <> struct vec4_of<float> { using type = float4; };
template <> struct vec4_of<double> { using type = double4; };
template <typename T> using vec4 = typename vec4_of<T>::type;

constexpr int kMaxWin = 64;
// Scale-axis boxcar of Morlet.smooth: out[i] = sum_k w[k] * T[i + up - k], rows outside
// [0, S) count as zero and the window is not renormalised (scipy convolve2d 'same').
struct ScaleWin {
  int K;          // taps
  int up;         // (K-1)/2
  double w[kMaxWin];
};

// Morlet.smooth: rect(int(round(deltaj0/dj*2)), normalize=True), deltaj0 = 0.6
inline int make_win(double dj, ScaleWin *win) {
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

}  // namespace wtb
