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

}  // namespace wtb
