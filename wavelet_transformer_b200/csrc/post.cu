// Batched post-processing of transform planes on the device (SURVEY 8f-2): the steps the reference
// runs in NumPy right after the library calls, for batches that stay in HBM.
//   ratio planes   power / signif[:, None]            src/cwt.py:118-133
//                  |coherence| / signif[:, None]      src/wct.py:120-125
//                  |W12|^2 and |W12|^2 / signif       src/utils/wavelet_helpers.py:60-78
//   phase arrows   u = cos(pi/2 - phase), v = sin(pi/2 - phase)   src/wct.py:143-158, src/xwt.py:142-154
// Pure streaming kernels: HBM-bound, one read and one write per element.
#include "common.cuh"

namespace wtb {

// plane: [batch, S, n0] real (COMPLEX: interleaved complex).  signif: [sig_rows, S] double with
// sig_rows = batch or 1.  ratio = |x| / signif (COMPLEX: |z|^2 / signif, power = |z|^2).
template <typename T, bool COMPLEX>
__global__ void k_ratio_planes(const T *__restrict__ plane, int64_t rows, int S, int n0, const double *__restrict__ signif,
                               int sig_per_batch, T *__restrict__ power, T *__restrict__ ratio) {
  const int64_t row = blockIdx.y + (int64_t)blockIdx.z * gridDim.y;     // (b, s) flattened
  if (row >= rows) return;
  const int s = (int)(row % S);
  const int64_t b = row / S;
  const double sg = signif[(sig_per_batch ? b * S : 0) + s];
  const T *src = plane + row * (int64_t)n0 * (COMPLEX ? 2 : 1);
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n0; t += gridDim.x * blockDim.x) {
    T p;
    if (COMPLEX) {
      const T re = src[2 * t], im = src[2 * t + 1];
      // numpy: np.abs(z) ** 2 -- hypot, then the square
      const T m = sizeof(T) == 8 ? (T)hypot((double)re, (double)im) : (T)hypotf((float)re, (float)im);
      p = m * m;
      if (power) power[row * (int64_t)n0 + t] = p;
    } else {
      p = fabs(src[t]);
    }
    if (ratio) ratio[row * (int64_t)n0 + t] = (T)((double)p / sg);
  }
}

template <typename T>
__global__ void k_phase_arrows(const T *__restrict__ phase, int64_t count, T *__restrict__ u, T *__restrict__ v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    const T angle = T(0.5 * kPi) - phase[i];       // the reference's expression, same rounding
    T sn, cs;
    if (sizeof(T) == 8) { double a, c; sincos((double)angle, &a, &c); sn = (T)a; cs = (T)c; }
    else { float a, c; sincosf((float)angle, &a, &c); sn = (T)a; cs = (T)c; }
    if (u) u[i] = cs;
    if (v) v[i] = sn;
  }
}

template <typename T>
static int ratio_impl(const void *plane, int64_t batch, int S, int n0, const double *signif, int64_t sig_rows, int flags,
                      void *power_out, void *ratio_out, cudaStream_t st) {
  const bool dev = flags & WTB_DEVICE_PTRS, cx = flags & WTB_PLANE_COMPLEX;
  const size_t in_row = sizeof(T) * (size_t)S * n0 * (cx ? 2 : 1), out_row = sizeof(T) * (size_t)S * n0;
  void *prm = nullptr;
  const double *d_sig = signif;
  // signif is small and always comes from the host side of the caller's pipeline unless DEVICE_PTRS
  if (!dev) {
    WTB_TRY(arena_reserve(align256(sizeof(double) * (size_t)sig_rows * S), &prm));
    WTB_CUDA(cudaMemcpyAsync(prm, signif, sizeof(double) * (size_t)sig_rows * S, cudaMemcpyHostToDevice, st));
    d_sig = (const double *)prm;
  }
  return stage_rows(batch, host_rows(batch, in_row + 2 * out_row, flags), flags, st, {{plane, in_row}},
                    {{power_out, out_row}, {ratio_out, out_row}}, 0,
                    [&](const void *const *in, void *const *out, void *, int64_t b0, int64_t nb) {
                      const int64_t rows = nb * S;
                      const unsigned gy = (unsigned)std::min<int64_t>(rows, 65535), gz = (unsigned)((rows + gy - 1) / gy);
                      WTB_REQUIRE(gz <= 65535, WTB_EUNSUPPORTED, "batch too large for one launch");
                      const dim3 grid((unsigned)std::min(8, (n0 + 255) / 256), gy, gz);
                      const double *sg = d_sig + (sig_rows > 1 ? b0 * S : 0);
                      const T *src = (const T *)in[0];
                      T *pw = (T *)out[0], *rt = (T *)out[1];
                      if (cx) k_ratio_planes<T, true><<<grid, 256, 0, st>>>(src, rows, S, n0, sg, sig_rows > 1, pw, rt);
                      else k_ratio_planes<T, false><<<grid, 256, 0, st>>>(src, rows, S, n0, sg, sig_rows > 1, pw, rt);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

template <typename T>
static int arrows_impl(const void *phase, int64_t count, int flags, void *u_out, void *v_out, cudaStream_t st) {
  return stage_rows(count, host_rows(count, 3 * sizeof(T), flags), flags, st, {{phase, sizeof(T)}},
                    {{u_out, sizeof(T)}, {v_out, sizeof(T)}}, 0,
                    [&](const void *const *in, void *const *out, void *, int64_t, int64_t n) {
                      const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 16);
                      k_phase_arrows<T><<<blocks, 256, 0, st>>>((const T *)in[0], n, (T *)out[0], (T *)out[1]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_ratio_planes(const void *plane, int64_t batch, int S, int n0, const double *signif, int64_t sig_rows,
                                int flags, void *power_out, void *ratio_out, void *stream) {
  WTB_REQUIRE(plane && signif && batch >= 0 && S > 0 && n0 > 0, WTB_EINVAL, "wtb_ratio_planes: bad arguments");
  WTB_REQUIRE(sig_rows == 1 || sig_rows == batch, WTB_EINVAL, "wtb_ratio_planes: signif has %lld rows, expected 1 or %lld",
              (long long)sig_rows, (long long)batch);
  WTB_REQUIRE(ratio_out || ((flags & WTB_PLANE_COMPLEX) && power_out), WTB_EINVAL, "wtb_ratio_planes: no output requested");
  WTB_REQUIRE(!power_out || (flags & WTB_PLANE_COMPLEX), WTB_EINVAL, "wtb_ratio_planes: power_out needs WTB_PLANE_COMPLEX");
  WTB_ENTER(flags, plane, stream);
  if (batch == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return ratio_impl<double>(plane, batch, S, n0, signif, sig_rows, flags, power_out, ratio_out, st);
  return ratio_impl<float>(plane, batch, S, n0, signif, sig_rows, flags, power_out, ratio_out, st);
}

extern "C" int wtb_phase_arrows(const void *phase, int64_t count, int flags, void *u_out, void *v_out, void *stream) {
  WTB_REQUIRE(phase && count >= 0 && (u_out || v_out), WTB_EINVAL, "wtb_phase_arrows: bad arguments");
  WTB_ENTER(flags, phase, stream);
  if (count == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & WTB_F64) return arrows_impl<double>(phase, count, flags, u_out, v_out, st);
  return arrows_impl<float>(phase, count, flags, u_out, v_out, st);
}
