// AR(1) red-noise surrogates generated on device (pycwt.helpers.rednoise as used
// by pycwt.wct_significance): y[t] = g*y[t-1] + eps[t], eps ~ N(0,1), with the
// first tau = ceil(-2/ln|g|) samples dropped.
//
// Philox4x32-10 keyed by `seed`; the counter is (sample block, series 0 .. K-1,
// GLOBAL realisation index lo/hi), so a realisation's noise does not depend on
// how realisations are partitioned over GPUs or chunks.  K = 2 for coherence
// pairs, K = 3 for the (y, x1, x2) triples of partial / multiple coherence.
#include "common.cuh"

namespace wtb {

struct Philox {
  static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  static constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  __device__ static uint4 run(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
      const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
      c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
      k.x += W0;
      k.y += W1;
    }
    return c;
  }
};

// two uniforms -> two standard normals (Box-Muller, full-precision functions)
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const float u1 = ((float)(a >> 8) + 0.5f) * (1.0f / 16777216.0f);  // (0,1)
  const float u2 = ((float)(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
  const float r = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  return make_float2(r * c, r * s);
}

constexpr int kNoiseThreads = 256;

// One CTA = one series (realisation m, which in [0, K)).  Each thread owns a
// contiguous chunk of the N+tau samples; chunk carries are chained in shared
// memory (a 256-step serial pass, negligible next to the transforms).
// out: [count, K, nsurr]; series `which` has coefficient g[which], burn-in tau[which].
template <typename T, int K>
__global__ void k_rednoise(double g0, double g1, double g2, int tau0, int tau1, int tau2, int nsurr,
                           int64_t first, uint64_t seed, int white, T *__restrict__ out) {
  __shared__ double s_end[kNoiseThreads];
  __shared__ double s_carry[kNoiseThreads];
  const int64_t local = blockIdx.x / K;
  const int which = blockIdx.x % K;
  const uint64_t real = (uint64_t)(first + local);
  const double g = which == 0 ? g0 : (which == 1 ? g1 : g2);
  const int tau = which == 0 ? tau0 : (which == 1 ? tau1 : tau2);
  const int M = nsurr + tau;
  int chunk = (M + kNoiseThreads - 1) / kNoiseThreads;
  chunk = (chunk + 3) & ~3;  // whole Philox blocks of 4 normals
  const int t0 = threadIdx.x * chunk;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  T *dst = out + ((int64_t)local * K + which) * nsurr;

  // pass 1: local recurrence with zero carry-in, remember the chunk-end value
  double y = 0.0;
  for (int i = 0; i < chunk && t0 + i < M; i += 4) {
    const uint4 r = Philox::run(make_uint4((uint32_t)((t0 + i) >> 2), (uint32_t)which,
                                           (uint32_t)real, (uint32_t)(real >> 32)), key);
    const float2 n01 = box_muller(r.x, r.y), n23 = box_muller(r.z, r.w);
    const float e[4] = {n01.x, n01.y, n23.x, n23.y};
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (t0 + i + q < M) y = white ? (double)e[q] : g * y + (double)e[q];
  }
  s_end[threadIdx.x] = y;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double gc = pow(g, (double)chunk);
    double c = 0.0;
    for (int i = 0; i < kNoiseThreads; ++i) {
      s_carry[i] = c;                       // value of y just before chunk i
      c = gc * c + s_end[i];
    }
  }
  __syncthreads();
  // pass 2: regenerate the same normals, now with the right carry-in, and store
  y = white ? 0.0 : s_carry[threadIdx.x];
  for (int i = 0; i < chunk && t0 + i < M; i += 4) {
    const uint4 r = Philox::run(make_uint4((uint32_t)((t0 + i) >> 2), (uint32_t)which,
                                           (uint32_t)real, (uint32_t)(real >> 32)), key);
    const float2 n01 = box_muller(r.x, r.y), n23 = box_muller(r.z, r.w);
    const float e[4] = {n01.x, n01.y, n23.x, n23.y};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int t = t0 + i + q;
      if (t < M) {
        y = white ? (double)e[q] : g * y + (double)e[q];
        if (t >= tau) dst[t - tau] = (T)y;
      }
    }
  }
}

static int burn_in(double g) {
  if (g == 0) return 0;
  return (int)std::ceil(-2.0 / std::log(std::fabs(g)));
}

template <typename T, int K>
static int rednoise_launch(const double (&g)[3], int nsurr, int64_t first, int64_t count, uint64_t seed, bool white,
                           T *d_out, cudaStream_t st) {
  WTB_REQUIRE(count * K < (1LL << 31), WTB_EUNSUPPORTED, "too many surrogates in one launch");
  k_rednoise<T, K><<<(unsigned)(count * K), kNoiseThreads, 0, st>>>(
      g[0], g[1], g[2], burn_in(g[0]), burn_in(g[1]), burn_in(g[2]), nsurr, first, seed, white ? 1 : 0, d_out);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

template <typename T>
int rednoise_device(double a1, double a2, int nsurr, int64_t first, int64_t count, uint64_t seed,
                    bool white, T *d_out, cudaStream_t st) {
  return rednoise_launch<T, 2>({a1, a2, 0.0}, nsurr, first, count, seed, white, d_out, st);
}
template int rednoise_device<float>(double, double, int, int64_t, int64_t, uint64_t, bool, float *, cudaStream_t);
template int rednoise_device<double>(double, double, int, int64_t, int64_t, uint64_t, bool, double *, cudaStream_t);

template <typename T>
int rednoise_triples_device(double ay, double a1, double a2, int nsurr, int64_t first, int64_t count,
                            uint64_t seed, bool white, T *d_out, cudaStream_t st) {
  return rednoise_launch<T, 3>({ay, a1, a2}, nsurr, first, count, seed, white, d_out, st);
}
template int rednoise_triples_device<float>(double, double, double, int, int64_t, int64_t, uint64_t, bool, float *,
                                            cudaStream_t);
template int rednoise_triples_device<double>(double, double, double, int, int64_t, int64_t, uint64_t, bool, double *,
                                             cudaStream_t);

}  // namespace wtb

using namespace wtb;

// wtb_rednoise (K = 2) and wtb_rednoise_triples (K = 3)
template <int K>
static int rednoise_entry(const char *name, const double (&g)[3], int nsurr, int64_t first, int64_t count,
                          uint64_t seed, int flags, void *out, void *stream) {
  WTB_REQUIRE(out && nsurr > 0 && count >= 0 && first >= 0, WTB_EINVAL, "%s: bad arguments", name);
  for (int i = 0; i < K; ++i)
    WTB_REQUIRE(fabs(g[i]) < 1, WTB_EINVAL, "AR(1) coefficients must lie in (-1, 1)");
  WTB_ENTER(flags, out, stream);
  if (count == 0) return WTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool f64 = flags & WTB_F64;
  const size_t bytes = (f64 ? 8 : 4) * (size_t)count * K * nsurr;
  void *d = out;
  if (!(flags & WTB_DEVICE_PTRS)) WTB_TRY(staging_reserve(bytes, &d));
  const bool white = flags & WTB_NOISE_WHITE;
  const int rc = f64 ? rednoise_launch<double, K>(g, nsurr, first, count, seed, white, (double *)d, st)
                     : rednoise_launch<float, K>(g, nsurr, first, count, seed, white, (float *)d, st);
  WTB_TRY(rc);
  if (!(flags & WTB_DEVICE_PTRS)) {
    WTB_TRY(copy_to_host(out, d, bytes, st));
    WTB_CUDA(cudaStreamSynchronize(st));
  }
  return WTB_OK;
}

extern "C" int wtb_rednoise(double a1, double a2, int nsurr, int64_t first, int64_t count, uint64_t seed,
                            int flags, void *out, void *stream) {
  return rednoise_entry<2>("wtb_rednoise", {a1, a2, 0.0}, nsurr, first, count, seed, flags, out, stream);
}

extern "C" int wtb_rednoise_triples(double ay, double a1, double a2, int nsurr, int64_t first, int64_t count,
                                    uint64_t seed, int flags, void *out, void *stream) {
  return rednoise_entry<3>("wtb_rednoise_triples", {ay, a1, a2}, nsurr, first, count, seed, flags, out, stream);
}
