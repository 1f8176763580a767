// FP32 fast path of the fused CWT+power kernel for nfft = 1024 (BASELINE cfg4).
//
// One warp owns one series at a time and never synchronises with other warps:
//   forward FFT(1024) -> X^ in shared memory (positive half only)
//   for every scale row s: Y = X^ * daughter_s (band-limited, one-sided)
//                          w = IFFT_1024(Y) as 32 x 32:  k = k1 + 32 k2,  t = t2 + 32 t1
//                          power = |w|^2 -> 128-byte coalesced streaming stores
// A 1024-point transform is two in-register 32-point DFTs per thread with one
// shared-memory transpose between them:
//   step A (lane = k1): A[k1][t2]  = sum_k2 Y[k1+32 k2] w32^(k2 t2), times w1024^(k1 t2)
//   step B (lane = t2): x[t2+32t1] = sum_k1 A'[k1][t2] w32^(k1 t1)
// Lanes map to t2, so for each t1 the warp stores 32 consecutive floats.
//
// Arithmetic is the sm_100a packed FP32x2 pipe (FFMA2/FADD2/FMUL2): registers hold
// (element p, element p+16) pairs in structure-of-arrays form (fft32_gen.cuh), so
// one instruction does two butterflies / two twiddle products / two |w|^2.
//
// Work that the Morlet daughter makes unnecessary is skipped exactly (to 1e-6 of
// the daughter peak, far inside the FP32 tolerance): negative frequencies, and
// bins above k_hi(s) = (f0 + 5.3) N dt / (2 pi s).  Rows with k_hi < 32 need no
// step A and no transpose; rows with fewer non-zero inputs skip butterfly stages.
#include "cwt_paths.cuh"
#include "fft32_gen.cuh"
#include "filterbank_common.cuh"
#include "spectral.cuh"

namespace wtb {

namespace {

using fft32::add2;
using fft32::bc;
using fft32::br4;
using fft32::fma2;
using fft32::mul2;

constexpr int kN = 1024;
constexpr int kWarps = 16;            // warps per CTA, one CTA per SM
constexpr int kTrStride = 34;         // floats per row of the transpose buffer (even, == 2 mod 32)

struct RowParam {
  float a;         // (s/dt) * 2*pi/N : s*w_k = a*k
  float lognorm;   // log2( sqrt(2*pi*s/dt) * pi^-1/4 / N )
  int L;           // log2(#non-zero inputs) of the first DFT that runs (>= 1)
  int multi;       // 1: k_hi >= 32 -> step A + transpose + full step B
};

struct WarpSmem {
  float2 xr[8][32];                 // xr[m][lane] = Re X^[lane + 32*(2m)], Re X^[lane + 32*(2m+1)]
  float2 xi[8][32];
  float trr[32 * kTrStride];        // transpose buffer, real parts:  [k1][2*(t2&15) + (t2>>4)]
  float tri[32 * kTrStride];
  float yr[32];                     // Y[k] of a single-pass row
  float yi[32];
};

struct CtaSmem {
  // exp(+2*pi*i*a*b/1024) tables, float4 = (re_0, re_1, im_0, im_1) for a packed pair
  float4 tw_a[16][32];              // pair (t2, t2+16) x k1=lane   : step A output twiddle
  float4 tw_b[16][32];              // pair (2m, 2m+1)  x t2=lane   : single-pass input twiddle
  RowParam row[kMaxRows];
  ushort2 coi[kMaxRows];            // COI only: samples [x, y] of row s lie inside the cone of influence
  WarpSmem w[kWarps];
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float2 neg2(float2 v) { return make_float2(-v.x, -v.y); }

// For a power of two M:  m < M  <=>  M > below_pow2(m), with below_pow2(m) the largest
// power of two <= m (and -1 for m = 0).  Unrolled loops over m then test M against only
// log2 distinct constants, one compare per block [2^k, 2^(k+1)).
__device__ __forceinline__ constexpr int below_pow2(int m) {
  return m == 0 ? -1 : (m < 2 ? 1 : (m < 4 ? 2 : (m < 8 ? 4 : 8)));
}

// One dit32 call site serves the forward transform (s = -1), step A and step B of
// every scale row: the hot code stays inside the instruction cache.
//
// HALF = true serves nfft = 512 (series of 257..512 samples) with the same 1024-point machinery,
// TWO SERIES per warp: series A takes the even bins of the 1024-point spectrum, series B the odd
// ones, Z[2k] = Y_A[k], Z[2k+1] = Y_B[k].  Then x[t] = a[t] + w1024^t b[t] and
// x[t+512] = a[t] - w1024^t b[t] with a, b the two 512-point inverse transforms, and t, t+512 are
// the two halves of one packed register: |a|^2 = |x[t] + x[t+512]|^2 / 4, |b|^2 likewise with
// the difference (the phase w^t drops out of the power).  The forward transforms of both real
// series come from one pass over A - iB repeated twice (even bins = the 512-point spectrum).
//
// COI = true fuses pycwt's cone-of-influence mask into the store loop (north_star (1); consumers:
// src/utils/wavelet_helpers.py:60-78, pycwt's `outsidecoi`): row s keeps samples coi[s].x ..
// coi[s].y and writes NaN elsewhere -- the interval is evaluated on the host in double exactly as
// the generic kernel evaluates `period > coi(t)`, so the mask is bit-equal and costs no traffic.
template <bool HALF, bool COI>
__global__ void __launch_bounds__(kWarps * 32, 1)
k_cwt_fast_1024(const float *__restrict__ x, int64_t batch, int n0, int S,
                const RowParam *__restrict__ rows, const ushort2 *__restrict__ coi, float f0,
                float *__restrict__ power, int split) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CtaSmem &sm = *reinterpret_cast<CtaSmem *>(smem_raw);
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 16 * 32; i += blockDim.x) {
    const int p = i >> 5, l = i & 31;
    float s0, c0, s1, c1;
    sincospif(2.0f * (float)(p * l) / (float)kN, &s0, &c0);
    sincospif(2.0f * (float)((p + 16) * l) / (float)kN, &s1, &c1);
    sm.tw_a[p][l] = make_float4(c0, c1, s0, s1);
    sincospif(2.0f * (float)(2 * p * l) / (float)kN, &s0, &c0);
    sincospif(2.0f * (float)((2 * p + 1) * l) / (float)kN, &s1, &c1);
    sm.tw_b[p][l] = make_float4(c0, c1, s0, s1);
  }
  for (int i = threadIdx.x; i < S; i += blockDim.x) {
    sm.row[i] = rows[i];
    if (COI) sm.coi[i] = coi[i];
  }
  __syncthreads();
  WarpSmem &ws = sm.w[warp];
  // consecutive series go to different SMs: a small batch spreads over the machine
  const int64_t gwarp = (int64_t)warp * gridDim.x + blockIdx.x;
  const int64_t nwarps = (int64_t)gridDim.x * kWarps;
  const bool full_row = (n0 == kN);
  // HALF: bin k = lane + 32 k2 belongs to series (lane & 1) and is its bin (k - (lane & 1)) / 2
  const float lanef = (float)(HALF ? (lane & ~1) : lane);
  const int tidx = 2 * (lane & 15) + (lane >> 4);   // column of this lane (as t2) in the transpose buffer
  float2 R[16], I[16];

  // One warp item = one series (HALF: series 2b and 2b + 1) and every split-th scale row from row c
  // on: a batch too small to give every warp of the machine a series is spread by rows instead
  // (each item repeats the forward transform, 1 / S of a series' work).  split = 1: all rows.
  const int64_t items = (HALF ? (batch + 1) / 2 : batch) * split;
  for (int64_t it = gwarp; it < items; it += nwarps) {
    const int64_t b = it / split;
    const int c = (int)(it - b * split);
    const float *xr = x + (HALF ? 2 * b : b) * n0;
    const bool has_b = !HALF || 2 * b + 1 < batch;
    float unscale_a = 1.0f, unscale_b = 1.0f;              // HALF: 4^exponent of each series' pre-scaling
    float *out = power + (HALF ? 2 * b : b) * (int64_t)S * n0 + lane;
#pragma unroll 1
    for (int s = -1; s < S; s = s < 0 ? c : s + split) {
      int L, two_pass;
      if (s < 0) {
        // forward FFT of the real series: X^[t] = conj(sum_k x[k] w^(+k t))
#pragma unroll
        for (int m = 0; m < 16; ++m) {
          const int k = lane + 64 * m;
          if (HALF) {
            // conj(z), z[t] = A[t mod 512] + i B[t mod 512]: the periodic repeat puts the 512-point
            // spectrum of z on the even bins
            const int t0 = k & 511, t1 = (k + 32) & 511;
            const float *xb = xr + n0;
            R[br4(m)] = make_float2(t0 < n0 ? __ldg(xr + t0) : 0.0f, t1 < n0 ? __ldg(xr + t1) : 0.0f);
            I[br4(m)] = make_float2(has_b && t0 < n0 ? -__ldg(xb + t0) : 0.0f, has_b && t1 < n0 ? -__ldg(xb + t1) : 0.0f);
          } else {
            R[br4(m)] = make_float2(k < n0 ? __ldg(xr + k) : 0.0f, k + 32 < n0 ? __ldg(xr + k + 32) : 0.0f);
            I[br4(m)] = make_float2(0.0f, 0.0f);
          }
        }
        if (HALF) {
          // The two series share one transform, so round-off scales with the LARGER of them: bring
          // each to [0.5, 1) by an exact power of two first and give the factor back to its power.
          float ma = 0.0f, mb = 0.0f;
#pragma unroll
          for (int m = 0; m < 16; ++m) {
            ma = fmaxf(ma, fmaxf(fabsf(R[m].x), fabsf(R[m].y)));
            mb = fmaxf(mb, fmaxf(fabsf(I[m].x), fabsf(I[m].y)));
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, o));
            mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, o));
          }
          int ea = 0, eb = 0;
          if (ma > 0.0f && ma < INFINITY) frexpf(ma, &ea);
          if (mb > 0.0f && mb < INFINITY) frexpf(mb, &eb);
          const float2 sa = bc(ldexpf(1.0f, -ea)), sb = bc(ldexpf(1.0f, -eb));
          unscale_a = ldexpf(1.0f, 2 * ea);
          unscale_b = ldexpf(1.0f, 2 * eb);
#pragma unroll
          for (int m = 0; m < 16; ++m) {
            R[m] = mul2(R[m], sa);
            I[m] = mul2(I[m], sb);
          }
        }
        L = 5;
        two_pass = 1;
      } else {
        const RowParam rp = sm.row[s];
        L = rp.L;
        two_pass = rp.multi;
        const float zl = fmaf(rp.a, lanef, -f0);   // s*w_k - f0 at k = lane
        if (two_pass) {
          // Y[lane + 32 k2] = X^ * daughter for k2 < 2^L, two k2 per packed op
          const int M = 1 << (rp.L - 1);
          const float2 zl2 = make_float2(zl, fmaf(rp.a, 32.0f, zl));
          const float2 a64 = bc(rp.a * 64.0f);
          const float2 ln2 = bc(rp.lognorm);
          // M is a power of two: blocks [0,1), [1,2), [2,4), [4,8) need one branch each
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            if (M > below_pow2(m)) {
              const float2 z = fma2(a64, bc((float)m), zl2);
              const float2 e = fma2(mul2(z, z), bc(-0.72134752044f), ln2);   // -0.5*log2(e)*z^2 + log2(norm)
              const float2 d = make_float2(ex2(e.x), ex2(e.y));
              R[br4(m)] = mul2(ws.xr[m][lane], d);
              I[br4(m)] = mul2(ws.xi[m][lane], d);
            }
          }
        } else {
          const float e = fmaf(zl * zl, -0.72134752044f, rp.lognorm);
          const float d = ex2(e);
          const float2 vr = ws.xr[0][lane], vi = ws.xi[0][lane];
          ws.yr[lane] = vr.x * d;
          ws.yi[lane] = vi.x * d;
          __syncwarp();
          // u[k1] = Y[k1] * w1024^(k1 * lane) for k1 < 2^L, two k1 per packed op
          const int M = 1 << (rp.L - 1);
#pragma unroll
          for (int m = 0; m < 16; ++m) {
            if (M > below_pow2(m)) {
              const float2 yr = *reinterpret_cast<const float2 *>(&ws.yr[2 * m]);
              const float2 yi = *reinterpret_cast<const float2 *>(&ws.yi[2 * m]);
              const float4 t = sm.tw_b[m][lane];
              const float2 twr = make_float2(t.x, t.y), twi = make_float2(t.z, t.w);
              R[br4(m)] = fma2(yi, neg2(twi), mul2(yr, twr));
              I[br4(m)] = fma2(yr, twi, mul2(yi, twr));
            }
          }
          __syncwarp();
        }
      }
      fft32::dit32(R, I, L);        // the pruned site: step A, or the only pass of a narrow row
      if (two_pass) {
        // step A done (lane = k1): twiddle by w1024^(k1 t2), transpose, reload with lane = t2
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          const float4 t = sm.tw_a[p][lane];
          const float2 twr = make_float2(t.x, t.y), twi = make_float2(t.z, t.w);
          const float2 vr = fma2(I[p], neg2(twi), mul2(R[p], twr));
          const float2 vi = fma2(R[p], twi, mul2(I[p], twr));
          *reinterpret_cast<float2 *>(&ws.trr[lane * kTrStride + 2 * p]) = vr;
          *reinterpret_cast<float2 *>(&ws.tri[lane * kTrStride + 2 * p]) = vi;
        }
        __syncwarp();
#pragma unroll
        for (int m = 0; m < 16; ++m) {
          R[br4(m)] = make_float2(ws.trr[(2 * m) * kTrStride + tidx], ws.trr[(2 * m + 1) * kTrStride + tidx]);
          I[br4(m)] = make_float2(ws.tri[(2 * m) * kTrStride + tidx], ws.tri[(2 * m + 1) * kTrStride + tidx]);
        }
        __syncwarp();
        fft32::dit32(R, I, 5);      // step B is always a full transform: its own straight-line site
      }
      if (s < 0 && HALF) {
        // FFT1024(z repeated)[2 kk] = 2 Z[kk] = 2 conj(u[2 kk]); even lanes hold kk = lane/2 + 16 t1.
        // Park Z/2 in the (now free) transpose buffer, then split it into the two real series'
        // spectra: A^ = (Z[kk] + conj Z[-kk]) / 2, B^ = (Z[kk] - conj Z[-kk]) / 2i, kk < 256.
        float *zr = ws.trr, *zi = ws.tri;
        if ((lane & 1) == 0) {
#pragma unroll
          for (int t1 = 0; t1 < 16; ++t1) {
            zr[(lane >> 1) + 16 * t1] = 0.25f * R[t1].x;
            zi[(lane >> 1) + 16 * t1] = -0.25f * I[t1].x;
            zr[(lane >> 1) + 16 * (t1 + 16)] = 0.25f * R[t1].y;
            zi[(lane >> 1) + 16 * (t1 + 16)] = -0.25f * I[t1].y;
          }
        }
        __syncwarp();
        const bool odd = lane & 1;
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          float vr[2], vi[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int kk = (lane >> 1) + 16 * (2 * m + h), j = (512 - kk) & 511;
            const float ar = zr[kk], ai = zi[kk], br = zr[j], bi = zi[j];   // Z[kk]/2 and Z[-kk]/2 (unconjugated)
            vr[h] = odd ? ai + bi : ar + br;
            vi[h] = odd ? br - ar : ai - bi;
          }
          ws.xr[m][lane] = make_float2(vr[0], vr[1]);
          ws.xi[m][lane] = make_float2(vi[0], vi[1]);
        }
        __syncwarp();
      } else if (s < 0) {
        // X^[lane + 32 t1] = conj(u[t1]), t1 < 16 (positive frequencies only)
        float *pr = reinterpret_cast<float *>(&ws.xr[0][0]);
        float *pi = reinterpret_cast<float *>(&ws.xi[0][0]);
#pragma unroll
        for (int t1 = 0; t1 < 16; ++t1) {
          pr[(t1 >> 1) * 64 + lane * 2 + (t1 & 1)] = R[t1].x;
          pi[(t1 >> 1) * 64 + lane * 2 + (t1 & 1)] = -I[t1].x;
        }
        __syncwarp();
      } else if (HALF) {
        // (x[t], x[t+512]) share a register: a = (sum)/2, b = (difference)/2 up to a phase; the 1/2
        // rides in lognorm (1/1024 instead of 1/512)
        float *orow = out + (int64_t)s * n0;
        const int tlo = COI ? sm.coi[s].x : 0, thi = COI ? sm.coi[s].y : kN;
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          const float sr = R[p].x + R[p].y, si = I[p].x + I[p].y;
          const float dr = R[p].x - R[p].y, di = I[p].x - I[p].y;
          if (lane + 32 * p < n0) {
            const bool in = !COI || (lane + 32 * p >= tlo && lane + 32 * p <= thi);
            __stcs(orow + 32 * p, in ? fmaf(sr, sr, si * si) * unscale_a : NAN);
            if (has_b) __stcs(orow + (int64_t)S * n0 + 32 * p, in ? fmaf(dr, dr, di * di) * unscale_b : NAN);
          }
        }
      } else {
        float *orow = out + (int64_t)s * n0;
        if (COI) {
          // outside [tlo, thi] (and past n0, where thi < n0 ends the row anyway) nothing valid exists
          const int tlo = sm.coi[s].x, thi = sm.coi[s].y;
#pragma unroll
          for (int p = 0; p < 16; ++p) {
            const float2 pw = fma2(R[p], R[p], mul2(I[p], I[p]));
            const int ta = lane + 32 * p, tb = ta + 512;
            if (ta < n0) __stcs(orow + 32 * p, (ta >= tlo && ta <= thi) ? pw.x : NAN);
            if (tb < n0) __stcs(orow + 32 * (p + 16), (tb >= tlo && tb <= thi) ? pw.y : NAN);
          }
        } else if (full_row) {
#pragma unroll
          for (int p = 0; p < 16; ++p) {
            const float2 pw = fma2(R[p], R[p], mul2(I[p], I[p]));
            __stcs(orow + 32 * p, pw.x);
            __stcs(orow + 32 * (p + 16), pw.y);
          }
        } else {
#pragma unroll
          for (int p = 0; p < 16; ++p) {
            const float2 pw = fma2(R[p], R[p], mul2(I[p], I[p]));
            if (lane + 32 * p < n0) __stcs(orow + 32 * p, pw.x);
            if (lane + 32 * (p + 16) < n0) __stcs(orow + 32 * (p + 16), pw.y);
          }
        }
      }
    }
  }
}


// ---- nfft = 2048 (series of 1025..2048 samples, e.g. the reference's 1346-month CPI series) ----
// Two warps per scale row (k_cwt_dif<2>).  Decimation in frequency: with E[u], G[u] the 1024-point
// inverse transforms of the even and of the odd bins of the one-sided spectrum Y[k], k < 1024,
//   x[u]        = E[u] + w2048^u G[u]
//   x[u + 1024] = E[u] - w2048^u G[u],          u < 1024.
// Warp h of a pair owns the bins of parity h: 512 of them, so step A of its 1024-point transform has at
// most 16 non-zero inputs (one butterfly stage less than a full pass) and a row is single-pass up to
// k_hi < 64 instead of 32.  The two warps swap half of their packed registers through mailboxes that alias
// the (by then idle) transpose buffers: warp 0 finishes register positions p < 8, warp 1 p >= 8; the twiddle
// w2048^u rides in the additions of the finishing warp (x[u] = e + w g as two FFMA2 per component,
// x[u + 1024] = 2 e - x[u]), so both warps do the same work, and each stores whole 128-byte lines of x[u],
// x[u + 512], x[u + 1024] and x[u + 1536] -- no strided stores, no staging, nothing past n0 is combined or stored.
// The eight pairs of a CTA work on ONE series: its spectrum X^ (8 KB, in the layout the warps load with one
// 16-byte access per packed pair) arrives by a TMA bulk copy into a ring of three slots (mbarrier full /
// done), so no row ever re-reads global memory, and the pairs draw rows from a shared counter (small scales
// first, they are the expensive ones).
// History: rounds 1-2 ran this shape as two time-decimated 1024-point passes per row in one warp (samples
// 2u + q, `k_cwt_fast_fold`: stride-2 or staged stores, X^ re-read through L1; 4.0e11 coeff/s at 1346
// samples, 5.6e11 at 2048 -- DESIGN.md section 4 keeps its measurements); this kernel is faster at every batch
// size (4.6e11 / 6.9e11, 0.040 ms against 0.055 ms for 12 series) and replaced it.
// nfft = 4096 (series of 2049..4096 samples) is the same kernel with D = 4 warps per row: warp r owns the bins
// k = 4 j + r of the one-sided spectrum (k < 2048, again 512 per warp), and
//   x[u + 1024 q] = sum_r i^(q r) w4096^(r u) G_r[u],   q = 0..3,
// is a radix-4 butterfly of the four twiddled 1024-point transforms: every warp deals its 16 register positions
// to the four mailboxes of the group (its own included, so that the finishing code has compile-time register
// indices), warp g finishes positions 4g .. 4g+3 and stores eight whole lines per position.
constexpr int kDifWarps = 16;

struct alignas(16) WarpSmemP {
  float trr[32 * kTrStride];        // transpose buffer; its first 32 floats double as Y[k] of a single-pass row,
  float tri[32 * kTrStride];        // its first 2 KB (D = 2) / 4 KB (D = 4) as the mailbox the group's warps fill
};

template <int D> struct CtaSmemP {
  static constexpr int kRing = D == 2 ? 3 : 2;
  static constexpr int kGroups = kDifWarps / D;
  float4 tw_a[16][32];              // as in CtaSmem: twiddles of the 1024-point transform
  float4 tw_b[16][32];
  float4 tw_o[D - 1][16][32];       // w_N^(r u), u = lane + 32 p, r = 1 .. D-1: (Re at u, Re at u + 512, Im at u, Im at u + 512)
  float4 xh[kRing][D][8][32];       // X^ of the series in flight in group layout (k_fwd_fft_pair2048 / k_dif_layout): [r][m][lane] =
                                    // (Re X^[k0], Re X^[k1], Im X^[k0], Im X^[k1]), k0 = D (lane + 64 m) + r, k1 = k0 + 32 D
  RowParam row[kMaxRowsF];
  ushort2 coi[kMaxRowsF];
  uint64_t full[kRing];             // TMA completion of a slot
  uint64_t done[kRing];             // every group has finished the slot's series
  int next_row[kRing];
  int group_row[2][kGroups];        // row drawn by the group's leader, by series parity (the other warps may still be
                                    // reading the last draw of one series when the leader draws for the next)
  WarpSmemP w[kDifWarps];
};
static_assert(sizeof(CtaSmemP<2>) <= 227 * 1024 && sizeof(CtaSmemP<4>) <= 227 * 1024,
              "the tables, ring and per-warp buffers of the decimation-in-frequency kernels must fit one CTA");

template <int D> __device__ __forceinline__ void group_sync(int group) {
  asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(32 * D) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t phase) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(phase)
      : "memory");
  return ok != 0;
}

template <int D, bool COI>
__global__ void __launch_bounds__(kDifWarps * 32, 1)
k_cwt_dif(const float2 *__restrict__ xhat, int64_t xhat_stride, int64_t batch, int n0, int S,
          const RowParam *__restrict__ rows, const ushort2 *__restrict__ coi, float f0,
          float *__restrict__ power, int split) {
  using Smem = CtaSmemP<D>;
  constexpr int kRing = Smem::kRing, kGroups = Smem::kGroups;
  constexpr int kNF = D * kN;
  constexpr uint32_t kSlotBytes = sizeof(float4) * D * 8 * 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int group = warp / D, h = warp % D;
  for (int i = threadIdx.x; i < 16 * 32; i += blockDim.x) {
    const int p = i >> 5, l = i & 31;
    float s0, c0, s1, c1;
    sincospif(2.0f * (float)(p * l) / (float)kN, &s0, &c0);
    sincospif(2.0f * (float)((p + 16) * l) / (float)kN, &s1, &c1);
    sm.tw_a[p][l] = make_float4(c0, c1, s0, s1);
    sincospif(2.0f * (float)(2 * p * l) / (float)kN, &s0, &c0);
    sincospif(2.0f * (float)((2 * p + 1) * l) / (float)kN, &s1, &c1);
    sm.tw_b[p][l] = make_float4(c0, c1, s0, s1);
#pragma unroll
    for (int r = 1; r < D; ++r) {
      sincospif(2.0f * (float)(r * (l + 32 * p)) / (float)kNF, &s0, &c0);
      sincospif(2.0f * (float)(r * (l + 32 * p + 512)) / (float)kNF, &s1, &c1);
      sm.tw_o[r - 1][p][l] = make_float4(c0, c1, s0, s1);
    }
  }
  for (int i = threadIdx.x; i < S; i += blockDim.x) {
    sm.row[i] = rows[i];
    if (COI) sm.coi[i] = coi[i];
  }
  const unsigned items = (unsigned)(batch * split);   // one CTA item = one series and every split-th row from row c on (host: < 2^31)
  int next_load = 0;                              // thread 0: local index of the next series to fetch
  auto issue_load = [&](int j) {
    const unsigned it = blockIdx.x + (unsigned)j * gridDim.x;
    const int slot = j % kRing;
    sm.next_row[slot] = 0;
    mbar_expect_tx(&sm.full[slot], kSlotBytes);
    tma_load_1d(&sm.xh[slot][0][0][0], xhat + (int64_t)(it / (unsigned)split) * xhat_stride, kSlotBytes, &sm.full[slot]);
  };
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRing; ++i) {
      mbar_init(&sm.full[i], 1);
      mbar_init(&sm.done[i], kGroups);
    }
    mbar_init_fence();
    for (; next_load < kRing && blockIdx.x + (unsigned)next_load * gridDim.x < items; ++next_load) issue_load(next_load);
  }
  __syncthreads();
  // refill every slot whose series all groups have left (thread 0, between rows: never blocks)
  auto refill = [&](bool block) {
    while (blockIdx.x + (unsigned)next_load * gridDim.x < items) {
      const int slot = next_load % kRing;
      const uint32_t ph = (uint32_t)((next_load / kRing - 1) & 1);
      if (block) mbar_wait(&sm.done[slot], ph);
      else if (!mbar_test(&sm.done[slot], ph)) break;
      issue_load(next_load);
      ++next_load;
      block = false;
    }
  };
  WarpSmemP &ws = sm.w[warp];
  float *const yr = ws.trr, *const yi = ws.tri;
  float2 *const my_mr = reinterpret_cast<float2 *>(ws.trr), *const my_mi = reinterpret_cast<float2 *>(ws.tri);
  const float kf = (float)(D * lane + h);           // this lane's first bin
  const int tidx = 2 * (lane & 15) + (lane >> 4);
  const bool leader = (h == 0 && lane == 0);
  float2 R[16], I[16];

  for (int i = 0;; ++i) {
    const unsigned it = blockIdx.x + (unsigned)i * gridDim.x;
    if (it >= items) break;
    const int slot = i % kRing;
    const unsigned b = it / (unsigned)split;
    const int c = (int)(it - b * (unsigned)split);
    const int nrows = (S - c + split - 1) / split;
    if (threadIdx.x == 0 && next_load <= i) refill(true);     // only when the groups ran a whole ring apart
    mbar_wait(&sm.full[slot], (uint32_t)((i / kRing) & 1));
    const float4 *xs = &sm.xh[slot][h][0][lane];
    volatile int *const my_row = &sm.group_row[i & 1][group];
    if (leader) *my_row = atomicAdd(&sm.next_row[slot], 1);
    __syncwarp();
    group_sync<D>(group);
#pragma unroll 1
    for (;;) {
      const int r = *my_row;
      if (r >= nrows) break;
      const int s = c + split * r;
      const RowParam rp = sm.row[s];
      const int L = rp.L, two_pass = rp.multi;
      const float zl = fmaf(rp.a, kf, -f0);         // s*w_k - f0 at k = D lane + h
      if (two_pass) {
        // Y[D (lane + 32 k2) + h] = X^ * daughter for k2 < 2^L <= 16, two k2 per packed op
        const int M = 1 << (rp.L - 1);
        const float2 zl2 = make_float2(zl, fmaf(rp.a, 32.0f * D, zl));
        const float2 a64 = bc(rp.a * (64.0f * D));
        const float2 ln2 = bc(rp.lognorm);
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          if (M > below_pow2(m)) {
            const float2 z = fma2(a64, bc((float)m), zl2);
            const float2 e = fma2(mul2(z, z), bc(-0.72134752044f), ln2);
            const float2 d = make_float2(ex2(e.x), ex2(e.y));
            const float4 v = xs[32 * m];
            R[br4(m)] = mul2(make_float2(v.x, v.y), d);
            I[br4(m)] = mul2(make_float2(v.z, v.w), d);
          }
        }
      } else {
        const float d = ex2(fmaf(zl * zl, -0.72134752044f, rp.lognorm));
        const float4 v0 = xs[0];
        yr[lane] = v0.x * d;
        yi[lane] = v0.z * d;
        __syncwarp();
        // u[j] = Y[j] * w1024^(j * lane) for j < 2^L, two j per packed op; nested warp-uniform branches,
        // not per-element predicates (a narrow row must not issue the whole unrolled loop)
        auto pre = [&](const int m) {
          const float2 y_r = *reinterpret_cast<const float2 *>(&yr[2 * m]);
          const float2 y_i = *reinterpret_cast<const float2 *>(&yi[2 * m]);
          const float4 t = sm.tw_b[m][lane];
          const float2 twr = make_float2(t.x, t.y), twi = make_float2(t.z, t.w);
          R[br4(m)] = fma2(y_i, neg2(twi), mul2(y_r, twr));
          I[br4(m)] = fma2(y_r, twi, mul2(y_i, twr));
        };
        pre(0);
        if (L >= 2) {
          pre(1);
          if (L >= 3) {
            pre(2); pre(3);
            if (L >= 4) {
              pre(4); pre(5); pre(6); pre(7);
              if (L >= 5) {
#pragma unroll
                for (int m = 8; m < 16; ++m) pre(m);
              }
            }
          }
        }
        __syncwarp();
      }
      if (L == 1) {
        // two non-zero inputs: out[t] = in0 + w32^t in1, straight from the definition (no replication
        // of registers, no scalar last stage)
        fft32::dft32_two_inputs(R, I);
      } else {
        __builtin_assume(L >= 2 && L <= 5);        // RowParam::L of this kernel: no single-input path
        fft32::dit32(R, I, L);
      }
      if (two_pass) {
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          const float4 t = sm.tw_a[p][lane];
          const float2 twr = make_float2(t.x, t.y), twi = make_float2(t.z, t.w);
          const float2 vr = fma2(I[p], neg2(twi), mul2(R[p], twr));
          const float2 vi = fma2(R[p], twi, mul2(I[p], twr));
          *reinterpret_cast<float2 *>(&ws.trr[lane * kTrStride + 2 * p]) = vr;
          *reinterpret_cast<float2 *>(&ws.tri[lane * kTrStride + 2 * p]) = vi;
        }
        __syncwarp();
#pragma unroll
        for (int m = 0; m < 16; ++m) {
          R[br4(m)] = make_float2(ws.trr[(2 * m) * kTrStride + tidx], ws.trr[(2 * m + 1) * kTrStride + tidx]);
          I[br4(m)] = make_float2(ws.tri[(2 * m) * kTrStride + tidx], ws.tri[(2 * m + 1) * kTrStride + tidx]);
        }
        __syncwarp();
        fft32::dit32(R, I, 5);
      }
      // position p holds u = lane + 32 p (.x) and u + 512 (.y) of this warp's 1024-point transform.
      // The mailboxes live in the transpose buffers: every warp of the group must be past its step-B loads.
      group_sync<D>(group);
      const int tlo = COI ? sm.coi[s].x : 0, thi = COI ? sm.coi[s].y : kNF;
      float *const orow0 = power + ((int64_t)b * S + s) * (int64_t)n0 + lane;
      if constexpr (D == 2) {
        float2 *const wp_mr = reinterpret_cast<float2 *>(sm.w[warp ^ 1].trr), *const wp_mi = reinterpret_cast<float2 *>(sm.w[warp ^ 1].tri);
        if (h) {
#pragma unroll
          for (int p = 0; p < 8; ++p) {               // warp 0 finishes positions p < 8
            wp_mr[p * 32 + lane] = R[p];
            wp_mi[p * 32 + lane] = I[p];
          }
        } else {
#pragma unroll
          for (int p = 0; p < 8; ++p) {               // warp 1 finishes positions p >= 8
            wp_mr[p * 32 + lane] = R[p + 8];
            wp_mi[p * 32 + lane] = I[p + 8];
          }
        }
      } else {
        // warp g of the group finishes positions 4 g .. 4 g + 3: slot [source h][position] of its mailbox
        WarpSmemP *const gw = &sm.w[warp - h];
#pragma unroll
        for (int g = 0; g < D; ++g) {
          float2 *const mr = reinterpret_cast<float2 *>(gw[g].trr) + (h * 4) * 32 + lane;
          float2 *const mi = reinterpret_cast<float2 *>(gw[g].tri) + (h * 4) * 32 + lane;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            mr[q * 32] = R[4 * g + q];
            mi[q * 32] = I[4 * g + q];
          }
        }
      }
      if (leader) {
        *my_row = atomicAdd(&sm.next_row[slot], 1);
        if (threadIdx.x == 0) refill(false);
      }
      __syncwarp();
      group_sync<D>(group);
      if constexpr (D == 2) {
        const int t0 = lane + 256 * h;
        float *orow = orow0 + 256 * h;
        // e = even-bin transform, g = odd-bin transform, both at u = t0 + 32 p (.x) and u + 512 (.y), w = w2048^u as
        // (Re | Im) of the two halves (w2048^(u+512) = i w2048^u):  x[u] = e + w g,  x[u + 1024] = e - w g = 2 e - x[u].
        // The twiddle rides in the additions (the receiving side applies it: both warps do the same work), and each
        // position leaves as four whole lines.
        auto finish = [&](const int p, const float2 er, const float2 ei, const float2 gr, const float2 gi, const float4 w) {
          const float2 wa = make_float2(w.x, w.y), wb = make_float2(w.z, w.w);
          const float2 lr = fma2(gr, wa, fma2(gi, neg2(wb), er)), li = fma2(gi, wa, fma2(gr, wb, ei));
          float2 lo = fma2(lr, lr, mul2(li, li));      // |x[u]|^2, |x[u + 512]|^2
          const int ta = t0 + 32 * p;
          if (COI) {
            if (ta < tlo || ta > thi) lo.x = NAN;
            if (ta + 512 < tlo || ta + 512 > thi) lo.y = NAN;
          }
          __stcs(orow + 32 * p, lo.x);                 // n0 > 1024: the first half is always inside the row
          __stcs(orow + 32 * p + 512, lo.y);
          if (kN + 256 * h + 32 * p < n0) {            // warp-uniform: some lane still has a sample in the second half
            const float2 hr = fma2(er, bc(2.0f), neg2(lr)), hi = fma2(ei, bc(2.0f), neg2(li));
            float2 hp = fma2(hr, hr, mul2(hi, hi));    // |x[u + 1024]|^2, |x[u + 1536]|^2
            if (COI) {
              if (ta + 1024 < tlo || ta + 1024 > thi) hp.x = NAN;
              if (ta + 1536 < tlo || ta + 1536 > thi) hp.y = NAN;
            }
            if (ta + 1024 < n0) __stcs(orow + 32 * p + 1024, hp.x);
            if (ta + 1536 < n0) __stcs(orow + 32 * p + 1536, hp.y);
          }
        };
        if (h) {
#pragma unroll
          for (int p = 0; p < 8; ++p)
            finish(p, my_mr[p * 32 + lane], my_mi[p * 32 + lane], R[p + 8], I[p + 8], sm.tw_o[0][p + 8][lane]);
        } else {
#pragma unroll
          for (int p = 0; p < 8; ++p) finish(p, R[p], I[p], my_mr[p * 32 + lane], my_mi[p * 32 + lane], sm.tw_o[0][p][lane]);
        }
      } else {
        // radix-4 butterfly of the twiddled transforms t_r = w4096^(r u) G_r at u = lane + 32 (4 h + q) (.x), u + 512 (.y):
        //   a0 = t0 + t2, a1 = t0 - t2, a2 = t1 + t3, a3 = t1 - t3;  x_0 = a0 + a2, x_2 = a0 - a2, x_1 = a1 + i a3, x_3 = a1 - i a3,
        // x_q = x[u + 1024 q]; the twiddles of t2 and t3 ride in the additions.
        const int t0 = lane + 128 * h;
        float *orow = orow0 + 128 * h;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 g0r = my_mr[(0 * 4 + q) * 32 + lane], g0i = my_mi[(0 * 4 + q) * 32 + lane];
          const float2 g1r = my_mr[(1 * 4 + q) * 32 + lane], g1i = my_mi[(1 * 4 + q) * 32 + lane];
          const float2 g2r = my_mr[(2 * 4 + q) * 32 + lane], g2i = my_mi[(2 * 4 + q) * 32 + lane];
          const float2 g3r = my_mr[(3 * 4 + q) * 32 + lane], g3i = my_mi[(3 * 4 + q) * 32 + lane];
          const float4 w1 = sm.tw_o[0][4 * h + q][lane], w2 = sm.tw_o[1][4 * h + q][lane], w3 = sm.tw_o[2][4 * h + q][lane];
          const float2 c1 = make_float2(w1.x, w1.y), s1 = make_float2(w1.z, w1.w);
          const float2 c2 = make_float2(w2.x, w2.y), s2 = make_float2(w2.z, w2.w);
          const float2 c3 = make_float2(w3.x, w3.y), s3 = make_float2(w3.z, w3.w);
          const float2 a0r = fma2(g2r, c2, fma2(g2i, neg2(s2), g0r)), a0i = fma2(g2i, c2, fma2(g2r, s2, g0i));
          const float2 a1r = fma2(g0r, bc(2.0f), neg2(a0r)), a1i = fma2(g0i, bc(2.0f), neg2(a0i));
          const float2 t1r = fma2(g1i, neg2(s1), mul2(g1r, c1)), t1i = fma2(g1r, s1, mul2(g1i, c1));
          const float2 a2r = fma2(g3r, c3, fma2(g3i, neg2(s3), t1r)), a2i = fma2(g3i, c3, fma2(g3r, s3, t1i));
          const float2 a3r = fma2(t1r, bc(2.0f), neg2(a2r)), a3i = fma2(t1i, bc(2.0f), neg2(a2i));
          const int ta = t0 + 32 * q;
          float *o = orow + 32 * q;
          auto put = [&](const int qq, const float2 xr, const float2 xi) {
            float2 pw = fma2(xr, xr, mul2(xi, xi));    // |x[u + 1024 qq]|^2, |x[u + 512 + 1024 qq]|^2
            const int tq = ta + kN * qq;
            if (COI) {
              if (tq < tlo || tq > thi) pw.x = NAN;
              if (tq + 512 < tlo || tq + 512 > thi) pw.y = NAN;
            }
            if (qq < 2) {                              // n0 > 2048: the first half is always inside the row
              __stcs(o + kN * qq, pw.x);
              __stcs(o + kN * qq + 512, pw.y);
            } else {
              if (tq < n0) __stcs(o + kN * qq, pw.x);
              if (tq + 512 < n0) __stcs(o + kN * qq + 512, pw.y);
            }
          };
          put(0, add2(a0r, a2r), add2(a0i, a2i));
          put(1, fma2(a3i, bc(-1.0f), a1r), add2(a1i, a3r));
          if (2 * kN + 128 * h + 32 * q < n0)          // warp-uniform, as in the pair kernel
            put(2, fma2(a2r, bc(-1.0f), a0r), fma2(a2i, bc(-1.0f), a0i));
          if (3 * kN + 128 * h + 32 * q < n0)
            put(3, add2(a1r, a3i), fma2(a3r, bc(-1.0f), a1i));
        }
      }
    }
    if (leader) mbar_arrive(&sm.done[slot]);
  }
}

}  // namespace

// Forward FFT (N = 2048) for k_cwt_dif<2>: the positive half of the spectrum leaves in the group layout
// (CtaSmemP::xh) -- per series 8 KB at the start of its xhat row: float4 [parity h][m < 8][lane] =
// (Re X^[k0], Re X^[k1], Im X^[k0], Im X^[k1]), k0 = 2 (lane + 64 m) + h, k1 = k0 + 64.
__global__ void k_fwd_fft_pair2048(const float *__restrict__ x, int n0, FftPlan<float> plan, float2 *__restrict__ xhat) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *a = reinterpret_cast<float2 *>(smem_raw);
  float2 *b = a + plan.M;
  const int N = plan.n;
  const int64_t row = blockIdx.x;
  const float *xr = x + row * n0;
  for (int t = threadIdx.x; t < N; t += blockDim.x) a[t] = make_float2(t < n0 ? xr[t] : 0.0f, 0.0f);
  __syncthreads();
  const float2 *r = plan_fft<float, -1>(a, b, plan);
  float4 *o = reinterpret_cast<float4 *>(xhat + row * N);
  for (int i = threadIdx.x; i < 2 * 8 * 32; i += blockDim.x) {
    const int lane = i & 31, m = (i >> 5) & 7, h = i >> 8;
    const float2 v0 = r[2 * (lane + 64 * m) + h], v1 = r[2 * (lane + 64 * m) + h + 64];
    o[i] = make_float4(v0.x, v1.x, v0.y, v1.y);
  }
}

// The same layout for N = 4096 (four warps per row: k0 = 4 (lane + 64 m) + r, k1 = k0 + 128, r < 4; 16 KB), built from
// the natural-order spectrum of the radix-16 forward kernel into the unused negative-frequency half of the row.
__global__ void k_dif_layout4096(float2 *__restrict__ xhat) {
  const float2 *r = xhat + (int64_t)blockIdx.x * 4096;
  float4 *o = reinterpret_cast<float4 *>(xhat + (int64_t)blockIdx.x * 4096 + 2048);
  for (int i = threadIdx.x; i < 4 * 8 * 32; i += blockDim.x) {
    const int lane = i & 31, m = (i >> 5) & 7, h = i >> 8;
    const float2 v0 = r[4 * (lane + 64 * m) + h], v1 = r[4 * (lane + 64 * m) + h + 128];
    o[i] = make_float4(v0.x, v1.x, v0.y, v1.y);
  }
}

// Per-row sample interval inside the cone of influence, evaluated in double with the expression
// the generic kernel (cwt.cu) and pycwt use -- period(s) > coi(t) is masked -- so that the fused
// mask is bit-equal.  Rows with no valid sample get the empty interval [1, 0].
void coi_row_ranges(int n0, double dt, const Axes &ax, double f0, std::vector<ushort2> *out) {
  const int S = ax.J + 1;
  const double fl = morlet_flambda(f0);
  const double c = fl * (1.0 / std::sqrt(2.0)) * dt;
  out->resize(S);
  // monotone on either side of the centre (exact subtractions, one multiplication by c > 0):
  // binary searches give the interval a scan over t would
  auto valid = [&](double period, int t) { return !(period > c * (n0 / 2.0 - std::fabs(t - (n0 - 1) / 2.0))); };
  const int mid_lo = (n0 - 1) / 2, mid_hi = n0 / 2;
  for (int s = 0; s < S; ++s) {
    const double period = 1.0 / (1.0 / (fl * ax.scales[s]));
    if (!valid(period, mid_lo) && !valid(period, mid_hi)) {
      (*out)[s] = make_ushort2(1, 0);
      continue;
    }
    int a = 0, b = mid_lo;
    while (a < b) {
      const int m = (a + b) / 2;
      if (valid(period, m)) b = m; else a = m + 1;
    }
    const int lo = a;
    a = mid_hi; b = n0 - 1;
    while (a < b) {
      const int m = (a + b + 1) / 2;
      if (valid(period, m)) a = m; else b = m - 1;
    }
    (*out)[s] = make_ushort2((unsigned short)lo, (unsigned short)a);
  }
}

// RowParam of every scale row for an n-point transform whose one-sided spectrum a group of D warps splits by residue
// mod D (k_cwt_fast_1024: n = 1024, D = 1; k_cwt_dif<D>: n = 1024 D).  `extra` moves the band edge one bin further
// out: for nfft = 512 two series share the interleaved 1024-point spectrum, where a series' bin kk sits at
// k = 2 kk + parity, so a, lognorm and the band edge are those of a 1024-point transform with the edge one bin on.
static std::vector<RowParam> row_params(int n, int D, int extra, double dt, const Axes &ax, double f0) {
  std::vector<RowParam> rows(ax.J + 1);
  for (size_t s = 0; s < rows.size(); ++s) {
    const double a = ax.scales[s] / dt * 2.0 * kPi / n;
    int khi = (int)std::floor((f0 + kZCut) / a) + extra;
    khi = std::max(1, std::min(khi, n / 2 - 1));
    RowParam &r = rows[s];
    r.a = (float)a;
    r.lognorm = (float)std::log2(std::sqrt(2.0 * kPi * ax.scales[s] / dt) * 0.75112554446494248286 / n);
    // a warp transforms the bins of one residue mod D, j = k / D <= jhi < 512: K2 = 2^L >= ceil((jhi+1)/32), at most
    // 16 (one-sided), for a two-pass row; K1 = 2^L >= jhi+1, at least 2, for a single-pass one
    const int jhi = khi / D;
    r.multi = jhi >= 32;
    r.L = r.multi ? std::max(1, std::min(4, ilog2(jhi / 32 + 1))) : std::max(1, ilog2(jhi + 1));
  }
  return rows;
}

int cwt_fast_1024(const CwtPlan &pl, const float *d_x, int64_t batch, int n0, double dt, const Axes &ax, double f0,
                  int flags, float *d_power, cudaStream_t st) {
  const int S = ax.J + 1;
  const bool half = pl.rows == Rows::kFast512Pairs;   // two series per warp (HALF)
  const bool coi = flags & WTB_COI_MASK;
  // fewer series than warps on the machine: split each series' rows over up to 16 warps
  const int64_t items = half ? (batch + 1) / 2 : batch;
  const int64_t machine_warps = (int64_t)sm_count() * kWarps;
  const int split = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(16, S), machine_warps / items));
  const std::vector<RowParam> rows = row_params(kN, 1, half ? 1 : 0, dt, ax, f0);
  void *scratch = nullptr;
  WTB_TRY(arena_reserve(sizeof(RowParam) * S + sizeof(ushort2) * S, &scratch));
  RowParam *d_rows = (RowParam *)scratch;
  ushort2 *d_coi = nullptr;
  // rows.data() is pageable: the copy is staged before the call returns
  WTB_CUDA(cudaMemcpyAsync(d_rows, rows.data(), sizeof(RowParam) * S, cudaMemcpyHostToDevice, st));
  if (coi) {
    std::vector<ushort2> rng;
    coi_row_ranges(n0, dt, ax, f0, &rng);
    d_coi = (ushort2 *)(d_rows + S);
    WTB_CUDA(cudaMemcpyAsync(d_coi, rng.data(), sizeof(ushort2) * S, cudaMemcpyHostToDevice, st));
  }
  auto launch = [&](auto kern) -> int {
    WTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CtaSmem)));
    const int grid = (int)std::min<int64_t>(items * split, (int64_t)sm_count());
    kern<<<grid, kWarps * 32, sizeof(CtaSmem), st>>>(d_x, batch, n0, S, d_rows, d_coi, (float)f0, d_power, split);
    WTB_LAUNCH_CHECK();
    return WTB_OK;
  };
  if (half) return coi ? launch(k_cwt_fast_1024<true, true>) : launch(k_cwt_fast_1024<true, false>);
  return coi ? launch(k_cwt_fast_1024<false, true>) : launch(k_cwt_fast_1024<false, false>);
}

int cwt_dif(const CwtPlan &pl, const float *d_x, float2 *d_xhat, int64_t batch, int n0, double dt, const Axes &ax,
            double f0, int flags, float *d_power, cudaStream_t st) {
  const int S = ax.J + 1;
  const int nfft = pl.rows == Rows::kDif2048 ? 2 * kN : 4 * kN;
  const int D = nfft / kN;
  const float2 *d_layout = d_xhat;
  if (pl.fwd == Fwd::kPair2048) {
    FftPlan<float> plan;
    WTB_TRY(make_plan<float>(nfft, &plan));
    const size_t smem = 2 * sizeof(float2) * (size_t)plan.M;
    WTB_CUDA(cudaFuncSetAttribute(k_fwd_fft_pair2048, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_fwd_fft_pair2048<<<(unsigned)batch, 256, smem, st>>>(d_x, n0, plan, d_xhat);
    WTB_LAUNCH_CHECK();
  } else {
    WTB_TRY(fwd_fft_4096(d_x, batch, n0, d_xhat, st));
    k_dif_layout4096<<<(unsigned)batch, 256, 0, st>>>(d_xhat);
    WTB_LAUNCH_CHECK();
    d_layout = d_xhat + 2048;
  }
  const bool coi = flags & WTB_COI_MASK;
  const std::vector<RowParam> rows = row_params(nfft, D, 0, dt, ax, f0);
  // the caller's arena holds xhat: row parameters go to the per-thread parameter buffer
  void *prm = nullptr;
  WTB_TRY(params_reserve((sizeof(RowParam) + sizeof(ushort2)) * kMaxRowsF, &prm));
  RowParam *d_rows = (RowParam *)prm;
  ushort2 *d_coi = nullptr;
  // rows.data() is pageable: the copy is staged before the call returns
  WTB_CUDA(cudaMemcpyAsync(d_rows, rows.data(), sizeof(RowParam) * S, cudaMemcpyHostToDevice, st));
  if (coi) {
    std::vector<ushort2> rng;
    coi_row_ranges(n0, dt, ax, f0, &rng);
    d_coi = (ushort2 *)(d_rows + kMaxRowsF);
    WTB_CUDA(cudaMemcpyAsync(d_coi, rng.data(), sizeof(ushort2) * S, cudaMemcpyHostToDevice, st));
  }
  // Fewer series than SMs: the rows of a series are dealt to up to 16 CTAs.  A few series per SM: CTAs take whole
  // items, so the last wave is only as full as ceil() leaves it (500 series on 148 SMs: 3.4 -> 4 rounds, 84 %);
  // dealing each series' rows to 2 .. 4 items evens that out (the X^ reload per item is 8 / 16 KB).
  const int64_t sms = sm_count();
  int split = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(16, S), sms / batch));
  if (batch >= sms && batch < 16 * sms) {
    double best = 0.0;
    for (int c = 1; c <= std::min(4, S); ++c) {
      const double waves = (double)(batch * c) / (double)sms;
      const double eff = waves / std::ceil(waves) * (1.0 - 0.01 * (c - 1));
      if (eff > best + 1e-9) { best = eff; split = c; }
    }
  }
  const int grid = (int)std::min<int64_t>(batch * split, sms);
  WTB_REQUIRE(batch * split < (1LL << 31), WTB_EUNSUPPORTED, "batch too large for one launch");
  auto run = [&](auto kern, size_t smem) -> int {
    WTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kDifWarps * 32, smem, st>>>(d_layout, nfft, batch, n0, S, d_rows, d_coi, (float)f0, d_power, split);
    WTB_LAUNCH_CHECK();
    return WTB_OK;
  };
  if (D == 2) return coi ? run(k_cwt_dif<2, true>, sizeof(CtaSmemP<2>)) : run(k_cwt_dif<2, false>, sizeof(CtaSmemP<2>));
  return coi ? run(k_cwt_dif<4, true>, sizeof(CtaSmemP<4>)) : run(k_cwt_dif<4, false>, sizeof(CtaSmemP<4>));
}

}  // namespace wtb
