// FP32 fast path of the coherence pipeline for nfft = 4096 (BASELINE cfg5 and the Monte
// Carlo inside cfg3: surrogates of 3351 samples padded to 4096).
//
// One CTA of 256 threads owns one (pair, scale) row and carries the row's TWO fields
// (two independent 4096-point FFTs) through every pass together: twiddles and index
// arithmetic are shared, and the shared-memory exchanges move both fields with one
// 64-bit access per real / imaginary pair.  A 4096-point transform is three radix-16 passes; every thread keeps
// its 2 x 16 points in registers (fft16_gen.cuh: Linzer-Feig FMA butterflies, literal
// twiddles); passes exchange data through two padded planes of float2 (real pairs, imaginary
// pairs; Stockham index maps, in place).  Forward transforms run the same inverse code on conjugated data, so
// one pass body (one copy of the code, instruction-cache resident) serves every round.
//
// The rounds of a row are chained through REGISTERS: pass 3 leaves thread j with
// elements j + 256 r', which are exactly the inputs of pass 1 of the next round.
//   kernel A  round 1  W1, W2 = IFFT(X^ * daughter_s)        (bins >= 2048 skipped, pass 1 pruned)
//             pointwise P = (|W1|^2 + i |W2|^2)/s, C = W1 conj(W2)/s, zero for t >= n0
//             round 2  P^, C^ = FFT(.)
//             store    G_s[k] = exp(-0.5 (s/dt)^2 k^2)/N * (P^, C^)[k]  for bins with filter > 1e-7
//   kernel B  load     sum_m w_m G_{i+m}[k]      scale boxcar of Morlet.smooth applied to spectra
//             round 3  S1 + i S2, S12 = IFFT(.)
//             |S12|^2 / (S1 S2) -> plane, or -> shared-memory histogram -> global
// The boxcar is a linear combination of rows, so it commutes with the inverse transform;
// applying it to the filtered spectra removes the time-domain plane round trip and the
// separate scale-smoothing pass of the generic path.
#include "cwt_paths.cuh"
#include "fft16_gen.cuh"

namespace wtb {

namespace {

using fft16::br4;

constexpr int kN = 4096;
constexpr int kThreads = 256;
constexpr int kBuf = kN + kN / 16;     // padded: index i lives at pad(i) = i + (i >> 4)

struct WRow {
  float a;        // (s/dt) * 2*pi/N : s*w_k = a*k
  float lognorm;  // log2( sqrt(2*pi*s/dt) * pi^-1/4 / N )
  float gcoef;    // -0.5 * log2(e) * a^2 : Gaussian exponent per squared bin index
  float inv_s;    // 1 / scale
  int R1;         // number of 256-bin blocks with daughter support (power of two, 1..8)
  int L1;         // log2(R1)
  float kc2;      // squared bin index beyond which the Gaussian filter is < 1e-7
  int kc;         // floor(sqrt(kc2))
};
static_assert(sizeof(WRow) == 32, "wct_device reserves 32 bytes of row parameters per scale");

struct CohWin {
  int K, up;
  float w[kMaxWin];
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

using fft32::bc;
using fft32::fma2;
using fft32::mul2;

// Registers: R[p] = (re of field 0, re of field 1), I[p] = (im of field 0, im of field 1):
// both fields of the row ride in the two lanes of every FFMA2 / FADD2 / FMUL2.
//
// Inverse 4096-point transforms of both fields.  On entry R/I[br4(r)] hold input
// j + 256 r (first 2^L of them non-zero); on exit R/I[r'] hold output j + 256 r'.
// Contains 4 CTA barriers and ends with the buffer free.
__device__ __forceinline__ void fft4096_inv2(float2 (&R)[16], float2 (&I)[16], int L, float2 *Bre, float2 *Bim,
                                             const float2 *__restrict__ tw2s,
                                             const float2 *__restrict__ tw3, int j) {
  // The real and the imaginary pairs travel through two planes of 8-byte elements: a register
  // pair goes out and comes back with one 64-bit access each, so no MOVs assemble 128-bit
  // vectors, and every index below is `base + immediate` (pad(i) = i + (i >> 4) is spelled out
  // per access pattern because the compiler cannot see that the shifts never carry).
  const int k2 = j & 15;
  fft16::dit16p_inv(R, I, L);
  // exchange 1: pass-1 output index 16 j + r'  ->  pad = 17 j + r'
  {
    float2 *wre = Bre + 17 * j, *wim = Bim + 17 * j;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      wre[r] = R[r];
      wim[r] = I[r];
    }
  }
  __syncthreads();
  // reads of index j + 256 r  ->  pad = j + (j >> 4) + 272 r
  const float2 *rre = Bre + j + (j >> 4), *rim = Bim + j + (j >> 4);
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const float2 qr = rre[272 * r], qi = rim[272 * r];
    const float2 w = tw2s[r * 16 + k2];
    R[br4(r)] = fma2(qi, bc(-w.y), mul2(qr, bc(w.x)));
    I[br4(r)] = fma2(qr, bc(w.y), mul2(qi, bc(w.x)));
  }
  __syncthreads();
  fft16::dit16p_inv(R, I, 4);
  // exchange 2: pass-2 output index (j - k2) * 16 + k2 + 16 r'  ->  pad = 17 (j - k2) + k2 + 17 r'
  {
    const int base = 17 * (j - k2) + k2;
    float2 *wre = Bre + base, *wim = Bim + base;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      wre[17 * r] = R[r];
      wim[17 * r] = I[r];
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const float2 qr = rre[272 * r], qi = rim[272 * r];
    const float2 w = __ldg(&tw3[r * 256 + j]);
    R[br4(r)] = fma2(qi, bc(-w.y), mul2(qr, bc(w.x)));
    I[br4(r)] = fma2(qr, bc(w.y), mul2(qi, bc(w.x)));
  }
  __syncthreads();   // buffer free again once every thread has loaded
  fft16::dit16p_inv(R, I, 4);
}

// Kernel A: rounds 1 and 2 of one (pair, scale) row, filtered spectra out.
// spec: [rows = pairs*S][4096] float4 = (P^.re, C^.re, P^.im, C^.im) * filter.
__global__ void __launch_bounds__(kThreads, 3)
k_wct_spec_4096(const float2 *__restrict__ xhat, int n0, int S, int S_run, const WRow *__restrict__ rows,
                const float2 *__restrict__ tw2, const float2 *__restrict__ tw3, float f0,
                float4 *__restrict__ spec, float *__restrict__ phase, float2 *__restrict__ w12,
                int smooth) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *Bre = reinterpret_cast<float2 *>(smem_raw);                // [kBuf] real pairs
  float2 *Bim = Bre + kBuf;                                          // [kBuf] imaginary pairs
  float2 *tw2s = Bim + kBuf;                                         // [256]
  const int j = threadIdx.x;
  tw2s[j] = tw2[j];
  // rows 0 .. S_run-1 of every pair (the larger scales go to k_wct_spec_direct)
  const int64_t pair = blockIdx.x / S_run;
  const int s = (int)(blockIdx.x % S_run);
  const int64_t row = pair * S + s;
  const WRow rp = rows[s];
  const float2 *x1 = xhat + (pair * 2) * (int64_t)kN;
  const float2 *x2 = x1 + kN;
  float2 R[16], I[16];

  // round 1, pass 1 inputs: Y[j + 256 r] for r < R1 (bins beyond the daughter's support are zero)
  {
    const float zl = fmaf(rp.a, (float)j, -f0);
    const float a256 = rp.a * 256.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      if (r < rp.R1) {
        const float z = fmaf(a256, (float)r, zl);
        const float2 dgt = bc(ex2(fmaf(z * z, -0.72134752044f, rp.lognorm)));
        const float2 p = __ldg(&x1[j + 256 * r]), q = __ldg(&x2[j + 256 * r]);
        R[br4(r)] = mul2(make_float2(p.x, q.x), dgt);
        I[br4(r)] = mul2(make_float2(p.y, q.y), dgt);
      }
    }
  }
  __syncthreads();   // tw2s visible
  // round 1: W1, W2 (pruned first pass); its own call site, so round 2 below is straight-line
  // code with a compile-time full first pass and no loop-carried copies of the 64 data registers
  fft4096_inv2(R, I, rp.L1, Bre, Bim, tw2s, tw3, j);
  {
    // pointwise step: lane 0 becomes P = (|W1|^2 + i |W2|^2)/s, lane 1 becomes
    // C = W1 conj(W2)/s.  Both are CONJUGATED so that round 2 (a forward transform) can
    // reuse the inverse code: FFT(x) = conj(IFFT(conj(x))).
    const int64_t obase = row * (int64_t)n0;
    float2 nR[16], nI[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int t = j + 256 * r;
      float2 pr = make_float2(0.0f, 0.0f), pi = pr;
      if (t < n0) {
        const float2 m2 = fma2(R[r], R[r], mul2(I[r], I[r]));          // (|W1|^2, |W2|^2)
        const float xr = fmaf(R[r].x, R[r].y, I[r].x * I[r].y);        // W1 conj(W2)
        const float xi = fmaf(I[r].x, R[r].y, -R[r].x * I[r].y);
        if (w12) w12[obase + t] = make_float2(xr, xi);
        if (phase) phase[obase + t] = atan2f(xi, xr);
        pr = mul2(make_float2(m2.x, xr), bc(rp.inv_s));
        pi = mul2(make_float2(m2.y, xi), bc(-rp.inv_s));
      }
      nR[br4(r)] = pr;
      nI[br4(r)] = pi;
    }
    if (!smooth) return;
#pragma unroll
    for (int r = 0; r < 16; ++r) { R[r] = nR[r]; I[r] = nI[r]; }
  }
  fft4096_inv2(R, I, 4, Bre, Bim, tw2s, tw3, j);   // round 2
  // (R, I) = conj(FFT(field)); Gaussian filter in the Fourier domain with the 1/N of the
  // inverse.  Bins where the filter is negligible are neither stored nor ever read.
  float4 *srow = spec + row * (int64_t)kN;
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int bin = j + 256 * r;
    const float kk = (float)(bin < kN / 2 ? bin : bin - kN);
    const float k2v = kk * kk;
    if (k2v <= rp.kc2) {
      const float g = ex2(fmaf(rp.gcoef, k2v, -12.0f));
      const float2 sr = mul2(R[r], bc(g)), si = mul2(I[r], bc(-g));
      srow[bin] = make_float4(sr.x, sr.y, si.x, si.y);
    }
  }
}

// Kernel A for the LARGE scales: the same filtered spectra without a single transform.
// A large-scale daughter keeps only B = O(10.6 / a) bins of X^ (a = s/dt * 2 pi / N), so
//   W(t) = sum_l W^[l] e^{+2 pi i l t / N}           with W^ = X^ * daughter on B bins,
//   |W1(t)|^2 = sum_m A1[m] e^{2 pi i m t / N},      A1[m]  = sum_l W1^[l+m] conj(W1^[l])   (|m| < B),
//   W1 conj(W2)(t) = sum_m A12[m] e^{2 pi i m t / N}, A12[m] = sum_l W1^[l+m] conj(W2^[l]),
// and the transform of such a field cut off at t < n0 (pycwt truncates before it smooths) is
//   FFT(f rect)[k] = sum_m A[m] Dn[k - m],            Dn[d] = sum_{t < n0} e^{-2 pi i d t / N}
// -- needed only for the |k| <= kc bins the row's Gaussian keeps.  That is 2 B^2 + 6 B (2 kc + 1)
// complex multiply-adds per row (kc ~ 0.54 B) against four 4096-point transforms: a few per cent
// of the work for the largest scales, break-even near B = 90.  Output: exactly the spectra
// k_wct_spec_4096 stores (same layout, same bins), so kernels C and B do not change.
constexpr int kDirB = 128;                   // widest band (bins) a row may have to come here
constexpr int kDirKc = 72;                   // largest kc of such a row (kc = 5.68 / a ~ 0.54 B)
constexpr int kDirDn = kDirB + kDirKc + 2;   // Dn is tabulated for |d| <= kDirDn
constexpr int kDirThreads = 128;
constexpr int kDirKp = (kDirKc + 2) / 2;     // pairs (k, k + 1), k >= 0
constexpr int kDirG = 8;                     // the sum over m is split over up to this many thread groups

struct DRow {
  int l0;    // first bin of the daughter's support
  int B;     // number of bins
};

// Work per row: correlations 2 B^2 and the Dirichlet convolution 4.3 B^2 complex multiply-adds.
// Both loops are arranged so that one thread owns several outputs that share their operands:
//   step 2  thread m >= 0 forms A1[m], A2[m], A12[m] and A12[-m] from the same four loads
//           (two of them warp-wide broadcasts): 4 loads per 4 multiply-adds;
//   step 3  thread (k pair, m chunk) forms P1^, P2^, C^ at k, k + 1 and C^ at -k, -k - 1 (the real
//           fields are Hermitian: P^[-k] = conj P^[k]) with two sliding windows over Dn: 5 loads
//           (3 broadcasts) per 8 multiply-adds; the chunks' partial sums meet in shared memory
//           and are added in a fixed order.
__global__ void __launch_bounds__(kDirThreads)
k_wct_spec_direct(const float2 *__restrict__ xhat, int S, int s_first, const WRow *__restrict__ rows,
                  const DRow *__restrict__ drows, const float2 *__restrict__ dn, float f0,
                  float4 *__restrict__ spec) {
  __shared__ float2 u1[2 * kDirB], u2[2 * kDirB];             // W^[l] of the two series, zero for l >= B
  __shared__ float2 a1[2 * kDirB], a2[2 * kDirB], a12[2 * kDirB];   // A[m] at index m + B - 1, |m| < B
  __shared__ float2 sdn[2 * kDirDn + 1];                      // sdn[d + dm], |d| <= dm = B + kc + 1
  __shared__ float2 part[kDirG][8][kDirKp];                   // partial sums of step 3
  const int tid = threadIdx.x;
  const int nrun = S - s_first;
  const int64_t pair = blockIdx.x / nrun;
  const int s = s_first + (int)(blockIdx.x % nrun);
  const WRow rp = rows[s];
  const int l0 = drows[s].l0, B = drows[s].B, kc = rp.kc;
  const int dm = B + kc + 1;
  const float2 *x1 = xhat + (pair * 2) * (int64_t)kN + l0;
  const float2 *x2 = x1 + kN;
  for (int l = tid; l < 2 * B; l += kDirThreads) {
    float2 p = make_float2(0.0f, 0.0f), q = p;
    if (l < B) {
      const float z = fmaf(rp.a, (float)(l0 + l), -f0);
      const float dgt = ex2(fmaf(z * z, -0.72134752044f, rp.lognorm));
      p = __ldg(&x1[l]);
      q = __ldg(&x2[l]);
      p = make_float2(p.x * dgt, p.y * dgt);
      q = make_float2(q.x * dgt, q.y * dgt);
    }
    u1[l] = p;
    u2[l] = q;
  }
  for (int d = tid; d <= 2 * dm; d += kDirThreads) sdn[d] = __ldg(&dn[d - dm + kDirDn]);
  __syncthreads();
  // ---- step 2: correlations of the band-limited spectra
  for (int m = tid; m < B; m += kDirThreads) {
    float a1r = 0.0f, a1i = 0.0f, a2r = 0.0f, a2i = 0.0f, pr = 0.0f, pi = 0.0f, nr = 0.0f, ni = 0.0f;
    for (int l = 0; l < B - m; ++l) {
      const float2 xa = u1[l + m], xb = u2[l + m];             // per lane
      const float2 ya = u1[l], yb = u2[l];                     // broadcast
      a1r = fmaf(xa.x, ya.x, fmaf(xa.y, ya.y, a1r));           // xa conj(ya)
      a1i = fmaf(xa.y, ya.x, fmaf(-xa.x, ya.y, a1i));
      a2r = fmaf(xb.x, yb.x, fmaf(xb.y, yb.y, a2r));           // xb conj(yb)
      a2i = fmaf(xb.y, yb.x, fmaf(-xb.x, yb.y, a2i));
      pr = fmaf(xa.x, yb.x, fmaf(xa.y, yb.y, pr));             // A12[m]  += u1[l + m] conj(u2[l])
      pi = fmaf(xa.y, yb.x, fmaf(-xa.x, yb.y, pi));
      nr = fmaf(ya.x, xb.x, fmaf(ya.y, xb.y, nr));             // A12[-m] += u1[l] conj(u2[l + m])
      ni = fmaf(ya.y, xb.x, fmaf(-ya.x, xb.y, ni));
    }
    a1[B - 1 + m] = make_float2(a1r, a1i);
    a1[B - 1 - m] = make_float2(a1r, -a1i);                    // real field: A[-m] = conj A[m]
    a2[B - 1 + m] = make_float2(a2r, a2i);
    a2[B - 1 - m] = make_float2(a2r, -a2i);
    a12[B - 1 + m] = make_float2(pr, pi);
    if (m) a12[B - 1 - m] = make_float2(nr, ni);
  }
  __syncthreads();
  // ---- step 3: the cut-off at t < n0 = convolution with the Dirichlet kernel, bins |k| <= kc only
  const int KP = (kc + 2) / 2;                                 // k pairs (0,1), (2,3), ... covering 0 .. kc
  const int M = 2 * B - 1;                                     // terms m = -(B-1) .. B-1
  int G = kDirThreads / KP;
  G = G < 1 ? 1 : (G > kDirG ? kDirG : G);
  const int chunk = (M + G - 1) / G;
  for (int item = tid; item < G * KP; item += kDirThreads) {
    const int g = item / KP, kp = item - g * KP;
    const int k0 = 2 * kp;
    const int mi0 = g * chunk, mi1 = min(M, mi0 + chunk);      // m index range (m = mi - (B - 1))
    float acc[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) acc[q] = 0.0f;
    // windows: dA0 = Dn[k0 - m], dA1 = Dn[k0 + 1 - m]; dB0 = Dn[-k0 - m], dB1 = Dn[-k0 - 1 - m]
    const int m_first = mi0 - (B - 1);
    const float2 *pa = sdn + dm + k0 - m_first;                // pa[-(mi - mi0)] = Dn[k0 - m]
    const float2 *pb = sdn + dm - k0 - m_first;                // pb[-(mi - mi0)] = Dn[-k0 - m]
    float2 dA1 = pa[1], dB0 = pb[0];
    for (int mi = mi0; mi < mi1; ++mi) {
      const int o = mi - mi0;
      const float2 dA0 = pa[-o], dB1 = pb[-o - 1];
      const float2 x1m = a1[mi], x2m = a2[mi], xc = a12[mi];   // broadcasts (a warp shares its chunk)
      // P1 at k0, k0 + 1
      acc[0] = fmaf(x1m.x, dA0.x, fmaf(-x1m.y, dA0.y, acc[0]));  acc[1] = fmaf(x1m.x, dA0.y, fmaf(x1m.y, dA0.x, acc[1]));
      acc[2] = fmaf(x1m.x, dA1.x, fmaf(-x1m.y, dA1.y, acc[2]));  acc[3] = fmaf(x1m.x, dA1.y, fmaf(x1m.y, dA1.x, acc[3]));
      // P2 at k0, k0 + 1
      acc[4] = fmaf(x2m.x, dA0.x, fmaf(-x2m.y, dA0.y, acc[4]));  acc[5] = fmaf(x2m.x, dA0.y, fmaf(x2m.y, dA0.x, acc[5]));
      acc[6] = fmaf(x2m.x, dA1.x, fmaf(-x2m.y, dA1.y, acc[6]));  acc[7] = fmaf(x2m.x, dA1.y, fmaf(x2m.y, dA1.x, acc[7]));
      // C at k0, k0 + 1, -k0, -k0 - 1
      acc[8] = fmaf(xc.x, dA0.x, fmaf(-xc.y, dA0.y, acc[8]));    acc[9] = fmaf(xc.x, dA0.y, fmaf(xc.y, dA0.x, acc[9]));
      acc[10] = fmaf(xc.x, dA1.x, fmaf(-xc.y, dA1.y, acc[10]));  acc[11] = fmaf(xc.x, dA1.y, fmaf(xc.y, dA1.x, acc[11]));
      acc[12] = fmaf(xc.x, dB0.x, fmaf(-xc.y, dB0.y, acc[12]));  acc[13] = fmaf(xc.x, dB0.y, fmaf(xc.y, dB0.x, acc[13]));
      acc[14] = fmaf(xc.x, dB1.x, fmaf(-xc.y, dB1.y, acc[14]));  acc[15] = fmaf(xc.x, dB1.y, fmaf(xc.y, dB1.x, acc[15]));
      dA1 = dA0;      // Dn[k0 + 1 - (m + 1)] = Dn[k0 - m]
      dB0 = dB1;      // Dn[-k0 - (m + 1)]    = Dn[-k0 - 1 - m]
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) part[g][q][kp] = make_float2(acc[2 * q], acc[2 * q + 1]);
  }
  __syncthreads();
  float4 *srow = spec + (pair * S + s) * (int64_t)kN;
  // bins 0 .. kc and -1 .. -kc: P = |W1|^2 + i |W2|^2 travels as one complex field; 1/s and the 1/N of
  // the inverse ride in g
  for (int kk = tid; kk <= 2 * kc; kk += kDirThreads) {
    const int k = kk <= kc ? kk : kc - kk;                     // 0 .. kc, then -1 .. -kc
    const int ka = k < 0 ? -k : k, kp = ka >> 1, odd = ka & 1;
    float2 p1 = make_float2(0.0f, 0.0f), p2 = p1, c = p1;
    for (int g = 0; g < G; ++g) {                              // fixed order: reproducible sums
      const float2 v1 = part[g][odd][kp], v2 = part[g][2 + odd][kp], vc = part[g][(k < 0 ? 6 : 4) + odd][kp];
      p1.x += v1.x; p1.y += v1.y; p2.x += v2.x; p2.y += v2.y; c.x += vc.x; c.y += vc.y;
    }
    if (k < 0) { p1.y = -p1.y; p2.y = -p2.y; }                 // Hermitian: P1^[-k] = conj P1^[k]
    const float g = ex2(fmaf(rp.gcoef, (float)(k * k), -12.0f)) * rp.inv_s;
    srow[k >= 0 ? k : kN + k] = make_float4((p1.x - p2.y) * g, c.x * g, (p1.y + p2.x) * g, c.y * g);
  }
}

// Forward transforms for this pipeline: two real series of a pair (or two neighbouring series of a
// batch) in the two FFMA2 lanes, through the same three radix-16 passes: for real y the inverse
// code gives sum_t y[t] e^{+2 pi i k t / N} = conj(X^[k]).  y: [nseries, n0], xhat: [nseries, 4096].
// (The generic shared-memory Stockham kernel spent 3.5 % of a Monte-Carlo step on these 2 of the
// 398 transforms of a realisation.)
__global__ void __launch_bounds__(kThreads, 3)
k_fwd_fft_4096(const float *__restrict__ y, int64_t nseries, int n0, const float2 *__restrict__ tw2,
               const float2 *__restrict__ tw3, float2 *__restrict__ xhat) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *Bre = reinterpret_cast<float2 *>(smem_raw);
  float2 *Bim = Bre + kBuf;
  float2 *tw2s = Bim + kBuf;
  const int j = threadIdx.x;
  tw2s[j] = tw2[j];
  const int64_t b0 = 2 * (int64_t)blockIdx.x;
  const bool second = b0 + 1 < nseries;
  const float *y1 = y + b0 * n0, *y2 = second ? y1 + n0 : y1;
  float2 R[16], I[16];
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int t = j + 256 * r;
    R[br4(r)] = t < n0 ? make_float2(__ldg(y1 + t), __ldg(y2 + t)) : make_float2(0.0f, 0.0f);
    I[br4(r)] = make_float2(0.0f, 0.0f);
  }
  __syncthreads();   // tw2s visible
  fft4096_inv2(R, I, 4, Bre, Bim, tw2s, tw3, j);
  float2 *o1 = xhat + b0 * kN + j, *o2 = o1 + kN;
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    o1[256 * r] = make_float2(R[r].x, -I[r].x);
    if (second) o2[256 * r] = make_float2(R[r].y, -I[r].y);
  }
}

// Plain CWT rows for nfft = 4096 (series of 2049..4096 samples): round 1 of kernel A on its own,
// with the two FFMA2 lanes carrying TWO SERIES instead of the two members of a pair.
// xhat: [batch, 4096]; outputs (either may be null): power / coef [batch, S, n0].
// coi (may be null): per-row sample interval inside the cone of influence; power outside it is NaN.
__global__ void __launch_bounds__(kThreads, 3)
k_cwt_rows_4096(const float2 *__restrict__ xhat, int64_t batch, int n0, int S, const WRow *__restrict__ rows,
                const float2 *__restrict__ tw2, const float2 *__restrict__ tw3, float f0,
                float *__restrict__ power, float2 *__restrict__ coef, const ushort2 *__restrict__ coi) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *Bre = reinterpret_cast<float2 *>(smem_raw);
  float2 *Bim = Bre + kBuf;
  float2 *tw2s = Bim + kBuf;
  const int j = threadIdx.x;
  tw2s[j] = tw2[j];
  const int64_t row = blockIdx.x;
  const int64_t b0 = 2 * (row / S);
  const int s = (int)(row % S);
  const bool second = b0 + 1 < batch;       // an odd batch ends with a half-empty CTA
  const WRow rp = rows[s];
  const float2 *x1 = xhat + b0 * (int64_t)kN;
  const float2 *x2 = second ? x1 + kN : x1;
  float2 R[16], I[16];
  {
    const float zl = fmaf(rp.a, (float)j, -f0);
    const float a256 = rp.a * 256.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      if (r < rp.R1) {
        const float z = fmaf(a256, (float)r, zl);
        const float2 dgt = bc(ex2(fmaf(z * z, -0.72134752044f, rp.lognorm)));
        const float2 p = __ldg(&x1[j + 256 * r]), q = __ldg(&x2[j + 256 * r]);
        R[br4(r)] = mul2(make_float2(p.x, q.x), dgt);
        I[br4(r)] = mul2(make_float2(p.y, q.y), dgt);
      }
    }
  }
  __syncthreads();   // tw2s visible
  fft4096_inv2(R, I, rp.L1, Bre, Bim, tw2s, tw3, j);
  const int64_t o1 = (b0 * S + s) * (int64_t)n0, o2 = o1 + (int64_t)S * n0;
  const int tlo = coi ? coi[s].x : 0, thi = coi ? coi[s].y : kN;
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int t = j + 256 * r;
    if (t < n0) {
      if (coef) {
        coef[o1 + t] = make_float2(R[r].x, I[r].x);
        if (second) coef[o2 + t] = make_float2(R[r].y, I[r].y);
      }
      if (power) {
        float2 pw = fma2(R[r], R[r], mul2(I[r], I[r]));
        if (t < tlo || t > thi) pw = make_float2(NAN, NAN);
        __stcs(power + o1 + t, pw.x);
        if (second) __stcs(power + o2 + t, pw.y);
      }
    }
  }
}

// Kernel C: scale-axis boxcar of Morlet.smooth applied to the filtered spectra, in place.
// One thread owns one frequency bin of one pair and slides over the scales with a ring of
// the last K input rows in shared memory (column-private, so in-place is safe): every
// spectrum is read once and every smoothed spectrum written once.
// H_i[bin] = sum_k w[k] * G_{i+up-k}[bin]; rows outside [0, S) and bins outside a row's
// pass band count as zero.  Row i is written for bins inside the widest band of its window.
__global__ void __launch_bounds__(kThreads)
k_wct_boxcar_4096(float4 *__restrict__ spec, int S, const WRow *__restrict__ rows, CohWin win) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *ring = reinterpret_cast<float4 *>(smem_raw);     // [K][kThreads]
  __shared__ int s_kc[kMaxRowsC];
  const int tid = threadIdx.x;
  for (int q = tid; q < S; q += kThreads) s_kc[q] = rows[q].kc;
  __syncthreads();
  const int64_t pair = blockIdx.x >> 4;
  const int bin = ((blockIdx.x & 15) << 8) + tid;
  const int akk = bin < kN / 2 ? bin : kN - bin;
  if (akk > s_kc[0]) return;                               // outside every row's pass band
  // pass bands shrink with scale: rows 0 .. s_max hold this bin
  int s_max = 0;
  while (s_max + 1 < S && akk <= s_kc[s_max + 1]) ++s_max;
  float4 *col = spec + pair * (int64_t)S * kN + bin;
  const int K = win.K, up = win.up;
  const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (int k = 0; k < K; ++k) ring[k * kThreads + tid] = zero;
  // outputs i <= s_max + (K-1) - up are the only ones whose window still holds this bin
  const int s_end = min(S + up, s_max + K);
  int slot = 0;                                             // ring slot of input row s_in
  for (int s0 = 0; s0 < s_end; s0 += 4) {
    float4 v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)                             // four independent loads in flight
      v[q] = (s0 + q <= s_max) ? col[(int64_t)(s0 + q) * kN] : zero;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int s_in = s0 + q;
      if (s_in < s_end) {
        ring[slot * kThreads + tid] = v[q];
        const int i = s_in - up;                            // output row completed by this input
        if (i >= 0 && i < S) {
          const int first = i + up - (K - 1);               // smallest-scale row of the window
          if (akk <= s_kc[first < 0 ? 0 : first]) {
            float4 acc = zero;
            int sl = slot;                                  // k = 0 <-> row i + up = s_in
            for (int k = 0; k < K; ++k) {
              const float4 g = ring[sl * kThreads + tid];
              const float w = win.w[k];
              acc.x = fmaf(w, g.x, acc.x); acc.y = fmaf(w, g.y, acc.y);
              acc.z = fmaf(w, g.z, acc.z); acc.w = fmaf(w, g.w, acc.w);
              sl = sl == 0 ? K - 1 : sl - 1;
            }
            col[(int64_t)i * kN] = acc;
          }
        }
        slot = slot + 1 == K ? 0 : slot + 1;
      }
    }
  }
}

// The same boxcar for a compile-time tap count: K input rows per trip of the outer loop, so the
// ring slot of every row is a compile-time index and the ring lives in REGISTERS (K float4):
// no shared-memory traffic at all, taps in registers too.  Same sums in the same order as the
// generic kernel above (bit-identical output).
template <int K, int H>
__global__ void __launch_bounds__(kThreads)
k_wct_boxcar_4096_t(float4 *__restrict__ spec, int S, const WRow *__restrict__ rows, CohWin win) {
  static_assert(K % H == 0, "loads are issued in K / H batches");
  __shared__ int s_kc[kMaxRowsC];
  const int tid = threadIdx.x;
  for (int q = tid; q < S; q += kThreads) s_kc[q] = rows[q].kc;
  __syncthreads();
  const int64_t pair = blockIdx.x >> 4;
  const int bin = ((blockIdx.x & 15) << 8) + tid;
  const int akk = bin < kN / 2 ? bin : kN - bin;
  if (akk > s_kc[0]) return;
  int s_max = 0;
  while (s_max + 1 < S && akk <= s_kc[s_max + 1]) ++s_max;
  float4 *col = spec + pair * (int64_t)S * kN + bin;
  constexpr int up = (K - 1) / 2;
  const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  float wk[K];
  float4 ring[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    wk[k] = win.w[k];
    ring[k] = zero;
  }
  const int s_end = min(S + up, s_max + K);
  for (int base = 0; base < s_end; base += K) {
#pragma unroll
    for (int half = 0; half < K; half += H) {
      float4 v[H];
#pragma unroll
      for (int q = 0; q < H; ++q)                            // H independent loads in flight
        v[q] = (base + half + q <= s_max) ? col[(int64_t)(base + half + q) * kN] : zero;
#pragma unroll
      for (int q = 0; q < H; ++q) {
        const int slot = half + q;                           // compile-time after unrolling
        const int s_in = base + slot;
        if (s_in < s_end) {
          ring[slot] = v[q];
          const int i = s_in - up;                           // output row completed by this input
          if (i >= 0 && i < S) {
            const int first = i + up - (K - 1);
            if (akk <= s_kc[first < 0 ? 0 : first]) {
              float2 lo = make_float2(0.0f, 0.0f), hi = lo;  // two FFMA2 per tap, same sums in the same order
#pragma unroll
              for (int k = 0; k < K; ++k) {                  // k = 0 <-> row s_in, then older rows
                const float4 g = ring[(slot - k + K) % K];
                lo = fma2(bc(wk[k]), make_float2(g.x, g.y), lo);
                hi = fma2(bc(wk[k]), make_float2(g.z, g.w), hi);
              }
              col[(int64_t)i * kN] = make_float4(lo.x, lo.y, hi.x, hi.y);
            }
          }
        }
      }
    }
  }
}

// Kernel B: one CTA = one (pair, scale i): boxcar over the neighbouring rows' filtered
// spectra, inverse transform, coherence -> plane (MODE 0) or per-scale histogram (MODE 1).
template <int MODE>
__global__ void __launch_bounds__(kThreads, 3)
k_wct_coh_4096(const float4 *__restrict__ spec, int n0, int S, const WRow *__restrict__ rows,
               const float2 *__restrict__ tw2, const float2 *__restrict__ tw3, CohWin win,
               float *__restrict__ wct, unsigned long long *__restrict__ hist,
               const int *__restrict__ tlo, const int *__restrict__ thi, int maxscale) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *Bre = reinterpret_cast<float2 *>(smem_raw);
  float2 *Bim = Bre + kBuf;
  float2 *tw2s = Bim + kBuf;
  unsigned int *shist = reinterpret_cast<unsigned int *>(tw2s + 256);   // MODE 1: 1000 bins
  const int j = threadIdx.x;
  const int64_t row = blockIdx.x;
  const int i = (int)(row % S);
  if (MODE == 1 && i >= maxscale) return;
  tw2s[j] = tw2[j];
  if (MODE == 1)
    for (int q = j; q < WTB_NBINS; q += kThreads) shist[q] = 0u;
  // smoothed spectrum of this row (kernel C): bins inside the widest pass band of its window
  const int first = i + win.up - (win.K - 1);
  const int kc = rows[first < 0 ? 0 : first].kc;
  const int r_lo = (kc - j) >> 8;                         // bins j + 256 r <= kc
  const int r_hi = (kN - kc - j + 255) >> 8;              // bins j + 256 r >= N - kc
  const float4 *srow = spec + row * (int64_t)kN + j;
  float2 R[16], I[16];
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    float4 g = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (r <= r_lo || r >= r_hi) g = __ldg(srow + 256 * r);
    R[br4(r)] = make_float2(g.x, g.y);
    I[br4(r)] = make_float2(g.z, g.w);
  }
  __syncthreads();   // tw2s / shist visible
  fft4096_inv2(R, I, 4, Bre, Bim, tw2s, tw3, j);
  // lane 0 = S1 + i S2 (two real fields), lane 1 = S12
  if (MODE == 0) {
    float *orow = wct + row * (int64_t)n0;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int t = j + 256 * r;
      if (t < n0) orow[t] = fmaf(R[r].y, R[r].y, I[r].y * I[r].y) / (R[r].x * I[r].x);
    }
  } else {
    const int lo = tlo[i], hi = thi[i];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int t = j + 256 * r;
      if (t >= lo && t <= hi) {
        // binning to 1/1000: the 2-ulp reciprocal-multiply is far inside the bin width
        const float r2 = __fdividef(fmaf(R[r].y, R[r].y, I[r].y * I[r].y), R[r].x * I[r].x);
        if (r2 >= 0.0f) {   // NaN (0/0) is skipped
          int bin = (int)floorf(r2 * (float)WTB_NBINS);
          bin = min(bin, WTB_NBINS - 1);
          atomicAdd(&shist[bin], 1u);
        }
      }
    }
    __syncthreads();
    unsigned long long *hrow = hist + (size_t)i * WTB_NBINS;
    for (int q = j; q < WTB_NBINS; q += kThreads) {
      const unsigned int c = shist[q];
      if (c) atomicAdd(&hrow[q], (unsigned long long)c);
    }
  }
}

struct Tables {
  float2 *tw2 = nullptr;   // [16][16]  exp(+2*pi*i*r*k/256)
  float2 *tw3 = nullptr;   // [16][256] exp(+2*pi*i*r*j/4096)
};
std::mutex g_tab_mu;
std::map<int, Tables> g_tab;   // per device (one process may drive several: wtb_init_multi)

int ensure_tables(const float2 **tw2, const float2 **tw3) {
  std::lock_guard<std::mutex> lk(g_tab_mu);
  const int dev = current_device();
  auto it = g_tab.find(dev);
  if (it == g_tab.end()) {
    std::vector<float2> h2(256), h3(4096);
    const long double two_pi = 2.0L * 3.141592653589793238462643383279502884L;
    for (int r = 0; r < 16; ++r) {
      for (int k = 0; k < 16; ++k) {
        const long double ang = two_pi * r * k / 256.0L;
        h2[r * 16 + k] = make_float2((float)cosl(ang), (float)sinl(ang));
      }
      for (int jj = 0; jj < 256; ++jj) {
        const long double ang = two_pi * r * jj / 4096.0L;
        h3[r * 256 + jj] = make_float2((float)cosl(ang), (float)sinl(ang));
      }
    }
    Tables t;
    WTB_CUDA(cudaMalloc(&t.tw2, sizeof(float2) * 256));
    WTB_CUDA(cudaMalloc(&t.tw3, sizeof(float2) * 4096));
    WTB_CUDA(cudaMemcpy(t.tw2, h2.data(), sizeof(float2) * 256, cudaMemcpyHostToDevice));
    WTB_CUDA(cudaMemcpy(t.tw3, h3.data(), sizeof(float2) * 4096, cudaMemcpyHostToDevice));
    it = g_tab.emplace(dev, t).first;   // kept until wtb_shutdown (34 KB)
  }
  *tw2 = it->second.tw2;
  *tw3 = it->second.tw3;
  return WTB_OK;
}

}  // namespace

// wtb_shutdown: the radix-16 twiddle tables go with the arenas
void wct_fast_release() {
  std::lock_guard<std::mutex> lk(g_tab_mu);
  for (auto &kv : g_tab) {
    if (kv.second.tw2) cudaFree(kv.second.tw2);
    if (kv.second.tw3) cudaFree(kv.second.tw3);
  }
  g_tab.clear();
}

static void fill_rows(const Axes &ax, double dt, double f0, std::vector<WRow> *rows) {
  const int S = ax.J + 1;
  rows->resize(S);
  for (int s = 0; s < S; ++s) {
    const double a = ax.scales[s] / dt * 2.0 * kPi / kN;
    int khi = (int)std::floor((f0 + 5.3) / a);          // daughter < 8e-7 of its peak beyond
    if (khi > kN / 2 - 1) khi = kN / 2 - 1;
    if (khi < 1) khi = 1;
    WRow &r = (*rows)[s];
    r.a = (float)a;
    r.lognorm = (float)std::log2(std::sqrt(2.0 * kPi * ax.scales[s] / dt) * 0.75112554446494248286 / kN);
    r.gcoef = (float)(-0.5 * 1.4426950408889634 * a * a);
    r.inv_s = (float)(1.0 / ax.scales[s]);
    r.L1 = ilog2(khi / 256 + 1);
    r.R1 = 1 << r.L1;               // whole power of two: every input the pruned DFT reads is set
    const double kc = 5.68 / a;     // exp(-0.5 (a k)^2) < 1e-7 beyond
    r.kc = (int)std::floor(kc);
    if (r.kc > kN / 2) r.kc = kN / 2;
    r.kc2 = (float)r.kc * (float)r.kc;   // kernel A stores exactly the bins kernel B reads
  }
}

int fwd_fft_4096(const float *d_y, int64_t nseries, int n0, float2 *d_xhat, cudaStream_t st) {
  const float2 *tw2 = nullptr, *tw3 = nullptr;
  WTB_TRY(ensure_tables(&tw2, &tw3));
  const size_t smem = 2 * sizeof(float2) * kBuf + sizeof(float2) * 256;
  const int64_t ctas = (nseries + 1) / 2;
  WTB_REQUIRE(ctas < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
  WTB_CUDA(cudaFuncSetAttribute(k_fwd_fft_4096, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_fwd_fft_4096<<<(unsigned)ctas, kThreads, smem, st>>>(d_y, nseries, n0, tw2, tw3, d_xhat);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

int cwt_rows_4096(const float2 *d_xhat, int64_t batch, int n0, double dt, const Axes &ax, double f0, int flags,
                  float *d_power, float2 *d_coef, cudaStream_t st) {
  const int S = ax.J + 1;
  std::vector<WRow> rows;
  fill_rows(ax, dt, f0, &rows);
  const float2 *tw2 = nullptr, *tw3 = nullptr;
  WTB_TRY(ensure_tables(&tw2, &tw3));
  // row parameters go to the per-thread parameter buffer (the caller's arena holds xhat)
  void *prm = nullptr;
  WTB_TRY(params_reserve((sizeof(WRow) + sizeof(ushort2)) * kMaxRowsC, &prm));
  WRow *d_rows = (WRow *)prm;
  WTB_CUDA(cudaMemcpyAsync(d_rows, rows.data(), sizeof(WRow) * S, cudaMemcpyHostToDevice, st));
  ushort2 *d_coi = nullptr;
  if ((flags & WTB_COI_MASK) && d_power) {
    std::vector<ushort2> rng;
    coi_row_ranges(n0, dt, ax, f0, &rng);
    d_coi = (ushort2 *)(d_rows + kMaxRowsC);
    WTB_CUDA(cudaMemcpyAsync(d_coi, rng.data(), sizeof(ushort2) * S, cudaMemcpyHostToDevice, st));
  }
  const int64_t nrows = (batch + 1) / 2 * S;
  WTB_REQUIRE(nrows < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
  const size_t smem = 2 * sizeof(float2) * kBuf + sizeof(float2) * 256;
  WTB_CUDA(cudaFuncSetAttribute(k_cwt_rows_4096, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_cwt_rows_4096<<<(unsigned)nrows, kThreads, smem, st>>>(d_xhat, batch, n0, S, d_rows, tw2, tw3, (float)f0, d_power,
                                                          d_coef, d_coi);
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

int wct_fast(const float2 *d_xhat, int64_t pairs, int n0, double dt, const Axes &ax, double f0, void *d_rows_scratch,
             float4 *d_spec, const ScaleWin &win, float *d_wct, float *d_phase, float2 *d_w12,
             unsigned long long *d_hist, const int *d_tlo, const int *d_thi, int maxscale, cudaStream_t st) {
  const int S = ax.J + 1;
  const bool smooth = d_wct || d_hist;
  std::vector<WRow> rows;
  fill_rows(ax, dt, f0, &rows);
  const float2 *tw2 = nullptr, *tw3 = nullptr;
  WTB_TRY(ensure_tables(&tw2, &tw3));
  WRow *d_rows = (WRow *)d_rows_scratch;
  WTB_CUDA(cudaMemcpyAsync(d_rows, rows.data(), sizeof(WRow) * S, cudaMemcpyHostToDevice, st));
  const size_t smem_a = sizeof(float4) * kBuf + sizeof(float2) * 256;
  const size_t smem_b = smem_a + sizeof(unsigned int) * WTB_NBINS;
  const int64_t nrows = pairs * S;
  WTB_REQUIRE(nrows < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
  float4 *spec = d_spec;
  // Rows whose daughter keeps at most `bmax` bins (the largest scales) skip the transforms: their
  // filtered spectra come from k_wct_spec_direct.  Bands shrink with scale, so they are the rows
  // from s_split on.  Only when nothing in the time domain is asked for (phase, cross spectrum).
  int s_split = S;
  std::vector<DRow> drows(S);
  if (smooth && !d_phase && !d_w12) {
    int bmax = 128;     // flat from 128 to 192 bins (measured); 128 keeps the kernel at 32 KB of shared memory (WTB_MC_DIRECT_B overrides, 0 = off)
    if (const char *e = std::getenv("WTB_MC_DIRECT_B")) bmax = std::min(std::atoi(e), kDirB);
    for (int q = S - 1; q >= 0; --q) {
      const double a = ax.scales[q] / dt * 2.0 * kPi / kN;
      int lo = (int)std::ceil((f0 - 5.3) / a), hi = (int)std::floor((f0 + 5.3) / a);
      lo = std::max(lo, 0);
      hi = std::min(hi, kN / 2 - 1);
      drows[q].l0 = lo;
      drows[q].B = hi - lo + 1;
      if (drows[q].B < 1 || drows[q].B > bmax || rows[q].kc > kDirKc || rows[q].kc >= kN / 2) break;
      s_split = q;
    }
  }
  if (s_split > 0) {
    WTB_CUDA(cudaFuncSetAttribute(k_wct_spec_4096, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a));
    k_wct_spec_4096<<<(unsigned)(pairs * s_split), kThreads, smem_a, st>>>(d_xhat, n0, S, s_split, d_rows, tw2, tw3,
                                                                        (float)f0, spec, d_phase, d_w12, smooth ? 1 : 0);
    WTB_LAUNCH_CHECK();
  }
  if (s_split < S) {
    // Dn[d] = sum_{t < n0} exp(-2 pi i d t / N) = exp(-i pi d (n0 - 1) / N) sin(pi d n0 / N) / sin(pi d / N)
    std::vector<float2> dn(2 * kDirDn + 1);
    for (int d = -kDirDn; d <= kDirDn; ++d) {
      double re = n0, im = 0.0;
      if (d != 0) {
        const double mag = std::sin(kPi * d * n0 / kN) / std::sin(kPi * d / kN), ph = -kPi * d * (n0 - 1.0) / kN;
        re = mag * std::cos(ph);
        im = mag * std::sin(ph);
      }
      dn[d + kDirDn] = make_float2((float)re, (float)im);
    }
    void *prm = nullptr;
    const size_t b_dn = align256(sizeof(float2) * dn.size());
    WTB_TRY(params_reserve(b_dn + sizeof(DRow) * kMaxRowsC, &prm));
    float2 *d_dn = (float2 *)prm;
    DRow *d_drows = (DRow *)((char *)prm + b_dn);
    WTB_CUDA(cudaMemcpyAsync(d_dn, dn.data(), sizeof(float2) * dn.size(), cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync(d_drows, drows.data(), sizeof(DRow) * S, cudaMemcpyHostToDevice, st));
    k_wct_spec_direct<<<(unsigned)(pairs * (S - s_split)), kDirThreads, 0, st>>>(d_xhat, S, s_split, d_rows, d_drows,
                                                                                d_dn, (float)f0, spec);
    WTB_LAUNCH_CHECK();
  }
  if (!smooth) return WTB_OK;
  CohWin cw;
  cw.K = win.K;
  cw.up = win.up;
  for (int k = 0; k < win.K; ++k) cw.w[k] = (float)win.w[k];
  {
    auto run = [&](auto kern, size_t smem_c) -> int {
      WTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
      kern<<<(unsigned)(pairs * 16), kThreads, smem_c, st>>>(spec, S, d_rows, cw);
      WTB_LAUNCH_CHECK();
      return WTB_OK;
    };
    // rect(round(0.6 / dj * 2)) taps: 10 at dj = 1/8, 14 at dj = 1/12, 5 at dj = 1/4
    if (cw.K == 10 && cw.up == 4) WTB_TRY(run(k_wct_boxcar_4096_t<10, 5>, 0));
    else if (cw.K == 14 && cw.up == 6) WTB_TRY(run(k_wct_boxcar_4096_t<14, 7>, 0));
    else if (cw.K == 5 && cw.up == 2) WTB_TRY(run(k_wct_boxcar_4096_t<5, 5>, 0));
    else WTB_TRY(run(k_wct_boxcar_4096, sizeof(float4) * (size_t)cw.K * kThreads));
  }
  if (d_hist) {
    WTB_CUDA(cudaFuncSetAttribute(k_wct_coh_4096<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    k_wct_coh_4096<1><<<(unsigned)nrows, kThreads, smem_b, st>>>(spec, n0, S, d_rows, tw2, tw3, cw, nullptr,
                                                                d_hist, d_tlo, d_thi, maxscale);
  } else {
    WTB_CUDA(cudaFuncSetAttribute(k_wct_coh_4096<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    k_wct_coh_4096<0><<<(unsigned)nrows, kThreads, smem_b, st>>>(spec, n0, S, d_rows, tw2, tw3, cw, d_wct,
                                                                nullptr, nullptr, nullptr, 0);
  }
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

}  // namespace wtb
