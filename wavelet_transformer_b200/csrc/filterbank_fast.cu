// Register-blocked MODWT / DWT kernels for compile-time tap counts (L = 2, 4, 6, 8: haar,
// db2, db3, db4 / sym4 = LA8 -- the reference's filters, src/modwt.py:30, dwt.py:71).
//
// One CTA owns one series (one (series, row) pair for the MRA); the row arrives by a 1-D
// TMA bulk load, every level runs in place in shared memory and coefficient rows leave
// through TMA bulk stores, so HBM sees exactly N in + (J+1) N out per series.
//
// What makes these paths HBM-bound instead of shared-memory- or issue-bound:
//  * an a-trous level with dilation d = 2^(j-1) only shares inputs between outputs that are d
//    apart, so a thread owns a chain of R outputs t0, t0+d, .., t0+(R-1)d and slides ONE
//    window of R+L-1 shared-memory loads over all of them (R*L FMAs per filter).  R is odd:
//    lanes then sit R*d elements apart (or 1 apart inside a residue class), which maps the 32
//    lanes of every load/store onto 32 distinct banks for any power-of-two d;
//  * the level index is a template parameter and the circular signal carries a wrap-around
//    halo in shared memory, so every window element is `LDS [base + immediate]` -- no modulo,
//    no address arithmetic in the inner loop; the threads that produce the samples next to
//    the seam also write the halo the next level needs;
//  * taps are (wavelet, scaling) pairs in the constant bank: one packed FFMA2 (FP32) feeds
//    both filters.
#include "filterbank_common.cuh"

namespace wtb {

constexpr int kRM = 9;         // MODWT outputs per thread
constexpr int kRA = 17;        // MRA cascade outputs per thread for long rows (n >= kLongRow): the one-filter
                               // passes are bound by shared-memory wavefronts and a longer chain reads
                               // (R+L-1)/R per output; short rows keep kRM so a CTA still has >= 4 warps
constexpr int kLongRow = 2048;
constexpr int kRD = 5;         // DWT outputs (analysis) / output pairs (synthesis) per thread
constexpr int kMaxFastJ = 10;  // a-trous levels with a compile-time dilation (d <= 512)
constexpr int kChainThreads = 512;  // CTA size limit of the a-trous kernels (<= 64 registers per thread)

template <typename T> struct vec2_of;
template <> struct vec2_of<float> { using type = float2; };
template <> struct vec2_of<double> { using type = double2; };
template <typename T> using vec2 = typename vec2_of<T>::type;

// acc += tap * (v, v) and acc += tap * v, component-wise; FP32 uses the packed FFMA2 pipe
__device__ __forceinline__ float2 fma_dup(float2 tap, float v, float2 acc) {
  return __ffma2_rn(tap, make_float2(v, v), acc);
}
__device__ __forceinline__ double2 fma_dup(double2 tap, double v, double2 acc) {
  acc.x = fma(tap.x, v, acc.x);
  acc.y = fma(tap.y, v, acc.y);
  return acc;
}
__device__ __forceinline__ float2 fma_pair(float2 tap, float2 v, float2 acc) { return __ffma2_rn(tap, v, acc); }
__device__ __forceinline__ double2 fma_pair(double2 tap, double2 v, double2 acc) {
  acc.x = fma(tap.x, v.x, acc.x);
  acc.y = fma(tap.y, v.y, acc.y);
  return acc;
}
template <typename T> __device__ __forceinline__ vec2<T> mk2(T x, T y) {
  vec2<T> r;
  r.x = x;
  r.y = y;
  return r;
}

// Taps in the kernel's precision as constant-bank operands.  hl[l] = (wavelet h[l], scaling
// g[l]); lo2 / hi2 hold consecutive taps (t[2e], t[2e+1]) for the DWT synthesis.
template <typename T, int L> struct TapsK {
  vec2<T> hl[L];
  vec2<T> lo2[L / 2];
  vec2<T> hi2[L / 2];
};
template <typename T, int L> inline TapsK<T, L> narrow_taps(const Taps &t) {
  TapsK<T, L> k;
  for (int i = 0; i < L; ++i) {
    k.hl[i].x = T(t.hi[i]);
    k.hl[i].y = T(t.lo[i]);
  }
  for (int e = 0; e < L / 2; ++e) {
    k.lo2[e].x = T(t.lo[2 * e]);
    k.lo2[e].y = T(t.lo[2 * e + 1]);
    k.hi2[e].x = T(t.hi[2 * e]);
    k.hi2[e].y = T(t.hi[2 * e + 1]);
  }
  return k;
}

// Chain owned by this thread at dilation d = 2^sh: outputs t0 + m d, m < R.  Computed with the
// runtime level so that the per-level template bodies hold nothing but immediate-offset
// loads, FMAs and stores (ptxas otherwise hoists ten copies of this above the level switch).
struct Chain {
  bool active;
  int t0;
  __device__ __forceinline__ Chain(int n, int sh, int R) {
    const int item = threadIdx.x;
    const int first = (item >> sh) * (R << sh) + (item & ((1 << sh) - 1));
    active = first < n;  // a chain that starts past the end has no output
    // idle threads run the window of chain 0 (in bounds, results dropped): keeping the
    // arithmetic unconditional keeps every accumulator in registers across the barrier
    t0 = active ? first : 0;
  }
};
// wrap-around halo (elements) a level with dilation 2^sh reads on one side, TMA-sized
__host__ __device__ __forceinline__ int halo_of(int L, int sh) { return (((L - 1) << sh) + 3) & ~3; }

// ---- rows at any element alignment --------------------------------------------------------
// A 1-D bulk copy needs 16-byte aligned addresses and sizes, but rows of an odd-length batch
// start 4, 8 or 12 bytes off.  The copy therefore covers the enclosing 16-byte aligned span
// (at most 15 bytes of the neighbouring rows on either side) and the row is addressed `shift`
// elements into its shared-memory slot; every shared-memory access of the kernels is scalar,
// so the slot's own alignment does not matter.  Stores mirror this: the row is staged at the
// shift of its global address, the aligned body leaves by TMA and the <= 3 elements on each
// end by plain stores.
template <typename T> __device__ __forceinline__ int shift_of(const T *p) {
  return (int)((reinterpret_cast<uintptr_t>(p) & 15) / sizeof(T));
}

template <typename T> struct RowIn {
  const T *src;
  int n, shift;
  bool aligned;  // no shift and a whole number of 16-byte units: halos can come by TMA too
  __device__ __forceinline__ RowIn(const T *src_, int n_) : src(src_), n(n_) {
    shift = shift_of(src);
    aligned = shift == 0 && (sizeof(T) * (size_t)n) % 16 == 0;
  }
  // thread 0.  slot: 16-byte aligned, room for tail + 4 + n + head elements around slot[0].
  // head / tail (multiples of 4): copies of the first / last elements after / before the row.
  __device__ __forceinline__ void issue(T *slot, int head, int tail, uint64_t *bar) const {
    const uint32_t s = sizeof(T);
    if (aligned) {
      mbar_expect_tx(bar, s * (uint32_t)(n + head + tail));
      tma_load_1d(slot, src, s * n, bar);
      if (head) tma_load_1d(slot + n, src, s * head, bar);
      if (tail) tma_load_1d(slot - tail, src + n - tail, s * tail, bar);
    } else {
      const uint32_t bytes = (uint32_t)((s * (size_t)(shift + n) + 15) & ~size_t(15));
      mbar_expect_tx(bar, bytes);
      tma_load_1d(slot, src - shift, bytes, bar);
    }
  }
  // all threads, after the barrier wait; returns the row pointer.  Unaligned rows build their
  // halos here (one extra CTA barrier).
  __device__ __forceinline__ T *finish(T *slot, int head, int tail) const {
    T *row = slot + shift;
    if (!aligned) {
      for (int k = threadIdx.x; k < head; k += blockDim.x) row[n + k] = row[k];
      for (int k = threadIdx.x; k < tail; k += blockDim.x) row[-1 - k] = row[n - 1 - k];
      __syncthreads();
    }
    return row;
  }
};

// All threads, after the barrier that published `row` (staged at shift_of(dst) in a 16-byte
// aligned slot) and a fence_smem_to_async().  Thread 0 owns the bulk group.
template <typename T>
__device__ __forceinline__ void store_row(T *dst, const T *row, int n) {
  const int per16 = 16 / (int)sizeof(T);
  const int head = min(n, (per16 - shift_of(dst)) & (per16 - 1));
  const int body = (n - head) & ~(per16 - 1);
  if (threadIdx.x == 0 && body) {
    tma_store_1d(dst + head, row + head, (uint32_t)(sizeof(T) * (size_t)body));
    tma_store_commit();
  }
  const int k = threadIdx.x;
  if (k < head) dst[k] = row[k];
  if (k < per16 && head + body + k < n) dst[head + body + k] = row[head + body + k];
}

// ---- MODWT analysis: w_j[t] = sum_l h[l] v[(t - d l) mod n], v_j with g ------------------
// v carries a left halo: v[-k] = v[n-k].  In place: window -> registers | barrier | write.
template <typename T, int L, int SH>
__device__ __forceinline__ void analysis_level(T *__restrict__ v, T *__restrict__ wb, int n, int mirror,
                                            const TapsK<T, L> &tp, bool wait_store, const Chain ch) {
  constexpr int R = kRM, d = 1 << SH;
  vec2<T> acc[R];
#pragma unroll
  for (int m = 0; m < R; ++m) acc[m] = mk2<T>(0, 0);
  const T *win = v + ch.t0 - (L - 1) * d;  // window element q sits at t0 + (q-(L-1)) d
#pragma unroll
  for (int q = R + L - 2; q >= 0; --q) {
    const T val = win[q * d];
#pragma unroll
    for (int m = 0; m < R; ++m) {
      const int l = m + L - 1 - q;  // ascending in l as q descends, like the reference sum
      if (l >= 0 && l < L) acc[m] = fma_dup(tp.hl[l], val, acc[m]);
    }
  }
  // the previous row's bulk store must have left wb before it is overwritten
  if (wait_store && threadIdx.x == 0) tma_store_wait_read();
  __syncthreads();
  if (ch.active) {
    if (ch.t0 + (R - 1) * d < n - mirror) {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        wb[ch.t0 + m * d] = acc[m].x;
        v[ch.t0 + m * d] = acc[m].y;
      }
    } else {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int t = ch.t0 + m * d;
        if (t < n) wb[t] = acc[m].x;
        if (t < n) v[t] = acc[m].y;
        if (t < n && t >= n - mirror) v[t - n] = acc[m].y;  // next level's halo
      }
    }
  }
}

template <typename T, int L>
__global__ void __launch_bounds__(kChainThreads, 2) k_modwt_blk(const T *__restrict__ x, int n, int J, TapsK<T, L> tp,
                                                                T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int HL = halo_of(L, J - 1);                              // left halo of the deepest level
  const int np = (n + (kRM - 1) * (1 << (J - 1)) + 4 + 3) & ~3;  // + discarded chain slots + shift
  T *v_slot = reinterpret_cast<T *>(smem_raw) + HL;
  T *w_slot = v_slot + np;
  const int64_t b = blockIdx.x;
  const RowIn<T> rin(x + b * n, n);
  T *o = out + b * (int64_t)(J + 1) * n;
  const int h0 = halo_of(L, 0);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) rin.issue(v_slot, 0, h0, &bar);
  mbar_wait(&bar, 0);
  T *v = rin.finish(v_slot, 0, h0);
  for (int j = 1; j <= J; ++j) {
    const int mirror = j < J ? halo_of(L, j) : 0;
    T *orow = o + (int64_t)(j - 1) * n;
    T *wb = w_slot + shift_of(orow);
    const Chain ch(n, j - 1, kRM);
    switch (j - 1) {
#define WTB_LEVEL(SH) \
  case SH: analysis_level<T, L, SH>(v, wb, n, mirror, tp, true, ch); break;
      WTB_LEVEL(0) WTB_LEVEL(1) WTB_LEVEL(2) WTB_LEVEL(3) WTB_LEVEL(4)
      WTB_LEVEL(5) WTB_LEVEL(6) WTB_LEVEL(7) WTB_LEVEL(8) WTB_LEVEL(9)
#undef WTB_LEVEL
    }
    fence_smem_to_async();
    __syncthreads();
    store_row(orow, wb, n);
  }
  T *vrow = o + (int64_t)J * n;
  if (shift_of(vrow) == rin.shift) {
    store_row(vrow, v, n);
  } else {
    for (int t = threadIdx.x; t < n; t += blockDim.x) vrow[t] = v[t];
  }
  if (threadIdx.x == 0) tma_store_wait_all();
}

// Write a chain in place; samples t < mirror are repeated at t + n (the right halo the next,
// finer level reads).  Three shapes: all inside and clear of the halo, all inside the halo,
// and the seam cases with per-sample predicates.
template <typename T, int R, int d>
__device__ __forceinline__ void store_chain(T *__restrict__ x, const T (&val)[R], int t0, int n, int mirror) {
  const int last = t0 + (R - 1) * d;
  if (last < n && t0 >= mirror) {
#pragma unroll
    for (int m = 0; m < R; ++m) x[t0 + m * d] = val[m];
  } else if (last < mirror) {
#pragma unroll
    for (int m = 0; m < R; ++m) {
      x[t0 + m * d] = val[m];
      x[t0 + m * d + n] = val[m];
    }
  } else {
#pragma unroll
    for (int m = 0; m < R; ++m) {
      const int t = t0 + m * d;
      if (t < n) x[t] = val[m];
      if (t < mirror) x[t + n] = val[m];
    }
  }
}

// ---- MODWT synthesis: v_{j-1}[t] = sum_l h[l] w_j[(t + d l) mod n] + g[l] v_j[(t + d l) mod n]
// v and the w_j row carry a right halo: x[n+k] = x[k].
template <typename T, int L, int SH>
__device__ __forceinline__ void synthesis_level(const T *__restrict__ wj, T *__restrict__ v, int n, int mirror,
                                             const TapsK<T, L> &tp, const Chain ch) {
  constexpr int R = kRM, d = 1 << SH;
  T res[R];
  {
    vec2<T> acc[R];
#pragma unroll
    for (int m = 0; m < R; ++m) acc[m] = mk2<T>(0, 0);
    const T *pw = wj + ch.t0, *pv = v + ch.t0;  // window element q sits at t0 + q d
#pragma unroll
    for (int q = 0; q < R + L - 1; ++q) {
      const vec2<T> val = mk2<T>(pw[q * d], pv[q * d]);
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int l = q - m;
        if (l >= 0 && l < L) acc[m] = fma_pair(tp.hl[l], val, acc[m]);
      }
    }
#pragma unroll
    for (int m = 0; m < R; ++m) res[m] = acc[m].x + acc[m].y;
  }
  __syncthreads();
  if (ch.active) store_chain<T, R, d>(v, res, ch.t0, n, mirror);
}

template <typename T, int L>
__global__ void __launch_bounds__(kChainThreads, 2) k_imodwt_blk(const T *__restrict__ w, int n, int J, TapsK<T, L> tp,
                                                                 T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar[3];  // w rows alternate on [0], [1]; v_J arrives on [2]
  // row + wrap halo + window tail of discarded chain slots + alignment shift
  const int np = (n + (kRM + L - 2) * (1 << (J - 1)) + 4 + 3) & ~3;
  T *v_slot = reinterpret_cast<T *>(smem_raw);
  T *w_slot = v_slot + np;  // [2][np]: w_j rows, the next one prefetched while this one is used
  const int64_t b = blockIdx.x;
  const T *wb = w + b * (int64_t)(J + 1) * n;
  if (threadIdx.x == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    mbar_init(&bar[2], 1);
    mbar_init_fence();
  }
  __syncthreads();
  const int hJ = halo_of(L, J - 1);
  const RowIn<T> rv(wb + (int64_t)J * n, n);
  if (threadIdx.x == 0) {
    rv.issue(v_slot, hJ, 0, &bar[2]);
    RowIn<T>(wb + (int64_t)(J - 1) * n, n).issue(w_slot, hJ, 0, &bar[0]);
  }
  mbar_wait(&bar[2], 0);
  T *v = rv.finish(v_slot, hJ, 0);
  for (int j = J; j >= 1; --j) {
    const int it = J - j, cur = it & 1;
    const RowIn<T> rw(wb + (int64_t)(j - 1) * n, n);
    // the other slot was last read in iteration it-1, which ended with a barrier
    if (threadIdx.x == 0 && j > 1)
      RowIn<T>(wb + (int64_t)(j - 2) * n, n).issue(w_slot + (cur ^ 1) * np, halo_of(L, j - 2), 0, &bar[cur ^ 1]);
    mbar_wait(&bar[cur], (it >> 1) & 1);
    const T *wj = rw.finish(w_slot + cur * np, halo_of(L, j - 1), 0);
    const int mirror = j > 1 ? halo_of(L, j - 2) : 0;
    const Chain ch(n, j - 1, kRM);
    switch (j - 1) {
#define WTB_LEVEL(SH) \
  case SH: synthesis_level<T, L, SH>(wj, v, n, mirror, tp, ch); break;
      WTB_LEVEL(0) WTB_LEVEL(1) WTB_LEVEL(2) WTB_LEVEL(3) WTB_LEVEL(4)
      WTB_LEVEL(5) WTB_LEVEL(6) WTB_LEVEL(7) WTB_LEVEL(8) WTB_LEVEL(9)
#undef WTB_LEVEL
    }
    if (j == 1) fence_smem_to_async();
    __syncthreads();
  }
  T *xrow = out + b * n;
  if (shift_of(xrow) == rv.shift) {
    store_row(xrow, v, n);
    if (threadIdx.x == 0) tma_store_wait_all();
  } else {
    for (int t = threadIdx.x; t < n; t += blockDim.x) xrow[t] = v[t];
  }
}

// ---- MODWT multiresolution analysis as a synthesis cascade ----------------------------------
// D_j = G_1' .. G_{j-1}' H_j' w_j and S_J = G_1' .. G_J' v_J, where X_k' is the one-filter
// synthesis step at dilation 2^(k-1).  Algebraically this is the reference's correlation with
// the periodised equivalent filter (src/modwt.py:163-194), at sum_j j*L instead of
// sum_j ((2^j - 1)(L-1) + 1) multiply-adds per sample.
template <typename T, int L, int R, int SH, bool HI>
__device__ __forceinline__ void cascade_level(T *__restrict__ a, int n, int mirror, const TapsK<T, L> &tp,
                                           const Chain ch) {
  constexpr int d = 1 << SH;
  T acc[R];
  {
#pragma unroll
    for (int m = 0; m < R; ++m) acc[m] = T(0);
    const T *win = a + ch.t0;
#pragma unroll
    for (int q = 0; q < R + L - 1; ++q) {
      const T val = win[q * d];
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int l = q - m;
        if (l >= 0 && l < L) acc[m] = fma(HI ? tp.hl[l].x : tp.hl[l].y, val, acc[m]);
      }
    }
  }
  __syncthreads();
  if (ch.active) store_chain<T, R, d>(a, acc, ch.t0, n, mirror);
}

template <typename T, int L, int R>
__global__ void __launch_bounds__(kChainThreads, 2) k_mra_blk(const T *__restrict__ w, int n, int J, TapsK<T, L> tp, T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  T *a_slot = reinterpret_cast<T *>(smem_raw);
  const int row = blockIdx.x % (J + 1);
  const int64_t off = (int64_t)blockIdx.x * n;  // (b (J+1) + row) n
  const int lev = row < J ? row + 1 : J;
  const RowIn<T> rin(w + off, n);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) rin.issue(a_slot, halo_of(L, lev - 1), 0, &bar);
  mbar_wait(&bar, 0);
  T *a = rin.finish(a_slot, halo_of(L, lev - 1), 0);
  for (int k = lev; k >= 1; --k) {
    const int mirror = k > 1 ? halo_of(L, k - 2) : 0;
    const bool first = k == lev && row < J;  // the detail rows enter through the wavelet filter
    const Chain ch(n, k - 1, R);
    switch (k - 1) {
#define WTB_LEVEL(SH)                                              \
  case SH:                                                         \
    if (first)                                                     \
      cascade_level<T, L, R, SH, true>(a, n, mirror, tp, ch);         \
    else                                                           \
      cascade_level<T, L, R, SH, false>(a, n, mirror, tp, ch);        \
    break;
      WTB_LEVEL(0) WTB_LEVEL(1) WTB_LEVEL(2) WTB_LEVEL(3) WTB_LEVEL(4)
      WTB_LEVEL(5) WTB_LEVEL(6) WTB_LEVEL(7) WTB_LEVEL(8) WTB_LEVEL(9)
#undef WTB_LEVEL
    }
    if (k == 1) fence_smem_to_async();
    __syncthreads();
  }
  if (shift_of(out + off) == rin.shift) {
    store_row(out + off, a, n);
    if (threadIdx.x == 0) tma_store_wait_all();
  } else {
    for (int t = threadIdx.x; t < n; t += blockDim.x) out[off + t] = a[t];
  }
}

// ---- DWT analysis (pywt.wavedec, symmetric): cA[i] = sum_j lo[j] xe[2i+1-j], cD with hi ----
// The signal sits in shared memory WITH its half-sample-symmetric halo (kHalo samples before
// index 0, L-1 mirrored samples after the end), so every window is a plain strided read; the
// threads that produce the first / last approximation samples also write their mirror images,
// which is the halo of the next level.  In place: window -> registers | barrier | write.
constexpr int kHalo = 8;  // >= L-1 and a multiple of 16 bytes in either precision

template <typename T, int L>
__global__ void k_wavedec_blk(const T *__restrict__ x, LevelPlan plan, TapsK<T, L> tp, T *__restrict__ coeffs) {
  constexpr int R = kRD;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int64_t b = blockIdx.x;
  T *o = coeffs + b * (int64_t)plan.total;
  const RowIn<T> rin(x + b * (int64_t)plan.n, plan.n);
  T *a_slot = reinterpret_cast<T *>(smem_raw) + kHalo;  // signal slot: [-kHalo .. plan.buf - kHalo)
  // the packed output row cA_L | cD_L | .. | cD_1, staged at the alignment of its global row
  T *pk = reinterpret_cast<T *>(smem_raw) + plan.buf + shift_of(o);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) rin.issue(a_slot, 0, 0, &bar);
  mbar_wait(&bar, 0);
  T *a = a_slot + rin.shift;
  int cur = plan.n;
  if ((int)threadIdx.x < L - 1) {
    const int k = threadIdx.x;
    a[-1 - k] = a[k];
    a[cur + k] = a[cur - 1 - k];
  }
  __syncthreads();
  for (int lev = 1; lev <= plan.level; ++lev) {
    const int slot = plan.level - lev + 1;  // cD_lev
    const int nout = plan.len[slot];
    const int i0 = threadIdx.x * R;
    const bool active = i0 < nout;
    vec2<T> acc[R];  // (cD, cA)
    if (active) {
#pragma unroll
      for (int m = 0; m < R; ++m) acc[m] = mk2<T>(0, 0);
      const T *win = a + (2 * i0 + 2 - L);  // leftmost input of output i0
#pragma unroll
      for (int q = 2 * R + L - 3; q >= 0; --q) {
        const T val = win[q];
#pragma unroll
        for (int m = 0; m < R; ++m) {
          const int j = 2 * m + L - 1 - q;
          if (j >= 0 && j < L) acc[m] = fma_dup(tp.hl[j], val, acc[m]);
        }
      }
    }
    __syncthreads();
    if (active) {
      T *od = pk + plan.off[slot];
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int i = i0 + m;
        if (i < nout) {
          od[i] = acc[m].x;
          a[i] = acc[m].y;
          if (i < L - 1) a[-1 - i] = acc[m].y;
          if (i >= nout - (L - 1)) a[2 * nout - 1 - i] = acc[m].y;
          if (lev == plan.level) pk[i] = acc[m].y;
        }
      }
    }
    if (lev == plan.level) fence_smem_to_async();
    __syncthreads();
    cur = nout;
  }
  if (plan.level == 0) {
    for (int i = threadIdx.x; i < cur; i += blockDim.x) pk[i] = a[i];
    fence_smem_to_async();
    __syncthreads();
  }
  store_row(o, pk, plan.total);
  if (threadIdx.x == 0) tma_store_wait_all();
}

// ---- DWT synthesis (pywt.waverec): full[p] = sum_k lo[p-2k] a[k] + hi[p-2k] d[k], kept
// p in [L-2, 2m).  Output pair u (samples 2u, 2u+1) uses a[u .. u+L/2-1] and d[same]:
// even samples take the even taps, odd samples the odd taps, and no index leaves [0, m).
template <typename T, int L>
__global__ void k_waverec_blk(const T *__restrict__ coeffs, LevelPlan plan, TapsK<T, L> tp, T *__restrict__ x) {
  constexpr int R = kRD, H = L / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int64_t b = blockIdx.x;
  T *o = x + b * (int64_t)plan.n;
  const RowIn<T> rin(coeffs + b * (int64_t)plan.total, plan.total);
  // ping-pong buffers staged at the alignment of the output row (an even shift: pair stores)
  const int so = shift_of(o) & ~1;
  T *a = reinterpret_cast<T *>(smem_raw) + so;
  T *an = a + plan.buf;
  T *pk_slot = reinterpret_cast<T *>(smem_raw) + 2 * plan.buf;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) rin.issue(pk_slot, 0, 0, &bar);
  mbar_wait(&bar, 0);
  const T *pk = pk_slot + rin.shift;
  const T *ap = pk;  // cA_L sits at the head of the packed row
  int cur = plan.len[0];
  for (int slot = 1; slot <= plan.level; ++slot) {
    const int m = plan.len[slot];  // == cur or cur-1 (pywt drops the extra approximation sample)
    const T *d = pk + plan.off[slot];
    const int npairs = m - H + 1;
    const int items = (npairs + R - 1) / R;
    for (int item = threadIdx.x; item < items; item += blockDim.x) {
      const int u0 = item * R;
      vec2<T> acc[R];  // (even sample, odd sample)
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = mk2<T>(0, 0);
#pragma unroll
      for (int q = 0; q < R + H - 1; ++q) {
        const int k = min(u0 + q, m - 1);  // only the unused tail pairs ever clamp
        const T av = ap[k], dv = d[k];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int e = r + H - 1 - q;
          if (e >= 0 && e < H) {
            acc[r] = fma_dup(tp.lo2[e], av, acc[r]);
            acc[r] = fma_dup(tp.hi2[e], dv, acc[r]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (u0 + r < npairs) reinterpret_cast<vec2<T> *>(an)[u0 + r] = acc[r];
    }
    fence_smem_to_async();
    __syncthreads();
    ap = an;
    an = (an == a) ? a + plan.buf : a;
    cur = 2 * npairs;
  }
  if (plan.level > 0 && so == shift_of(o)) {
    store_row(o, ap, plan.n);
    if (threadIdx.x == 0) tma_store_wait_all();
  } else {
    for (int i = threadIdx.x; i < cur; i += blockDim.x) o[i] = ap[i];
  }
}

// ---- launchers --------------------------------------------------------------------------------
static int round_threads(int64_t items) {
  const int64_t t = (items + 31) / 32 * 32;
  return (int)std::max<int64_t>(32, std::min<int64_t>(1024, t));
}

#define WTB_TAPS_SWITCH(L, ...)                             \
  switch (L) {                                              \
    case 2: { constexpr int LT = 2; __VA_ARGS__; } break;   \
    case 4: { constexpr int LT = 4; __VA_ARGS__; } break;   \
    case 6: { constexpr int LT = 6; __VA_ARGS__; } break;   \
    case 8: { constexpr int LT = 8; __VA_ARGS__; } break;   \
    default: return WTB_EUNSUPPORTED;                       \
  }

// CTA size for the a-trous kernels: one chain per thread at every level.  0 = not coverable:
// too many levels for the compile-time dilations, a dilated filter longer than the series
// (the halo would wrap more than once), or more chains than a CTA has threads.
static int chain_threads(int n, int L, int J, int R = kRM) {
  if (J > kMaxFastJ || halo_of(L, J - 1) > n) return 0;
  int64_t most = 0;
  for (int j = 1; j <= J; ++j) {
    const int64_t d = int64_t(1) << (j - 1), span = d * R;
    most = std::max<int64_t>(most, ((n + span - 1) / span) * d);
  }
  return most <= kChainThreads ? round_threads(most) : 0;
}

template <typename T>
int modwt_fast(const void *x, int64_t batch, int n, const Taps &taps, int J, void *out, cudaStream_t st) {
  if (!fast_taps_ok(taps.L)) return WTB_EUNSUPPORTED;
  const int threads = chain_threads(n, taps.L, J);
  if (!threads) return WTB_EUNSUPPORTED;
  const size_t v_len = (size_t)halo_of(taps.L, J - 1) + (size_t)((n + (kRM - 1) * (1 << (J - 1)) + 4 + 3) & ~3);
  const size_t smem = sizeof(T) * (v_len + (size_t)((n + 4 + 3) & ~3));
  if (smem > kSmemLimit) return WTB_EUNSUPPORTED;
  WTB_TAPS_SWITCH(taps.L, {
    WTB_TRY(set_smem(k_modwt_blk<T, LT>, smem));
    k_modwt_blk<T, LT><<<(unsigned)batch, threads, smem, st>>>((const T *)x, n, J, narrow_taps<T, LT>(taps), (T *)out);
  });
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

template <typename T>
int imodwt_fast(const void *w, int64_t batch, int n, const Taps &taps, int J, void *out, cudaStream_t st) {
  if (!fast_taps_ok(taps.L)) return WTB_EUNSUPPORTED;
  const int threads = chain_threads(n, taps.L, J);
  if (!threads) return WTB_EUNSUPPORTED;
  const size_t np = (size_t)((n + (kRM + taps.L - 2) * (1 << (J - 1)) + 4 + 3) & ~3);
  const size_t smem = sizeof(T) * 3 * np;
  if (smem > kSmemLimit) return WTB_EUNSUPPORTED;
  WTB_TAPS_SWITCH(taps.L, {
    WTB_TRY(set_smem(k_imodwt_blk<T, LT>, smem));
    k_imodwt_blk<T, LT><<<(unsigned)batch, threads, smem, st>>>((const T *)w, n, J, narrow_taps<T, LT>(taps), (T *)out);
  });
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

// shared memory of k_mra_blk<T, L, R> (elem = sizeof(T)) for this shape; 0 when its chains do not cover it
static size_t mra_blk_smem(int n, int L, int J, int R, size_t elem) {
  if (!chain_threads(n, L, J, R)) return 0;
  return elem * (size_t)((n + (R + L - 2) * (1 << (J - 1)) + 4 + 3) & ~3);
}

// mra_fast's choice below, without a launch (its batch * (J + 1) < 2^31 test cannot fail at a length that the
// generic kernel's shared memory refuses)
bool mra_fast_covers(int n, int L, int J, size_t elem) {
  auto fits = [&](int R) {
    const size_t smem = mra_blk_smem(n, L, J, R, elem);
    return smem && smem <= kSmemLimit;
  };
  return fast_taps_ok(L) && ((n >= kLongRow && fits(kRA)) || fits(kRM));
}

template <typename T, int R>
static int mra_fast_r(const void *w, int64_t batch, int n, const Taps &taps, int J, void *out, cudaStream_t st) {
  const int threads = chain_threads(n, taps.L, J, R);
  const size_t smem = mra_blk_smem(n, taps.L, J, R, sizeof(T));
  if (!smem || smem > kSmemLimit) return WTB_EUNSUPPORTED;
  WTB_TAPS_SWITCH(taps.L, {
    WTB_TRY(set_smem(k_mra_blk<T, LT, R>, smem));
    k_mra_blk<T, LT, R><<<(unsigned)(batch * (J + 1)), threads, smem, st>>>((const T *)w, n, J,
                                                                           narrow_taps<T, LT>(taps), (T *)out);
  });
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

template <typename T>
int mra_fast(const void *w, int64_t batch, int n, const Taps &taps, int J, void *out, cudaStream_t st) {
  if (!fast_taps_ok(taps.L) || batch * (J + 1) >= (1LL << 31)) return WTB_EUNSUPPORTED;
  if (n >= kLongRow) {
    const int rc = mra_fast_r<T, kRA>(w, batch, n, taps, J, out, st);
    if (rc != WTB_EUNSUPPORTED) return rc;   // e.g. the longer chains' halo no longer fits
  }
  return mra_fast_r<T, kRM>(w, batch, n, taps, J, out, st);
}

template <typename T>
int wavedec_fast(const void *x, int64_t batch, const LevelPlan &plan_in, const Taps &taps, void *coeffs,
                 cudaStream_t st) {
  if (!fast_taps_ok(taps.L)) return WTB_EUNSUPPORTED;
  LevelPlan plan = plan_in;
  // every level's input must hold one whole mirror image of the filter overhang
  int cur = plan.n;
  for (int lev = 1; lev <= plan.level; ++lev) {
    if (cur < taps.L - 1) return WTB_EUNSUPPORTED;
    cur = plan.len[plan.level - lev + 1];
  }
  const int64_t items = ((plan.n + taps.L - 1) / 2 + kRD - 1) / kRD;
  if (items > 1024) return WTB_EUNSUPPORTED;
  plan.buf = (kHalo + plan.n + taps.L + 2 * kRD + 4 + 3) & ~3;  // halo | shift | signal | mirror + discarded tail
  const size_t smem = sizeof(T) * ((size_t)plan.buf + (size_t)((plan.total + 4 + 3) & ~3));
  if (smem > kSmemLimit) return WTB_EUNSUPPORTED;
  const int threads = round_threads(items);
  WTB_TAPS_SWITCH(taps.L, {
    WTB_TRY(set_smem(k_wavedec_blk<T, LT>, smem));
    k_wavedec_blk<T, LT><<<(unsigned)batch, threads, smem, st>>>((const T *)x, plan, narrow_taps<T, LT>(taps), (T *)coeffs);
  });
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

template <typename T>
int waverec_fast(const void *coeffs, int64_t batch, const LevelPlan &plan_in, const Taps &taps, void *x,
                 cudaStream_t st) {
  if (!fast_taps_ok(taps.L)) return WTB_EUNSUPPORTED;
  LevelPlan plan = plan_in;
  int longest = plan.n;
  for (int i = 0; i <= plan.level; ++i) {
    longest = std::max(longest, plan.len[i]);
    if (i > 0 && plan.len[i] < taps.L / 2) return WTB_EUNSUPPORTED;  // no full output pair
  }
  plan.buf = (longest + taps.L + 4 + 3) & ~3;
  const size_t smem = sizeof(T) * (2 * (size_t)plan.buf + (size_t)((plan.total + 4 + 3) & ~3));
  if (smem > kSmemLimit) return WTB_EUNSUPPORTED;
  const int threads = round_threads((plan.n / 2 + kRD - 1) / kRD);
  WTB_TAPS_SWITCH(taps.L, {
    WTB_TRY(set_smem(k_waverec_blk<T, LT>, smem));
    k_waverec_blk<T, LT><<<(unsigned)batch, threads, smem, st>>>((const T *)coeffs, plan, narrow_taps<T, LT>(taps), (T *)x);
  });
  WTB_LAUNCH_CHECK();
  return WTB_OK;
}

#define WTB_INSTANTIATE(T)                                                                               \
  template int modwt_fast<T>(const void *, int64_t, int, const Taps &, int, void *, cudaStream_t);       \
  template int imodwt_fast<T>(const void *, int64_t, int, const Taps &, int, void *, cudaStream_t);      \
  template int mra_fast<T>(const void *, int64_t, int, const Taps &, int, void *, cudaStream_t);         \
  template int wavedec_fast<T>(const void *, int64_t, const LevelPlan &, const Taps &, void *, cudaStream_t); \
  template int waverec_fast<T>(const void *, int64_t, const LevelPlan &, const Taps &, void *, cudaStream_t);
WTB_INSTANTIATE(float)
WTB_INSTANTIATE(double)

}  // namespace wtb
