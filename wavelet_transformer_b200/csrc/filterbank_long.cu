// MODWT, inverse MODWT, MRA and symmetric-mode DWT of long series: the shapes whose ping-pong buffers do not fit
// one CTA's shared memory (filterbank.cu routes here exactly when its generic kernel's buffer passes kSmemLimit).
//
// Each level is one launch over a grid of (output tile, series[, row]); a thread computes one output with the
// per-output arithmetic of the one-CTA kernel it stands in for (same taps, same order, same accumulators) and
// gathers its inputs through L1 / L2: a warp's reads for one tap are contiguous.  The level-to-level
// intermediates live in two arena buffers, and series run in waves whose two buffers fit 64 MiB (half the
// B200's 126 MB L2), so level j+1 finds level j's output in L2.  A series' arithmetic does not depend on its
// wave, so results do not depend on the batch, the host chunk of run_batched, the pool or the pointers.
//
//   k_modwt_long     w_j, v_j from v_{j-1} (k_modwt)                      J launches per wave
//   k_synth_long     h / g synthesis at one dilation: the inverse MODWT     J launches per wave (wtb_imodwt)
//                    step (k_imodwt) and one level of the MRA cascade     J launches per wave (wtb_modwtmra_taps)
//                    of every active row (k_mra_blk)
//   k_dwt_long       cA, cD of one symmetric-mode level (k_wavedec)        `level` launches per wave
//   k_idwt_long      one level of pywt's waverec (k_waverec)               `level` launches per wave
//   k_mra_filt_long  correlation with explicit periodised filters over    1 launch per wave (wtb_modwtmra)
//                    each row's non-zero taps only (k_modwtmra)
#include <vector>

#include "filterbank_common.cuh"

namespace wtb {

constexpr int kLongThreads = 256;
constexpr size_t kLongWaveBytes = size_t(64) << 20;

// Series per wave: those whose two intermediate buffers (per_series bytes together) fit 64 MiB, at least one, at
// most the batch.  At the lengths routed here that is at most 64 MiB / (2 * 4 B * 14529) = 577 series, well
// inside gridDim.y.
static int64_t long_wave(size_t per_series, int64_t batch) {
  return std::min<int64_t>(batch, std::max<int64_t>(1, (int64_t)(kLongWaveBytes / per_series)));
}

static dim3 long_grid(int64_t n, int64_t series, int rows = 1) {
  return dim3((unsigned)((n + kLongThreads - 1) / kLongThreads), (unsigned)series, (unsigned)rows);
}

static size_t al256(size_t b) { return (b + 255) / 256 * 256; }

// Taps in the kernel's precision and the level's circular offsets (2^(j-1) l) mod n, from 64-bit host arithmetic
// so that a dilated filter that wraps the series several times is exact.
template <typename T> struct LongTaps {
  int L;
  T lo[kMaxTaps];
  T hi[kMaxTaps];
  int off[kMaxTaps];
};

template <typename T> static LongTaps<T> long_taps(const Taps &t, int j, int n) {
  LongTaps<T> k;
  k.L = t.L;
  for (int l = 0; l < t.L; ++l) {
    k.lo[l] = T(t.lo[l]);
    k.hi[l] = T(t.hi[l]);
    k.off[l] = j > 0 ? (int)(((int64_t(1) << (j - 1)) * l) % n) : 0;
  }
  return k;
}

// ---- MODWT analysis level: w[t] = sum_l hi[l] v[(t - off_l) mod n], vn[t] with lo (k_modwt's order) -------------
template <typename T>
__global__ void __launch_bounds__(kLongThreads) k_modwt_long(const T *__restrict__ v, int64_t v_ser, int n,
                                                             LongTaps<T> tp, T *__restrict__ w, int64_t w_ser,
                                                             T *__restrict__ vn, int64_t vn_ser) {
  const int64_t t = (int64_t)blockIdx.x * kLongThreads + threadIdx.x;
  if (t >= n) return;
  const int64_t s = blockIdx.y;
  const T *vr = v + s * v_ser;
  T a = 0, b = 0;
  for (int l = 0; l < tp.L; ++l) {
    int64_t idx = t - tp.off[l];
    idx += idx < 0 ? n : 0;
    const T val = vr[idx];
    a = fma(tp.hi[l], val, a);
    b = fma(tp.lo[l], val, b);
  }
  w[s * w_ser + t] = a;
  vn[s * vn_ser + t] = b;
}

// ---- synthesis level: out[t] = sum_l hi[l] a[(t + off_l) mod n] + sum_l lo[l] b[(t + off_l) mod n] ---------------
// Row z = blockIdx.z of series s = blockIdx.y.  Row 0 reads a (when given); rows z >= zb read row z - zb of b's
// series (when given).  Accumulators as k_imodwt (acc_h, acc_g, then their sum); a row with one input keeps its
// accumulator as is, which is k_mra_blk's single accumulator.
template <typename T> struct SynthRows {
  const T *a;
  int64_t a_ser;
  const T *b;
  int64_t b_ser;
  int zb;
  T *out;  // row z of series s: out + s out_ser + z n
  int64_t out_ser;
};

template <typename T>
__global__ void __launch_bounds__(kLongThreads) k_synth_long(SynthRows<T> r, int n, LongTaps<T> tp) {
  const int64_t t = (int64_t)blockIdx.x * kLongThreads + threadIdx.x;
  if (t >= n) return;
  const int64_t s = blockIdx.y;
  const int z = blockIdx.z;
  const T *a = (r.a && z == 0) ? r.a + s * r.a_ser : nullptr;
  const T *b = (r.b && z >= r.zb) ? r.b + s * r.b_ser + (int64_t)(z - r.zb) * n : nullptr;
  T acc_h = 0, acc_g = 0;
  for (int l = 0; l < tp.L; ++l) {
    int64_t idx = t + tp.off[l];
    idx -= idx >= n ? n : 0;
    if (a) acc_h = fma(tp.hi[l], a[idx], acc_h);
    if (b) acc_g = fma(tp.lo[l], b[idx], acc_g);
  }
  r.out[s * r.out_ser + (int64_t)z * n + t] = (a && b) ? acc_h + acc_g : (a ? acc_h : acc_g);
}

// ---- DWT analysis level (symmetric): cA[i] = sum_j lo[j] a[sym(2i+1-j)], cD with hi (k_wavedec's order) ---------
// half-sample symmetric extension of reflect_sym, in 64-bit: 2i + 1 passes 2^31 for n close to it
__device__ __forceinline__ int64_t reflect_sym_long(int64_t p, int64_t n) {
  if (p >= 0 && p < n) return p;
  if (p < 0 && p >= -n) return -1 - p;
  if (p >= n && p < 2 * n) return 2 * n - 1 - p;
  const int64_t period = 2 * n;
  int64_t m = p % period;
  if (m < 0) m += period;
  return m >= n ? period - 1 - m : m;
}

template <typename T>
__global__ void __launch_bounds__(kLongThreads) k_dwt_long(const T *__restrict__ a, int64_t a_ser, int cur, int nout,
                                                           LongTaps<T> tp, T *__restrict__ cd, int64_t cd_ser,
                                                           T *__restrict__ ca, int64_t ca_ser) {
  const int64_t i = (int64_t)blockIdx.x * kLongThreads + threadIdx.x;
  if (i >= nout) return;
  const int64_t s = blockIdx.y;
  const T *ar = a + s * a_ser;
  T sa = 0, sd = 0;
  for (int j = 0; j < tp.L; ++j) {
    const T val = ar[reflect_sym_long(2 * i + 1 - j, cur)];
    sa += tp.lo[j] * val;
    sd += tp.hi[j] * val;
  }
  cd[s * cd_ser + i] = sd;
  ca[s * ca_ser + i] = sa;
}

// ---- DWT synthesis level: full[p] = sum_k lo[p-2k] a[k] + hi[p-2k] d[k], kept p in [L-2, L-2+nout) (k_waverec) ---
template <typename T>
__global__ void __launch_bounds__(kLongThreads) k_idwt_long(const T *__restrict__ a, int64_t a_ser,
                                                            const T *__restrict__ d, int64_t d_ser, int m, int nout,
                                                            LongTaps<T> tp, T *__restrict__ out, int64_t out_ser) {
  const int64_t o = (int64_t)blockIdx.x * kLongThreads + threadIdx.x;
  if (o >= nout) return;
  const int64_t s = blockIdx.y;
  const T *ar = a + s * a_ser, *dr = d + s * d_ser;
  const int L = tp.L;
  const int64_t nn = o + L - 2;
  int64_t k_lo = (nn - L + 2) / 2;  // ceil((nn-L+1)/2) for nn-L+1 >= -1
  if (nn - L + 1 < 0) k_lo = 0;
  const int64_t k_hi = nn / 2 < m - 1 ? nn / 2 : m - 1;
  T acc = 0;
  for (int64_t k = k_lo; k <= k_hi; ++k) {
    const int idx = (int)(nn - 2 * k);
    acc += tp.lo[idx] * ar[k] + tp.hi[idx] * dr[k];
  }
  out[s * out_ser + o] = acc;
}

// ---- MRA with explicit periodised filters: out[s,j,t] = sum over the non-zero taps (l, f) of row j, in increasing
// l, of f w[s,j,(t+l) mod n] (k_modwtmra without its +0 terms) -----------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kLongThreads) k_mra_filt_long(const T *__restrict__ w, int n, int rows,
                                                                const int *__restrict__ first,
                                                                const int *__restrict__ off,
                                                                const T *__restrict__ val, T *__restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * kLongThreads + threadIdx.x;
  if (t >= n) return;
  const int j = blockIdx.z;
  const int64_t base = ((int64_t)blockIdx.y * rows + j) * n;
  const T *row = w + base;
  T acc = 0;
  for (int k = first[j]; k < first[j + 1]; ++k) {
    int64_t idx = t + off[k];
    idx -= idx >= n ? n : 0;
    acc += val[k] * row[idx];
  }
  out[base + t] = acc;
}

// ---- host side -------------------------------------------------------------------------------------------------
template <typename T>
int modwt_long(const void *x, int64_t batch, int n, const Taps &taps, int J, int flags, void *out, cudaStream_t st) {
  const int64_t ser = (int64_t)(J + 1) * n;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)n, batch);
  const size_t b_buf = al256(sizeof(T) * (size_t)cap * n);
  T *buf[2] = {nullptr, nullptr};
  if (J > 1) {
    void *scratch = nullptr;
    WTB_TRY(arena_reserve(2 * b_buf, &scratch));
    buf[0] = (T *)scratch;
    buf[1] = (T *)((char *)scratch + b_buf);
  }
  return run_batched(x, out, batch, sizeof(T) * n, sizeof(T) * (size_t)ser, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         const T *xin = (const T *)di + b0 * n;
                         T *o = (T *)dout + b0 * ser;
                         // level j reads v_{j-1} (x, then buf[(j-1)&1]) and writes v_j to buf[j&1], v_J to row J
                         for (int j = 1; j <= J; ++j) {
                           const T *src = j == 1 ? xin : buf[(j - 1) & 1];
                           T *dst = j == J ? o + (int64_t)J * n : buf[j & 1];
                           k_modwt_long<T><<<long_grid(n, nw), kLongThreads, 0, st>>>(
                               src, n, n, long_taps<T>(taps, j, n), o + (int64_t)(j - 1) * n, ser, dst,
                               j == J ? ser : n);
                           WTB_LAUNCH_CHECK();
                         }
                       }
                       return WTB_OK;
                     });
}

template <typename T>
int imodwt_long(const void *w, int64_t batch, int n, const Taps &taps, int J, int flags, void *out, cudaStream_t st) {
  const int64_t ser = (int64_t)(J + 1) * n;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)n, batch);
  const size_t b_buf = al256(sizeof(T) * (size_t)cap * n);
  T *buf[2] = {nullptr, nullptr};
  if (J > 1) {
    void *scratch = nullptr;
    WTB_TRY(arena_reserve(2 * b_buf, &scratch));
    buf[0] = (T *)scratch;
    buf[1] = (T *)((char *)scratch + b_buf);
  }
  return run_batched(w, out, batch, sizeof(T) * (size_t)ser, sizeof(T) * n, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         const T *wi = (const T *)di + b0 * ser;
                         // level j reads v_j (row J, then buf[(j+1)&1]) and writes v_{j-1} to buf[j&1], x at j = 1
                         for (int j = J; j >= 1; --j) {
                           SynthRows<T> r;
                           r.a = wi + (int64_t)(j - 1) * n;
                           r.a_ser = ser;
                           r.b = j == J ? wi + (int64_t)J * n : buf[(j + 1) & 1];
                           r.b_ser = j == J ? ser : n;
                           r.zb = 0;
                           r.out = j == 1 ? (T *)dout + b0 * n : buf[j & 1];
                           r.out_ser = n;
                           k_synth_long<T><<<long_grid(n, nw), kLongThreads, 0, st>>>(r, n, long_taps<T>(taps, j, n));
                           WTB_LAUNCH_CHECK();
                         }
                       }
                       return WTB_OK;
                     });
}

// D_j = G_1' .. G_{j-1}' H_j' w_j and S_J = G_1' .. G_J' v_J, level k = J .. 1 in one launch each: row k-1 enters
// through H_k' from w_{k}; rows k .. J apply G_k' to their intermediates (S_J enters from v_J at k = J).
template <typename T>
int mra_taps_long(const void *w, int64_t batch, int n, const Taps &taps, int J, int flags, void *out,
                  cudaStream_t st) {
  const int64_t ser = (int64_t)(J + 1) * n;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)ser, batch);
  const size_t b_buf = al256(sizeof(T) * (size_t)(cap * ser));
  T *buf[2] = {nullptr, nullptr};
  if (J > 1) {
    void *scratch = nullptr;
    WTB_TRY(arena_reserve(2 * b_buf, &scratch));
    buf[0] = (T *)scratch;
    buf[1] = (T *)((char *)scratch + b_buf);
  }
  return run_batched(w, out, batch, sizeof(T) * (size_t)ser, sizeof(T) * (size_t)ser, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         const T *wi = (const T *)di + b0 * ser;
                         // level k writes rows k-1 .. J to buf[k&1] (the output at k = 1) in the [J+1, n] layout
                         for (int k = J; k >= 1; --k) {
                           SynthRows<T> r;
                           r.a = wi + (int64_t)(k - 1) * n;
                           r.a_ser = ser;
                           r.b = k == J ? wi + (int64_t)J * n : buf[(k + 1) & 1] + (int64_t)k * n;
                           r.b_ser = ser;
                           r.zb = 1;
                           r.out = (k == 1 ? (T *)dout + b0 * ser : buf[k & 1]) + (int64_t)(k - 1) * n;
                           r.out_ser = ser;
                           k_synth_long<T><<<long_grid(n, nw, J - k + 2), kLongThreads, 0, st>>>(
                               r, n, long_taps<T>(taps, k, n));
                           WTB_LAUNCH_CHECK();
                         }
                       }
                       return WTB_OK;
                     });
}

template <typename T>
int mra_filt_long(const void *w, int64_t batch, int n, const double *filt, int J, int flags, void *out,
                  cudaStream_t st) {
  // (offset, value) of each row's non-zero taps in increasing offset; for finite input the skipped taps add +0
  std::vector<int> first(J + 2, 0), off;
  std::vector<T> val;
  for (int j = 0; j <= J; ++j) {
    for (int l = 0; l < n; ++l) {
      const double f = filt[(size_t)j * n + l];
      if (f != 0.0) {
        off.push_back(l);
        val.push_back(T(f));
      }
    }
    first[j + 1] = (int)off.size();
  }
  const size_t nnz = std::max<size_t>(1, off.size());
  const size_t b_first = al256(sizeof(int) * (J + 2)), b_off = al256(sizeof(int) * nnz);
  void *scratch = nullptr;
  WTB_TRY(arena_reserve(b_first + b_off + sizeof(T) * nnz, &scratch));
  int *d_first = (int *)scratch, *d_off = (int *)((char *)scratch + b_first);
  T *d_val = (T *)((char *)scratch + b_first + b_off);
  WTB_CUDA(cudaMemcpyAsync(d_first, first.data(), sizeof(int) * (J + 2), cudaMemcpyHostToDevice, st));
  if (!off.empty()) {
    WTB_CUDA(cudaMemcpyAsync(d_off, off.data(), sizeof(int) * off.size(), cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaMemcpyAsync(d_val, val.data(), sizeof(T) * val.size(), cudaMemcpyHostToDevice, st));
  }
  WTB_CUDA(cudaStreamSynchronize(st));  // the tables are locals
  const int64_t ser = (int64_t)(J + 1) * n;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)ser, batch);
  return run_batched(w, out, batch, sizeof(T) * (size_t)ser, sizeof(T) * (size_t)ser, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         k_mra_filt_long<T><<<long_grid(n, nw, J + 1), kLongThreads, 0, st>>>(
                             (const T *)di + b0 * ser, n, J + 1, d_first, d_off, d_val, (T *)dout + b0 * ser);
                         WTB_LAUNCH_CHECK();
                       }
                       return WTB_OK;
                     });
}

template <typename T>
int wavedec_long(const void *x, int64_t batch, const LevelPlan &plan, const Taps &taps, int flags, void *coeffs,
                 cudaStream_t st) {
  const int n = plan.n;
  const int64_t total = plan.total;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)n, batch);
  const int64_t mid = plan.level > 0 ? plan.len[plan.level] : 0;  // cA_1, the longest intermediate
  const size_t b_buf = al256(sizeof(T) * (size_t)(cap * mid));
  T *buf[2] = {nullptr, nullptr};
  if (plan.level > 1) {
    void *scratch = nullptr;
    WTB_TRY(arena_reserve(2 * b_buf, &scratch));
    buf[0] = (T *)scratch;
    buf[1] = (T *)((char *)scratch + b_buf);
  }
  return run_batched(x, coeffs, batch, sizeof(T) * n, sizeof(T) * (size_t)total, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       if (plan.level == 0) {  // cA_0 is the signal
                         WTB_CUDA(cudaMemcpyAsync(dout, di, sizeof(T) * (size_t)(nb * n), cudaMemcpyDeviceToDevice, st));
                         return WTB_OK;
                       }
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         T *o = (T *)dout + b0 * total;
                         int cur = n;
                         // level lev reads cA_{lev-1} (x, then buf[(lev-1)&1]) and writes cA_lev to buf[lev&1],
                         // cA_L to slot 0
                         for (int lev = 1; lev <= plan.level; ++lev) {
                           const int slot = plan.level - lev + 1;  // cD_lev
                           const int nout = plan.len[slot];
                           const bool last = lev == plan.level;
                           const T *src = lev == 1 ? (const T *)di + b0 * n : buf[(lev - 1) & 1];
                           k_dwt_long<T><<<long_grid(nout, nw), kLongThreads, 0, st>>>(
                               src, lev == 1 ? n : mid, cur, nout, long_taps<T>(taps, 0, 1), o + plan.off[slot], total,
                               last ? o : buf[lev & 1], last ? total : mid);
                           WTB_LAUNCH_CHECK();
                           cur = nout;
                         }
                       }
                       return WTB_OK;
                     });
}

template <typename T>
int waverec_long(const void *coeffs, int64_t batch, const LevelPlan &plan, const Taps &taps, int flags, void *x,
                 cudaStream_t st) {
  const int nout = plan.n;
  const int64_t total = plan.total;
  const int64_t cap = long_wave(2 * sizeof(T) * (size_t)nout, batch);
  int64_t mid = 0;  // longest intermediate approximation
  for (int slot = 1; slot < plan.level; ++slot) mid = std::max<int64_t>(mid, 2 * (int64_t)plan.len[slot] - taps.L + 2);
  const size_t b_buf = al256(sizeof(T) * (size_t)(cap * mid));
  T *buf[2] = {nullptr, nullptr};
  if (plan.level > 1) {
    void *scratch = nullptr;
    WTB_TRY(arena_reserve(2 * b_buf, &scratch));
    buf[0] = (T *)scratch;
    buf[1] = (T *)((char *)scratch + b_buf);
  }
  return run_batched(coeffs, x, batch, sizeof(T) * (size_t)total, sizeof(T) * (size_t)nout, flags, st,
                     [&](const void *di, void *dout, int64_t nb) -> int {
                       if (plan.level == 0) {  // the signal is cA_0
                         WTB_CUDA(cudaMemcpyAsync(dout, di, sizeof(T) * (size_t)(nb * nout), cudaMemcpyDeviceToDevice, st));
                         return WTB_OK;
                       }
                       for (int64_t b0 = 0; b0 < nb; b0 += cap) {
                         const int64_t nw = std::min(cap, nb - b0);
                         const T *c = (const T *)di + b0 * total;
                         // slot s reads cA (slot 0, then buf[(s-1)&1]) and cD (slot s) and writes buf[s&1], x last
                         for (int slot = 1; slot <= plan.level; ++slot) {
                           const int m = plan.len[slot];
                           const int len = 2 * m - taps.L + 2;
                           const bool last = slot == plan.level;
                           k_idwt_long<T><<<long_grid(len, nw), kLongThreads, 0, st>>>(
                               slot == 1 ? c : buf[(slot - 1) & 1], slot == 1 ? total : mid, c + plan.off[slot], total,
                               m, len, long_taps<T>(taps, 0, 1), last ? (T *)dout + b0 * nout : buf[slot & 1],
                               last ? nout : mid);
                           WTB_LAUNCH_CHECK();
                         }
                       }
                       return WTB_OK;
                     });
}

#define WTB_INSTANTIATE(T)                                                                                         \
  template int modwt_long<T>(const void *, int64_t, int, const Taps &, int, int, void *, cudaStream_t);            \
  template int imodwt_long<T>(const void *, int64_t, int, const Taps &, int, int, void *, cudaStream_t);           \
  template int mra_taps_long<T>(const void *, int64_t, int, const Taps &, int, int, void *, cudaStream_t);         \
  template int mra_filt_long<T>(const void *, int64_t, int, const double *, int, int, void *, cudaStream_t);       \
  template int wavedec_long<T>(const void *, int64_t, const LevelPlan &, const Taps &, int, void *, cudaStream_t); \
  template int waverec_long<T>(const void *, int64_t, const LevelPlan &, const Taps &, int, void *, cudaStream_t);
WTB_INSTANTIATE(float)
WTB_INSTANTIATE(double)

}  // namespace wtb
