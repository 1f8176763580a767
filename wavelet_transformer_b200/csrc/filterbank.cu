// MODWT (reference src/modwt.py:86-194, own arithmetic) and decimated DWT
// (pywt.wavedec / pywt.waverec, mode='symmetric') filterbank kernels.
//
// One CTA owns one series.  The row is staged into shared memory with a 1-D TMA
// bulk copy (cp.async.bulk + mbarrier) when it is 16-byte aligned, all pyramid
// levels run out of shared memory, and only coefficients leave the SM.  These
// paths are HBM-bound: bytes in = N, bytes out = (J+1) N per series.  A shape whose generic kernel would need more
// than kSmemLimit of shared memory, its static tables included, runs level by level instead (filterbank_long.cu);
// each *_impl decides that from the shape before any launch.
#include "filterbank_common.cuh"

namespace wtb {

// Filter taps (in precision T) and the per-level circular offsets (2^(j-1) l) mod N live in
// shared memory: the inner loops are then one LDS + compare + 2 FMA per tap, with no
// integer division and no double->T conversion.
template <typename T> struct TapSmem {
  T lo[kMaxTaps];
  T hi[kMaxTaps];
  int off[kMaxTaps];
};

template <typename T>
__device__ __forceinline__ void load_taps(TapSmem<T> &ts, const Taps &taps) {
  if (threadIdx.x < taps.L) {
    ts.lo[threadIdx.x] = T(taps.lo[threadIdx.x]);
    ts.hi[threadIdx.x] = T(taps.hi[threadIdx.x]);
  }
}
// call with all threads; ends with a barrier
template <typename T>
__device__ __forceinline__ void set_offsets(TapSmem<T> &ts, int L, int j, int n) {
  if (threadIdx.x < L) ts.off[threadIdx.x] = (int)(((1LL << (j - 1)) * threadIdx.x) % n);
  __syncthreads();
}

// ---- MODWT analysis: w_j[t] = sum_l h[l] v[(t - 2^(j-1) l) mod N] ---------------------
// LT: compile-time tap count (0 = runtime taps.L)
template <typename T, int LT>
__global__ void k_modwt(const T *__restrict__ x, int n, int J, Taps taps, T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ TapSmem<T> ts;
  T *v = reinterpret_cast<T *>(smem_raw);
  T *vn = v + ((n + 3) & ~3);
  const int64_t b = blockIdx.x;
  const int L = LT ? LT : taps.L;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  load_taps(ts, taps);
  __syncthreads();
  uint32_t phase = 0;
  stage_row<T>(v, x + b * n, n, &bar, phase);
  T *o = out + b * (int64_t)(J + 1) * n;
  for (int j = 1; j <= J; ++j) {
    set_offsets(ts, L, j, n);
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      T w = 0, s = 0;
#pragma unroll
      for (int l = 0; l < L; ++l) {
        int idx = t - ts.off[l];
        idx += idx < 0 ? n : 0;
        const T val = v[idx];
        w = fma(ts.hi[l], val, w);
        s = fma(ts.lo[l], val, s);
      }
      o[(int64_t)(j - 1) * n + t] = w;
      vn[t] = s;
    }
    __syncthreads();
    T *tmp = v; v = vn; vn = tmp;
  }
  for (int t = threadIdx.x; t < n; t += blockDim.x) o[(int64_t)J * n + t] = v[t];
}

// ---- MODWT synthesis: v_{j-1}[t] = sum_l h[l] w_j[(t+2^(j-1) l) mod N] + g[l] v_j[...] ---
template <typename T, int LT>
__global__ void k_imodwt(const T *__restrict__ w, int n, int J, Taps taps, T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ TapSmem<T> ts;
  const int np = (n + 3) & ~3;
  T *v = reinterpret_cast<T *>(smem_raw);
  T *vn = v + np;
  T *wj = vn + np;
  const int64_t b = blockIdx.x;
  const int L = LT ? LT : taps.L;
  const T *wb = w + b * (int64_t)(J + 1) * n;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  load_taps(ts, taps);
  __syncthreads();
  uint32_t phase = 0;
  stage_row<T>(v, wb + (int64_t)J * n, n, &bar, phase);
  for (int j = J; j >= 1; --j) {
    stage_row<T>(wj, wb + (int64_t)(j - 1) * n, n, &bar, phase);
    set_offsets(ts, L, j, n);
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      T acc_h = 0, acc_g = 0;
#pragma unroll
      for (int l = 0; l < L; ++l) {
        int idx = t + ts.off[l];
        idx -= idx >= n ? n : 0;
        acc_h = fma(ts.hi[l], wj[idx], acc_h);
        acc_g = fma(ts.lo[l], v[idx], acc_g);
      }
      vn[t] = acc_h + acc_g;
    }
    __syncthreads();
    T *tmp = v; v = vn; vn = tmp;
  }
  for (int t = threadIdx.x; t < n; t += blockDim.x) out[b * n + t] = v[t];
}

// ---- MODWT MRA: out[b,j,t] = sum_{l<len_j} filt[j,l] w[b,j,(t+l) mod N] --------------
template <typename T>
__global__ void k_modwtmra(const T *__restrict__ w, int n, int J, const double *__restrict__ filt,
                           const int *__restrict__ flen, T *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int np = (n + 3) & ~3;
  T *row = reinterpret_cast<T *>(smem_raw);
  T *f = row + np;
  const int64_t b = blockIdx.x / (J + 1);
  const int j = blockIdx.x % (J + 1);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t phase = 0;
  const int len = flen[j];
  for (int l = threadIdx.x; l < len; l += blockDim.x) f[l] = T(filt[(int64_t)j * n + l]);
  stage_row<T>(row, w + (b * (J + 1) + j) * (int64_t)n, n, &bar, phase);
  __syncthreads();
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    T acc = 0;
    int idx = t;
    for (int l = 0; l < len; ++l) {
      acc += f[l] * row[idx];
      if (++idx == n) idx = 0;
    }
    out[(b * (J + 1) + j) * (int64_t)n + t] = acc;
  }
}

// ---- DWT (symmetric) ---------------------------------------------------------------------
// cA[i] = sum_j lo[j] xe[2i+1-j]; cD with hi.  cA stays in smem for the next level.
template <typename T>
__global__ void k_wavedec(const T *__restrict__ x, LevelPlan plan, Taps taps, T *__restrict__ coeffs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  T *a = reinterpret_cast<T *>(smem_raw);
  T *an = a + plan.buf;
  const int64_t b = blockIdx.x;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t phase = 0;
  stage_row<T>(a, x + b * (int64_t)plan.n, plan.n, &bar, phase);
  T *o = coeffs + b * (int64_t)plan.total;
  int cur = plan.n;
  for (int lev = 1; lev <= plan.level; ++lev) {
    const int slot = plan.level - lev + 1;  // cD_lev
    const int nout = plan.len[slot];
    T *od = o + plan.off[slot];
    for (int i = threadIdx.x; i < nout; i += blockDim.x) {
      T ca = 0, cd = 0;
      for (int j = 0; j < taps.L; ++j) {
        const T val = a[reflect_sym(2 * i + 1 - j, cur)];
        ca += T(taps.lo[j]) * val;
        cd += T(taps.hi[j]) * val;
      }
      od[i] = cd;
      an[i] = ca;
    }
    __syncthreads();
    T *tmp = a; a = an; an = tmp;
    cur = nout;
  }
  for (int i = threadIdx.x; i < cur; i += blockDim.x) o[i] = a[i];
}

// a <- idwt(a, d): full[n] = sum_k lo[n-2k] a[k] + hi[n-2k] d[k]; keep full[L-2 : L-2+2m-L+2]
template <typename T>
__global__ void k_waverec(const T *__restrict__ coeffs, LevelPlan plan, Taps taps, T *__restrict__ x) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T *a = reinterpret_cast<T *>(smem_raw);
  T *an = a + plan.buf;
  const int64_t b = blockIdx.x;
  const T *c = coeffs + b * (int64_t)plan.total;
  int cur = plan.len[0];
  for (int i = threadIdx.x; i < cur; i += blockDim.x) a[i] = c[i];
  __syncthreads();
  const int L = taps.L;
  for (int slot = 1; slot <= plan.level; ++slot) {
    const int m = plan.len[slot];  // == cur or cur-1 (pywt drops the extra approximation sample)
    const T *d = c + plan.off[slot];
    const int nout = 2 * m - L + 2;
    for (int o = threadIdx.x; o < nout; o += blockDim.x) {
      const int nn = o + L - 2;
      int k_lo = (nn - L + 2) / 2;  // ceil((nn-L+1)/2) for nn-L+1 >= -1
      if (nn - L + 1 < 0) k_lo = 0;
      int k_hi = nn / 2;
      if (k_hi > m - 1) k_hi = m - 1;
      T acc = 0;
      for (int k = k_lo; k <= k_hi; ++k) {
        const int idx = nn - 2 * k;
        acc += T(taps.lo[idx]) * a[k] + T(taps.hi[idx]) * d[k];
      }
      an[o] = acc;
    }
    __syncthreads();
    T *tmp = a; a = an; an = tmp;
    cur = nout;
  }
  for (int i = threadIdx.x; i < cur; i += blockDim.x) x[b * (int64_t)plan.n + i] = a[i];
}

// ---- host side -----------------------------------------------------------------------------
int make_taps(const double *lo, const double *hi, int L, double scale, Taps *t) {
  WTB_REQUIRE(lo && hi && L >= 2 && L <= kMaxTaps, WTB_EUNSUPPORTED, "filter length %d outside [2,%d]", L, kMaxTaps);
  t->L = L;
  for (int i = 0; i < L; ++i) {
    t->lo[i] = lo[i] * scale;
    t->hi[i] = hi[i] * scale;
  }
  return WTB_OK;
}

static int threads_for(int n) { return n >= 2048 ? 512 : (n >= 512 ? 256 : 128); }

enum class FbPath { kBlocked, kGeneric, kLong };
struct FbPlan { FbPath path; BlkShape cta; };  // cta: the launch of the chosen one-CTA kernel

// The kernels for a call of `op` on series of n samples (DWT: of *dwt, whose buf it sets), from the shape alone:
// kBlocked (filterbank_fast.cu) where blk_shape covers the shape, unless WTB_GENERIC_ONLY; else kGeneric, the
// one-CTA kernel `generic` (for the MRA from taps: k_modwtmra with the host-built equivalent filters), if it fits
// kSmemLimit with its static shared memory; else kLong (filterbank_long.cu).  The blocked kernels are asked only
// where `generic` fits, except for the MRA from taps, whose cascade kernel keeps every shape it covers.
template <typename T, typename K>
static int fb_plan(FbOp op, K generic, int n, int L, int J, LevelPlan *dwt, int flags, FbPlan *p) {
  int buf = (n + 3) & ~3;  // generic kernels: two ping-pong buffers, three for the inverse MODWT
  if (op == FbOp::kWaverec) {
    int longest = n;
    for (int i = 0; i <= dwt->level; ++i) longest = std::max(longest, dwt->len[i]);
    buf = (longest + L + 3) & ~3;
  }
  const size_t smem = sizeof(T) * (op == FbOp::kImodwt ? 3 : 2) * (size_t)buf;
  bool fits;
  WTB_TRY(fits_one_cta(generic, smem, &fits));
  const bool ask = !(flags & WTB_GENERIC_ONLY) && (fits || op == FbOp::kMraTaps);
  const BlkShape blk = ask ? blk_shape(op, n, L, J, dwt, sizeof(T)) : BlkShape{};
  *p = {FbPath::kGeneric, {threads_for(n), smem, 0, buf}};
  if (blk.threads)
    *p = {FbPath::kBlocked, blk};
  else if (!fits)
    p->path = FbPath::kLong;
  if (dwt) dwt->buf = p->cta.buf;
  return WTB_OK;
}

template <typename T>
static int modwt_impl(const void *x, int64_t batch, int n, const Taps &taps, int J, int flags, void *out,
                      cudaStream_t st) {
  auto kern = taps.L == 8 ? k_modwt<T, 8> : taps.L == 4 ? k_modwt<T, 4> : taps.L == 2 ? k_modwt<T, 2> : k_modwt<T, 0>;
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kModwt, kern, n, taps.L, J, nullptr, flags, &p));
  if (p.path == FbPath::kLong) return modwt_long<T>(x, batch, n, taps, J, flags, out, st);
  if (p.path == FbPath::kGeneric) WTB_TRY(set_smem(kern, p.cta.smem));
  const size_t in_row = sizeof(T) * n, out_row = sizeof(T) * (size_t)(J + 1) * n;
  return stage_rows(batch, host_rows(batch, in_row + out_row, flags), flags, st, {{x, in_row}}, {{out, out_row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
                      if (p.path == FbPath::kBlocked) return modwt_fast<T>(p.cta, di[0], nb, n, taps, J, dout[0], st);
                      kern<<<(unsigned)nb, p.cta.threads, p.cta.smem, st>>>((const T *)di[0], n, J, taps, (T *)dout[0]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

template <typename T>
int modwt_device(const T *x, int64_t batch, int n, const Taps &taps, int J, int flags, T *out, cudaStream_t st) {
  return modwt_impl<T>(x, batch, n, taps, J, flags | WTB_DEVICE_PTRS, out, st);
}
template int modwt_device<float>(const float *, int64_t, int, const Taps &, int, int, float *, cudaStream_t);
template int modwt_device<double>(const double *, int64_t, int, const Taps &, int, int, double *, cudaStream_t);

template <typename T>
static int imodwt_impl(const void *w, int64_t batch, int n, const Taps &taps, int J, int flags, void *out,
                       cudaStream_t st) {
  auto kern = taps.L == 8 ? k_imodwt<T, 8> : taps.L == 4 ? k_imodwt<T, 4> : taps.L == 2 ? k_imodwt<T, 2> : k_imodwt<T, 0>;
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kImodwt, kern, n, taps.L, J, nullptr, flags, &p));
  if (p.path == FbPath::kLong) return imodwt_long<T>(w, batch, n, taps, J, flags, out, st);
  if (p.path == FbPath::kGeneric) WTB_TRY(set_smem(kern, p.cta.smem));
  const size_t in_row = sizeof(T) * (size_t)(J + 1) * n, out_row = sizeof(T) * n;
  return stage_rows(batch, host_rows(batch, in_row + out_row, flags), flags, st, {{w, in_row}}, {{out, out_row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
                      if (p.path == FbPath::kBlocked) return imodwt_fast<T>(p.cta, di[0], nb, n, taps, J, dout[0], st);
                      kern<<<(unsigned)nb, p.cta.threads, p.cta.smem, st>>>((const T *)di[0], n, J, taps, (T *)dout[0]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

// k_modwtmra over the batch with the periodised filters filt [J+1, n] (host), on a kGeneric plan
template <typename T>
static int mra_generic(const FbPlan &p, const void *w, int64_t batch, int n, const double *filt, int J, int flags,
                       void *out, cudaStream_t st) {
  WTB_TRY(set_smem(k_modwtmra<T>, p.cta.smem));
  // effective filter length per level (trailing zeros of the periodised filter are skipped)
  std::vector<int> flen(J + 1);
  for (int j = 0; j <= J; ++j) {
    int len = n;
    while (len > 0 && filt[(size_t)j * n + len - 1] == 0.0) --len;
    flen[j] = len;
  }
  void *scratch = nullptr;
  const size_t b_f = align256(sizeof(double) * (size_t)(J + 1) * n);
  WTB_TRY(arena_reserve(b_f + sizeof(int) * (J + 1), &scratch));
  double *d_filt = (double *)scratch;
  int *d_flen = (int *)((char *)scratch + b_f);
  WTB_CUDA(cudaMemcpyAsync(d_filt, filt, sizeof(double) * (size_t)(J + 1) * n, cudaMemcpyHostToDevice, st));
  WTB_CUDA(cudaMemcpyAsync(d_flen, flen.data(), sizeof(int) * (J + 1), cudaMemcpyHostToDevice, st));
  WTB_CUDA(cudaStreamSynchronize(st));  // flen is a local
  const size_t row = sizeof(T) * (size_t)(J + 1) * n;
  return stage_rows(batch, host_rows(batch, 2 * row, flags), flags, st, {{w, row}}, {{out, row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
    WTB_REQUIRE(nb * (J + 1) < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
    k_modwtmra<T><<<(unsigned)(nb * (J + 1)), p.cta.threads, p.cta.smem, st>>>((const T *)di[0], n, J, d_filt, d_flen,
                                                                               (T *)dout[0]);
    WTB_LAUNCH_CHECK();
    return WTB_OK;
  });
}

template <typename T>
static int mra_impl(const void *w, int64_t batch, int n, const double *filt, int J, int flags, void *out,
                    cudaStream_t st) {
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kMra, k_modwtmra<T>, n, 0, J, nullptr, flags, &p));
  if (p.path == FbPath::kLong) return mra_filt_long<T>(w, batch, n, filt, J, flags, out, st);
  return mra_generic<T>(p, w, batch, n, filt, J, flags, out, st);
}

// Periodised equivalent filters [h_1 .. h_J, g_J] of the reference's modwtmra
// (src/modwt.py:56-83, 172-193) from the UNSCALED taps g = dec_lo, h = dec_hi.
static void equivalent_filters(const double *g, const double *h, int L, int J, int n, std::vector<double> *filt) {
  auto dilate = [&](const double *taps, int j) {  // upArrow_op: 2^(j-1)-1 zeros between taps; j == 0 -> [1]
    if (j == 0) return std::vector<double>{1.0};
    const size_t step = size_t(1) << (j - 1);
    std::vector<double> out(step * (L - 1) + 1, 0.0);
    for (int l = 0; l < L; ++l) out[step * l] = taps[l];
    return out;
  };
  auto conv = [](const std::vector<double> &a, const std::vector<double> &b) {
    std::vector<double> out(a.size() + b.size() - 1, 0.0);
    for (size_t i = 0; i < a.size(); ++i)
      for (size_t k = 0; k < b.size(); ++k) out[i + k] += a[i] * b[k];
    return out;
  };
  filt->assign((size_t)(J + 1) * n, 0.0);
  auto fold = [&](const std::vector<double> &f, double scale, int row) {  // period_list
    for (size_t i = 0; i < f.size(); ++i) (*filt)[(size_t)row * n + i % n] += f[i] * scale;
  };
  std::vector<double> g_part{1.0};
  for (int j = 0; j < J; ++j) {
    g_part = conv(g_part, dilate(g, j));
    if (j == 0)
      fold(std::vector<double>(h, h + L), 1.0 / std::sqrt(2.0), 0);
    else
      fold(conv(g_part, dilate(h, j + 1)), std::pow(2.0, -(j + 1) / 2.0), j);
  }
  fold(conv(g_part, dilate(g, J)), std::pow(2.0, -J / 2.0), J);
}

template <typename T>
static int mra_taps_impl(const void *w, int64_t batch, int n, const Taps &taps, const double *g, const double *h,
                         int J, int flags, void *out, cudaStream_t st) {
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kMraTaps, k_modwtmra<T>, n, taps.L, J, nullptr, flags, &p));
  if (p.path == FbPath::kLong) return mra_taps_long<T>(w, batch, n, taps, J, flags, out, st);
  if (p.path == FbPath::kGeneric) {  // shape outside the cascade kernel: correlate with the periodised filters
    std::vector<double> filt;
    equivalent_filters(g, h, taps.L, J, n, &filt);
    return mra_generic<T>(p, w, batch, n, filt.data(), J, flags, out, st);
  }
  const size_t row = sizeof(T) * (size_t)(J + 1) * n;
  return stage_rows(batch, host_rows(batch, 2 * row, flags), flags, st, {{w, row}}, {{out, row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
    WTB_REQUIRE(nb * (J + 1) < (1LL << 31), WTB_EUNSUPPORTED, "batch too large");
    return mra_fast<T>(p.cta, di[0], nb, n, taps, J, dout[0], st);
  });
}

static int make_plan(int n, int L, int level, const int *lens_in, LevelPlan *p) {
  WTB_REQUIRE(level >= 0 && level <= kMaxLevels, WTB_EUNSUPPORTED, "level %d outside [0,%d]", level, kMaxLevels);
  p->level = level;
  p->n = n;
  if (lens_in) {
    for (int i = 0; i <= level; ++i) p->len[i] = lens_in[i];
  } else {
    WTB_TRY(wtb_dwt_coeff_lens(n, L, level, p->len));
  }
  int off = 0;
  for (int i = 0; i <= level; ++i) {
    WTB_REQUIRE(p->len[i] > 0, WTB_EINVAL, "empty coefficient block %d", i);
    p->off[i] = off;
    off += p->len[i];
  }
  p->total = off;
  return WTB_OK;
}

template <typename T>
static int wavedec_impl(const void *x, int64_t batch, int n, const Taps &taps, int level, int flags,
                        void *coeffs, cudaStream_t st) {
  LevelPlan plan;
  WTB_TRY(make_plan(n, taps.L, level, nullptr, &plan));
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kWavedec, k_wavedec<T>, n, taps.L, level, &plan, flags, &p));
  if (p.path == FbPath::kLong) return wavedec_long<T>(x, batch, plan, taps, flags, coeffs, st);
  if (p.path == FbPath::kGeneric) WTB_TRY(set_smem(k_wavedec<T>, p.cta.smem));
  const size_t in_row = sizeof(T) * n, out_row = sizeof(T) * (size_t)plan.total;
  return stage_rows(batch, host_rows(batch, in_row + out_row, flags), flags, st, {{x, in_row}}, {{coeffs, out_row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
                      if (p.path == FbPath::kBlocked) return wavedec_fast<T>(p.cta, di[0], nb, plan, taps, dout[0], st);
                      k_wavedec<T><<<(unsigned)nb, p.cta.threads, p.cta.smem, st>>>((const T *)di[0], plan, taps,
                                                                                   (T *)dout[0]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

template <typename T>
static int waverec_impl(const void *coeffs, int64_t batch, const int *lens, int level, const Taps &taps,
                        int flags, void *x, cudaStream_t st) {
  const int nout = wtb_waverec_len(lens, level, taps.L);
  if (nout < 0) return nout;
  LevelPlan plan;
  WTB_TRY(make_plan(nout, taps.L, level, lens, &plan));
  FbPlan p;
  WTB_TRY(fb_plan<T>(FbOp::kWaverec, k_waverec<T>, nout, taps.L, level, &plan, flags, &p));
  if (p.path == FbPath::kLong) return waverec_long<T>(coeffs, batch, plan, taps, flags, x, st);
  if (p.path == FbPath::kGeneric) WTB_TRY(set_smem(k_waverec<T>, p.cta.smem));
  const size_t in_row = sizeof(T) * (size_t)plan.total, out_row = sizeof(T) * (size_t)nout;
  return stage_rows(batch, host_rows(batch, in_row + out_row, flags), flags, st, {{coeffs, in_row}}, {{x, out_row}}, 0,
                    [&](const void *const *di, void *const *dout, void *, int64_t, int64_t nb) -> int {
                      if (p.path == FbPath::kBlocked) return waverec_fast<T>(p.cta, di[0], nb, plan, taps, dout[0], st);
                      k_waverec<T><<<(unsigned)nb, p.cta.threads, p.cta.smem, st>>>((const T *)di[0], plan, taps,
                                                                                   (T *)dout[0]);
                      WTB_LAUNCH_CHECK();
                      return WTB_OK;
                    });
}

}  // namespace wtb

using namespace wtb;

#define DISPATCH(fn, ...) ((flags & WTB_F64) ? fn<double>(__VA_ARGS__) : fn<float>(__VA_ARGS__))

extern "C" int wtb_modwt(const void *x, int64_t batch, int n, const double *g, const double *h, int L,
                         int J, int flags, void *w_out, void *stream) {
  WTB_REQUIRE(x && w_out && batch >= 0 && n > 0 && J >= 1 && J < 31, WTB_EINVAL, "wtb_modwt: bad arguments");
  Taps taps;
  WTB_TRY(make_taps(g, h, L, 1.0 / std::sqrt(2.0), &taps));
  WTB_ENTER(flags, x, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    return DISPATCH(modwt_impl, (const char *)x + first * e * n, nb, n, taps, J, flags,
                    (char *)w_out + first * e * (J + 1) * n, st);
  });
}

extern "C" int wtb_imodwt(const void *w, int64_t batch, int n, const double *g, const double *h, int L,
                          int J, int flags, void *x_out, void *stream) {
  WTB_REQUIRE(w && x_out && batch >= 0 && n > 0 && J >= 1 && J < 31, WTB_EINVAL, "wtb_imodwt: bad arguments");
  Taps taps;
  WTB_TRY(make_taps(g, h, L, 1.0 / std::sqrt(2.0), &taps));
  WTB_ENTER(flags, w, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    return DISPATCH(imodwt_impl, (const char *)w + first * e * (J + 1) * n, nb, n, taps, J, flags,
                    (char *)x_out + first * e * n, st);
  });
}

extern "C" int wtb_modwtmra(const void *w, int64_t batch, int n, const double *filt, int J, int flags,
                            void *out, void *stream) {
  WTB_REQUIRE(w && out && filt && batch >= 0 && n > 0 && J >= 1, WTB_EINVAL, "wtb_modwtmra: bad arguments");
  WTB_ENTER(flags, w, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    const size_t at = first * e * (J + 1) * n;
    return DISPATCH(mra_impl, (const char *)w + at, nb, n, filt, J, flags, (char *)out + at, st);
  });
}

extern "C" int wtb_modwtmra_taps(const void *w, int64_t batch, int n, const double *g, const double *h, int L,
                                 int J, int flags, void *out, void *stream) {
  WTB_REQUIRE(w && out && batch >= 0 && n > 0 && J >= 1 && J < 31, WTB_EINVAL, "wtb_modwtmra_taps: bad arguments");
  Taps taps;
  WTB_TRY(make_taps(g, h, L, 1.0 / std::sqrt(2.0), &taps));
  WTB_ENTER(flags, w, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    const size_t at = first * e * (J + 1) * n;
    return DISPATCH(mra_taps_impl, (const char *)w + at, nb, n, taps, g, h, J, flags, (char *)out + at, st);
  });
}

extern "C" int wtb_wavedec(const void *x, int64_t batch, int n, const double *dec_lo, const double *dec_hi,
                           int L, int level, int flags, void *coeffs, void *stream) {
  WTB_REQUIRE(x && coeffs && batch >= 0 && n > 0 && level >= 0, WTB_EINVAL, "wtb_wavedec: bad arguments");
  Taps taps;
  WTB_TRY(make_taps(dec_lo, dec_hi, L, 1.0, &taps));
  WTB_ENTER(flags, x, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  std::vector<int> lens(level + 1);
  WTB_TRY(wtb_dwt_coeff_lens(n, L, level, lens.data()));
  size_t total = 0;
  for (int v : lens) total += (size_t)v;
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    return DISPATCH(wavedec_impl, (const char *)x + first * e * n, nb, n, taps, level, flags,
                    (char *)coeffs + first * e * total, st);
  });
}

extern "C" int wtb_waverec(const void *coeffs, int64_t batch, const int *lens, int level, const double *rec_lo,
                           const double *rec_hi, int L, int flags, void *x_out, void *stream) {
  WTB_REQUIRE(coeffs && x_out && lens && batch >= 0 && level >= 0, WTB_EINVAL, "wtb_waverec: bad arguments");
  Taps taps;
  WTB_TRY(make_taps(rec_lo, rec_hi, L, 1.0, &taps));
  WTB_ENTER(flags, coeffs, stream);
  if (batch == 0) return WTB_OK;
  const size_t e = ((flags & WTB_F64) ? 8 : 4);
  size_t total = 0;
  for (int l = 0; l <= level; ++l) total += (size_t)lens[l];
  const int nout = wtb_waverec_len(lens, level, L);
  if (nout < 0) return nout;
  return shard_host_rows(batch, flags, (cudaStream_t)stream, [&](int64_t first, int64_t nb, cudaStream_t st) {
    return DISPATCH(waverec_impl, (const char *)coeffs + first * e * total, nb, lens, level, taps, flags,
                    (char *)x_out + first * e * nout, st);
  });
}
