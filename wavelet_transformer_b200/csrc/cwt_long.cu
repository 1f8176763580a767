// CWT of long series: power-of-two transforms whose two shared-memory buffers do not fit one CTA
// (nfft >= 16384 in FP32, >= 8192 in FP64), up to nfft = 2^22.  cwt_device (cwt.cu) branches here.
//
// The four-step transforms and their launch shapes are in long_fft.cuh.
//
// One call: the forward transform of every series into X^ [batch, N] (natural order), then per flattened
// (series, scale) row the inverse transform of X^ * daughter (pass 1 forms the product on the fly, with
// k_cwt_rows' arithmetic) and power / coefficients for t < n0 (pass 2).  Rows run in waves whose
// intermediate Y fits half the B200's 126 MB L2 (long_wave_rows); a row's arithmetic does not depend on
// its wave, so results do not depend on the batch, the host chunk or the pool.
#include "long_fft.cuh"

namespace wtb {

// The long path takes exactly the power-of-two lengths whose two shared-memory buffers exceed 227 KB
// (nfft > 2^22 included: cwt_long refuses them).
bool cwt_long_takes(int N, size_t elem) { return is_pow2(N) && 2 * 2 * elem * (size_t)N > 227 * 1024; }

// exp(-2 pi i j / N) for j < 2048, then exp(-2 pi i 2048 j / N) for j < N / 2048; cached per (device, N), kept
// until wtb_shutdown (at most 48 KB in FP64 at N = 2^22).
namespace {
template <typename T> struct LongTables {
  std::mutex mu;
  std::map<std::pair<int, int>, void *> tab;
};
template <typename T> LongTables<T> &long_tables() {
  static LongTables<T> t;
  return t;
}
template <typename T> void release_tables() {
  LongTables<T> &c = long_tables<T>();
  std::lock_guard<std::mutex> lk(c.mu);
  for (auto &kv : c.tab) cudaFree(kv.second);
  c.tab.clear();
}
}  // namespace

template <typename T> static int long_twiddles(int N, cudaStream_t st, const cplx<T> **lo, const cplx<T> **hi) {
  LongTables<T> &c = long_tables<T>();
  std::lock_guard<std::mutex> lk(c.mu);
  const auto key = std::make_pair(current_device(), N);
  auto it = c.tab.find(key);
  if (it == c.tab.end()) {
    const int nhi = N / 2048;
    std::vector<cplx<T>> h(2048 + nhi);
    const long double two_pi = 2.0L * 3.141592653589793238462643383279502884L;
    for (int j = 0; j < 2048; ++j) {
      const long double a = -two_pi * j / N;
      h[j] = mk<T>((T)cosl(a), (T)sinl(a));
    }
    for (int j = 0; j < nhi; ++j) {
      const long double a = -two_pi * j / nhi;
      h[2048 + j] = mk<T>((T)cosl(a), (T)sinl(a));
    }
    void *d = nullptr;
    WTB_CUDA(cudaMalloc(&d, sizeof(cplx<T>) * h.size()));
    WTB_CUDA(cudaMemcpyAsync(d, h.data(), sizeof(cplx<T>) * h.size(), cudaMemcpyHostToDevice, st));
    WTB_CUDA(cudaStreamSynchronize(st));    // the table is shared with every later call, on any stream
    it = c.tab.emplace(key, d).first;
  }
  *lo = (const cplx<T> *)it->second;
  *hi = *lo + 2048;
  return WTB_OK;
}

// Split, block_fft tables and inter-pass twiddles of one power-of-two length; refuses nfft > 2^22.
template <typename T> int long_plan(int N, cudaStream_t st, LongPlan<T> *p) {
  WTB_REQUIRE(N <= kLongMaxN, WTB_EUNSUPPORTED,
              "nfft=%d: power-of-two transforms go up to nfft = 2^22 = %d (pad the series to at most 2^22 points)", N,
              kLongMaxN);
  const int L = ilog2(N);
  p->N = N;
  p->log2N1 = L / 2;
  p->log2N2 = L - L / 2;
  p->N1 = 1 << p->log2N1;
  p->N2 = 1 << p->log2N2;
  WTB_TRY(twiddles<T>(p->N1, &p->tw1));
  WTB_TRY(twiddles<T>(p->N2, &p->tw2));
  return long_twiddles<T>(N, st, &p->tlo, &p->thi);
}
template int long_plan<float>(int, cudaStream_t, LongPlan<float> *);
template int long_plan<double>(int, cudaStream_t, LongPlan<double> *);

void cwt_long_release() {
  release_tables<float>();
  release_tables<double>();
}

template <typename T>
int cwt_long(const T *d_x, int64_t batch, int n0, int N, double dt, const Axes &ax, const Mother &mo, int flags,
             T *d_power, cplx<T> *d_coef, cudaStream_t st) {
  LongPlan<T> p;
  WTB_TRY(long_plan<T>(N, st, &p));
  const int S = ax.J + 1;
  const int64_t rows = batch * S;
  const int64_t wave_fwd = long_wave_rows(N, sizeof(cplx<T>), batch), wave = long_wave_rows(N, sizeof(cplx<T>), rows);
  // one reservation: a slot that grows is moved
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t b_sc = al(sizeof(double) * S), b_xhat = al(sizeof(cplx<T>) * (size_t)batch * N);
  void *scratch = nullptr;
  WTB_TRY(arena_reserve(b_sc + b_xhat + sizeof(cplx<T>) * (size_t)wave * N, &scratch));
  double *d_scales = (double *)scratch;
  cplx<T> *d_xhat = (cplx<T> *)((char *)scratch + b_sc);
  cplx<T> *d_y = (cplx<T> *)((char *)scratch + b_sc + b_xhat);
  WTB_CUDA(cudaMemcpyAsync(d_scales, ax.scales.data(), sizeof(double) * S, cudaMemcpyHostToDevice, st));
  const LongLaunch l1 = long_launch<T>(1, p.N2), l2 = long_launch<T>(2, p.N1);
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass1<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass1<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass2<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2.smem));
  WTB_CUDA(cudaFuncSetAttribute(k_long_pass2<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l2.smem));
  const unsigned g1 = p.N1 / long_cols<T>(1), g2 = p.N2 / long_cols<T>(2);
  for (int64_t r0 = 0; r0 < batch; r0 += wave_fwd) {
    const unsigned nw = (unsigned)std::min(wave_fwd, batch - r0);
    k_long_pass1<T, false><<<dim3(g1, nw), l1.block, l1.smem, st>>>(p, r0, d_x, n0, nullptr, S, nullptr, dt, 0.0, 0, 0,
                                                                     T(0), T(0), d_y);
    WTB_LAUNCH_CHECK();
    k_long_pass2<T, false><<<dim3(g2, nw), l2.block, l2.smem, st>>>(p, r0, d_y, n0, S, nullptr, d_xhat, nullptr,
                                                                     nullptr, 0, 0.0, 0.0);
    WTB_LAUNCH_CHECK();
  }
  double pre_re, pre_im;
  mother_prefactor(mo, &pre_re, &pre_im);
  const double f0 = mo.kind == WTB_MORLET ? mo.param : 0.0;
  const int coi_mask = (flags & WTB_COI_MASK) ? 1 : 0;
  for (int64_t r0 = 0; r0 < rows; r0 += wave) {
    const unsigned nw = (unsigned)std::min(wave, rows - r0);
    k_long_pass1<T, true><<<dim3(g1, nw), l1.block, l1.smem, st>>>(p, r0, nullptr, n0, d_xhat, S, d_scales, dt, f0,
                                                                    mo.kind, (int)mo.param, T(pre_re), T(pre_im), d_y);
    WTB_LAUNCH_CHECK();
    k_long_pass2<T, true><<<dim3(g2, nw), l2.block, l2.smem, st>>>(
        p, r0, d_y, n0, S, d_scales, nullptr, d_power, d_coef, coi_mask, mother_flambda(mo) * mother_coi(mo) * dt,
        mother_flambda(mo));
    WTB_LAUNCH_CHECK();
  }
  return WTB_OK;
}
template int cwt_long<float>(const float *, int64_t, int, int, double, const Axes &, const Mother &, int, float *,
                             float2 *, cudaStream_t);
template int cwt_long<double>(const double *, int64_t, int, int, double, const Axes &, const Mother &, int, double *,
                              double2 *, cudaStream_t);

}  // namespace wtb
