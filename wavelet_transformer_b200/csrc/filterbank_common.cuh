// Pieces shared by the generic (filterbank.cu) and the register-blocked
// (filterbank_fast.cu) MODWT / DWT kernels: tap tables, the DWT level plan and 1-D TMA
// bulk copies (cp.async.bulk + mbarrier / bulk_group).
#pragma once

#include <algorithm>

#include "common.cuh"

namespace wtb {

constexpr int kMaxTaps = 32;
struct Taps {
  int L;
  double lo[kMaxTaps];  // scaling (g) taps as used by the kernel
  double hi[kMaxTaps];  // wavelet (h) taps
};

constexpr int kMaxLevels = 32;
struct LevelPlan {
  int level;
  int n;                     // signal length (wavedec) / output length (waverec)
  int buf;                   // elements per shared-memory ping-pong buffer
  int total;                 // packed coefficient count per series
  int len[kMaxLevels + 1];   // cA_L, cD_L, ..., cD_1
  int off[kMaxLevels + 1];   // offsets of those blocks in the packed row
};

// ---- 1-D TMA bulk copies ---------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(phase)
      : "memory");
}
// global -> shared, completion counted on `bar` (bytes multiple of 16, both sides 16B aligned)
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// shared -> global, tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void tma_store_1d(void *dst, const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's bulk stores have finished READING shared memory
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy shared-memory writes become visible to the async (TMA) proxy
__device__ __forceinline__ void fence_smem_to_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__host__ __device__ __forceinline__ bool tma_row_ok(const void *base, size_t row_bytes) {
  return (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(base) & 15) == 0) && row_bytes < (1u << 20);
}

// Stage `n` elements of a row into shared memory.  All threads call it.
template <typename T>
__device__ void stage_row(T *dst, const T *__restrict__ src, int n, uint64_t *bar, uint32_t &phase) {
  const size_t bytes = sizeof(T) * (size_t)n;
  if (tma_row_ok(src, bytes)) {
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, (uint32_t)bytes);
      tma_load_1d(dst, src, (uint32_t)bytes, bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    // No thread may lag a whole phase behind: if thread 0 re-armed the barrier and the next
    // copy landed before a slow thread had tested this phase, that thread would wait forever.
    __syncthreads();
  } else {
    for (int t = threadIdx.x; t < n; t += blockDim.x) dst[t] = src[t];
    __syncthreads();
  }
}

// half-sample symmetric extension (pywt mode='symmetric'), repeated when |p| runs past a period
__device__ __forceinline__ int reflect_sym(int p, int n) {
  if (p >= 0 && p < n) return p;
  if (p < 0 && p >= -n) return -1 - p;
  if (p >= n && p < 2 * n) return 2 * n - 1 - p;
  const int period = 2 * n;
  int m = p % period;
  if (m < 0) m += period;
  return m >= n ? period - 1 - m : m;
}

// ---- host side -------------------------------------------------------------------------
template <typename K> static int set_smem(K kernel, size_t bytes) {
  WTB_REQUIRE(bytes <= kSmemLimit, WTB_EUNSUPPORTED,
              "series too long for the in-shared-memory filterbank (%zu B > 227 KB per CTA)", bytes);
  WTB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return WTB_OK;
}

// Whether `kernel` runs with `dyn` bytes of dynamic shared memory: its static shared memory (tap tables, barrier)
// counts against the same 227 KB.  A shape whose generic kernel does not fit runs the long path (filterbank_long.cu).
template <typename K> static int fits_one_cta(K kernel, size_t dyn, bool *fits) {
  cudaFuncAttributes a;
  WTB_CUDA(cudaFuncGetAttributes(&a, kernel));
  *fits = dyn + a.sharedSizeBytes <= kSmemLimit;
  return WTB_OK;
}

// Taps of the kernels from the caller's lo / hi, each multiplied by `scale` (1/sqrt 2 for the MODWT);
// WTB_EUNSUPPORTED for L outside [2, kMaxTaps] (filterbank.cu)
int make_taps(const double *lo, const double *hi, int L, double scale, Taps *t);

// wtb_modwt, wtb_imodwt, wtb_modwtmra, wtb_modwtmra_taps, wtb_wavedec, wtb_waverec
enum class FbOp { kModwt, kImodwt, kMra, kMraTaps, kWavedec, kWaverec };
// One-CTA launch of a shape: CTA size (0: not covered), dynamic shared memory, k_mra_blk's chain length R and the
// DWT's LevelPlan::buf
struct BlkShape { int threads; size_t smem; int R, buf; };

// ---- register-blocked kernels (filterbank_fast.cu).  blk_shape: whether they cover a shape and how they launch
// for it, from host arithmetic alone (`dwt`: the DWT ops' level plan, read instead of n and J; nullptr for the
// others).  The launchers take its result and launch ----------------------------------------------------------------
BlkShape blk_shape(FbOp op, int n, int L, int J, const LevelPlan *dwt, size_t elem);
template <typename T> int modwt_fast(const BlkShape &s, const void *x, int64_t batch, int n, const Taps &taps, int J,
                                     void *out, cudaStream_t st);
template <typename T> int imodwt_fast(const BlkShape &s, const void *w, int64_t batch, int n, const Taps &taps, int J,
                                      void *out, cudaStream_t st);
template <typename T> int mra_fast(const BlkShape &s, const void *w, int64_t batch, int n, const Taps &taps, int J,
                                   void *out, cudaStream_t st);
template <typename T> int wavedec_fast(const BlkShape &s, const void *x, int64_t batch, const LevelPlan &plan,
                                       const Taps &taps, void *coeffs, cudaStream_t st);
template <typename T> int waverec_fast(const BlkShape &s, const void *coeffs, int64_t batch, const LevelPlan &plan,
                                       const Taps &taps, void *x, cudaStream_t st);

// ---- wtb_modwt on device rows x [batch, n] -> out [batch, J+1, n], enqueued on st (filterbank.cu): the plan and
// every kernel of wtb_modwt, bit for bit.  It reserves no staging (stage_rows takes none for device pointers), so a
// caller may hold staging across it; the long path takes the arena.
template <typename T>
int modwt_device(const T *x, int64_t batch, int n, const Taps &taps, int J, int flags, T *out, cudaStream_t st);

// ---- long series (filterbank_long.cu): one launch per level per wave of series, for the shapes whose generic
// kernel above needs more than kSmemLimit of shared memory.  Each runs the whole call, host chunks included ----
template <typename T>
int modwt_long(const void *x, int64_t batch, int n, const Taps &taps, int J, int flags, void *out, cudaStream_t st);
template <typename T>
int imodwt_long(const void *w, int64_t batch, int n, const Taps &taps, int J, int flags, void *out, cudaStream_t st);
template <typename T>
int mra_taps_long(const void *w, int64_t batch, int n, const Taps &taps, int J, int flags, void *out,
                  cudaStream_t st);
template <typename T>
int mra_filt_long(const void *w, int64_t batch, int n, const double *filt, int J, int flags, void *out,
                  cudaStream_t st);
template <typename T>
int wavedec_long(const void *x, int64_t batch, const LevelPlan &plan, const Taps &taps, int flags, void *coeffs,
                 cudaStream_t st);
template <typename T>
int waverec_long(const void *coeffs, int64_t batch, const LevelPlan &plan, const Taps &taps, int flags, void *x,
                 cudaStream_t st);

}  // namespace wtb
