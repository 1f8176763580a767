// Shared host/device helpers for libwavelet_sm100a.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/wtb.h"

namespace wtb {

// ---- error plumbing ---------------------------------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define WTB_CUDA(call)                                                        \
  do {                                                                        \
    cudaError_t e__ = (call);                                                 \
    if (e__ != cudaSuccess) return ::wtb::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

// after every kernel launch: count it (wtb_kernel_launches) and surface launch errors
void note_launch();
#define WTB_LAUNCH_CHECK()            \
  do {                                \
    ::wtb::note_launch();             \
    WTB_CUDA(cudaGetLastError());     \
  } while (0)

#define WTB_REQUIRE(cond, code, ...)   \
  do {                                 \
    if (!(cond)) {                     \
      ::wtb::set_error(__VA_ARGS__);   \
      return (code);                   \
    }                                  \
  } while (0)

// WTB_TRACE=1: host wall-clock per phase of a call, each closed with a stream synchronisation
// (stderr).  A debugging aid for latency work; it serialises the call, never time with it on.
struct TracePoint {
  static bool on() {
    static const bool v = std::getenv("WTB_TRACE") && std::atoi(std::getenv("WTB_TRACE"));
    return v;
  }
  static void mark(cudaStream_t st, const char *label);
};
#define WTB_TRACE_POINT(st, label)                          \
  do {                                                      \
    if (::wtb::TracePoint::on()) ::wtb::TracePoint::mark((st), (label)); \
  } while (0)

#define WTB_TRY(expr)          \
  do {                         \
    int rc__ = (expr);         \
    if (rc__ != WTB_OK) return rc__; \
  } while (0)

// ---- complex arithmetic -----------------------------------------------------
template <typename T> struct cplx_of;
template <> struct cplx_of<float> { using type = float2; };
template <> struct cplx_of<double> { using type = double2; };
template <typename T> using cplx = typename cplx_of<T>::type;

template <typename T> __host__ __device__ __forceinline__ cplx<T> mk(T x, T y) {
  cplx<T> r; r.x = x; r.y = y; return r;
}
template <typename C> __device__ __forceinline__ C cadd(C a, C b) { a.x += b.x; a.y += b.y; return a; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { a.x -= b.x; a.y -= b.y; return a; }
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
  C r; r.x = a.x * b.x - a.y * b.y; r.y = a.x * b.y + a.y * b.x; return r;
}
// a * conj(b)
template <typename C> __device__ __forceinline__ C cmulc(C a, C b) {
  C r; r.x = a.x * b.x + a.y * b.y; r.y = a.y * b.x - a.x * b.y; return r;
}

constexpr double kPi = 3.14159265358979323846264338327950288;
constexpr size_t kSmemLimit = 227 << 10;   // shared memory of one CTA on sm_100 (B200), static and dynamic

// ---- per-call context, device scratch, tables (host side) -----------------------
// Every C-ABI entry point opens a CallScope first.  It decides which device the call runs on
//   1. the device of a multi-GPU pool worker thread (wtb_init_multi, multi.cu),
//   2. with WTB_DEVICE_PTRS: the device that owns the data pointer,
//   3. the device given to wtb_init() / WTB_DEVICE,
//   4. otherwise the calling thread's current CUDA device,
// checks once per device that it is sm_100, makes it current for the call and puts the
// caller's device back on return.  It also records the (device, stream) pair that keys scratch.
class CallScope {
 public:
  CallScope(int flags, const void *data_ptr, void *stream);
  ~CallScope();
  CallScope(const CallScope &) = delete;
  CallScope &operator=(const CallScope &) = delete;
  int rc() const { return rc_; }
  int device() const { return device_; }

 private:
  int rc_ = WTB_OK;
  int device_ = -1;
  int restore_ = -1;         // device to make current again on exit (-1: nothing to undo)
  int outer_device_ = -1;    // enclosing scope's key (entry points may nest)
  cudaStream_t outer_stream_ = nullptr;
  bool nested_ = false;
};
#define WTB_ENTER(flags, ptr, stream)                \
  ::wtb::CallScope scope__((flags), (ptr), (stream)); \
  WTB_TRY(scope__.rc())

int current_device();         // device of the innermost CallScope on this thread
cudaStream_t current_stream();

// Grow-only device scratch owned by the library, keyed by (host thread, device, stream): two
// calls only ever share scratch when they are ordered on the same stream of the same thread, so
// concurrent Streamlit sessions (threads) and concurrent torch streams never see each other's
// intermediates.  Memory is stream-ordered (cudaMallocAsync / cudaFreeAsync), so growing an
// arena neither synchronises the device nor frees memory a queued kernel still uses.  A thread's
// arenas are released when the thread exits, everything that is left by wtb_shutdown().
int arena_reserve(size_t bytes, void **out);  // intermediates, 256B aligned
// Second independent arena (I/O staging for host-pointer calls).
int staging_reserve(size_t bytes, void **out);
// small buffer for kernel parameter tables, separate from the two arenas above so a callee can
// fill it while its caller's arena holds live data
int params_reserve(size_t bytes, void **out);
// An internal copy stream of the calling thread on the current device (created once, destroyed
// when the thread exits): host-to-device copies of the next chunk run there while the kernels of
// the current chunk occupy the caller's stream.
int copy_stream(cudaStream_t *out);

// small page-locked host buffer of the calling thread (results that go back to pageable caller
// memory bounce through it); grow-only, freed when the thread exits
int pinned_reserve(size_t bytes, void **out);
// Device -> caller's host buffer.  Results up to 4 MiB (every single-series request of the
// reference) go through the thread's pinned buffer and a memcpy -- the call returns with the
// data in place; larger ones are one cudaMemcpyAsync straight into the caller's memory, which
// the caller's stream synchronisation completes.
int copy_to_host(void *dst, const void *d_src, size_t bytes, cudaStream_t st);
// bytes of device scratch the library holds right now, over all threads (leak tests)
size_t scratch_bytes_held();

// Twiddle table exp(-2*pi*i*k/N), k in [0,N), in precision T; cached per (device,N).
template <typename T> int twiddles(int N, const cplx<T> **out);

// Chirp tables of Bluestein's algorithm for length n over work length M (fft_block.cuh), cached
// per (device, n, M) like the twiddles.
template <typename T> int bluestein_tables(int n, int M, const cplx<T> **chirp, const cplx<T> **chat);

int sm_count();               // SMs of current_device()

// ---- multi-GPU pool (multi.cu): one worker thread + stream per device -------------------
int pool_size();              // 1 unless wtb_init_multi() made a pool
// Runs fn(part, first, count, stream) for a split of [0, total) into contiguous blocks, one per
// pool device, each on that device's worker thread (device current, scratch keyed by the worker's
// stream) and waits for all of them.  Returns the first failure (its message becomes the caller's
// wtb_last_error()).  With no pool, or total < min_total, fn runs once on the calling thread.
using ShardFn = int (*)(void *ctx, int part, int64_t first, int64_t count, cudaStream_t stream);
int run_sharded(int64_t total, int64_t min_total, cudaStream_t caller_stream, ShardFn fn, void *ctx);
template <typename F> int run_sharded_fn(int64_t total, int64_t min_total, cudaStream_t st, F &&f) {
  using Fn = typename std::remove_reference<F>::type;
  return run_sharded(total, min_total, st,
                     [](void *ctx, int part, int64_t first, int64_t count, cudaStream_t s) -> int {
                       return (*static_cast<Fn *>(ctx))(part, first, count, s);
                     },
                     (void *)&f);
}
const char *last_error();     // this thread's message (workers hand theirs to the caller)

// ---- batches of rows: the split over the pool and the host staging of every batched entry point -------------------
inline size_t align256(size_t bytes) { return (bytes + 255) / 256 * 256; }

// Host-buffer batches with a pool of two or more devices (wtb_init_multi) and at least two rows per device:
// call(first, count, stream) once per device for a contiguous block of rows, on that device's worker thread.
// Otherwise call(0, batch, stream) once.  The caller offsets its pointers by `first`; the worker runs `call` itself
// and never comes back here, so a block is never split again.
template <typename F> int shard_host_rows(int64_t batch, int flags, cudaStream_t st, F &&call) {
  if ((flags & WTB_DEVICE_PTRS) || pool_size() < 2 || batch < 2 * pool_size()) return call(int64_t(0), batch, st);
  return run_sharded_fn(batch, 2, st, [&](int, int64_t first, int64_t count, cudaStream_t s) {
    return call(first, count, s);
  });
}

// Rows per host chunk: as many as keep `row_bytes` each within 1 GiB of staging, at least one, at most the batch;
// with device pointers the whole batch
inline int64_t host_rows(int64_t batch, size_t row_bytes, int flags) {
  if (flags & WTB_DEVICE_PTRS) return batch;
  return std::max<int64_t>(1, std::min<int64_t>(batch, (int64_t)((size_t(1) << 30) / row_bytes)));
}

// One buffer of the caller's batch: rows of row_bytes bytes each.  ptr is null for an output not asked for.
template <typename P> struct RowBuf {
  P *ptr;
  size_t row_bytes;
  RowBuf at(int64_t row) const { return {ptr ? (P *)((const char *)ptr + row * row_bytes) : nullptr, row_bytes}; }
};
using InRows = RowBuf<const void>;
using OutRows = RowBuf<void>;

// Runs launch(in, out, extra, b0, nb) over [0, batch) in chunks of `rows` (the caller's chunk rule).  in[i] / out[i]
// are the device rows b0 .. b0 + nb of ins[i] / outs[i], null where the caller's pointer is; extra is extra_bytes of
// staging scratch (null when 0).
//   Host buffers: the inputs go up with cudaMemcpyAsync before the launch, the outputs come back through copy_to_host,
//   then the stream is synchronised, chunk by chunk.
//   WTB_DEVICE_PTRS: the caller's pointers, offset by b0; nothing is copied or synchronised.
// The staging slot is reserved once for the whole call (every non-null port at `rows` rows and extra_bytes, each
// region 256-byte aligned): a second reservation that grew the slot would move it under the first one's data, so
// nothing inside `launch` may take staging.
template <typename F>
int stage_rows(int64_t batch, int64_t rows, int flags, cudaStream_t st, std::initializer_list<InRows> ins,
               std::initializer_list<OutRows> outs, size_t extra_bytes, F &&launch) {
  const bool dev = flags & WTB_DEVICE_PTRS;
  const size_t n_in = ins.size(), n_out = outs.size();
  const InRows *in = ins.begin();
  const OutRows *out = outs.begin();
  size_t bytes = align256(extra_bytes);
  for (size_t i = 0; i < n_in && !dev; ++i) bytes += in[i].ptr ? align256(in[i].row_bytes * rows) : 0;
  for (size_t i = 0; i < n_out && !dev; ++i) bytes += out[i].ptr ? align256(out[i].row_bytes * rows) : 0;
  char *stage = nullptr;
  if (bytes) WTB_TRY(staging_reserve(bytes, (void **)&stage));
  void *extra = extra_bytes ? stage : nullptr;
  std::vector<const void *> d_in(n_in, nullptr);
  std::vector<void *> d_out(n_out, nullptr);
  char *p = stage + align256(extra_bytes);
  for (size_t i = 0; i < n_in && !dev; ++i)
    if (in[i].ptr) { d_in[i] = p; p += align256(in[i].row_bytes * rows); }
  for (size_t i = 0; i < n_out && !dev; ++i)
    if (out[i].ptr) { d_out[i] = p; p += align256(out[i].row_bytes * rows); }
  for (int64_t b0 = 0; b0 < batch; b0 += rows) {
    const int64_t nb = std::min(rows, batch - b0);
    for (size_t i = 0; i < n_in; ++i) {
      if (dev) d_in[i] = in[i].at(b0).ptr;
      else if (in[i].ptr)
        WTB_CUDA(cudaMemcpyAsync((void *)d_in[i], in[i].at(b0).ptr, in[i].row_bytes * nb, cudaMemcpyHostToDevice, st));
    }
    for (size_t i = 0; i < n_out && dev; ++i) d_out[i] = out[i].at(b0).ptr;
    WTB_TRY(launch(d_in.data(), d_out.data(), extra, b0, nb));
    if (dev) continue;   // every chunk is ordered on st
    for (size_t i = 0; i < n_out; ++i)
      if (out[i].ptr) WTB_TRY(copy_to_host(out[i].at(b0).ptr, d_out[i], out[i].row_bytes * nb, st));
    WTB_CUDA(cudaStreamSynchronize(st));
  }
  return WTB_OK;
}

inline int ilog2(int n) { int l = 0; while ((int64_t(1) << l) < n) ++l; return l; }   // ceil(log2 n), any int n
inline bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }
// make_plan's work length, any int nfft: a power of two itself, else Bluestein's 2^m >= 2 nfft - 1 (2 << ilog2)
inline int64_t work_length(int nfft) { return is_pow2(nfft) ? nfft : int64_t(2) << ilog2(nfft); }

// Morlet constants (pycwt.mothers.Morlet)
inline double morlet_flambda(double f0) { return 4.0 * kPi / (f0 + std::sqrt(2.0 + f0 * f0)); }

// pycwt.mothers: kind = WTB_MORLET / WTB_PAUL / WTB_DOG, param = f0 or the order m
struct Mother {
  int kind = WTB_MORLET;
  double param = 6.0;
};
inline double mother_flambda(const Mother &m) {
  if (m.kind == WTB_PAUL) return 4.0 * kPi / (2.0 * m.param + 1.0);
  if (m.kind == WTB_DOG) return 2.0 * kPi / std::sqrt(m.param + 0.5);
  return morlet_flambda(m.param);
}
// e-folding factor of the cone of influence (Torrence & Compo table 1)
inline double mother_coi(const Mother &m) { return m.kind == WTB_PAUL ? std::sqrt(2.0) : 1.0 / std::sqrt(2.0); }
// conj of the constant complex prefactor of psi_ft (1 for Morlet: pi^-1/4 stays in the kernel)
inline void mother_prefactor(const Mother &m, double *re, double *im) {
  *re = 1.0;
  *im = 0.0;
  const int order = (int)m.param;
  if (m.kind == WTB_PAUL) {
    double fact = 1.0;  // (2m-1)!
    for (int k = 2; k <= 2 * order - 1; ++k) fact *= k;
    *re = std::pow(2.0, order) / std::sqrt(order * fact);
  } else if (m.kind == WTB_DOG) {
    const double c = 1.0 / std::sqrt(std::tgamma(m.param + 0.5));
    // -i^m: m%4 = 0 -> -1, 1 -> -i, 2 -> +1, 3 -> +i; conjugated here
    switch (order & 3) {
      case 0: *re = -c; break;
      case 1: *re = 0; *im = c; break;
      case 2: *re = c; break;
      default: *re = 0; *im = -c; break;
    }
  }
}

struct Axes {
  int J = 0;
  std::vector<double> scales, freqs;
};
int resolve_axes(int n0, double dt, double dj, double s0, int J, double f0, Axes *ax);
int resolve_axes(int n0, double dt, double dj, double s0, int J, const Mother &m, Axes *ax);

}  // namespace wtb
