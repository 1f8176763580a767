// Runtime plumbing of libwavelet_sm100a.so: errors, device binding, scratch
// arenas, twiddle tables, and the small host-side pieces of the C ABI.
#include <atomic>
#include <tuple>
#include <chrono>
#include <cstdarg>

#include "common.cuh"

namespace wtb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
  set_error("CUDA error %s (%d) at %s:%d: %s", cudaGetErrorName(e), (int)e, file, line, what);
  return WTB_ECUDA;
}

void TracePoint::mark(cudaStream_t st, const char *label) {
  static thread_local std::chrono::steady_clock::time_point last = std::chrono::steady_clock::now();
  const auto t_host = std::chrono::steady_clock::now();
  cudaStreamSynchronize(st);
  const auto t_dev = std::chrono::steady_clock::now();
  fprintf(stderr, "[wtb trace] %-28s host +%8.1f us, device drained +%8.1f us\n", label,
          std::chrono::duration<double, std::micro>(t_host - last).count(),
          std::chrono::duration<double, std::micro>(t_dev - t_host).count());
  last = std::chrono::steady_clock::now();
}

static std::atomic<uint64_t> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
uint64_t launches() { return g_launches.load(std::memory_order_relaxed); }

// ---- device selection --------------------------------------------------------------
static std::mutex g_mu;
static int g_default_device = -1;   // wtb_init(device) / WTB_DEVICE; -1: follow the caller's current device
constexpr int kMaxDevices = 64;
struct DeviceInfo {
  int state = 0;   // 0 unknown, 1 usable sm_100, -1 rejected
  int sms = 0;
};
static DeviceInfo g_devinfo[kMaxDevices];

thread_local int tl_worker_device = -1;      // set by multi.cu's pool threads
static thread_local int tl_device = -1;      // innermost CallScope
static thread_local cudaStream_t tl_stream = nullptr;
static thread_local int tl_depth = 0;

static int check_device(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device visible (%s); libwavelet_sm100a has no CPU fallback",
              e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
    cudaGetLastError();
    return WTB_ENODEVICE;
  }
  WTB_REQUIRE(device >= 0 && device < count && device < kMaxDevices, WTB_EINVAL, "device %d out of range [0,%d)",
              device, count);
  std::lock_guard<std::mutex> lk(g_mu);
  DeviceInfo &di = g_devinfo[device];
  if (di.state == 0) {
    int major = 0, minor = 0, sms = 0;
    WTB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    WTB_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
    WTB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    di.sms = sms;
    di.state = major == 10 ? 1 : -(100 + major * 10 + minor);
  }
  WTB_REQUIRE(di.state == 1, WTB_ENODEVICE, "device %d is sm_%d; this library is built for sm_100a only", device,
              -di.state - 100);
  return WTB_OK;
}

CallScope::CallScope(int flags, const void *data_ptr, void *stream) {
  nested_ = tl_depth > 0;
  outer_device_ = tl_device;
  outer_stream_ = tl_stream;
  ++tl_depth;
  if (nested_) {          // an entry point called from another one: same device, same scratch key
    device_ = tl_device;
    return;
  }
  int cur = -1;
  cudaError_t e = cudaGetDevice(&cur);
  if (e != cudaSuccess) {
    set_error("no CUDA device visible (%s); libwavelet_sm100a has no CPU fallback", cudaGetErrorString(e));
    cudaGetLastError();
    rc_ = WTB_ENODEVICE;
    return;
  }
  int want = -1;
  if (tl_worker_device >= 0) {
    want = tl_worker_device;
  } else if ((flags & WTB_DEVICE_PTRS) && data_ptr) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, data_ptr) == cudaSuccess &&
        (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged)) {
      want = attr.device;
    } else {
      cudaGetLastError();
      set_error("WTB_DEVICE_PTRS: %p is not a device pointer", data_ptr);
      rc_ = WTB_EINVAL;
      return;
    }
  } else if (g_default_device >= 0) {
    want = g_default_device;
  } else if (const char *env = getenv("WTB_DEVICE")) {
    want = atoi(env);
  } else {
    want = cur;
  }
  rc_ = check_device(want);
  if (rc_ != WTB_OK) return;
  if (want != cur) {
    e = cudaSetDevice(want);
    if (e != cudaSuccess) {
      rc_ = cuda_fail(e, "cudaSetDevice", __FILE__, __LINE__);
      return;
    }
    restore_ = cur;
  }
  device_ = want;
  tl_device = want;
  tl_stream = (cudaStream_t)stream;
}

CallScope::~CallScope() {
  --tl_depth;
  if (nested_) return;
  tl_device = outer_device_;
  tl_stream = outer_stream_;
  if (restore_ >= 0) cudaSetDevice(restore_);
}

int current_device() { return tl_device; }
cudaStream_t current_stream() { return tl_stream; }

int sm_count() {
  const int d = tl_device;
  return (d >= 0 && d < kMaxDevices && g_devinfo[d].sms > 0) ? g_devinfo[d].sms : 148;
}

const char *last_error() { return g_err; }

// ---- arenas ------------------------------------------------------------------------
// One ArenaSet per (thread, device, stream); a thread keeps at most kMaxSetsPerThread of them
// (least recently used goes first), so a caller that keeps making new streams cannot grow the
// footprint without bound.
struct Arena {
  void *ptr = nullptr;
  size_t cap = 0;
};
struct ArenaSet {
  int device = -1;
  cudaStream_t stream = nullptr;
  uint64_t last_use = 0;
  Arena a[3];   // intermediates, staging, parameters
};
constexpr int kMaxSetsPerThread = 8;

static std::mutex g_arena_mu;
static std::vector<ArenaSet *> g_sets;   // every live set, for wtb_shutdown and the byte count
static std::atomic<size_t> g_scratch_bytes{0};

static void release_set(ArenaSet *s) {
  // cudaFree is valid for stream-ordered allocations and waits for the work that uses them
  int cur = -1;
  const bool have = cudaGetDevice(&cur) == cudaSuccess;
  bool any = false;
  for (Arena &a : s->a) any = any || a.ptr;
  if (any && have && cur != s->device) cudaSetDevice(s->device);
  for (Arena &a : s->a) {
    if (a.ptr) {
      cudaFree(a.ptr);
      g_scratch_bytes.fetch_sub(a.cap, std::memory_order_relaxed);
    }
    a.ptr = nullptr;
    a.cap = 0;
  }
  if (any && have && cur != s->device) cudaSetDevice(cur);
  cudaGetLastError();   // at process exit the runtime may already be unloading: nothing to report
}

struct ThreadArenas {
  std::vector<ArenaSet *> sets;
  uint64_t tick = 0;
  ~ThreadArenas() {
    std::lock_guard<std::mutex> lk(g_arena_mu);
    for (ArenaSet *s : sets) {
      release_set(s);
      for (size_t i = 0; i < g_sets.size(); ++i)
        if (g_sets[i] == s) { g_sets[i] = g_sets.back(); g_sets.pop_back(); break; }
      delete s;
    }
  }
  ArenaSet *get(int device, cudaStream_t stream) {
    ++tick;
    for (ArenaSet *s : sets)
      if (s->device == device && s->stream == stream) { s->last_use = tick; return s; }
    std::lock_guard<std::mutex> lk(g_arena_mu);
    ArenaSet *s = nullptr;
    if ((int)sets.size() >= kMaxSetsPerThread) {
      s = sets[0];
      for (ArenaSet *c : sets) if (c->last_use < s->last_use) s = c;
      release_set(s);
    } else {
      s = new ArenaSet();
      sets.push_back(s);
      g_sets.push_back(s);
    }
    s->device = device;
    s->stream = stream;
    s->last_use = tick;
    return s;
  }
};
static thread_local ThreadArenas tl_arenas;

static int reserve(int which, size_t bytes, void **out) {
  WTB_REQUIRE(tl_device >= 0, WTB_ECUDA, "internal: scratch requested outside a call scope");
  ArenaSet *set = tl_arenas.get(tl_device, tl_stream);
  Arena &a = set->a[which];
  if (bytes == 0) bytes = 256;
  if (a.cap < bytes) {
    if (a.ptr) {
      // stream-ordered: the old block is released once the work queued so far on this stream
      // (the only work that can be using it) has finished; nothing blocks here
      WTB_CUDA(cudaFreeAsync(a.ptr, set->stream));
      g_scratch_bytes.fetch_sub(a.cap, std::memory_order_relaxed);
      a.ptr = nullptr;
      a.cap = 0;
    }
    size_t want = bytes + bytes / 8;
    want = (want + (1u << 20) - 1) & ~size_t((1u << 20) - 1);
    cudaError_t e = cudaMallocAsync(&a.ptr, want, set->stream);
    if (e != cudaSuccess) {
      a.ptr = nullptr;
      return cuda_fail(e, "cudaMallocAsync(scratch)", __FILE__, __LINE__);
    }
    a.cap = want;
    g_scratch_bytes.fetch_add(want, std::memory_order_relaxed);
  }
  *out = a.ptr;
  return WTB_OK;
}

struct CopyStreams {
  struct Entry { int device; cudaStream_t s; };
  std::vector<Entry> entries;
  ~CopyStreams() {
    for (Entry &e : entries) cudaStreamDestroy(e.s);
    cudaGetLastError();
  }
};
static thread_local CopyStreams tl_copy;

int copy_stream(cudaStream_t *out) {
  for (auto &e : tl_copy.entries)
    if (e.device == tl_device) { *out = e.s; return WTB_OK; }
  CopyStreams::Entry e;
  e.device = tl_device;
  WTB_CUDA(cudaStreamCreateWithFlags(&e.s, cudaStreamNonBlocking));
  tl_copy.entries.push_back(e);
  *out = e.s;
  return WTB_OK;
}

struct PinnedBuf {
  void *ptr = nullptr;
  size_t cap = 0;
  ~PinnedBuf() {
    if (ptr) cudaFreeHost(ptr);
    cudaGetLastError();
  }
};
static thread_local PinnedBuf tl_pinned;

int pinned_reserve(size_t bytes, void **out) {
  if (tl_pinned.cap < bytes) {
    if (tl_pinned.ptr) WTB_CUDA(cudaFreeHost(tl_pinned.ptr));
    tl_pinned.ptr = nullptr;
    tl_pinned.cap = 0;
    const size_t want = (bytes + 4095) & ~size_t(4095);
    WTB_CUDA(cudaHostAlloc(&tl_pinned.ptr, want, cudaHostAllocDefault));
    tl_pinned.cap = want;
  }
  *out = tl_pinned.ptr;
  return WTB_OK;
}

int copy_to_host(void *dst, const void *d_src, size_t bytes, cudaStream_t st) {
  if (bytes == 0) return WTB_OK;
  if (bytes <= (size_t(4) << 20)) {
    cudaPointerAttributes attr;
    const bool pageable = cudaPointerGetAttributes(&attr, dst) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if (pageable) {
      void *pin = nullptr;
      WTB_TRY(pinned_reserve(bytes, &pin));
      WTB_CUDA(cudaMemcpyAsync(pin, d_src, bytes, cudaMemcpyDeviceToHost, st));
      WTB_CUDA(cudaStreamSynchronize(st));
      std::memcpy(dst, pin, bytes);
      return WTB_OK;
    }
  }
  WTB_CUDA(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
  return WTB_OK;
}

int arena_reserve(size_t bytes, void **out) { return reserve(0, bytes, out); }
int staging_reserve(size_t bytes, void **out) { return reserve(1, bytes, out); }
int params_reserve(size_t bytes, void **out) { return reserve(2, bytes, out); }
size_t scratch_bytes_held() { return g_scratch_bytes.load(std::memory_order_relaxed); }

// ---- twiddles ----------------------------------------------------------------------
template <typename T> struct TwCache {
  std::mutex mu;
  std::map<std::pair<int, int>, void *> tab;
};
template <typename T> static TwCache<T> &tw_cache() {
  static TwCache<T> c;
  return c;
}

template <typename T> int twiddles(int N, const cplx<T> **out) {
  TwCache<T> &c = tw_cache<T>();
  std::lock_guard<std::mutex> lk(c.mu);
  auto key = std::make_pair(tl_device, N);
  auto it = c.tab.find(key);
  if (it == c.tab.end()) {
    std::vector<cplx<T>> h(N);
    for (int k = 0; k < N; ++k) {
      // exact octant symmetry is not needed; long double keeps the table
      // correctly rounded in T
      long double a = -2.0L * 3.141592653589793238462643383279502884L * (long double)k / (long double)N;
      h[k] = mk<T>((T)cosl(a), (T)sinl(a));
    }
    void *d = nullptr;
    WTB_CUDA(cudaMalloc(&d, sizeof(cplx<T>) * N));
    WTB_CUDA(cudaMemcpy(d, h.data(), sizeof(cplx<T>) * N, cudaMemcpyHostToDevice));
    it = c.tab.emplace(key, d).first;
  }
  *out = (const cplx<T> *)it->second;
  return WTB_OK;
}
template int twiddles<float>(int, const cplx<float> **);
template int twiddles<double>(int, const cplx<double> **);

// ---- Bluestein tables ----------------------------------------------------------------
namespace {
void host_fft(std::vector<long double> &re, std::vector<long double> &im) {   // in place, radix 2, forward
  const size_t n = re.size();
  for (size_t i = 1, j = 0; i < n; ++i) {
    size_t bit = n >> 1;
    for (; j & bit; bit >>= 1) j ^= bit;
    j ^= bit;
    if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
  }
  const long double pi = 3.141592653589793238462643383279502884L;
  for (size_t len = 2; len <= n; len <<= 1) {
    const long double ang = -2.0L * pi / (long double)len;
    for (size_t i = 0; i < n; i += len) {
      for (size_t k = 0; k < len / 2; ++k) {
        const long double wr = cosl(ang * k), wi = sinl(ang * k);
        const size_t a = i + k, b = i + k + len / 2;
        const long double xr = re[b] * wr - im[b] * wi, xi = re[b] * wi + im[b] * wr;
        re[b] = re[a] - xr; im[b] = im[a] - xi;
        re[a] += xr; im[a] += xi;
      }
    }
  }
}
template <typename T> struct BsCache {
  std::mutex mu;
  std::map<std::tuple<int, int, int>, std::pair<void *, void *>> tab;
};
template <typename T> BsCache<T> &bs_cache() {
  static BsCache<T> c;
  return c;
}
}  // namespace

template <typename T> int bluestein_tables(int n, int M, const cplx<T> **chirp, const cplx<T> **chat) {
  BsCache<T> &c = bs_cache<T>();
  std::lock_guard<std::mutex> lk(c.mu);
  const auto key = std::make_tuple(tl_device, n, M);
  auto it = c.tab.find(key);
  if (it == c.tab.end()) {
    const long double pi = 3.141592653589793238462643383279502884L;
    std::vector<cplx<T>> hc(n), hh(M);
    std::vector<long double> br(M, 0.0L), bi(M, 0.0L);
    for (int t = 0; t < n; ++t) {
      // pi t^2 / n with t^2 reduced modulo 2n in integers: the phase stays exact for any t
      const long long q = ((long long)t * t) % (2LL * n);
      const long double ang = pi * (long double)q / (long double)n;
      hc[t] = mk<T>((T)cosl(ang), (T)-sinl(ang));          // exp(-i pi t^2 / n)
      br[t] = cosl(ang); bi[t] = sinl(ang);                // conj chirp, wrapped: b[M - t] = b[t]
      if (t) { br[M - t] = br[t]; bi[M - t] = bi[t]; }
    }
    host_fft(br, bi);
    for (int k = 0; k < M; ++k) hh[k] = mk<T>((T)(br[k] / M), (T)(bi[k] / M));
    void *d1 = nullptr, *d2 = nullptr;
    WTB_CUDA(cudaMalloc(&d1, sizeof(cplx<T>) * n));
    WTB_CUDA(cudaMalloc(&d2, sizeof(cplx<T>) * M));
    WTB_CUDA(cudaMemcpy(d1, hc.data(), sizeof(cplx<T>) * n, cudaMemcpyHostToDevice));
    WTB_CUDA(cudaMemcpy(d2, hh.data(), sizeof(cplx<T>) * M, cudaMemcpyHostToDevice));
    it = c.tab.emplace(key, std::make_pair(d1, d2)).first;
  }
  *chirp = (const cplx<T> *)it->second.first;
  *chat = (const cplx<T> *)it->second.second;
  return WTB_OK;
}
template int bluestein_tables<float>(int, int, const cplx<float> **, const cplx<float> **);
template int bluestein_tables<double>(int, int, const cplx<double> **, const cplx<double> **);

void wct_fast_release();  // wct_fast.cu: the radix-16 twiddle tables
void cwt_long_release();  // cwt_long.cu: the inter-pass twiddle tables
void pool_shutdown();      // multi.cu

static void free_tables() {
  {
    BsCache<float> &c = bs_cache<float>();
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto &kv : c.tab) { cudaFree(kv.second.first); cudaFree(kv.second.second); }
    c.tab.clear();
  }
  {
    BsCache<double> &c = bs_cache<double>();
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto &kv : c.tab) { cudaFree(kv.second.first); cudaFree(kv.second.second); }
    c.tab.clear();
  }
  {
    TwCache<float> &c = tw_cache<float>();
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto &kv : c.tab) cudaFree(kv.second);
    c.tab.clear();
  }
  {
    TwCache<double> &c = tw_cache<double>();
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto &kv : c.tab) cudaFree(kv.second);
    c.tab.clear();
  }
}

// ---- axes --------------------------------------------------------------------------
int resolve_axes(int n0, double dt, double dj, double s0, int J, double f0, Axes *ax) {
  Mother m;
  m.param = f0;
  return resolve_axes(n0, dt, dj, s0, J, m, ax);
}

int resolve_axes(int n0, double dt, double dj, double s0, int J, const Mother &m, Axes *ax) {
  WTB_REQUIRE(n0 > 0 && dt > 0 && dj > 0, WTB_EINVAL, "n0, dt and dj must be positive");
  WTB_REQUIRE(m.kind == WTB_MORLET || m.kind == WTB_PAUL || m.kind == WTB_DOG, WTB_EINVAL, "unknown mother wavelet %d", m.kind);
  WTB_REQUIRE(m.kind == WTB_MORLET ? m.param > 0 : (m.param >= 1 && m.param <= 40 && m.param == std::floor(m.param)),
              WTB_EINVAL, "mother wavelet parameter %g out of range", m.param);
  const double fl = mother_flambda(m);
  if (s0 == -1) s0 = 2 * dt / fl;
  WTB_REQUIRE(s0 > 0, WTB_EINVAL, "s0 must be positive (or -1)");
  if (J == -1) J = (int)std::nearbyint(std::log2(n0 * dt / s0) / dj);
  WTB_REQUIRE(J >= 0 && J < 4096, WTB_EINVAL, "J=%d out of range", J);
  ax->J = J;
  ax->scales.resize(J + 1);
  ax->freqs.resize(J + 1);
  for (int j = 0; j <= J; ++j) {
    ax->scales[j] = s0 * std::pow(2.0, j * dj);
    ax->freqs[j] = 1.0 / (fl * ax->scales[j]);
  }
  return WTB_OK;
}

}  // namespace wtb

using namespace wtb;

extern "C" {

int wtb_version(void) { return 100; }

uint64_t wtb_kernel_launches(void) { return wtb::launches(); }

int wtb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int wtb_init(int device) {
  WTB_TRY(check_device(device));
  {
    std::lock_guard<std::mutex> lk(g_mu);
    g_default_device = device;
  }
  // one process per GPU (torchrun): also make it the calling thread's current device
  WTB_CUDA(cudaSetDevice(device));
  return WTB_OK;
}

void wtb_shutdown(void) {
  pool_shutdown();
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  {
    // the sets stay with their threads (they are reused if the thread calls again); their
    // memory goes now.  release_set's cudaFree waits for the work that uses each block.
    std::lock_guard<std::mutex> lk(g_arena_mu);
    for (ArenaSet *s : g_sets) release_set(s);
  }
  free_tables();
  wct_fast_release();
  cwt_long_release();
  cudaSetDevice(cur);
  std::lock_guard<std::mutex> lk(g_mu);
  g_default_device = -1;
}

uint64_t wtb_scratch_bytes(void) { return (uint64_t)scratch_bytes_held(); }

const char *wtb_last_error(void) { return g_err; }

int wtb_cwt_axes_mother(int n0, double dt, double dj, double s0, int J, int mother, double param, int *J_out,
                        double *scales, double *freqs, double *coi) {
  Axes ax;
  Mother m;
  m.kind = mother;
  m.param = param;
  WTB_TRY(resolve_axes(n0, dt, dj, s0, J, m, &ax));
  if (J_out) *J_out = ax.J;
  for (int j = 0; j <= ax.J; ++j) {
    if (scales) scales[j] = ax.scales[j];
    if (freqs) freqs[j] = ax.freqs[j];
  }
  if (coi) {
    // pycwt.cwt: flambda * coi() * dt * (n0/2 - |t - (n0-1)/2|), coi() = 1/sqrt(2) for Morlet
    const double c = mother_flambda(m) * mother_coi(m) * dt;
    for (int t = 0; t < n0; ++t) coi[t] = c * (n0 / 2.0 - std::fabs(t - (n0 - 1) / 2.0));
  }
  return WTB_OK;
}

int wtb_cwt_axes(int n0, double dt, double dj, double s0, int J, double f0, int *J_out,
                 double *scales, double *freqs, double *coi) {
  return wtb_cwt_axes_mother(n0, dt, dj, s0, J, WTB_MORLET, f0, J_out, scales, freqs, coi);
}

int wtb_wct_mc_geometry(double dt, double dj, double s0, int J, double f0, int *nsurr, int *maxscale) {
  WTB_REQUIRE(J >= 0, WTB_EINVAL, "wct_significance needs a resolved J >= 0");
  const double fl = morlet_flambda(f0);
  if (s0 == -1) s0 = 2 * dt / fl;
  const double ms = s0 * std::pow(2.0, J * dj) / dt;
  const int N = (int)std::ceil(ms * 6);
  WTB_REQUIRE(N > 1, WTB_EINVAL, "degenerate surrogate length %d", N);
  if (nsurr) *nsurr = N;
  if (maxscale) {
    // largest s with any t such that period[s] <= coi[t]; max coi is at the centre
    const double c = fl / std::sqrt(2.0) * dt;
    double coimax = 0;
    for (int t = 0; t < N; ++t) coimax = std::fmax(coimax, c * (N / 2.0 - std::fabs(t - (N - 1) / 2.0)));
    int m = 0;
    for (int j = 0; j <= J; ++j) {
      const double freq = 1.0 / (fl * (s0 * std::pow(2.0, j * dj)));
      const double period = 1.0 / freq;  // same rounding path as pycwt
      if (period <= coimax) m = j;
    }
    *maxscale = m;
  }
  return WTB_OK;
}

int wtb_wct_sig_from_hist(const uint64_t *hist, int S, int maxscale, double level,
                          const uint8_t *row_has_points, double *sig95) {
  WTB_REQUIRE(hist && sig95 && S > 0, WTB_EINVAL, "null argument");
  WTB_REQUIRE(maxscale >= 0 && maxscale <= S, WTB_EINVAL, "maxscale out of range");
  const int nb = WTB_NBINS;
  for (int s = 0; s < S; ++s) sig95[s] = (row_has_points && row_has_points[s]) ? NAN : 0.0;
  std::vector<double> P, Y;
  for (int s = 0; s < maxscale; ++s) {
    P.clear();
    Y.clear();
    double cum = 0;
    for (int b = 0; b < nb; ++b) {
      const uint64_t c = hist[(size_t)s * nb + b];
      if (c == 0) continue;
      cum += (double)c;
      P.push_back(cum);
      Y.push_back((b + 0.5) / nb);
    }
    if (P.empty()) { sig95[s] = NAN; continue; }
    const double tot = P.back();
    for (double &p : P) p = (p - 0.5) / tot;
    // np.interp(level, P, Y): clamps outside, linear inside
    double v;
    if (level <= P.front()) v = Y.front();
    else if (level >= P.back()) v = Y.back();
    else {
      size_t i = 1;
      while (P[i] < level) ++i;
      // numpy picks the interval [i-1, i] with P[i-1] <= level < P[i] (ties -> later)
      while (i + 1 < P.size() && P[i] <= level) ++i;
      const double slope = (Y[i] - Y[i - 1]) / (P[i] - P[i - 1]);
      v = slope * (level - P[i - 1]) + Y[i - 1];
    }
    sig95[s] = v;
  }
  return WTB_OK;
}

int wtb_dwt_max_level(int n, int L) {
  if (L < 2 || n < L - 1) return 0;
  int lev = (int)std::floor(std::log2((double)n / (L - 1.0)));
  return lev < 0 ? 0 : lev;
}

int wtb_dwt_coeff_lens(int n, int L, int level, int *lens) {
  WTB_REQUIRE(n > 0 && L >= 2 && level >= 0 && lens, WTB_EINVAL, "bad dwt_coeff_lens arguments");
  int cur = n;
  for (int l = 0; l < level; ++l) {
    cur = (cur + L - 1) / 2;
    lens[level - l] = cur;  // cD_{l+1}
  }
  lens[0] = cur;  // cA_level (== n when level == 0)
  return WTB_OK;
}

int wtb_waverec_len(const int *lens, int level, int L) {
  if (!lens || level < 0) return WTB_EINVAL;
  int a = lens[0];
  for (int l = 1; l <= level; ++l) {
    const int d = lens[l];
    if (a == d + 1) a -= 1;
    if (a != d) { set_error("waverec: coefficient lengths %d and %d do not match", a, d); return WTB_EINVAL; }
    a = 2 * d - L + 2;
    if (a <= 0) { set_error("waverec: level too short for the filter"); return WTB_EINVAL; }
  }
  return a;
}

}  // extern "C"
