// One call, every GPU of the box (SURVEY 8e: the reference's only call sites are single-process --
// src/wct.py:106-118 `wavelet.wct(..., sig=True)` and the batched runners of
// src/utils/transform_helpers.py -- so the sharding lives inside the library, not in a launcher).
//
//   wtb_init_multi(n)        one worker thread + one stream per device, peer access enabled
//   run_sharded(...)         contiguous blocks of a batch (series, pairs, realisations) per device
//   wtb_wct_significance     Monte-Carlo realisation blocks keyed by GLOBAL index on every device,
//                            per-device uint64 histograms, summed by ONE kernel on device 0 that
//                            reads its peers' histograms directly over NVLink (P2P loads through
//                            NVSwitch: 8 x 528 KB), then the percentile step.
// The exchange is 528 KB per device once per call: a peer-load kernel is one launch (~10 us); a
// ring/tree collective would add protocol latency and a dependency for nothing.  Without peer
// access (PCIe-only boxes) the histograms are summed on the host.
#include <condition_variable>
#include <functional>
#include <memory>
#include <thread>

#include "cwt_paths.cuh"

namespace wtb {

extern thread_local int tl_worker_device;   // runtime.cu: CallScope picks this device on pool threads

namespace {

constexpr int kMaxPool = 16;

struct Worker {
  int device = -1;
  cudaStream_t stream = nullptr;
  unsigned long long *d_hist = nullptr;   // Monte-Carlo histogram of this device (plain cudaMalloc: peer-mappable)
  size_t hist_cap = 0;
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  bool has_job = false, done = false, stop = false;
  int rc = WTB_OK;
  int init_rc = WTB_OK;
  bool ready = false;
  char err[512] = "";
};

struct Pool {
  std::vector<std::unique_ptr<Worker>> w;
  bool peer = false;       // device 0 can load from every other pool device
};

std::mutex g_pool_mu;       // guards g_pool itself
std::mutex g_call_mu;       // one sharded call at a time (workers and their streams are shared)
Pool *g_pool = nullptr;

void worker_main(Worker *w) {
  tl_worker_device = w->device;
  cudaError_t e = cudaSetDevice(w->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking);
  {
    std::lock_guard<std::mutex> lk(w->mu);
    if (e != cudaSuccess) {
      w->init_rc = WTB_ECUDA;
      snprintf(w->err, sizeof(w->err), "device %d: %s", w->device, cudaGetErrorString(e));
    }
    w->ready = true;
  }
  w->cv.notify_all();
  if (e != cudaSuccess) return;
  for (;;) {
    std::function<int()> job;
    {
      std::unique_lock<std::mutex> lk(w->mu);
      w->cv.wait(lk, [&] { return w->has_job || w->stop; });
      if (w->stop) break;
      job = std::move(w->job);
      w->has_job = false;
    }
    int rc;
    {
      CallScope scope(0, nullptr, w->stream);   // device + scratch key of this worker
      rc = scope.rc();
      if (rc == WTB_OK) rc = job();
      if (rc == WTB_OK) {
        cudaError_t se = cudaStreamSynchronize(w->stream);
        if (se != cudaSuccess) rc = cuda_fail(se, "cudaStreamSynchronize(worker)", __FILE__, __LINE__);
      }
    }
    {
      std::lock_guard<std::mutex> lk(w->mu);
      w->rc = rc;
      if (rc != WTB_OK) snprintf(w->err, sizeof(w->err), "%s", last_error());
      w->done = true;
    }
    w->cv.notify_all();
  }
  if (w->d_hist) cudaFree(w->d_hist);
  cudaStreamDestroy(w->stream);
}

void submit(Worker *w, std::function<int()> job) {
  {
    std::lock_guard<std::mutex> lk(w->mu);
    w->job = std::move(job);
    w->has_job = true;
    w->done = false;
  }
  w->cv.notify_all();
}

int wait(Worker *w) {
  std::unique_lock<std::mutex> lk(w->mu);
  w->cv.wait(lk, [&] { return w->done; });
  return w->rc;
}

// first failure wins; its text becomes the calling thread's wtb_last_error()
int wait_all(Pool *p, int n) {
  int rc = WTB_OK;
  for (int i = 0; i < n; ++i) {
    const int r = wait(p->w[i].get());
    if (r != WTB_OK && rc == WTB_OK) {
      rc = r;
      set_error("GPU %d: %s", p->w[i]->device, p->w[i]->err);
    }
  }
  return rc;
}

void destroy_pool(Pool *p) {
  for (auto &w : p->w) {
    {
      std::lock_guard<std::mutex> lk(w->mu);
      w->stop = true;
    }
    w->cv.notify_all();
    if (w->th.joinable()) w->th.join();
  }
  delete p;
}

// dst[i] += sum over peers of src_p[i]: device 0 pulls its peers' histograms through NVLink
struct PeerPtrs {
  const unsigned long long *p[kMaxPool];
};
__global__ void k_hist_reduce_peers(unsigned long long *__restrict__ dst, PeerPtrs peers, int n_peers, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long acc = dst[i];
  for (int q = 0; q < n_peers; ++q) acc += __ldcv(peers.p[q] + i);   // remote, never cached
  dst[i] = acc;
}

}  // namespace

int pool_size() {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  return g_pool ? (int)g_pool->w.size() : 1;
}

void pool_shutdown() {
  std::lock_guard<std::mutex> call(g_call_mu);
  Pool *p = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    p = g_pool;
    g_pool = nullptr;
  }
  if (p) destroy_pool(p);
}

int run_sharded(int64_t total, int64_t min_total, cudaStream_t caller_stream, ShardFn fn, void *ctx) {
  // a pool worker that reaches a sharding entry point runs its block on its own device
  if (pool_size() < 2 || tl_worker_device >= 0 || total < min_total || total < 2)
    return fn(ctx, 0, 0, total, caller_stream);
  // the pool is only read under the call lock: wtb_init_multi / wtb_shutdown take the same lock
  // before they tear it down
  std::lock_guard<std::mutex> call(g_call_mu);
  Pool *p = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    p = g_pool;
  }
  if (!p) return fn(ctx, 0, 0, total, caller_stream);
  const int G = (int)std::min<int64_t>((int64_t)p->w.size(), total);
  for (int r = 0; r < G; ++r) {
    const int64_t first = total * r / G, count = total * (r + 1) / G - first;
    Worker *w = p->w[r].get();
    submit(w, [=]() { return fn(ctx, r, first, count, w->stream); });
  }
  return wait_all(p, G);
}

}  // namespace wtb

using namespace wtb;

extern "C" int wtb_gpu_count(void) { return pool_size(); }

extern "C" int wtb_init_multi(int n_gpus) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device visible (%s); libwavelet_sm100a has no CPU fallback",
              e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
    cudaGetLastError();
    return WTB_ENODEVICE;
  }
  if (n_gpus <= 0) {
    n_gpus = count;
    if (const char *env = getenv("WTB_GPUS")) n_gpus = atoi(env);
  }
  // WTB_POOL_SHARE_DEVICES=1 lets the pool be larger than the box (workers r and r + count share
  // device r % count): the sharding, the per-worker scratch and the peer reduction can then be
  // exercised on a single-GPU machine.  Not a performance mode.
  const bool share = getenv("WTB_POOL_SHARE_DEVICES") && atoi(getenv("WTB_POOL_SHARE_DEVICES"));
  WTB_REQUIRE(n_gpus >= 1 && (n_gpus <= count || share) && n_gpus <= kMaxPool, WTB_EINVAL,
              "wtb_init_multi: %d GPUs requested, %d visible (at most %d)", n_gpus, count, kMaxPool);
  pool_shutdown();
  if (n_gpus == 1) return WTB_OK;     // a single device needs no workers
  int cur = 0;
  WTB_CUDA(cudaGetDevice(&cur));
  Pool *p = new Pool();
  for (int r = 0; r < n_gpus; ++r) {
    const int d = r % count;
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d);
    if (major != 10) {
      destroy_pool(p);
      set_error("device %d is sm_%dx; this library is built for sm_100a only", d, major);
      return WTB_ENODEVICE;
    }
    auto w = std::make_unique<Worker>();
    w->device = d;
    w->th = std::thread(worker_main, w.get());
    p->w.push_back(std::move(w));
  }
  for (auto &w : p->w) {
    std::unique_lock<std::mutex> lk(w->mu);
    w->cv.wait(lk, [&] { return w->ready; });
    if (w->init_rc != WTB_OK) {
      set_error("wtb_init_multi: %s", w->err);
      lk.unlock();
      destroy_pool(p);
      return WTB_ECUDA;
    }
  }
  // device 0 reads its peers' histograms directly: enable the mappings once
  p->peer = true;
  cudaSetDevice(0);
  for (int d = 1; d < std::min(n_gpus, count); ++d) {
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, 0, d) != cudaSuccess || !can) {
      p->peer = false;
      break;
    }
    e = cudaDeviceEnablePeerAccess(d, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) p->peer = false;
    cudaGetLastError();
  }
  if (const char *env = getenv("WTB_NO_PEER")) {
    if (atoi(env)) p->peer = false;
  }
  cudaSetDevice(cur);
  std::lock_guard<std::mutex> lk(g_pool_mu);
  g_pool = p;
  return WTB_OK;
}

// ---- Monte-Carlo significance in one call: replaces pycwt.wct_significance as reached from
// pycwt.wct(sig=True) (src/wct.py:106-118) ------------------------------------------------------
extern "C" int wtb_wct_significance(double a1, double a2, double dt, double dj, double s0, int J, double f0,
                                    double level, int64_t mc_count, uint64_t seed, const void *surrogates,
                                    int flags, double *sig95, uint64_t *hist_out) {
  WTB_REQUIRE(sig95 && mc_count >= 0, WTB_EINVAL, "wtb_wct_significance: bad arguments");
  WTB_REQUIRE(!(flags & WTB_DEVICE_PTRS), WTB_EINVAL, "wtb_wct_significance takes host buffers only");
  WTB_REQUIRE(J >= 0, WTB_EINVAL, "wtb_wct_significance needs a resolved J");
  int nsurr = 0, maxscale = 0;
  WTB_TRY(wtb_wct_mc_geometry(dt, dj, s0, J, f0, &nsurr, &maxscale));
  Axes ax;
  WTB_TRY(resolve_axes(nsurr, dt, dj, s0, J, f0, &ax));
  const int S = J + 1;
  const size_t cells = (size_t)S * WTB_NBINS;
  std::vector<uint8_t> any;
  mc_row_has_points(nsurr, dt, ax, f0, &any);
  std::vector<uint64_t> hist(cells, 0);

  const int G = (int)std::min<int64_t>(pool_size(), std::max<int64_t>(mc_count, 1));
  if (G < 2) {
    WTB_TRY(wtb_wct_mc_hist(a1, a2, dt, dj, s0, J, f0, 0, mc_count, seed, surrogates, flags, hist.data(), nullptr));
  } else if (surrogates) {
    // host-injected series (parity mode): each device takes a block, histograms meet on the host
    std::vector<std::vector<uint64_t>> part(G, std::vector<uint64_t>(cells, 0));
    const size_t pair_bytes = ((flags & WTB_F64) ? 8 : 4) * 2 * (size_t)nsurr;
    const int rc = run_sharded_fn(mc_count, 2, nullptr, [&](int r, int64_t first, int64_t count, cudaStream_t st) {
      if (r >= G) { set_error("the GPU pool changed during the call"); return WTB_EINVAL; }
      return wtb_wct_mc_hist(a1, a2, dt, dj, s0, J, f0, first, count, seed, (const char *)surrogates + first * pair_bytes,
                             flags, part[r].data(), st);
    });
    if (rc != WTB_OK) return rc;
    for (int r = 0; r < G; ++r)
      for (size_t i = 0; i < cells; ++i) hist[i] += part[r][i];
  } else {
    std::lock_guard<std::mutex> call(g_call_mu);      // the pool is only read (and torn down) under this lock
    Pool *p = nullptr;
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      p = g_pool;
    }
    if (!p || (int)p->w.size() < G) {                 // the pool went away between the two looks
      WTB_TRY(wtb_wct_mc_hist(a1, a2, dt, dj, s0, J, f0, 0, mc_count, seed, nullptr, flags, hist.data(), nullptr));
      if (hist_out) std::memcpy(hist_out, hist.data(), sizeof(uint64_t) * cells);
      return wtb_wct_sig_from_hist(hist.data(), S, maxscale, level, any.data(), sig95);
    }
    // phase 1: every device bins its block of realisations into its own histogram
    for (int r = 0; r < G; ++r) {
      Worker *w = p->w[r].get();
      const int64_t first = mc_count * r / G, count = mc_count * (r + 1) / G - first;
      submit(w, [=]() -> int {
        if (w->hist_cap < cells) {
          if (w->d_hist) WTB_CUDA(cudaFree(w->d_hist));
          w->d_hist = nullptr;
          WTB_CUDA(cudaMalloc(&w->d_hist, sizeof(uint64_t) * cells));
          w->hist_cap = cells;
        }
        WTB_CUDA(cudaMemsetAsync(w->d_hist, 0, sizeof(uint64_t) * cells, w->stream));
        return wtb_wct_mc_hist(a1, a2, dt, dj, s0, J, f0, first, count, seed, nullptr, flags | WTB_DEVICE_PTRS,
                               (uint64_t *)w->d_hist, w->stream);
      });
    }
    WTB_TRY(wait_all(p, G));
    // phase 2: the exchange.  Device 0 sums its peers' histograms with direct NVLink loads.
    Worker *w0 = p->w[0].get();
    uint64_t *h = hist.data();
    if (p->peer) {
      PeerPtrs peers;
      for (int r = 1; r < G; ++r) peers.p[r - 1] = p->w[r]->d_hist;
      submit(w0, [=]() -> int {
        k_hist_reduce_peers<<<(unsigned)((cells + 255) / 256), 256, 0, w0->stream>>>(w0->d_hist, peers, G - 1, (int)cells);
        WTB_LAUNCH_CHECK();
        WTB_TRY(copy_to_host(h, w0->d_hist, sizeof(uint64_t) * cells, w0->stream));
        return WTB_OK;
      });
      WTB_TRY(wait(w0) == WTB_OK ? WTB_OK : (set_error("GPU 0: %s", w0->err), w0->rc));
    } else {
      std::vector<uint64_t> tmp(cells);
      for (int r = 0; r < G; ++r) {
        Worker *w = p->w[r].get();
        uint64_t *t = tmp.data();
        submit(w, [=]() -> int {
          WTB_TRY(copy_to_host(t, w->d_hist, sizeof(uint64_t) * cells, w->stream));
          return WTB_OK;
        });
        WTB_TRY(wait(w) == WTB_OK ? WTB_OK : (set_error("GPU %d: %s", w->device, w->err), w->rc));
        for (size_t i = 0; i < cells; ++i) hist[i] += tmp[i];
      }
    }
  }
  if (hist_out) std::memcpy(hist_out, hist.data(), sizeof(uint64_t) * cells);
  return wtb_wct_sig_from_hist(hist.data(), S, maxscale, level, any.data(), sig95);
}

// ---- Monte-Carlo significance of partial and multiple coherence in one call: every pool device bins its block of
// realisations into its own histogram, the host sums them (1 MB each at most: no peer reduction needed) and runs the
// percentile step on each half.
extern "C" int wtb_partial_wct_significance(double ay, double a1, double a2, double dt, double dj, double s0, int J,
                                            double f0, double level, int64_t mc_count, uint64_t seed,
                                            const void *surrogates, int flags, double *sig_pwc, double *sig_mwc,
                                            uint64_t *hist_out) {
  WTB_REQUIRE(sig_pwc && sig_mwc && mc_count >= 0, WTB_EINVAL, "wtb_partial_wct_significance: bad arguments");
  WTB_REQUIRE(!(flags & WTB_DEVICE_PTRS), WTB_EINVAL, "wtb_partial_wct_significance takes host buffers only");
  WTB_REQUIRE(J >= 0, WTB_EINVAL, "wtb_partial_wct_significance needs a resolved J");
  int nsurr = 0, maxscale = 0;
  WTB_TRY(wtb_wct_mc_geometry(dt, dj, s0, J, f0, &nsurr, &maxscale));
  Axes ax;
  WTB_TRY(resolve_axes(nsurr, dt, dj, s0, J, f0, &ax));
  const int S = J + 1;
  const size_t cells = 2 * (size_t)S * WTB_NBINS;
  std::vector<uint8_t> any;
  mc_row_has_points(nsurr, dt, ax, f0, &any);
  const int G = (int)std::min<int64_t>(pool_size(), std::max<int64_t>(mc_count, 1));
  std::vector<std::vector<uint64_t>> part(G, std::vector<uint64_t>(cells, 0));
  const size_t triple_bytes = ((flags & WTB_F64) ? 8 : 4) * 3 * (size_t)nsurr;
  WTB_TRY(run_sharded_fn(mc_count, 2, nullptr, [&](int r, int64_t first, int64_t count, cudaStream_t st) {
    if (r >= G) { set_error("the GPU pool changed during the call"); return WTB_EINVAL; }
    const void *sur = surrogates ? (const char *)surrogates + first * triple_bytes : nullptr;
    return wtb_partial_wct_mc_hist(ay, a1, a2, dt, dj, s0, J, f0, first, count, seed, sur, flags, part[r].data(), st);
  }));
  std::vector<uint64_t> hist(cells, 0);
  for (int r = 0; r < G; ++r)
    for (size_t i = 0; i < cells; ++i) hist[i] += part[r][i];
  if (hist_out) std::memcpy(hist_out, hist.data(), sizeof(uint64_t) * cells);
  WTB_TRY(wtb_wct_sig_from_hist(hist.data(), S, maxscale, level, any.data(), sig_pwc));
  return wtb_wct_sig_from_hist(hist.data() + (size_t)S * WTB_NBINS, S, maxscale, level, any.data(), sig_mwc);
}
