// api.cu -- host side of libkmergpu: the C ABI of include/kmergpu.h over the kernels in
// sort.cuh / csr.cuh / probe.cuh.  No CPU implementation of any step lives here: without a
// CUDA device every entry point fails with KMG_ERR_NODEV / KMG_ERR_CUDA.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <initializer_list>
#include <thread>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/kmergpu.h"
#include "common.cuh"
#include "csr.cuh"
#include "lookback.cuh"
#include "probe.cuh"
#include "segments.cuh"
#include "sort.cuh"
#include "windows.cuh"

using namespace kmg;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      int code_ = (e_ == cudaErrorMemoryAllocation) ? KMG_ERR_NOMEM                                \
                  : (e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver) ? KMG_ERR_NODEV \
                                                                                   : KMG_ERR_CUDA; \
      return fail(code_, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);     \
    }                                                                                              \
  } while (0)
#define TRY(call)            \
  do {                       \
    int rc_ = (call);        \
    if (rc_ != KMG_OK) return rc_; \
  } while (0)

extern "C" const char *kmg_last_error(void) { return g_err; }
extern "C" int kmg_version(void) { return 100; }

// ------------------------------------------------------------------------------------------------
// per-thread execution context
// ------------------------------------------------------------------------------------------------
struct Ctx {
  int device = 0;
  bool ready = false;
  cudaStream_t own = nullptr, copy = nullptr;   // compute stream, second stream for overlapped copies
  cudaStream_t user = nullptr;
  bool use_user = false;
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [0..1] kernel done, [2..3] copy done, [4..6] staging slot done
  int sms = 148;
  cudaStream_t stream() const { return use_user ? user : own; }
};
static thread_local Ctx g_ctx;

static int ctx_init() {
  Ctx &c = g_ctx;
  if (c.ready) {
    CU(cudaSetDevice(c.device));
    return KMG_OK;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(KMG_ERR_NODEV, "no CUDA device: %s (libkmergpu has no CPU path)", cudaGetErrorString(e));
  if (c.device >= n) return fail(KMG_ERR_ARG, "device %d out of range (have %d)", c.device, n);
  CU(cudaSetDevice(c.device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, c.device));
  if (prop.major != 10 || prop.minor != 0)     // the library carries sm_100a SASS only (no PTX): other parts cannot run it
    return fail(KMG_ERR_NODEV, "device %d is sm_%d%d; libkmergpu is built for sm_100a (B200) only", c.device, prop.major, prop.minor);
  c.sms = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&c.own, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c.copy, cudaStreamNonBlocking));
  for (auto &ev : c.ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  c.ready = true;
  return KMG_OK;
}

extern "C" int kmg_device_count(int *n) {
  if (!n) return fail(KMG_ERR_ARG, "n is NULL");
  cudaError_t e = cudaGetDeviceCount(n);
  if (e != cudaSuccess) { *n = 0; return fail(KMG_ERR_NODEV, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
  return KMG_OK;
}
extern "C" int kmg_set_device(int device) {
  if (device < 0) return fail(KMG_ERR_ARG, "negative device");
  if (g_ctx.ready && g_ctx.device != device) {   // new device: new streams
    g_ctx = Ctx();
  }
  g_ctx.device = device;
  return ctx_init();
}
extern "C" int kmg_set_stream(void *s) {
  g_ctx.user = (cudaStream_t)s;
  g_ctx.use_user = true;                          // NULL = the legacy default stream
  return KMG_OK;
}
extern "C" int kmg_unset_stream(void) { g_ctx.use_user = false; return KMG_OK; }
extern "C" void *kmg_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (ctx_init() != KMG_OK) return nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { fail(KMG_ERR_NOMEM, "cudaMallocHost(%zu) failed", bytes); return nullptr; }
  return p;
}
extern "C" void kmg_host_free(void *p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------------
// profiling: optional CUDA-event bracket around every kernel launch
// ------------------------------------------------------------------------------------------------
struct ProfEntry { double ms = 0; uint64_t launches = 0; double bytes = 0; };
struct ProfPending { std::string name; cudaEvent_t a, b; };
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::map<std::string, ProfEntry> g_prof;
static std::vector<ProfPending> g_prof_pending;
static std::vector<cudaEvent_t> g_prof_free;
static uint64_t g_launches = 0;

static cudaEvent_t prof_event() {
  if (!g_prof_free.empty()) { cudaEvent_t e = g_prof_free.back(); g_prof_free.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
static void prof_resolve() {   // caller holds the mutex; pending events must have completed
  for (auto &p : g_prof_pending) {
    float ms = 0;
    if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
      g_prof[p.name].ms += ms;
    }
    g_prof_free.push_back(p.a);
    g_prof_free.push_back(p.b);
  }
  g_prof_pending.clear();
}
struct LaunchScope {
  const char *name;
  cudaStream_t s;
  cudaEvent_t a = nullptr, b = nullptr;
  bool on;
  LaunchScope(const char *n, cudaStream_t st) : name(n), s(st) {
    std::lock_guard<std::mutex> g(g_prof_mu);
    on = g_prof_on;
    ++g_launches;
    if (on) { a = prof_event(); b = prof_event(); cudaEventRecord(a, s); }
  }
  ~LaunchScope() {
    if (!on) return;
    cudaEventRecord(b, s);
    std::lock_guard<std::mutex> g(g_prof_mu);
    g_prof[name].launches++;
    g_prof_pending.push_back({name, a, b});
  }
};
static void prof_bytes(const char *name, double bytes) {
  std::lock_guard<std::mutex> g(g_prof_mu);
  if (g_prof_on) g_prof[name].bytes += bytes;
}
#define LAUNCH(name, stream, ...)                                                              \
  do {                                                                                         \
    { LaunchScope ls_(name, stream); __VA_ARGS__; }                                            \
    cudaError_t le_ = cudaGetLastError();                                                      \
    if (le_ != cudaSuccess) return fail(KMG_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(le_)); \
  } while (0)

extern "C" int kmg_profile_enable(int on) { std::lock_guard<std::mutex> g(g_prof_mu); g_prof_on = on != 0; return KMG_OK; }
extern "C" int kmg_profile_reset(void) {
  std::lock_guard<std::mutex> g(g_prof_mu);
  prof_resolve();
  g_prof.clear();
  return KMG_OK;
}
extern "C" int kmg_profile_count(void) {
  std::lock_guard<std::mutex> g(g_prof_mu);
  prof_resolve();
  return (int)g_prof.size();
}
extern "C" int kmg_profile_get(int i, const char **name, double *total_ms, uint64_t *launches, double *algo_bytes) {
  std::lock_guard<std::mutex> g(g_prof_mu);
  prof_resolve();
  if (i < 0 || i >= (int)g_prof.size()) return fail(KMG_ERR_ARG, "profile index out of range");
  auto it = g_prof.begin();
  std::advance(it, i);
  if (name) *name = it->first.c_str();
  if (total_ms) *total_ms = it->second.ms;
  if (launches) *launches = it->second.launches;
  if (algo_bytes) *algo_bytes = it->second.bytes;
  return KMG_OK;
}
extern "C" uint64_t kmg_launch_count(void) { std::lock_guard<std::mutex> g(g_prof_mu); return g_launches; }

// ------------------------------------------------------------------------------------------------
// memory helpers
// ------------------------------------------------------------------------------------------------
// Device memory comes from a small caching arena (per device, thread safe): freed blocks are kept
// and handed back to requests of (nearly) the same size.  Index builds repeat the same sizes, so
// after the first build nothing touches the driver allocator.  (The driver's stream-ordered pool
// was tried first: its block reuse across differing request patterns stalled builds for 10 ms to
// seconds, see profiles/r01_notes.md.)
struct Arena {
  struct Block { void *p; size_t cap; cudaStream_t last; bool synced; };
  std::mutex mu;
  std::multimap<size_t, Block> cache;            // free blocks by capacity
  std::map<void *, Block> live;
  size_t cached_bytes = 0, limit = 0;

  static size_t round_up(size_t bytes) {
    if (bytes < (size_t(1) << 20)) return (bytes + 511) & ~size_t(511);
    return (bytes + (size_t(2) << 20) - 1) & ~((size_t(2) << 20) - 1);
  }
  void trim_locked() {
    for (auto &kv : cache) cudaFree(kv.second.p);
    cache.clear();
    cached_bytes = 0;
  }
  int get(void **out, size_t bytes, cudaStream_t s) {
    const size_t cap = round_up(bytes ? bytes : 1);
    std::unique_lock<std::mutex> g(mu);
    auto it = cache.lower_bound(cap);
    if (it != cache.end() && it->first <= cap + std::max(cap / 4, size_t(1) << 20)) {
      Block b = it->second;
      cache.erase(it);
      cached_bytes -= b.cap;
      g.unlock();
      if (!b.synced && b.last != s) cudaStreamSynchronize(b.last);   // last user was another stream
      g.lock();
      b.last = s; b.synced = false;
      live[b.p] = b;
      *out = b.p;
      return KMG_OK;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, cap);
    if (e != cudaSuccess) {                       // give the cache back to the driver and retry once
      cudaGetLastError();
      trim_locked();
      e = cudaMalloc(&p, cap);
    }
    if (e != cudaSuccess) { cudaGetLastError(); return fail(KMG_ERR_NOMEM, "device allocation of %zu bytes failed: %s", cap, cudaGetErrorString(e)); }
    live[p] = Block{p, cap, s, false};
    *out = p;
    return KMG_OK;
  }
  void put(void *p, cudaStream_t s, bool synced) {
    if (!p) return;
    std::lock_guard<std::mutex> g(mu);
    auto it = live.find(p);
    if (it == live.end()) {
      for (auto &kv : cache) if (kv.second.p == p) return;   // already given back: a second put must not free a cached block
      cudaFree(p);                                            // not from this arena (or from before a trim)
      return;
    }
    Block b = it->second;
    live.erase(it);
    b.last = s; b.synced = synced;
    if (limit == 0) {                                   // KMERGPU_CACHE_MB, else a quarter of the device
      const char *e = getenv("KMERGPU_CACHE_MB");
      size_t fr = 0, tot = 0;
      if (e && atoll(e) >= 0) limit = (size_t)atoll(e) << 20;
      else limit = cudaMemGetInfo(&fr, &tot) == cudaSuccess ? tot / 4 : (size_t(32) << 30);
      if (limit == 0) limit = 1;
    }
    if (cached_bytes + b.cap > limit) trim_locked();
    cache.emplace(b.cap, b);
    cached_bytes += b.cap;
  }
};
static Arena g_arena[64];

// Give the cached device blocks of this thread's device back to the driver (live indexes are untouched).  An R
// session calls it (or sets KMERGPU_CACHE_MB=0) when it wants the memory of freed indexes returned at once.
static void stage_release();
extern "C" int kmg_trim(void) {
  TRY(ctx_init());
  cudaStreamSynchronize(g_ctx.stream());
  Arena &a = g_arena[g_ctx.device & 63];
  std::lock_guard<std::mutex> g(a.mu);
  for (auto &kv : a.cache) if (!kv.second.synced && kv.second.last && kv.second.last != g_ctx.stream()) cudaStreamSynchronize(kv.second.last);
  a.trim_locked();
  stage_release();
  return KMG_OK;
}
extern "C" uint64_t kmg_cached_bytes(void) {
  Arena &a = g_arena[g_ctx.device & 63];
  std::lock_guard<std::mutex> g(a.mu);
  return a.cached_bytes;
}

template <typename T>
static int dalloc(T **p, size_t count, cudaStream_t s) {
  *p = nullptr;
  return g_arena[g_ctx.device & 63].get((void **)p, (count ? count : 1) * sizeof(T), s);
}
template <typename T>
static void dfree(T *&p, cudaStream_t s) {
  if (p) g_arena[g_ctx.device & 63].put((void *)p, s, false);
  p = nullptr;
}

// One arena block of T owned by a scope: given back on the stream it was taken on when the scope ends, earlier by
// reset(), never once release() has handed it to an index or handle.  It cannot be copied, so a block has one owner;
// kernels and the emit lambdas of stream_rows take the raw pointer.  The unnamed namespace keeps
// these helpers out of the library's exported symbols.
namespace {
template <typename T>
class DevBuf {
  T *p_ = nullptr;
  cudaStream_t s_;
 public:
  explicit DevBuf(cudaStream_t s, T *owned = nullptr) : p_(owned), s_(s) {}
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { reset(); }
  int alloc(size_t count) { reset(); return dalloc(&p_, count, s_); }   // gives back the block it held first
  void reset(T *owned = nullptr) { dfree(p_, s_); p_ = owned; }
  T *release() { T *p = p_; p_ = nullptr; return p; }
  T *get() const { return p_; }
  operator T *() const { return p_; }
};

// Handles owned by a scope until they are handed out: freed by their kmg_*_free on every other path.
template <auto Free>
struct Freer { template <class H> void operator()(H *h) const { Free(h); } };
using IndexPtr = std::unique_ptr<kmg_index, Freer<kmg_free>>;
using QueryPtr = std::unique_ptr<kmg_query, Freer<kmg_query_free>>;
using JoinPtr = std::unique_ptr<kmg_join, Freer<kmg_join_free>>;
using SegmentsPtr = std::unique_ptr<kmg_segments, Freer<kmg_segments_free>>;
using ChainsPtr = std::unique_ptr<kmg_chains, Freer<kmg_chains_free>>;
using ReadsPtr = std::unique_ptr<kmg_reads, Freer<kmg_reads_free>>;
}  // namespace

// A handle's arrays back to the arena of its device.  May run on a finaliser thread that never used the library, so the
// device's work is waited for first and the blocks are made reusable by any stream.
static void release_on_device(int device, std::initializer_list<void *> ptrs) {
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(device);
  const bool mine = g_ctx.ready && g_ctx.device == device;
  if (mine) cudaStreamSynchronize(g_ctx.stream()); else cudaDeviceSynchronize();
  for (void *p : ptrs) g_arena[device & 63].put(p, nullptr, true);
  cudaGetLastError();
  if (prev >= 0) cudaSetDevice(prev);
}

// A handle is used on the device it lives on: this thread's streams, events and arena belong to its current device
// (kmg_set_device), so a handle of another device is refused rather than driven with the wrong resources.
static int use_device(int device, const char *what) {
  TRY(ctx_init());
  if (device == g_ctx.device) return KMG_OK;
  return fail(KMG_ERR_ARG, "%s on device %d but this thread works on device %d: call kmg_set_device(%d) first", what, device, g_ctx.device, device);
}

// ------------------------------------------------------------------------------------------------
// pageable host buffers at PCIe speed: pinned staging + host copy threads
// ------------------------------------------------------------------------------------------------
// R hands the glue ordinary (pageable) memory: CHAR(STRING_ELT()) for the sequence, INTEGER(allocMatrix()) for the
// results (src/kmer_hash.c:1127-1140 of the reference memcpy's into the same kind).  A cudaMemcpy to or from pageable
// memory is staged by the driver in small pieces at a fraction of the link rate, so large transfers go through three
// pinned slots instead: the DMA fills (drains) one slot while a few host threads memcpy another to (from) the caller's
// buffer.  Worker threads touch caller memory only between entry and return of the library call that started them.
extern "C" void kmg_host_copy(void *dst, const void *src, size_t n);   // hostcopy.c: non-temporal stores for large pieces
class CopyPool {
  struct Task { char *dst; const char *src; size_t n; int group; };
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  std::deque<Task> q;
  int pending[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::vector<std::thread> th;
  bool stop = false;
  void run() {
    for (;;) {
      Task t;
      {
        std::unique_lock<std::mutex> l(mu);
        cv_work.wait(l, [&] { return stop || !q.empty(); });
        if (q.empty()) return;
        t = q.front();
        q.pop_front();
      }
      kmg_host_copy(t.dst, t.src, t.n);
      {
        std::lock_guard<std::mutex> l(mu);
        if (--pending[t.group & 7] == 0) cv_done.notify_all();
      }
    }
  }
 public:
  int threads() {
    std::lock_guard<std::mutex> l(mu);
    if (th.empty()) {
      const char *e = getenv("KMERGPU_COPY_THREADS");
      int n = e ? atoi(e) : (int)std::thread::hardware_concurrency() / 2;
      n = std::max(1, std::min(n, 8));
      for (int i = 0; i < n; ++i) th.emplace_back([this] { run(); });
    }
    return (int)th.size();
  }
  void submit(int group, void *dst, const void *src, size_t n) {       // split into one piece per thread
    const int parts = threads();
    const size_t piece = ((n + parts - 1) / parts + 4095) & ~size_t(4095);
    std::lock_guard<std::mutex> l(mu);
    for (size_t off = 0; off < n; off += piece) {
      q.push_back(Task{(char *)dst + off, (const char *)src + off, std::min(piece, n - off), group});
      ++pending[group & 7];
    }
    cv_work.notify_all();
  }
  void wait(int group) {
    std::unique_lock<std::mutex> l(mu);
    cv_done.wait(l, [&] { return pending[group & 7] == 0; });
  }
  ~CopyPool() {
    { std::lock_guard<std::mutex> l(mu); stop = true; }
    cv_work.notify_all();
    for (auto &t : th) t.join();
  }
};
static CopyPool g_pool;
constexpr size_t STAGE_BYTES = size_t(64) << 20;
constexpr int STAGE_SLOTS = 3;
struct Staging {
  std::mutex mu;                       // one staged transfer at a time per process
  char *slot[STAGE_SLOTS] = {nullptr, nullptr, nullptr};
  int ensure() {
    for (auto &p : slot)
      if (!p && cudaMallocHost((void **)&p, STAGE_BYTES) != cudaSuccess) { cudaGetLastError(); return fail(KMG_ERR_NOMEM, "pinned staging allocation failed"); }
    return KMG_OK;
  }
  void release() { for (auto &p : slot) { if (p) cudaFreeHost(p); p = nullptr; } }
};
static Staging g_stage;
static void stage_release() { std::lock_guard<std::mutex> gs(g_stage.mu); g_stage.release(); }
static bool staged_transfers() {
  static int on = -1;
  if (on < 0) { const char *e = getenv("KMERGPU_STAGING"); on = !(e && e[0] == '0'); }
  return on == 1;
}

// host (pageable) -> device through the slots: memcpy of piece c+1 overlaps the DMA of piece c
static int staged_upload(void *d_dst, const void *h_src, size_t bytes, cudaStream_t s) {
  std::lock_guard<std::mutex> g(g_stage.mu);
  TRY(g_stage.ensure());
  cudaEvent_t *ev = g_ctx.ev + 4;
  int c = 0;
  for (size_t off = 0; off < bytes; off += STAGE_BYTES, ++c) {
    const int sl = c % STAGE_SLOTS;
    const size_t n = std::min(STAGE_BYTES, bytes - off);
    if (c >= STAGE_SLOTS) CU(cudaEventSynchronize(ev[sl]));          // the DMA that last read this slot is done
    g_pool.submit(c, g_stage.slot[sl], (const char *)h_src + off, n);
    g_pool.wait(c);
    CU(cudaMemcpyAsync((char *)d_dst + off, g_stage.slot[sl], n, cudaMemcpyHostToDevice, s));
    CU(cudaEventRecord(ev[sl], s));
  }
  CU(cudaStreamSynchronize(s));                                        // the slots are reusable by the next call
  return KMG_OK;
}

enum PtrKind { PK_HOST_PAGEABLE, PK_HOST_PINNED, PK_DEVICE };
static PtrKind ptr_kind(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return PK_HOST_PAGEABLE; }
  if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return PK_DEVICE;
  if (a.type == cudaMemoryTypeHost) return PK_HOST_PINNED;
  return PK_HOST_PAGEABLE;
}

// A sequence on the device: 16 bytes of front padding (so base[-1] exists), len bytes from base = buf + 16, zero
// padding to a multiple of 16 plus one spare group.
static int seq_alloc(DevBuf<uint8_t> &buf, int64_t len, cudaStream_t s) {
  const size_t cap = 16 + (size_t)((len + 15) / 16) * 16 + 16;
  TRY(buf.alloc(cap));
  CU(cudaMemsetAsync(buf, 0, 16, s));
  CU(cudaMemsetAsync(buf + cap - 32, 0, 32, s));
  return KMG_OK;
}
static int upload_seq(const void *src, int64_t len, cudaStream_t s, DevBuf<uint8_t> &buf) {
  TRY(seq_alloc(buf, len, s));
  if (len > (int64_t)(8 << 20) && staged_transfers() && ptr_kind(src) == PK_HOST_PAGEABLE) return staged_upload(buf + 16, src, (size_t)len, s);
  if (len > 0) CU(cudaMemcpyAsync(buf + 16, src, (size_t)len, cudaMemcpyDefault, s));
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// the index
// ------------------------------------------------------------------------------------------------
struct kmg_index {
  int device = 0;
  int k = 0;
  uint64_t U = 0, N = 0;
  uint64_t P = 0, multi = 0;    // sum n(n-1)/2, k-mers with more than one position, longest list: made on first use (ensure_stats)
  uint32_t maxc = 0;
  bool have_stats = false;
  bool grouped = false;         // k-mers in the order of the grouped build instead of ascending key
  int hbits = 0;                // grouped: the records were sorted on the low hbits bits of mix64(key), then by mix64(key)
  bool unstable = false;        // a position list was found not ascending (never true of an index handed out)
  uint64_t *ukeys = nullptr;    // [U]
  uint32_t *ustart = nullptr;   // [U+1]
  uint32_t *pos = nullptr;      // [N]
  // made on first use
  std::mutex mu;
  uint4 *hash = nullptr;        // key table of the probe (probe.cuh), made on the first query
  uint64_t hash_nb = 0;         // buckets of the key table
  int hash_hbits = 0;           // 0: bucket = hash & (nb-1); else the monotone bucket function of a grouped index (probe.cuh)
  uint32_t *multi_u = nullptr;
  uint64_t *pair_off = nullptr;
};
struct kmg_query {
  const kmg_index *idx = nullptr;
  uint64_t H = 0, M = 0;
  int32_t *hit_i = nullptr;
  uint32_t *hit_start = nullptr;
  uint64_t *row_off = nullptr;
};

constexpr int HIST_THREADS = 512, HIST_ITEMS = 16, HIST_TILE = HIST_THREADS * HIST_ITEMS;
constexpr int RLE_THREADS = 256, RLE_ITEMS = 16, RLE_TILE = RLE_THREADS * RLE_ITEMS;
constexpr int PROBE_THREADS = 256, PROBE_ITEMS = 8, PROBE_TILE = PROBE_THREADS * PROBE_ITEMS;
constexpr int COMPACT_ITEMS = 8, COMPACT_TILE = PROBE_THREADS * COMPACT_ITEMS;
constexpr int EMIT_THREADS = 256, EMIT_TILE = EMIT_THREADS * 8;
constexpr int PIDX_THREADS = 256, PIDX_ITEMS = 8, PIDX_TILE = PIDX_THREADS * PIDX_ITEMS;

// ---- the sort pass: shape x rank variant x digit width ------------------------------------------------------
// Shapes <threads, records per thread, CTAs per SM> (kmg_tune "sort_shape", tuning runs): 0 = 256 x 24 x 2 (default),
// 1 = 256 x 28 x 2, 2 = 256 x 20 x 3 (8-bit digits only: three tiles must fit an SM's shared memory).
// Rank variant: 3 = one shared-memory atomic per record (needs lane-ordered atomics: checked per device, and every
// finished index is checked for ascending position lists), 0 = bitmap match (assumes nothing).
// Digit width: chosen per build (SortPlan).
static int g_sort_shape = -1;                  // kmg_tune "sort_shape": -1 auto (28 records per thread for 8-bit digits, else 24), 0..2 as above
static int g_rank_override = -1;               // kmg_tune "sort_cfg": -1 auto, 0 bitmap, 3 one-atomic
static std::atomic<int> g_rank_dev[64];        // per device: 0 unknown, 1 bitmap, 2 one-atomic
static std::atomic<uint64_t> g_unstable_rebuilds{0};
static std::atomic<uint64_t> g_region_rebuilds{0};   // grouped builds redone because a first-pass bin outgrew its region
static uint32_t g_sort_dbg = 0;
static int lane_order_failures(uint32_t *failures);
static bool log_on();

static int rank_variant() {
  if (g_rank_override >= 0) return g_rank_override;
  const int dev = g_ctx.device & 63;
  int v = g_rank_dev[dev].load(std::memory_order_acquire);
  if (v == 0) {
    const char *e = getenv("KMG_SORT_RANK");
    if (e) v = atoi(e) == 3 ? 2 : 1;
    else {
      uint32_t f = 1;
      v = (lane_order_failures(&f) == KMG_OK && f == 0) ? 2 : 1;
      if (log_on()) fprintf(stderr, "[kmergpu] device %d lane-order self-test: %u failures -> rank variant %d\n", dev, f, v == 2 ? 3 : 0);
    }
    int expect = 0;
    g_rank_dev[dev].compare_exchange_strong(expect, v, std::memory_order_acq_rel);   // a concurrent thread found the same answer
    v = g_rank_dev[dev].load(std::memory_order_acquire);
  }
  return v == 2 ? 3 : 0;
}
// An index built with the one-atomic variant had a descending position pair: never use that variant on this device again.
static void demote_rank_variant() {
  g_rank_dev[g_ctx.device & 63].store(1, std::memory_order_release);
  g_unstable_rebuilds.fetch_add(1);
  if (g_rank_override >= 3) g_rank_override = -1;
  if (log_on()) fprintf(stderr, "[kmergpu] device %d: position lists not ascending after a one-atomic sort pass; switching to the bitmap variant\n", g_ctx.device);
}

// Digits of one build: `passes` passes of `rb` bits each.
struct SortPlan { int rb, passes; int bits() const { return rb * passes; } };
// Bits of mix64(key) the grouped build sorts on (kmg_tune "hash_bits": 0 = chosen from the record count, else a multiple
// of 8 or 9; tests lower it to force collisions).  With b bits ~N^2 / 2^(b+1) pairs of distinct k-mers collide and are
// fixed up afterwards: 32 bits (4 passes of 8) up to 48 M records, 36 bits (4 passes of 9) up to 2^26, 40 bits (5 x 8) beyond.
static int g_hash_bits = 0;
static int g_hash_rb = 0;      // kmg_tune "hash_rb": force the digit width (tuning runs)
static int g_no_regions = 0;     // kmg_tune "no_regions": 1 = the grouped build's first pass takes its bin sizes from a histogram sweep (tests, tuning)
static int g_scatter_shape = 0;
static int g_scatter_bitmap = 0; // kmg_tune "scatter_bitmap": 1 = region scatter ranks by bitmap match even where the one-atomic variant is valid
static int g_hash_cas = 0;     // kmg_tune "hash_cas": 1 = always build the probe's key table by CAS (tests, tuning)
static int g_fix_cap = 0;      // kmg_tune "fix_cap": capacity of the short-group task list (0 = max(2^20, N/8)); tests shrink it
static SortPlan grouped_plan(int64_t n_upper) {
  if (g_hash_bits > 0) {
    const int rb = g_hash_rb > 0 && g_hash_bits % g_hash_rb == 0 ? g_hash_rb : (g_hash_bits % 8 == 0 ? 8 : 9);
    return SortPlan{rb, g_hash_bits / rb};
  }
  if (g_hash_rb > 0) return SortPlan{g_hash_rb, (36 + g_hash_rb - 1) / g_hash_rb};
  // measured on B200 (profiles/r02_sortbench_*): a 9-bit pass costs 1.18x an 8-bit one, 10-bit 1.66x, so 8-bit digits it is;
  // b sorted bits leave ~N^2 / 2^(b+1) pairs of k-mers that share them.  Since only groups whose k-mers INTERLEAVE are fixed
  // (a few per cent of the pairs: group_detect_kernel), 32 bits carry a 250 M-record build (7 M pairs) at 4 passes instead of 5.
  return n_upper <= (int64_t)400000000 ? SortPlan{8, 4} : SortPlan{8, 5};
}
// is the grouped build used for this k and requested order?  From k = 21 on (keys of more than 40 bits: a sort by key would
// need 6+ passes): independent of the size, so that every rank of a sharded build decides alike.
static bool grouped_for(int k, int order, int64_t /*n_upper*/) {
  return order == KMG_ORDER_GROUPED && 2 * k > 40;
}

static unsigned long long *g_trace = nullptr;
static int g_trace_tiles = 0;
extern "C" int kmg_trace_read(unsigned long long *host, int tiles) {
  if (!g_trace || tiles > g_trace_tiles) return -1;
  return cudaMemcpy(host, g_trace, (size_t)tiles * 64, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -4;
}
extern "C" int kmg_tune(const char *key, int value) {
  if (key && !strcmp(key, "sort_cfg")) {              // rank variant: -1 auto, 0 bitmap, 3 one atomic per record
    if (value != -1 && value != 0 && value != 3 && value != 4) return fail(KMG_ERR_ARG, "sort_cfg must be -1 (auto), 0 (bitmap), 3 (one atomic) or 4 (tests: unstable on purpose)");
    g_rank_override = value;
    return KMG_OK;
  }
  if (key && !strcmp(key, "sort_shape")) {
    if (value < -1 || value > 2) return fail(KMG_ERR_ARG, "sort_shape out of range");
    g_sort_shape = value;
    return KMG_OK;
  }
  if (key && !strcmp(key, "sort_dbg")) { g_sort_dbg = (uint32_t)value; return KMG_OK; }
  if (key && !strcmp(key, "fix_cap")) { g_fix_cap = value > 0 ? value : 0; return KMG_OK; }
  if (key && !strcmp(key, "hash_cas")) { g_hash_cas = value != 0; return KMG_OK; }
  if (key && !strcmp(key, "scatter_bitmap")) { g_scatter_bitmap = value != 0; return KMG_OK; }
  if (key && !strcmp(key, "scatter_shape")) { g_scatter_shape = value; return KMG_OK; }
  if (key && !strcmp(key, "no_regions")) { g_no_regions = value; return KMG_OK; }    // 0 auto, 1 never, 2 always (tests: skips the sampled check)
  if (key && !strcmp(key, "hash_bits")) {
    if (value != 0 && (value < 8 || value > 56 || (value % 8 && value % 9 && value % 10))) return fail(KMG_ERR_ARG, "hash_bits must be 0 (auto) or a multiple of 8, 9 or 10 in [8,56]");
    g_hash_bits = value;
    return KMG_OK;
  }
  if (key && !strcmp(key, "hash_rb")) {
    if (value != 0 && (value < 8 || value > 10)) return fail(KMG_ERR_ARG, "hash_rb must be 0, 8, 9 or 10");
    g_hash_rb = value;
    return KMG_OK;
  }
  if (key && !strcmp(key, "reset_rank")) {            // tests: forget what this device's self-test / index checks said
    for (auto &v : g_rank_dev) v.store(0);
    return KMG_OK;
  }
  if (key && !strcmp(key, "sort_trace")) {          // value = tiles to trace (0 = off); buffer read by kmg_trace_read
    if (g_trace) { cudaFree(g_trace); g_trace = nullptr; }
    g_trace_tiles = value;
    if (value > 0) { if (cudaMalloc(&g_trace, (size_t)value * 64) != cudaSuccess) return fail(KMG_ERR_NOMEM, "trace alloc"); cudaMemset(g_trace, 0, (size_t)value * 64); }
    return KMG_OK;
  }
  return fail(KMG_ERR_ARG, "unknown tuning key");
}
// what the library decided: "rank_variant" (0/3 for the current device), "unstable_rebuilds", "hash_bits" for n records
extern "C" int64_t kmg_tune_get(const char *key, int64_t arg) {
  if (key && !strcmp(key, "rank_variant")) return ctx_init() == KMG_OK ? rank_variant() : -1;
  if (key && !strcmp(key, "unstable_rebuilds")) return (int64_t)g_unstable_rebuilds.load();
  if (key && !strcmp(key, "region_rebuilds")) return (int64_t)g_region_rebuilds.load();
  if (key && !strcmp(key, "hash_bits")) return grouped_plan(arg).bits();
  if (key && !strcmp(key, "hash_rb")) return grouped_plan(arg).rb;
  return -1;
}
// RANK 3's precondition, checked on the current device: failures = 0 means the lanes of one shared-memory
// atomic instruction that collide on an address are applied in ascending lane order.
static int lane_order_failures(uint32_t *failures) {
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint32_t> bad(s);
  TRY(bad.alloc(1));
  CU(cudaMemsetAsync(bad, 0, 4, s));
  LAUNCH("lane_order_selftest", s, lane_order_selftest_kernel<<<g_ctx.sms * 4, 256, 0, s>>>(bad));
  CU(cudaMemcpyAsync(failures, bad, 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return KMG_OK;
}
extern "C" int kmg_selftest_lane_order(uint32_t *failures) {
  if (!failures) return fail(KMG_ERR_ARG, "failures is NULL");
  return lane_order_failures(failures);
}
// Two tiles of the default record pass fit the 196 KB shared-memory carve-out (1 KB per block is reserved).  With register
// loads, one step further (228 KB) left 28 KB of L1 for the loads in flight and cost every pass 8 % (profiles/r02_notes.md);
// since keys and positions arrive by bulk copy (no L1 lines) a 30-record tile at 228 KB runs as fast as this one -- and no
// faster (profiles/r02_sortbench_30.log), so the tile stays where register loads (partial tiles, dbg runs) are safe too.
static_assert(2 * (sizeof(PassSmem<PassCfg<256, 28, 2, 3, 4, 8>, false>) + 1024) <= 196 * 1024, "the record pass's tile outgrew the 196 KB carve-out");
constexpr int REGION_SAMPLE_STRIDE = 251;   // prime: tandem arrays are sampled in all their phases
constexpr int SORT_TILE_MIN = 4096;   // status sizing: smallest tile of any shape

template <class Cfg, bool FROM_SEQ, class BinFn, class NextFn, bool HAS_NEXT, bool PEER = false, bool SEGS = false>
static int launch_pass_cfg(const char *name, const PassParams<BinFn, NextFn> &P, int64_t n_upper, cudaStream_t s, int extra_tiles = 0) {
  using S = PassSmem<Cfg, FROM_SEQ>;
  if constexpr (!FROM_SEQ && !PEER && !SEGS) {             // a segmented record source runs the separately compiled variant
    if (P.segs) return launch_pass_cfg<Cfg, FROM_SEQ, BinFn, NextFn, HAS_NEXT, PEER, true>(name, P, n_upper, s, extra_tiles);
  }
  auto kern = scatter_pass_kernel<Cfg, FROM_SEQ, BinFn, NextFn, HAS_NEXT, PEER, SEGS>;
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S)));
  const int64_t tiles = ceil_div<int64_t>(n_upper, Cfg::TILE) + extra_tiles;   // extra: a segmented source has one partial tile per segment
  if (tiles == 0) return KMG_OK;
  LAUNCH(name, s, kern<<<(unsigned)tiles, Cfg::THREADS, sizeof(S), s>>>(P));
  return KMG_OK;
}
// rb: digit width of the pass (bins = 2^rb); P.bin / P.next must carry the matching mask
template <bool FROM_SEQ, class BinFn, class NextFn, bool HAS_NEXT>
static int launch_pass(const char *name, const PassParams<BinFn, NextFn> &P, int64_t n_upper, cudaStream_t s, int rb = RADIX_BITS, int extra_tiles = 0) {
  const int rank = rank_variant();
  // the fused encode + first pass gains 4 % from 28 records per thread (its positions are 16-bit in shared memory), the record passes nothing
  // 28 records per thread where the digit is 8 bits wide (measured at 250 M records: last pass 1.40 against 1.48 ms, the others 1 %)
  const int shape = g_sort_shape < 0 ? (rb == 8 ? 1 : 0)
                                     : (rb == 8) ? ((FROM_SEQ && g_sort_shape == 0) ? 1 : g_sort_shape) : (g_sort_shape == 2 ? 0 : g_sort_shape);
#define KMG_GO(T, I, M, RK, RB) return launch_pass_cfg<PassCfg<T, I, M, RK, (RK >= 3 ? 4 : 8), RB>, FROM_SEQ, BinFn, NextFn, HAS_NEXT>(name, P, n_upper, s, extra_tiles)
#define KMG_SHAPES(RK, RB)                         \
  do {                                             \
    if (shape == 1) KMG_GO(256, 28, 2, RK, RB);    \
    KMG_GO(256, 24, 2, RK, RB);                    \
  } while (0)
  if (rb == 8) {
    if (rank == 4) KMG_GO(256, 24, 2, 4, 8);       // tests: deliberately unstable
    if (shape == 2) { if (rank == 3) KMG_GO(256, 20, 3, 3, 8); else KMG_GO(256, 20, 3, 0, 8); }
    if (rank == 3) KMG_SHAPES(3, 8); else KMG_SHAPES(0, 8);
  } else if (rb == 9) {
    if (rank == 4) KMG_GO(256, 24, 2, 4, 9);
    if (rank == 3) KMG_SHAPES(3, 9); else KMG_SHAPES(0, 9);
  } else if (rb == 10) {
    if (rank == 3) KMG_GO(256, 24, 2, 3, 10); else KMG_GO(256, 24, 2, 0, 10);
  }
#undef KMG_SHAPES
#undef KMG_GO
  return fail(KMG_ERR_ARG, "bad sort configuration");
}

// records per tile of a RECORD pass with digits of rb bits (mirrors launch_pass's choice of shape)
static uint32_t record_tile(int rb) {
  const int shape = g_sort_shape < 0 ? (rb == 8 ? 1 : 0) : (rb == 8) ? g_sort_shape : (g_sort_shape == 2 ? 0 : g_sort_shape);
  if (rank_variant() == 4 || rb == 10) return 256 * 24;
  return shape == 1 ? 256 * 28 : shape == 2 ? 256 * 20 : 256 * 24;
}

// Scratch shared by the sort passes of one build.
struct SortScratch {
  DevBuf<uint32_t> small;        // hist[(MAX_PASSES+1)][MAX_NB] | gbase[(MAX_PASSES+1)][MAX_NB] | common[RADIX] | tickets[16] | IndexStats
  DevBuf<uint64_t> status;       // [tiles][bins]
  size_t small_words = 0, status_words = 0;
  static constexpr size_t H = (size_t)(MAX_PASSES + 1) * MAX_NB;
  explicit SortScratch(cudaStream_t s) : small(s), status(s) {}
  uint32_t *hist(int r) const { return small + (size_t)r * MAX_NB; }
  uint32_t *gbase(int r) const { return small + H + (size_t)r * MAX_NB; }
  uint32_t *common() const { return small + 2 * H; }
  uint32_t *ticket(int i) const { return small + 2 * H + RADIX + i; }
  IndexStats *stats() const { return reinterpret_cast<IndexStats *>(small + 2 * H + RADIX + 16); }
};
static int scratch_clear(SortScratch &sc, cudaStream_t s) {
  CU(cudaMemsetAsync(sc.small, 0, sc.small_words * 4, s));
  CU(cudaMemsetAsync(sc.status, 0, sc.status_words * sizeof(uint64_t), s));
  return KMG_OK;
}
static int scratch_alloc(SortScratch &sc, int64_t n_upper, cudaStream_t s, int rb = RADIX_BITS) {
  sc.small_words = 2 * SortScratch::H + RADIX + 16 + sizeof(IndexStats) / 4;
  TRY(sc.small.alloc(sc.small_words));
  const size_t tiles = (size_t)ceil_div<int64_t>(n_upper > 0 ? n_upper : 1, SORT_TILE_MIN) + MAX_SEGS + 1;   // segment-aligned tiles: one partial tile per segment
  sc.status_words = tiles << rb;
  TRY(sc.status.alloc(sc.status_words));
  return scratch_clear(sc, s);
}

template <class... A>
static int launch_scan_hist(int rb, cudaStream_t s, A... args) {
  if (rb == 8) LAUNCH("scan_hist", s, scan_hist_kernel<256><<<1, 256, 0, s>>>(args...));
  else if (rb == 9) LAUNCH("scan_hist", s, scan_hist_kernel<512><<<1, 512, 0, s>>>(args...));
  else if (rb == 10) LAUNCH("scan_hist", s, scan_hist_kernel<1024><<<1, 1024, 0, s>>>(args...));
  else return fail(KMG_ERR_ARG, "bad digit width");
  return KMG_OK;
}

// Sorted records -> CSR; reads the stats back (one synchronisation) and fills the handle.  The same sweep checks that
// positions ascend inside every k-mer (IndexStats::unstable): what a stable sort guarantees and the reference's
// insertion order gives; the caller rebuilds with the order-independent rank variant if it ever fails.
static int finish_index(kmg_index *ix, SortScratch &sc, uint64_t *keys_sorted, uint32_t *pos_sorted,
                        int64_t n_upper, cudaStream_t s, bool hashed = false) {
  IndexStats *st = sc.stats();
  DevBuf<uint64_t> ukeys(s);
  DevBuf<uint32_t> ustart(s);
  DevBuf<Pair64> status2(s);
  const int64_t tiles = ceil_div<int64_t>(n_upper > 0 ? n_upper : 1, RLE_TILE);
  TRY(ukeys.alloc((size_t)n_upper));
  TRY(ustart.alloc((size_t)n_upper + 1));
  TRY(status2.alloc((size_t)tiles));
  CU(cudaMemsetAsync(status2, 0, (size_t)tiles * sizeof(Pair64), s));
  LAUNCH("rle", s, rle_kernel<RLE_THREADS, RLE_ITEMS><<<(unsigned)tiles, RLE_THREADS, 0, s>>>(
                       keys_sorted, pos_sorted, st, ukeys, ustart, status2, sc.ticket(MAX_PASSES + 1), hashed));
  IndexStats h;
  CU(cudaMemcpyAsync(&h, st, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  ix->N = h.n; ix->U = h.U; ix->unstable = h.unstable != 0;
  ix->have_stats = false;       // P, multi, max count: on first demand (ensure_stats)
  status2.reset();
  // keep exact-size arrays when the over-allocation is large
  if (h.U * 2 < (uint64_t)n_upper) {
    DevBuf<uint64_t> uk2(s);
    DevBuf<uint32_t> us2(s);
    TRY(uk2.alloc((size_t)h.U));
    TRY(us2.alloc((size_t)h.U + 1));
    CU(cudaMemcpyAsync(uk2, ukeys, h.U * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    CU(cudaMemcpyAsync(us2, ustart, (h.U + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
    ukeys.reset(uk2.release()); ustart.reset(us2.release());
  }
  ix->ukeys = ukeys.release(); ix->ustart = ustart.release(); ix->pos = pos_sorted;
  const double N = (double)h.n, U = (double)h.U;
  prof_bytes("rle", 12 * N + 12 * U);
  return KMG_OK;
}

// LSD passes first_pass..plan.passes-1 over record buffers, digits of plan.rb bits.  has_next: only hist/gbase of
// first_pass exist, each pass takes the next one's histogram as it writes (grouped builds, builds from records);
// otherwise every pass's gbase is already there (sorted builds from the sequence, hist_all_kernel).
// final_pos (optional): the last pass writes its positions there instead of into the ping-pong buffer
// (the array the index keeps), so `pa` is meaningless afterwards.
static int sort_tail(SortScratch &sc, SortPlan plan, int first_pass, bool has_next, uint64_t *&ka, uint32_t *&pa, uint64_t *&kb,
                     uint32_t *&pb, int64_t n_upper, cudaStream_t s, uint32_t *final_pos = nullptr, const TileSegs *seg0 = nullptr, int nsegs0 = 0,
                     int end_pass = -1) {
  const int R = plan.passes, rb = plan.rb;
  const uint32_t mask = (1u << rb) - 1;
  for (int r = first_pass; r < (end_pass > 0 ? end_pass : R); ++r) {
    PassParams<DigitBin, DigitBin> P{};
    P.keys_in = ka; P.pos_in = pa; P.keys_out = kb; P.pos_out = (final_pos && r == R - 1) ? final_pos : pb;
    P.gbase = sc.gbase(r); P.hist_next = sc.hist(r + 1);
    P.status = sc.status; P.ticket = sc.ticket(r); P.epoch = (uint32_t)(r + 1);
    P.n_records = &sc.stats()->n;
    P.segs = r == first_pass ? seg0 : nullptr;              // the first pass may read a segmented source (TileSegs)
    const int extra = r == first_pass && seg0 ? nsegs0 : 0;
    P.bin = DigitBin{r * rb, mask}; P.next = DigitBin{(r + 1) * rb, mask};
    P.dbg = g_sort_dbg;
    P.trace = (r == 2 && g_trace && ceil_div<int64_t>(n_upper, SORT_TILE_MIN) <= g_trace_tiles) ? g_trace : nullptr;   // trace the third pass
    if (has_next && r + 1 < R) {
      TRY((launch_pass<false, DigitBin, DigitBin, true>("sort_pass_hist", P, n_upper, s, rb, extra)));
      TRY(launch_scan_hist(rb, s, sc.hist(r + 1), sc.gbase(r + 1), (uint64_t *)nullptr));
    } else {
      TRY((launch_pass<false, DigitBin, DigitBin, false>("sort_pass", P, n_upper, s, rb, extra)));
    }
    std::swap(ka, kb);
    std::swap(pa, pb);
  }
  return KMG_OK;
}

// Collisions of the low bits of the mix: partition those groups by the whole mix (sk, sp: scratch of the
// same size).  Returns the detect counters through h_cnt after the caller's next synchronisation; the task lists are in
// fixmem until then.
static int fix_groups(SortScratch &sc, int bits, uint64_t *keys, uint32_t *pos, uint64_t *sk, uint32_t *sp, int64_t n_upper, cudaStream_t s,
                      uint32_t *h_cnt /* [4], pinned or stack read after a sync */, DevBuf<uint32_t> &fixmem) {
  FixLists fl{};
  fl.small_cap = g_fix_cap > 0 ? (uint32_t)g_fix_cap : (uint32_t)std::max<int64_t>(1 << 20, n_upper / 8);
  fl.big_cap = 1 << 16;
  const size_t words = 4 + CLAIM_SLOTS + 2 * (size_t)fl.small_cap + 2 * (size_t)fl.big_cap;
  TRY(fixmem.alloc(words));
  CU(cudaMemsetAsync(fixmem, 0, (4 + CLAIM_SLOTS) * sizeof(uint32_t), s));
  fl.counters = fixmem; fl.claim = fixmem + 4;
  fl.small_tasks = reinterpret_cast<uint2 *>(fixmem + 4 + CLAIM_SLOTS);
  fl.big_tasks = fl.small_tasks + fl.small_cap;
  const unsigned dgrid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n_upper, 256 * 8), (int64_t)g_ctx.sms * 16);
  if (bits == 32) LAUNCH("group_detect", s, group_detect_kernel<true><<<dgrid, 256, 0, s>>>(keys, sc.stats(), bits, fl));
  else LAUNCH("group_detect", s, group_detect_kernel<false><<<dgrid, 256, 0, s>>>(keys, sc.stats(), bits, fl));
  LAUNCH("small_fix", s, small_fix_kernel<<<g_ctx.sms * 4, 128, 0, s>>>(keys, pos, fl));
  LAUNCH("big_fix", s, big_fix_kernel<1024><<<g_ctx.sms, 1024, 0, s>>>(keys, pos, sk, sp, fl));   // 1024 threads: config 2's long groups 87 -> 50 us
  CU(cudaMemcpyAsync(h_cnt, fl.counters, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  return KMG_OK;
}

// Grouped build: equal k-mers contiguous, k-mers in the order of (low bits of mix64(key), mix64(key)).
// regions (the default): the first pass needs no histogram of its digit -- the mixed digit is uniform, so every bin gets its
// own region of 1.25x the mean bin size and the pass writes bin b from b * cap on; its last tile leaves the bins' sizes,
// from which the second pass reads the regions tile by tile (TileSegs).  This drops the histogram sweep over the sequence
// (hist_seq_kernel: 0.41 ms of 11.7 at 250 Mbp).  A bin that outgrows its region (a k-mer with more copies than a quarter of
// a mean bin) sets a flag, the tile's records are dropped, and the caller redoes the build with the histogram.
static int build_grouped(const SeqView &sv, SortPlan plan, kmg_index *ix, SortScratch &sc, uint64_t *&ka, uint32_t *&pa, uint64_t *&kb,
                         uint32_t *&pb, int64_t n_upper, cudaStream_t s, bool *overflow, bool regions, bool *region_overflow) {
  const int R = plan.passes, rb = plan.rb, NB = 1 << rb;
  const uint32_t mask = (1u << rb) - 1;
  DevBuf<uint64_t> kr(s), d_counts(s);
  DevBuf<uint32_t> pr(s), d_over(s);
  DevBuf<TileSegs> segs(s);
  uint32_t h_over = 0;
  regions = regions && R > 1 && NB <= MAX_SEGS && n_upper <= (int64_t)1600000000;   // region offsets are 32-bit signed in the pass
  const uint32_t cap = (uint32_t)(((uint64_t)(n_upper / NB) * 5 / 4 + 4096 + 15) & ~uint64_t(15));
  if (regions && g_no_regions == 2) {
    // tests: regions whatever the sample would say
  } else if (regions && n_upper >= (int64_t)REGION_SAMPLE_STRIDE * 4096) {
    // A repeat-rich sequence puts a k-mer's every copy into one bin: ask a 1-in-251 sample whether the heaviest bin stays
    // clear of a region's size; if not, take the histogram path right away instead of finding out the expensive way.
    DevBuf<uint32_t> d_s(s);
    uint32_t h_est = 0;
    TRY(d_s.alloc((size_t)MAX_NB + 1));
    if (cudaMemsetAsync(d_s, 0, (MAX_NB + 1) * sizeof(uint32_t), s) != cudaSuccess) return fail(KMG_ERR_CUDA, "memset failed");
    const unsigned g = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n_upper / REGION_SAMPLE_STRIDE, 256), (int64_t)g_ctx.sms * 8);
    region_sample_kernel<<<g, 256, 0, s>>>(sv, REGION_SAMPLE_STRIDE, mask, d_s);
    region_estimate_kernel<<<1, 256, 0, s>>>(d_s, NB, REGION_SAMPLE_STRIDE, d_s + MAX_NB);
    if (cudaMemcpyAsync(&h_est, d_s + MAX_NB, 4, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess)
      return fail(KMG_ERR_CUDA, "region estimate failed: %s", cudaGetErrorString(cudaGetLastError()));
    if ((uint64_t)h_est * 10 > (uint64_t)cap * 9) regions = false;       // within 10 % of a region: not worth the risk
  } else if (regions) {
    regions = false;                                       // small inputs: the sweep is cheap and the slack relatively small
  }
  PassParams<DigitBin, DigitBin> P{};
  P.sv = sv; P.keys_out = ka; P.pos_out = pa;
  P.gbase = sc.gbase(0); P.hist_next = sc.hist(1);
  P.status = sc.status; P.ticket = sc.ticket(0); P.epoch = 1;
  P.hashed = 1;
  P.dbg = g_sort_dbg;
  P.bin = DigitBin{0, mask}; P.next = DigitBin{rb, mask};
  if (regions) {
    TRY(kr.alloc((size_t)NB * cap));
    TRY(pr.alloc((size_t)NB * cap));
    TRY(d_counts.alloc((size_t)MAX_SEGS));
    TRY(d_over.alloc(4));
    TRY(segs.alloc(1));
    CU(cudaMemsetAsync(d_counts, 0, MAX_SEGS * sizeof(uint64_t), s));
    LAUNCH("region_gbase", s, region_gbase_kernel<<<1, 256, 0, s>>>(sc.gbase(0), NB, cap, d_over));
    P.keys_out = kr; P.pos_out = pr;
    P.bin_counts = d_counts; P.bin_cap = cap; P.bin_overflow = d_over;
    TRY((launch_pass<true, DigitBin, DigitBin, true>("sort_pass_seq", P, n_upper, s, rb)));
    TRY(launch_scan_hist(rb, s, sc.hist(1), sc.gbase(1), (uint64_t *)nullptr));
    LAUNCH("tile_segs", s, tile_segs_kernel<<<1, MAX_SEGS, 0, s>>>(d_counts, NB, (uint64_t)cap, record_tile(rb), segs, &sc.stats()->n));
    CU(cudaMemcpyAsync(&h_over, d_over, 4, cudaMemcpyDeviceToHost, s));
    // second pass: regions -> (ka, pa); afterwards the region arrays are free
    uint64_t *rk = kr;
    uint32_t *rp = pr;
    TRY(sort_tail(sc, plan, 1, true, rk, rp, ka, pa, n_upper, s, nullptr, segs, NB, 2));
    std::swap(rk, ka); std::swap(rp, pa);                  // sort_tail swapped (in, out): the data is in what it calls `rk`
    TRY(sort_tail(sc, plan, 2, true, ka, pa, kb, pb, n_upper, s));
  } else {
    const int64_t tiles = ceil_div<int64_t>(n_upper, HIST_TILE);
    const unsigned hgrid = (unsigned)std::min<int64_t>(tiles, (int64_t)g_ctx.sms * 2);
    LAUNCH("hist_seq", s, hist_seq_kernel<HIST_THREADS, HIST_ITEMS, HashDigitBin><<<hgrid, HIST_THREADS, 0, s>>>(sv, sc.hist(0), HashDigitBin{0, mask}));
    TRY(launch_scan_hist(rb, s, sc.hist(0), sc.gbase(0), &sc.stats()->n));
    if (R > 1) {
      TRY((launch_pass<true, DigitBin, DigitBin, true>("sort_pass_seq", P, n_upper, s, rb)));
      TRY(launch_scan_hist(rb, s, sc.hist(1), sc.gbase(1), (uint64_t *)nullptr));
    } else {
      TRY((launch_pass<true, DigitBin, DigitBin, false>("sort_pass_seq", P, n_upper, s, rb)));
    }
    TRY(sort_tail(sc, plan, 1, true, ka, pa, kb, pb, n_upper, s));   // records ordered by the low bits of the mix, in (ka, pa)
  }
  uint32_t h_cnt[4] = {0, 0, 0, 0};
  DevBuf<uint32_t> fixmem(s);
  TRY(fix_groups(sc, plan.bits(), ka, pa, kb, pb, n_upper, s, h_cnt, fixmem));   // kb, pb are free: scratch
  TRY(finish_index(ix, sc, ka, pa, n_upper, s, true));      // synchronises
  *overflow = h_cnt[2] != 0;
  *region_overflow = h_over != 0;
  if (log_on()) fprintf(stderr, "[kmergpu] grouped build on %d bits: %u short and %u long groups fixed\n", plan.bits(), h_cnt[0], h_cnt[1]);
  ix->hbits = plan.bits();
  const double N = (double)ix->N, L = (double)sv.avail;
  if (!regions) prof_bytes("hist_seq", L);
  prof_bytes("sort_pass_seq", L + 12 * N);
  if (R > 2) prof_bytes("sort_pass_hist", 24 * N * (R - 2));
  if (R > 1) prof_bytes("sort_pass", 24 * N);
  prof_bytes("group_detect", 8 * N);
  return KMG_OK;
}

static void release_index_arrays(kmg_index *ix, cudaStream_t s) {
  void *ptrs[3] = {ix->ukeys, ix->ustart, ix->pos};
  for (void *p : ptrs) g_arena[ix->device & 63].put(p, s, false);
  ix->ukeys = nullptr; ix->ustart = nullptr; ix->pos = nullptr;
  ix->grouped = false; ix->hbits = 0; ix->unstable = false;
}

// One attempt at an index of the windows of `sv` (the caller retries once if the position lists came out unordered).
static int build_attempt(const SeqView &sv, int k, kmg_index *ix, int order, cudaStream_t s) {
  const int64_t n_upper = sv.nstarts;
  const int R = num_passes(k);
  const bool grouped = grouped_for(k, order, n_upper);
  const SortPlan gp = grouped_plan(n_upper);
  SortScratch sc(s);
  DevBuf<uint64_t> k0(s), k1(s);
  DevBuf<uint32_t> p0(s), p1(s);
  TRY(scratch_alloc(sc, n_upper, s, grouped ? gp.rb : RADIX_BITS));
  TRY(k0.alloc((size_t)n_upper));
  TRY(p0.alloc((size_t)n_upper));
  if (R > 1) { TRY(k1.alloc((size_t)n_upper)); TRY(p1.alloc((size_t)n_upper)); }
  uint64_t *ka = k0, *kb = k1;                             // the passes ping-pong between the two pairs
  uint32_t *pa = p0, *pb = p1;
  if (grouped) {
    bool overflow = false, region_overflow = false;
    TRY(build_grouped(sv, gp, ix, sc, ka, pa, kb, pb, n_upper, s, &overflow, g_no_regions != 1, &region_overflow));
    if (region_overflow) {                              // a bin outgrew its region (a huge repeat): once more with the histogram
      g_region_rebuilds.fetch_add(1);
      if (log_on()) fprintf(stderr, "[kmergpu] a first-pass bin outgrew its region: rebuilding with the histogram sweep\n");
      ix->pos = nullptr;                                // pa: still ours
      release_index_arrays(ix, s);
      TRY(scratch_clear(sc, s));
      overflow = false;
      TRY(build_grouped(sv, gp, ix, sc, ka, pa, kb, pb, n_upper, s, &overflow, false, &region_overflow));
    }
    if (!overflow) { (pa == p0.get() ? p0 : p1).release(); ix->grouped = true; return KMG_OK; }
    // more colliding groups than the task lists hold (not seen in practice): rebuild sorted by key
    ix->pos = nullptr;
    release_index_arrays(ix, s);
    sc.small.reset(); sc.status.reset();
    TRY(scratch_alloc(sc, n_upper, s, RADIX_BITS));
  }
  const int64_t tiles = ceil_div<int64_t>(n_upper, HIST_TILE);
  const unsigned hgrid = (unsigned)std::min<int64_t>(tiles, (int64_t)g_ctx.sms * 2);
  LAUNCH("hist_all", s, hist_all_kernel<HIST_THREADS, HIST_ITEMS><<<hgrid, HIST_THREADS, 0, s>>>(sv, sc.common(), sc.hist(0), MAX_NB));
  LAUNCH("hist_finish", s, hist_finish_kernel<<<R, RADIX, 0, s>>>(k, sc.common(), sc.hist(0), sc.gbase(0), MAX_NB, &sc.stats()->n));
  {
    PassParams<DigitBin, DigitBin> P{};
    P.sv = sv; P.keys_out = ka; P.pos_out = pa;
    P.gbase = sc.gbase(0);
    P.status = sc.status; P.ticket = sc.ticket(0); P.epoch = 1;
    P.dbg = g_sort_dbg;
    P.bin = DigitBin{0}; P.next = DigitBin{RADIX_BITS};
    TRY((launch_pass<true, DigitBin, DigitBin, false>("sort_pass_seq", P, n_upper, s)));
  }
  TRY(sort_tail(sc, SortPlan{RADIX_BITS, R}, 1, false, ka, pa, kb, pb, n_upper, s));   // result ends in (ka, pa)
  TRY(finish_index(ix, sc, ka, pa, n_upper, s));
  (pa == p0.get() ? p0 : p1).release();                    // now owned by the index
  const double N = (double)ix->N, L = (double)sv.avail;
  prof_bytes("hist_all", L);
  prof_bytes("sort_pass_seq", L + 12 * N);
  if (R > 1) prof_bytes("sort_pass", 24 * N * (R - 1));
  return KMG_OK;
}

static int build_from_view(const SeqView &sv, int k, kmg_index **out, int order = KMG_ORDER_SORTED) {
  cudaStream_t s = g_ctx.stream();
  const int64_t n_upper = sv.nstarts;
  if (n_upper > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "%lld windows exceed the 32-bit coordinates of the reference", (long long)n_upper);
  IndexPtr ix(new (std::nothrow) kmg_index());
  if (!ix) return fail(KMG_ERR_NOMEM, "host allocation failed");
  ix->device = g_ctx.device;
  ix->k = k;
  if (n_upper <= 0) {                      // shorter than k: an empty index, as the C core gives
    TRY(dalloc(&ix->ustart, 1, s));
    if (cudaMemsetAsync(ix->ustart, 0, 4, s) != cudaSuccess) return fail(KMG_ERR_CUDA, "memset failed");
    cudaStreamSynchronize(s);
    *out = ix.release();
    return KMG_OK;
  }
  TRY(build_attempt(sv, k, ix.get(), order, s));
  if (ix->unstable) {
    // A k-mer's positions are not ascending: the one-atomic rank variant's hardware assumption failed here.
    // Never use it on this device again and redo the build with the bitmap variant, which assumes nothing.
    const bool was_atomic = rank_variant() >= 3;
    release_index_arrays(ix.get(), s);
    if (!was_atomic) return fail(KMG_ERR_CUDA, "internal error: position lists not ascending after a stable sort");
    demote_rank_variant();
    TRY(build_attempt(sv, k, ix.get(), order, s));
    if (ix->unstable) return fail(KMG_ERR_CUDA, "internal error: position lists not ascending after a stable sort");
  }
  *out = ix.release();
  return KMG_OK;
}

static double wall_ms() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
static bool log_on() {
  static int on = -1;
  if (on < 0) { const char *e = getenv("KMERGPU_LOG"); on = e && e[0] == '1'; }
  return on == 1;
}

extern "C" int kmg_build(const char *seq, int64_t len, int k, kmg_index **out) {
  return kmg_build_ordered(seq, len, k, KMG_ORDER_GROUPED, out);
}
extern "C" int kmg_index_order(const kmg_index *ix) { return !ix ? fail(KMG_ERR_ARG, "index is NULL") : (ix->grouped ? KMG_ORDER_GROUPED : KMG_ORDER_SORTED); }

extern "C" int kmg_build_ordered(const char *seq, int64_t len, int k, int order, kmg_index **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  if (order != KMG_ORDER_SORTED && order != KMG_ORDER_GROUPED) return fail(KMG_ERR_ARG, "order must be KMG_ORDER_SORTED or KMG_ORDER_GROUPED");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be a positive integer less than 1+MAX_K");
  if (len < 0 || (len > 0 && !seq)) return fail(KMG_ERR_ARG, "bad sequence pointer/length");
  const double t0 = wall_ms();
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint8_t> dseq(s);
  TRY(upload_seq(seq, len, s, dseq));
  const double t1 = wall_ms();
  SeqView sv;
  sv.base = dseq + 16; sv.nstarts = len - k + 1 > 0 ? len - k + 1 : 0; sv.avail = len; sv.s0 = 0; sv.L = len; sv.k = k;
  const int rc = build_from_view(sv, k, out, order);
  if (log_on())
    fprintf(stderr, "[kmergpu] build len=%lld k=%d: upload(enqueue) %.3f ms, build %.3f ms (host wall clock)\n", (long long)len, k, t1 - t0, wall_ms() - t1);
  return rc;
}

extern "C" int kmg_free(kmg_index *ix) {
  if (!ix) return KMG_OK;
  release_on_device(ix->device, {ix->ukeys, ix->ustart, ix->pos, ix->hash, ix->multi_u, ix->pair_off});
  delete ix;
  return KMG_OK;
}

static int use_index(const kmg_index *ix) { return ix ? use_device(ix->device, "the index lives") : fail(KMG_ERR_ARG, "index is NULL"); }
// P, multi and the longest list: one sweep of ustart (4U bytes), taken the first time something asks for them -- the pair
// matrix's extent (kmg_sizes with P != NULL), kmg_index_stats, kmg_pairs*.  make.kmer.hash + kmer.pos(2|8) never does.
static int ensure_stats(const kmg_index *cix) {
  kmg_index *ix = const_cast<kmg_index *>(cix);
  std::lock_guard<std::mutex> g(ix->mu);
  if (ix->have_stats) return KMG_OK;
  if (ix->U == 0) { ix->P = 0; ix->multi = 0; ix->maxc = 0; ix->have_stats = true; return KMG_OK; }
  TRY(use_index(ix));
  cudaStream_t s = g_ctx.stream();
  DevBuf<IndexStats> st(s);
  IndexStats h;
  TRY(st.alloc(1));
  CU(cudaMemsetAsync(st, 0, sizeof(IndexStats), s));
  const unsigned sgrid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(ix->U, 256 * 16), (uint64_t)g_ctx.sms * 8);
  LAUNCH("stats", s, stats_kernel<256><<<sgrid, 256, 0, s>>>(ix->ustart, ix->U, st));
  CU(cudaMemcpyAsync(&h, st, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  ix->P = h.P; ix->multi = h.multi; ix->maxc = h.maxc;
  ix->have_stats = true;
  prof_bytes("stats", 4.0 * (double)ix->U);
  return KMG_OK;
}

// P may be NULL: the number of pair rows costs a sweep of the index the first time it is asked for (ensure_stats)
extern "C" int kmg_sizes(const kmg_index *ix, uint64_t *U, uint64_t *N, uint64_t *P) {
  if (!ix) return fail(KMG_ERR_ARG, "index is NULL");
  if (P) { TRY(ensure_stats(ix)); *P = ix->P; }
  if (U) *U = ix->U;
  if (N) *N = ix->N;
  return KMG_OK;
}
extern "C" int kmg_index_k(const kmg_index *ix) { return ix ? ix->k : fail(KMG_ERR_ARG, "index is NULL"); }
extern "C" int kmg_index_stats(const kmg_index *ix, uint64_t *multi, uint32_t *max_count) {
  if (!ix) return fail(KMG_ERR_ARG, "index is NULL");
  TRY(ensure_stats(ix));
  if (multi) *multi = ix->multi;
  if (max_count) *max_count = ix->maxc;
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// extraction
// ------------------------------------------------------------------------------------------------
// Run `emit(first, rows, d_dst)` over [0,total) rows of `row_bytes` each and land them at `out`.
// Device destinations are written in place; host destinations go through two device chunks so the
// copy of chunk c overlaps the kernel of chunk c+1.
// stream_rows for a large pageable destination: device chunk -> pinned slot (DMA) -> caller's buffer (host threads), the
// three stages of consecutive chunks overlapping.
template <class Emit>
static int stream_rows_staged(uint64_t total, size_t row_bytes, void *out, Emit emit) {
  std::lock_guard<std::mutex> g(g_stage.mu);
  TRY(g_stage.ensure());
  cudaStream_t s = g_ctx.stream(), cs = g_ctx.copy;
  const uint64_t chunk_rows = std::max<uint64_t>(1, STAGE_BYTES / row_bytes);
  const int64_t nchunks = (int64_t)ceil_div<uint64_t>(total, chunk_rows);
  DevBuf<uint64_t> blk(s);
  DevBuf<char> buf0(s), buf1(s);
  TRY(blk.alloc((size_t)ceil_div<uint64_t>(chunk_rows, EMIT_TILE)));
  TRY(buf0.alloc(chunk_rows * row_bytes));
  if (nchunks > 1) TRY(buf1.alloc(chunk_rows * row_bytes));
  char *buf[2] = {buf0, buf1};
  cudaEvent_t *ev = g_ctx.ev;                          // ev[0..1] kernel done, ev[4..6] slot filled (= device buffer free again)
  int64_t issued = 0, retired = 0;
  int rc = KMG_OK;                                     // on a failure the copies in flight are still drained
  while (rc == KMG_OK && retired < nchunks) {
    while (rc == KMG_OK && issued < nchunks && issued - retired < 2) {
      const int64_t c = issued;
      const int b = (int)(c & 1), sl = (int)(c % STAGE_SLOTS);
      const uint64_t first = (uint64_t)c * chunk_rows, rows = std::min<uint64_t>(chunk_rows, total - first);
      if (c >= STAGE_SLOTS) g_pool.wait((int)(c - STAGE_SLOTS));       // the slot's previous contents have reached the caller
      if (c >= 2) cudaStreamWaitEvent(s, ev[4 + (int)((c - 2) % STAGE_SLOTS)], 0);   // device buffer b has been drained
      rc = emit(first, rows, (void *)buf[b], blk, s);
      if (rc != KMG_OK) break;
      cudaEventRecord(ev[b], s);
      cudaStreamWaitEvent(cs, ev[b], 0);
      if (cudaMemcpyAsync(g_stage.slot[sl], buf[b], rows * row_bytes, cudaMemcpyDeviceToHost, cs) != cudaSuccess)
        rc = fail(KMG_ERR_CUDA, "device->host copy failed: %s", cudaGetErrorString(cudaGetLastError()));
      cudaEventRecord(ev[4 + sl], cs);
      ++issued;
    }
    if (rc != KMG_OK) break;
    const int64_t c = retired;
    const int sl = (int)(c % STAGE_SLOTS);
    const uint64_t first = (uint64_t)c * chunk_rows, rows = std::min<uint64_t>(chunk_rows, total - first);
    if (cudaEventSynchronize(ev[4 + sl]) != cudaSuccess) { rc = fail(KMG_ERR_CUDA, "device->host copy failed: %s", cudaGetErrorString(cudaGetLastError())); break; }
    g_pool.submit((int)c, (char *)out + first * row_bytes, g_stage.slot[sl], rows * row_bytes);
    ++retired;
  }
  for (int64_t c = std::max<int64_t>(0, retired - STAGE_SLOTS); c < retired; ++c) g_pool.wait((int)c);
  cudaStreamSynchronize(cs);
  cudaStreamSynchronize(s);
  if (rc == KMG_OK) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail(KMG_ERR_CUDA, "extraction failed: %s", cudaGetErrorString(e));
  }
  return rc;
}

template <class Emit>
static int stream_rows(uint64_t total, size_t row_bytes, void *out, uint64_t chunk_rows, Emit emit) {
  if (total == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  const bool to_device = ptr_kind(out) == PK_DEVICE;
  if (!to_device) chunk_rows = std::min<uint64_t>(chunk_rows, total);
  DevBuf<uint64_t> blk(s);                             // first segment of every EMIT_TILE-row block of the chunk being emitted
  TRY(blk.alloc((size_t)ceil_div<uint64_t>(to_device ? total : chunk_rows, EMIT_TILE)));
  if (to_device) {
    TRY(emit((uint64_t)0, total, out, blk, s));
    if (cudaStreamSynchronize(s) != cudaSuccess) return fail(KMG_ERR_CUDA, "extraction failed: %s", cudaGetErrorString(cudaGetLastError()));
    return KMG_OK;
  }
  if (staged_transfers() && total * row_bytes > (uint64_t)(8 << 20) && ptr_kind(out) == PK_HOST_PAGEABLE) {
    blk.reset();
    return stream_rows_staged(total, row_bytes, out, emit);
  }
  DevBuf<char> buf0(s), buf1(s);
  TRY(buf0.alloc(chunk_rows * row_bytes));
  if (total > chunk_rows) TRY(buf1.alloc(chunk_rows * row_bytes));
  char *buf[2] = {buf0, buf1};
  cudaStream_t cs = g_ctx.copy;
  cudaEvent_t *ev = g_ctx.ev;                        // ev[0..1] kernel done, ev[2..3] copy done
  uint64_t done = 0;
  int rc = KMG_OK;                                   // on a failure the copies in flight are still drained
  for (int c = 0; done < total && rc == KMG_OK; ++c, done += chunk_rows) {
    const int b = c & 1;
    const uint64_t rows = std::min<uint64_t>(chunk_rows, total - done);
    if (c >= 2) cudaStreamWaitEvent(s, ev[2 + b], 0);          // buffer b free again
    rc = emit(done, rows, (void *)buf[b], blk, s);
    if (rc != KMG_OK) break;
    cudaEventRecord(ev[b], s);
    cudaStreamWaitEvent(cs, ev[b], 0);
    if (cudaMemcpyAsync((char *)out + done * row_bytes, buf[b], rows * row_bytes, cudaMemcpyDeviceToHost, cs) != cudaSuccess)
      rc = fail(KMG_ERR_CUDA, "device->host copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaEventRecord(ev[2 + b], cs);
  }
  cudaStreamSynchronize(cs);
  cudaStreamSynchronize(s);
  if (rc == KMG_OK) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail(KMG_ERR_CUDA, "extraction failed: %s", cudaGetErrorString(e));
  }
  return rc;
}
constexpr uint64_t CHUNK_BYTES = uint64_t(256) << 20;

// first segment of every EMIT_TILE-row block of a chunk (see segment_starts_kernel) into stream_rows' scratch
template <typename OffT>
static int block_starts(const OffT *off, uint64_t cnt, uint64_t first, uint64_t rows, cudaStream_t s, uint64_t *blk) {
  const uint64_t nb = ceil_div<uint64_t>(rows, EMIT_TILE);
  LAUNCH("segment_starts", s, segment_starts_kernel<OffT><<<(unsigned)ceil_div<uint64_t>(nb, 128), 128, 0, s>>>(off, cnt, first, EMIT_TILE, nb, blk));
  return KMG_OK;
}

extern "C" int kmg_kmers_u64(const kmg_index *ix, uint64_t *keys) {
  TRY(use_index(ix));
  if (!keys && ix->U) return fail(KMG_ERR_ARG, "keys is NULL");
  if (ix->U == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  CU(cudaMemcpyAsync(keys, ix->ukeys, ix->U * sizeof(uint64_t), cudaMemcpyDefault, s));
  CU(cudaStreamSynchronize(s));
  return KMG_OK;
}

extern "C" int kmg_kmers_ascii(const kmg_index *ix, char *out) {
  TRY(use_index(ix));
  if (!out && ix->U) return fail(KMG_ERR_ARG, "buf is NULL");
  const size_t stride = (size_t)ix->k + 1;
  const int k = ix->k;
  const uint64_t *ukeys = ix->ukeys;
  const int sms = g_ctx.sms;
  int rc = stream_rows(ix->U, stride, out, CHUNK_BYTES / stride, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(rows * stride, 256), (uint64_t)sms * 16);
    LAUNCH("kmers_ascii", s, kmers_ascii_kernel<<<grid, 256, 0, s>>>(ukeys + first, rows, k, (char *)dst));
    return KMG_OK;
  });
  prof_bytes("kmers_ascii", (double)ix->U * (8 + stride));
  return rc;
}

extern "C" int kmg_counts(const kmg_index *ix, int32_t *out) {
  TRY(use_index(ix));
  if (!out && ix->U) return fail(KMG_ERR_ARG, "counts is NULL");
  const uint32_t *ustart = ix->ustart;            // a count is at most N <= INT32_MAX
  const int sms = g_ctx.sms;
  int rc = stream_rows(ix->U, 4, out, CHUNK_BYTES / 4, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(rows, 256), (uint64_t)sms * 16);
    LAUNCH("counts", s, counts_kernel<<<grid, 256, 0, s>>>(ustart + first, rows, (int32_t *)dst));
    return KMG_OK;
  });
  prof_bytes("counts", 8.0 * ix->U);
  return rc;
}

extern "C" int kmg_positions(const kmg_index *ix, int32_t *out) { return kmg_positions_base(ix, 0, out); }

// kmg_positions with the k-mer number offset by i_base: a rank of a sharded index writes its slice of one caller
// matrix with GLOBAL k-mer numbers (i_base = distinct k-mers held by the owners before it; SURVEY.md 8e "Extraction")
extern "C" int kmg_positions_base(const kmg_index *ix, uint64_t i_base, int32_t *out) {
  TRY(use_index(ix));
  if (!out && ix->N) return fail(KMG_ERR_ARG, "out is NULL");
  if (i_base + ix->U > (uint64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "k-mer numbers exceed int");
  const uint32_t *ustart = ix->ustart, *pos = ix->pos;
  const uint64_t U = ix->U, N = ix->N;
  int rc = stream_rows(N, 8, out, CHUNK_BYTES / 8, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *blk, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)ceil_div<uint64_t>(rows, EMIT_TILE);
    TRY(block_starts(ustart, U, first, rows, s, blk));
    LAUNCH("positions", s, positions_kernel<EMIT_THREADS><<<grid, EMIT_THREADS, 0, s>>>(ustart, U, pos, first, rows, blk, (int2 *)dst, (uint32_t)i_base));
    return KMG_OK;
  });
  prof_bytes("positions", 4.0 * U + 12.0 * N);
  return rc;
}

static int ensure_pair_index(kmg_index *ix) {
  TRY(ensure_stats(ix));
  std::lock_guard<std::mutex> g(ix->mu);
  if (ix->pair_off || ix->multi == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint32_t> multi_u(s), ticket(s);
  DevBuf<uint64_t> pair_off(s);
  DevBuf<Pair64> status(s);
  const uint64_t tiles = ceil_div<uint64_t>(ix->U, PIDX_TILE);
  TRY(multi_u.alloc(ix->multi));
  TRY(pair_off.alloc(ix->multi));
  TRY(status.alloc(tiles));
  TRY(ticket.alloc(1));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  LAUNCH("pair_index", s, pair_index_kernel<PIDX_THREADS, PIDX_ITEMS><<<(unsigned)tiles, PIDX_THREADS, 0, s>>>(
                              ix->ustart, ix->U, multi_u, pair_off, status, ticket));
  CU(cudaStreamSynchronize(s));
  ix->multi_u = multi_u.release(); ix->pair_off = pair_off.release();
  prof_bytes("pair_index", 4.0 * ix->U + 12.0 * ix->multi);
  return KMG_OK;
}

extern "C" int kmg_pairs_chunk(const kmg_index *cix, uint64_t first, uint64_t n, int32_t *out) { return kmg_pairs_chunk_base(cix, 0, first, n, out); }

extern "C" int kmg_pairs_chunk_base(const kmg_index *cix, uint64_t i_base, uint64_t first, uint64_t n, int32_t *out) {
  TRY(use_index(cix));
  if (i_base + cix->U > (uint64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "k-mer numbers exceed int");
  kmg_index *ix = const_cast<kmg_index *>(cix);
  TRY(ensure_stats(ix));
  if (first > ix->P || n > ix->P - first) return fail(KMG_ERR_ARG, "pair rows [%llu,+%llu) outside [0,%llu)", (unsigned long long)first, (unsigned long long)n, (unsigned long long)ix->P);
  if (n == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  TRY(ensure_pair_index(ix));
  const uint32_t *ustart = ix->ustart, *pos = ix->pos, *multi_u = ix->multi_u;
  const uint64_t *pair_off = ix->pair_off;
  const uint64_t n_multi = ix->multi;
  int rc = stream_rows(n, 12, out, CHUNK_BYTES / 12, [=](uint64_t f, uint64_t rows, void *dst, uint64_t *blk, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)ceil_div<uint64_t>(rows, EMIT_TILE);
    TRY(block_starts(pair_off, n_multi, first + f, rows, s, blk));
    LAUNCH("pairs", s, pairs_kernel<EMIT_THREADS><<<grid, EMIT_THREADS, 0, s>>>(ustart, pos, multi_u, pair_off, n_multi, first + f, rows, blk, (int32_t *)dst, (uint32_t)i_base));
    return KMG_OK;
  });
  prof_bytes("pairs", 12.0 * n);
  return rc;
}
extern "C" int kmg_pairs(const kmg_index *ix, int32_t *out) {
  if (!ix) return fail(KMG_ERR_ARG, "index is NULL");
  TRY(ensure_stats(ix));
  return kmg_pairs_chunk(ix, 0, ix->P, out);
}

// ------------------------------------------------------------------------------------------------
// probe
// ------------------------------------------------------------------------------------------------
static int ensure_hash(kmg_index *ix) {
  std::lock_guard<std::mutex> g(ix->mu);
  if (ix->hash || ix->U == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(ix->U, 256), (uint64_t)g_ctx.sms * 32);
  DevBuf<uint4> slots(s);
  // grouped index: the k-mers are in ascending order of the sorted bits of their mix, which a monotone bucket function
  // turns into ascending bucket order: the table is streamed out (one bucket per k-mer on average = load 0.5)
  const bool stream = ix->grouped && ix->hbits >= 8 && ix->hbits <= 56 && !g_hash_cas && (ix->hbits >= 40 || ix->U + ix->U / 4 <= (uint64_t(1) << ix->hbits));
  if (stream) {
    const uint64_t nb = std::max<uint64_t>(ix->U + ix->U / 4, 4);      // 1.25 buckets of two slots per k-mer: load 0.4
    DevBuf<uint64_t> d_last(s);
    TRY(slots.alloc(nb * BUCKET_SLOTS));
    TRY(d_last.alloc(1));
    KeyHash kt{slots, nb, ix->hbits};
    uint64_t h_last = 0;
    LAUNCH("hash_stream", s, hash_stream_kernel<<<grid, 256, 0, s>>>(ix->ukeys, ix->ustart, ix->U, kt, d_last));
    CU(cudaMemcpyAsync(&h_last, d_last, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (h_last + 1 < nb) CU(cudaMemsetAsync(slots + (h_last + 1) * BUCKET_SLOTS, 0, (nb - h_last - 1) * BUCKET_SLOTS * sizeof(uint4), s));
    constexpr int OV_ITEMS = 8;
    const unsigned ogrid = (unsigned)ceil_div<uint64_t>(ix->U, 256 * OV_ITEMS);
    LAUNCH("hash_insert", s, hash_overflow_kernel<OV_ITEMS><<<ogrid, 256, 0, s>>>(ix->ukeys, ix->ustart, ix->U, kt));
    CU(cudaStreamSynchronize(s));
    ix->hash = slots.release(); ix->hash_nb = nb; ix->hash_hbits = ix->hbits;
    prof_bytes("hash_stream", 12.0 * ix->U + 16.0 * BUCKET_SLOTS * nb);
    prof_bytes("hash_insert", 8.0 * ix->U);
    return KMG_OK;
  }
  uint64_t cap = 4 * BUCKET_SLOTS;
  while (cap < 2 * ix->U) cap <<= 1;                          // load <= 0.5
  TRY(slots.alloc(cap));
  CU(cudaMemsetAsync(slots, 0, cap * sizeof(uint4), s));
  LAUNCH("hash_insert", s, hash_insert_kernel<<<grid, 256, 0, s>>>(ix->ukeys, IndexPayload{ix->ustart}, ix->U, KeyHash{slots, cap / BUCKET_SLOTS, 0}, false));
  CU(cudaStreamSynchronize(s));
  ix->hash = slots.release(); ix->hash_nb = cap / BUCKET_SLOTS; ix->hash_hbits = 0;
  prof_bytes("hash_insert", 12.0 * ix->U + 16.0 * ix->U);
  return KMG_OK;
}

static int query_common(const kmg_index *cix, bool from_seq, const SeqView &sv, const uint64_t *d_keys,
                        const int32_t *d_i, int64_t n, kmg_query **out, uint64_t *M, const uint64_t *d_n = nullptr, bool mixed = false,
                        uint32_t max_count = UINT32_MAX) {
  kmg_index *ix = const_cast<kmg_index *>(cix);
  cudaStream_t s = g_ctx.stream();
  QueryPtr q(new (std::nothrow) kmg_query());
  if (!q) return fail(KMG_ERR_NOMEM, "host allocation failed");
  q->idx = ix;
  const int64_t total = from_seq ? sv.nstarts : n;
  if (total <= 0 || ix->U == 0) { if (M) *M = 0; *out = q.release(); return KMG_OK; }
  TRY(ensure_hash(ix));
  DevBuf<QueryStats> qs(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  DevBuf<uint2> found(s);
  const uint64_t tiles = ceil_div<uint64_t>((uint64_t)total, COMPACT_TILE);
  TRY(dalloc(&q->hit_i, (size_t)total, s));
  TRY(dalloc(&q->hit_start, (size_t)total, s));
  TRY(dalloc(&q->row_off, (size_t)total, s));
  TRY(qs.alloc(1));
  TRY(status.alloc(tiles));
  TRY(ticket.alloc(1));
  CU(cudaMemsetAsync(qs, 0, sizeof(QueryStats), s));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  KeyHash kt{ix->hash, ix->hash_nb, ix->hash_hbits};
  TRY(found.alloc((size_t)total));
  const unsigned ltiles = (unsigned)ceil_div<uint64_t>((uint64_t)total, PROBE_TILE);
  if (from_seq) {
    LAUNCH("probe_lookup", s, probe_lookup_kernel<PROBE_THREADS, PROBE_ITEMS, true><<<ltiles, PROBE_THREADS, 0, s>>>(sv, nullptr, 0, nullptr, kt, found));
    LAUNCH("probe_compact", s, probe_compact_kernel<PROBE_THREADS, COMPACT_ITEMS, true><<<(unsigned)tiles, PROBE_THREADS, 0, s>>>(
                                   found, sv.s0 + sv.k, nullptr, total, nullptr, q->hit_i, q->hit_start, q->row_off, qs, status, ticket, max_count));
  } else {
    LAUNCH("probe_lookup_rec", s, probe_lookup_kernel<PROBE_THREADS, PROBE_ITEMS, false><<<ltiles, PROBE_THREADS, 0, s>>>(sv, d_keys, n, d_n, kt, found, mixed));
    LAUNCH("probe_compact", s, probe_compact_kernel<PROBE_THREADS, COMPACT_ITEMS, false><<<(unsigned)tiles, PROBE_THREADS, 0, s>>>(
                                   found, 0, d_i, n, d_n, q->hit_i, q->hit_start, q->row_off, qs, status, ticket, max_count));
  }
  QueryStats h;
  CU(cudaMemcpyAsync(&h, qs, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  q->H = h.H; q->M = h.M;
  // a lookup moves one 128-byte line of HBM (measured: tools/micro/gups.cu), whatever it uses of it
  prof_bytes(from_seq ? "probe_lookup" : "probe_lookup_rec", (from_seq ? (double)sv.avail : 8.0 * total) + 128.0 * total + 8.0 * total);
  prof_bytes("probe_compact", 8.0 * total + 16.0 * q->H);
  if (M) *M = q->M;
  *out = q.release();
  return KMG_OK;
}

// seq.kmer.pos of q (rc: of reverseComplement(q), taken on the device); k-mers with more than max_count positions give no rows
static int query_seq(const kmg_index *ix, const char *qseq, int64_t qlen, int k, bool rc, uint32_t max_count, kmg_query **st, uint64_t *M) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (qlen < 0 || (qlen > 0 && !qseq)) return fail(KMG_ERR_ARG, "bad query pointer/length");
  if (qlen + 1 > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "query longer than int coordinates");
  TRY(use_index(ix));
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint8_t> fwd(s), rev(s);
  TRY(upload_seq(qseq, qlen, s, fwd));
  const uint8_t *base = fwd + 16;
  if (rc) {
    TRY(seq_alloc(rev, qlen, s));
    if (qlen > 0) {
      const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(qlen, 256), (int64_t)g_ctx.sms * 16);
      LAUNCH("revcomp", s, revcomp_kernel<<<grid, 256, 0, s>>>(fwd + 16, qlen, rev + 16));
      prof_bytes("revcomp", 2.0 * qlen);
    }
    base = rev + 16;
  }
  SeqView sv;
  sv.base = base; sv.nstarts = qlen - k + 1 > 0 ? qlen - k + 1 : 0; sv.avail = qlen; sv.s0 = 0; sv.L = qlen; sv.k = k;
  return query_common(ix, true, sv, nullptr, nullptr, 0, st, M, nullptr, false, max_count);
}

extern "C" int kmg_query_begin(const kmg_index *ix, const char *qseq, int64_t qlen, int k, kmg_query **st, uint64_t *M) {
  return query_seq(ix, qseq, qlen, k, false, UINT32_MAX, st, M);
}

// seq.kmer.pos(idx, reverseComplement(q), k) with the reverse complement taken on the device
extern "C" int kmg_query_begin_rc(const kmg_index *ix, const char *qseq, int64_t qlen, int k, kmg_query **st, uint64_t *M) {
  return query_seq(ix, qseq, qlen, k, true, UINT32_MAX, st, M);
}

extern "C" int kmg_query_records(const kmg_index *ix, const uint64_t *d_keys, const int32_t *d_i, int64_t n, kmg_query **st, uint64_t *M) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (n < 0 || (n > 0 && (!d_keys || !d_i))) return fail(KMG_ERR_ARG, "bad record arrays");
  TRY(use_index(ix));
  SeqView sv{};
  return query_common(ix, false, sv, d_keys, d_i, n, st, M);
}

extern "C" int kmg_query_emit_chunk(kmg_query *q, uint64_t first, uint64_t n, int32_t *out) {
  if (!q) return fail(KMG_ERR_ARG, "query is NULL");
  TRY(use_index(q->idx));
  if (first > q->M || n > q->M - first) return fail(KMG_ERR_ARG, "rows outside the result");
  if (n == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  const kmg_index *ix = q->idx;
  const int32_t *hit_i = q->hit_i;
  const uint32_t *hit_start = q->hit_start, *pos = ix->pos;
  const uint64_t *row_off = q->row_off;
  const uint64_t H = q->H;
  int rc = stream_rows(n, 8, out, CHUNK_BYTES / 8, [=](uint64_t f, uint64_t rows, void *dst, uint64_t *blk, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)ceil_div<uint64_t>(rows, EMIT_TILE);
    TRY(block_starts(row_off, H, first + f, rows, s, blk));
    LAUNCH("probe_emit", s, probe_emit_kernel<EMIT_THREADS><<<grid, EMIT_THREADS, 0, s>>>(hit_i, hit_start, row_off, H, pos, first + f, rows, blk, (int2 *)dst));
    return KMG_OK;
  });
  prof_bytes("probe_emit", 12.0 * n);
  return rc;
}
extern "C" int kmg_query_emit(kmg_query *q, int32_t *out) {
  if (!q) return fail(KMG_ERR_ARG, "query is NULL");
  return kmg_query_emit_chunk(q, 0, q->M, out);
}
extern "C" int kmg_query_free(kmg_query *q) {
  if (!q) return KMG_OK;
  release_on_device(q->idx ? q->idx->device : g_ctx.device, {q->hit_i, q->hit_start, q->row_off});
  delete q;
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// kmer.pairs
// ------------------------------------------------------------------------------------------------
struct kmg_join {
  const kmg_index *a = nullptr, *b = nullptr;
  uint64_t H = 0, M = 0;
  uint32_t *hit_astart = nullptr, *hit_bstart = nullptr, *hit_cb = nullptr;
  uint64_t *row_off = nullptr;
};

extern "C" int kmg_join_free(kmg_join *j) {
  if (!j) return KMG_OK;
  release_on_device(j->a ? j->a->device : g_ctx.device, {j->hit_astart, j->hit_bstart, j->hit_cb, j->row_off});
  delete j;
  return KMG_OK;
}

static int join_begin(const kmg_index *a, const kmg_index *cb, uint32_t max_count, kmg_join **out, uint64_t *M) {
  if (!out) return fail(KMG_ERR_ARG, "st is NULL");
  *out = nullptr;
  if (!a || !cb) return fail(KMG_ERR_ARG, "index is NULL");
  if (a->device != cb->device) return fail(KMG_ERR_ARG, "the two indexes live on different devices (%d, %d)", a->device, cb->device);
  TRY(use_index(a));
  kmg_index *b = const_cast<kmg_index *>(cb);
  cudaStream_t s = g_ctx.stream();
  JoinPtr j(new (std::nothrow) kmg_join());
  if (!j) return fail(KMG_ERR_NOMEM, "host allocation failed");
  j->a = a; j->b = b;
  if (a->U == 0 || b->U == 0) { if (M) *M = 0; *out = j.release(); return KMG_OK; }
  TRY(ensure_hash(b));
  DevBuf<QueryStats> qs(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  DevBuf<uint2> found(s);
  const uint64_t U = a->U;
  const uint64_t tiles = ceil_div<uint64_t>(U, PROBE_TILE);
  TRY(dalloc(&j->hit_astart, (size_t)U, s));
  TRY(dalloc(&j->hit_bstart, (size_t)U, s));
  TRY(dalloc(&j->hit_cb, (size_t)U, s));
  TRY(dalloc(&j->row_off, (size_t)U, s));
  TRY(found.alloc((size_t)U));
  TRY(qs.alloc(1));
  TRY(status.alloc(tiles));
  TRY(ticket.alloc(1));
  CU(cudaMemsetAsync(qs, 0, sizeof(QueryStats), s));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  KeyHash kt{b->hash, b->hash_nb, b->hash_hbits};
  SeqView sv{};
  LAUNCH("probe_lookup_rec", s, probe_lookup_kernel<PROBE_THREADS, PROBE_ITEMS, false><<<(unsigned)tiles, PROBE_THREADS, 0, s>>>(
                                    sv, a->ukeys, (int64_t)U, nullptr, kt, found));
  LAUNCH("join_compact", s, join_compact_kernel<PROBE_THREADS, PROBE_ITEMS><<<(unsigned)tiles, PROBE_THREADS, 0, s>>>(
                                found, a->ustart, U, j->hit_astart, j->hit_bstart, j->hit_cb, j->row_off, qs, status, ticket, max_count));
  QueryStats h;
  CU(cudaMemcpyAsync(&h, qs, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  j->H = h.H; j->M = h.M;
  prof_bytes("probe_lookup_rec", 8.0 * U + 128.0 * U + 8.0 * U);
  prof_bytes("join_compact", 12.0 * U + 20.0 * j->H);
  if (M) *M = j->M;
  *out = j.release();
  return KMG_OK;
}

extern "C" int kmg_join_begin(const kmg_index *a, const kmg_index *b, kmg_join **out, uint64_t *M) {
  return join_begin(a, b, UINT32_MAX, out, M);
}

extern "C" int kmg_join_emit_chunk(kmg_join *j, uint64_t first, uint64_t n, int32_t *out) {
  if (!j) return fail(KMG_ERR_ARG, "join is NULL");
  TRY(use_index(j->a));
  if (first > j->M || n > j->M - first) return fail(KMG_ERR_ARG, "rows outside the result");
  if (n == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  const uint32_t *ha = j->hit_astart, *hb = j->hit_bstart, *hc = j->hit_cb, *pa = j->a->pos, *pb = j->b->pos;
  const uint64_t *row_off = j->row_off;
  const uint64_t H = j->H;
  int rc = stream_rows(n, 8, out, CHUNK_BYTES / 8, [=](uint64_t f, uint64_t rows, void *dst, uint64_t *blk, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)ceil_div<uint64_t>(rows, EMIT_TILE);
    TRY(block_starts(row_off, H, first + f, rows, s, blk));
    LAUNCH("join_emit", s, join_emit_kernel<EMIT_THREADS><<<grid, EMIT_THREADS, 0, s>>>(ha, hb, hc, row_off, H, pa, pb, first + f, rows, blk, (int2 *)dst));
    return KMG_OK;
  });
  prof_bytes("join_emit", 16.0 * n);
  return rc;
}
extern "C" int kmg_join_emit(kmg_join *j, int32_t *out) {
  if (!j) return fail(KMG_ERR_ARG, "join is NULL");
  return kmg_join_emit_chunk(j, 0, j->M, out);
}

// ------------------------------------------------------------------------------------------------
// dot plots: the 2-D histogram of a probe's or a join's rows, counted on the device
// ------------------------------------------------------------------------------------------------
// Rows are walked in slices of DOT_SLICE_ROWS, so the block-start scratch stays 4 MB however many rows there are.
constexpr uint64_t DOT_SLICE_ROWS = uint64_t(1) << 30;

static DotAxis dot_axis(int64_t lo, int64_t hi, int n) {
  const uint64_t range = (uint64_t)(hi - lo);
  return DotAxis{(uint64_t)lo, range, ~uint64_t(0) / range, (uint32_t)n};
}

static int dotplot_args(int64_t x0, int64_t x1, int nx, int64_t y0, int64_t y1, int ny, const double *out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  if (nx < 1 || ny < 1) return fail(KMG_ERR_ARG, "bin counts must be at least 1 (nx = %d, ny = %d)", nx, ny);
  const int64_t top = int64_t(1) << 31;
  if (x0 < 0 || x1 <= x0 || x1 > top) return fail(KMG_ERR_ARG, "x window [%lld, %lld) is not inside [0, 2^31]", (long long)x0, (long long)x1);
  if (y0 < 0 || y1 <= y0 || y1 > top) return fail(KMG_ERR_ARG, "y window [%lld, %lld) is not inside [0, 2^31]", (long long)y0, (long long)y1);
  if ((int64_t)nx * ny > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "an image of %d x %d bins exceeds 2^31 - 1 cells", nx, ny);
  return KMG_OK;
}

// The rows [0, M) of `rows` (hits' row offsets row_off[0, H)) binned into an nx x ny image, written to out as doubles.
template <class Rows>
static int dotplot_run(const Rows &rows, const uint64_t *row_off, uint64_t H, uint64_t M, double row_bytes, DotAxis ax, DotAxis ay,
                       double *out) {
  cudaStream_t s = g_ctx.stream();
  const uint64_t cells = (uint64_t)ax.n * ay.n;
  DevBuf<unsigned long long> img(s);
  DevBuf<uint64_t> blk(s);
  TRY(img.alloc(cells));
  CU(cudaMemsetAsync(img, 0, cells * sizeof(unsigned long long), s));
  if (M) TRY(blk.alloc((size_t)ceil_div<uint64_t>(std::min(M, DOT_SLICE_ROWS), EMIT_TILE)));
  for (uint64_t first = 0; first < M; first += DOT_SLICE_ROWS) {
    const uint64_t n = std::min(DOT_SLICE_ROWS, M - first);
    TRY(block_starts(row_off, H, first, n, s, blk));
    LAUNCH("dotplot_bin", s, dotplot_bin_kernel<EMIT_THREADS, Rows><<<(unsigned)ceil_div<uint64_t>(n, EMIT_TILE), EMIT_THREADS, 0, s>>>(
                                 rows, row_off, H, first, n, blk, ax, ay, img));
  }
  const int sms = g_ctx.sms;
  const unsigned long long *im = img;
  TRY(stream_rows(cells, 8, out, CHUNK_BYTES / 8, [=](uint64_t f, uint64_t n, void *dst, uint64_t *, cudaStream_t st) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(n, 256), (uint64_t)sms * 16);
    LAUNCH("dotplot_finish", st, dotplot_finish_kernel<<<grid, 256, 0, st>>>(im + f, n, (double *)dst));
    return KMG_OK;
  }));
  cudaStreamSynchronize(s);
  prof_bytes("dotplot_bin", row_bytes * (double)M + 8.0 * (double)cells);
  prof_bytes("dotplot_finish", 16.0 * (double)cells);
  return KMG_OK;
}

extern "C" int kmg_query_dotplot(const kmg_index *ix, const char *q, int64_t qlen, int k, int rc, int64_t x0, int64_t x1, int nx,
                                 int64_t y0, int64_t y1, int ny, uint32_t max_count, double *out) {
  if (!ix) return fail(KMG_ERR_ARG, "index is NULL");
  if (rc != 0 && rc != 1) return fail(KMG_ERR_ARG, "rc must be 0 or 1");
  TRY(dotplot_args(x0, x1, nx, y0, y1, ny, out));
  kmg_query *st = nullptr;
  uint64_t M = 0;
  TRY(query_seq(ix, q, qlen, k, rc == 1, max_count ? max_count : UINT32_MAX, &st, &M));
  const QueryPtr probe(st);
  const ProbeRows rows{st->hit_i, st->hit_start, ix->pos};
  return dotplot_run(rows, st->row_off, st->H, M, 4.0, dot_axis(x0, x1, nx), dot_axis(y0, y1, ny), out);
}

extern "C" int kmg_join_dotplot(const kmg_index *a, const kmg_index *b, int64_t x0, int64_t x1, int nx, int64_t y0, int64_t y1, int ny,
                                uint32_t max_count, double *out) {
  if (!a || !b) return fail(KMG_ERR_ARG, "index is NULL");
  TRY(dotplot_args(x0, x1, nx, y0, y1, ny, out));
  kmg_join *j = nullptr;
  uint64_t M = 0;
  TRY(join_begin(a, b, max_count ? max_count : UINT32_MAX, &j, &M));
  const JoinPtr join(j);
  const JoinRows rows{j->hit_astart, j->hit_bstart, j->hit_cb, a->pos, b->pos};
  return dotplot_run(rows, j->row_off, j->H, M, 8.0, dot_axis(x0, x1, nx), dot_axis(y0, y1, ny), out);
}

// ------------------------------------------------------------------------------------------------
// match segments: maximal diagonal runs of a probe's rows (segments.cuh)
// ------------------------------------------------------------------------------------------------
struct kmg_segments {
  int device = 0;
  bool anti = false;            // antiparallel runs (kmg_join_segments_begin with rc = 1): the chains' orientation
  uint64_t R = 0;
  int32_t *rows = nullptr;      // [3R]: (i, j, n) per run
};
constexpr uint64_t SEG_SLICE_ROWS = uint64_t(1) << 30;   // rows per mark launch: the block-start and status scratch stay small
constexpr uint64_t SEG_CAP0 = uint64_t(1) << 26;         // starts / ends held before the first resize (20 bytes each)
constexpr int SEG_PAIR_ITEMS = 8, SEG_PAIR_TILE = 256 * SEG_PAIR_ITEMS;

// p[0, keep) moved into a fresh array of cap elements
template <typename T>
static int seg_grow(DevBuf<T> &p, uint64_t keep, uint64_t cap, cudaStream_t s) {
  DevBuf<T> q(s);
  TRY(q.alloc((size_t)cap));
  if (keep) CU(cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s));
  p.reset(q.release());
  return KMG_OK;
}

// Run starts (i, j) and run ends (diagonal key, i) of the probe st, each in row order, into arrays of at least R0 entries.
template <bool ANTI>
static int segments_mark(const kmg_query *st, const uint32_t *pos, DevBuf<int2> &starts, DevBuf<uint64_t> &ekey, DevBuf<uint32_t> &ei,
                         uint64_t *R0) {
  cudaStream_t s = g_ctx.stream();
  const uint64_t M = st->M;
  const uint64_t slice_tiles = ceil_div<uint64_t>(std::min(M, SEG_SLICE_ROWS), EMIT_TILE);
  uint64_t cap = std::min(M, SEG_CAP0), bs = 0, be = 0;
  DevBuf<uint64_t> blk(s), tot(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  TRY(starts.alloc((size_t)cap));
  TRY(ekey.alloc((size_t)cap));
  TRY(ei.alloc((size_t)cap));
  TRY(blk.alloc((size_t)slice_tiles));
  TRY(status.alloc((size_t)slice_tiles));
  TRY(ticket.alloc(1));
  TRY(tot.alloc(2));
  for (uint64_t first = 0; first < M;) {
    const uint64_t n = std::min(SEG_SLICE_ROWS, M - first);
    const uint64_t tiles = ceil_div<uint64_t>(n, EMIT_TILE);
    CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
    CU(cudaMemsetAsync(ticket, 0, 4, s));
    TRY(block_starts(st->row_off, st->H, first, n, s, blk));
    LAUNCH("segments_mark", s, segments_mark_kernel<EMIT_THREADS, ANTI><<<(unsigned)tiles, EMIT_THREADS, 0, s>>>(
                                   st->hit_i, st->hit_start, st->row_off, st->H, M, pos, first, n, blk, status, ticket, bs, be,
                                   cap, starts, ekey, ei, tot));
    uint64_t h[2];
    CU(cudaMemcpyAsync(h, tot, sizeof h, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const uint64_t need = std::max(bs + h[0], be + h[1]);
    if (need > (uint64_t)INT32_MAX)
      return fail(KMG_ERR_RANGE, "more than 2^31 - 1 runs (%llu so far) to pair", (unsigned long long)need);
    if (need > cap) {                                   // the slice did not fit: keep what is done, make room, run it again
      const uint64_t ncap = std::min<uint64_t>(std::min(M, (uint64_t)INT32_MAX), need + need / 4);
      TRY(seg_grow(starts, bs, ncap, s));
      TRY(seg_grow(ekey, be, ncap, s));
      TRY(seg_grow(ei, be, ncap, s));
      cap = ncap;
      continue;
    }
    bs += h[0]; be += h[1];
    first += n;
  }
  if (bs != be)
    return fail(KMG_ERR_CUDA, "internal error: %llu run starts but %llu run ends", (unsigned long long)bs, (unsigned long long)be);
  // rows (4 B) and one neighbouring position on either side; hits (16 B); the starts (8 B) and ends (12 B) written
  prof_bytes("segments_mark", 12.0 * M + 16.0 * st->H + 20.0 * bs);
  *R0 = bs;
  return KMG_OK;
}

// The runs of the probe st (freed here, on every path) with at least min_rows rows, as (i, j, n) triples in the order of
// their first rows: *rows (device, 12 * *R bytes) or nullptr when *R = 0.  ANTI: antiparallel runs (segments.cuh).
template <bool ANTI>
static int segments_of(kmg_query *st, uint32_t min_rows, int32_t **rows, uint64_t *R) {
  *rows = nullptr;
  *R = 0;
  QueryPtr probe(st);
  const uint64_t M = st->M;
  if (M == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  DevBuf<int2> starts(s);
  DevBuf<uint64_t> ekey(s);
  DevBuf<uint32_t> ei(s);
  uint64_t R0 = 0;
  TRY(segments_mark<ANTI>(st, st->idx->pos, starts, ekey, ei, &R0));
  probe.reset();                                          // the probe is done with: only the runs stay
  // the ends sorted by diagonal, i ascending inside one: keys below 2^32 (segment_key) are the 32 bits of a 16-mer
  kmg_index *e = nullptr;
  TRY(kmg_build_records(ekey, ei, (int64_t)R0, 16, &e));
  const IndexPtr ends(e);
  ekey.reset(); ei.reset();
  const uint64_t tiles = ceil_div<uint64_t>(R0, SEG_PAIR_TILE);
  DevBuf<int32_t> tmp(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  DevBuf<uint64_t> tot(s);
  TRY(tmp.alloc((size_t)(3 * R0)));
  TRY(status.alloc((size_t)tiles));
  TRY(ticket.alloc(1));
  TRY(tot.alloc(2));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  LAUNCH("segments_pair", s, segments_pair_kernel<256, SEG_PAIR_ITEMS, ANTI><<<(unsigned)tiles, 256, 0, s>>>(
                                 starts, R0, ends->ukeys, ends->U, ends->ustart, ends->pos, min_rows, status, ticket, tmp, tot));
  uint64_t h[2];
  CU(cudaMemcpyAsync(h, tot, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (h[1] != M)
    return fail(KMG_ERR_CUDA, "internal error: the runs hold %llu rows, the probe %llu", (unsigned long long)h[1], (unsigned long long)M);
  prof_bytes("segments_pair", 8.0 * R0 + 12.0 * R0 + 12.0 * h[0]);   // starts; the diagonal's key and end; the triples
  DevBuf<int32_t> out(s);
  if (h[0] == R0) out.reset(tmp.release());
  else if (h[0]) {                                        // keep exactly the runs that passed min_rows
    TRY(out.alloc((size_t)(3 * h[0])));
    CU(cudaMemcpyAsync(out, tmp, 12 * h[0], cudaMemcpyDeviceToDevice, s));
    CU(cudaStreamSynchronize(s));
  }
  cudaStreamSynchronize(s);
  *rows = out.release();
  *R = h[0];
  return KMG_OK;
}

// The runs of the probe (idx, q, qlen, k, rc, max_count), as segments_of
static int segments_run(const kmg_index *ix, const char *q, int64_t qlen, int k, int rc, uint32_t max_count, uint32_t min_rows,
                        int32_t **rows, uint64_t *R) {
  *rows = nullptr;
  *R = 0;
  kmg_query *st = nullptr;
  uint64_t M = 0;
  TRY(query_seq(ix, q, qlen, k, rc == 1, max_count ? max_count : UINT32_MAX, &st, &M));
  return segments_of<false>(st, min_rows, rows, R);
}

// kmer.pairs(a, b) as a probe of b (probe.cuh, "kmer.pairs.segments"): the hits are a's positions x, ascending, whose k-mer
// b holds (rc: whose code-space reverse complement b holds), each with b's position list of it, so the rows come out in
// (x, y) order.  max_count: a k-mer with more positions in a, or whose match has more in b, gives no hit.
static int join_probe(const kmg_index *a, const kmg_index *cb, bool rc, uint32_t max_count, kmg_query **out) {
  *out = nullptr;
  kmg_index *b = const_cast<kmg_index *>(cb);
  cudaStream_t s = g_ctx.stream();
  QueryPtr q(new (std::nothrow) kmg_query());
  if (!q) return fail(KMG_ERR_NOMEM, "host allocation failed");
  q->idx = b;
  if (a->U == 0 || b->U == 0) { *out = q.release(); return KMG_OK; }
  TRY(ensure_hash(b));
  const uint64_t U = a->U, N = a->N;
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(U, 256), (uint64_t)g_ctx.sms * 16);
  uint32_t X = 0;                                         // a's largest position: found_pos has one entry per x in [1, X]
  DevBuf<uint32_t> d_last(s);
  TRY(d_last.alloc(1));
  CU(cudaMemsetAsync(d_last, 0, 4, s));
  LAUNCH("last_pos", s, last_pos_kernel<<<grid, 256, 0, s>>>(a->ustart, a->pos, U, d_last));
  CU(cudaMemcpyAsync(&X, d_last, 4, cudaMemcpyDeviceToHost, s));
  const uint64_t *keys = a->ukeys;
  DevBuf<uint64_t> rkeys(s);
  if (rc) {
    TRY(rkeys.alloc((size_t)U));
    LAUNCH("revcomp_keys", s, revcomp_keys_kernel<<<grid, 256, 0, s>>>(a->ukeys, U, a->k, rkeys));
    keys = rkeys;
  }
  DevBuf<uint2> found(s);
  TRY(found.alloc((size_t)U));
  const KeyHash kt{b->hash, b->hash_nb, b->hash_hbits};
  const SeqView sv{};
  LAUNCH("probe_lookup_rec", s, probe_lookup_kernel<PROBE_THREADS, PROBE_ITEMS, false><<<(unsigned)ceil_div<uint64_t>(U, PROBE_TILE), PROBE_THREADS, 0, s>>>(
                                    sv, keys, (int64_t)U, nullptr, kt, found));
  CU(cudaStreamSynchronize(s));
  rkeys.reset();
  DevBuf<uint2> found_pos(s);
  TRY(found_pos.alloc((size_t)X));
  CU(cudaMemsetAsync(found_pos, 0, (size_t)X * sizeof(uint2), s));
  DevBuf<uint64_t> blk(s);
  TRY(blk.alloc((size_t)ceil_div<uint64_t>(std::min(N, SEG_SLICE_ROWS), EMIT_TILE)));
  for (uint64_t first = 0; first < N; first += SEG_SLICE_ROWS) {
    const uint64_t n = std::min(SEG_SLICE_ROWS, N - first);
    TRY(block_starts(a->ustart, U, first, n, s, blk));
    LAUNCH("join_scatter", s, join_scatter_kernel<EMIT_THREADS><<<(unsigned)ceil_div<uint64_t>(n, EMIT_TILE), EMIT_THREADS, 0, s>>>(
                                  a->ustart, U, a->pos, found, max_count, first, n, blk, found_pos));
  }
  const uint64_t tiles = ceil_div<uint64_t>(X, COMPACT_TILE);
  DevBuf<QueryStats> qs(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  TRY(dalloc(&q->hit_i, (size_t)X, s));
  TRY(dalloc(&q->hit_start, (size_t)X, s));
  TRY(dalloc(&q->row_off, (size_t)X, s));
  TRY(qs.alloc(1));
  TRY(status.alloc((size_t)tiles));
  TRY(ticket.alloc(1));
  CU(cudaMemsetAsync(qs, 0, sizeof(QueryStats), s));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  LAUNCH("probe_compact", s, probe_compact_kernel<PROBE_THREADS, COMPACT_ITEMS, true><<<(unsigned)tiles, PROBE_THREADS, 0, s>>>(
                                 found_pos, 1, nullptr, (int64_t)X, nullptr, q->hit_i, q->hit_start, q->row_off, qs, status, ticket,
                                 max_count));
  QueryStats h;
  CU(cudaMemcpyAsync(&h, qs, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  q->H = h.H; q->M = h.M;
  cudaStreamSynchronize(s);
  prof_bytes("last_pos", 8.0 * U);
  if (rc) prof_bytes("revcomp_keys", 16.0 * U);
  prof_bytes("probe_lookup_rec", 8.0 * U + 128.0 * U + 8.0 * U);
  // per position: its k-mer's found entry and list bounds (read once per k-mer), the position, one 8-byte write (a
  // 32-byte sector of DRAM when it scatters) for a shared k-mer; the memset of found_pos
  prof_bytes("join_scatter", 16.0 * U + 4.0 * N + 32.0 * (double)q->H + 8.0 * X);
  prof_bytes("probe_compact", 8.0 * X + 16.0 * q->H);
  *out = q.release();
  return KMG_OK;
}

// The runs of the rows of kmer.pairs(a, b) (rc: of a's k-mers reverse-complemented, antiparallel runs), as segments_of
static int join_segments_run(const kmg_index *a, const kmg_index *b, int rc, uint32_t max_count, uint32_t min_rows,
                             int32_t **rows, uint64_t *R) {
  *rows = nullptr;
  *R = 0;
  kmg_query *st = nullptr;
  TRY(join_probe(a, b, rc == 1, max_count ? max_count : UINT32_MAX, &st));
  return rc ? segments_of<true>(st, min_rows, rows, R) : segments_of<false>(st, min_rows, rows, R);
}

extern "C" int kmg_segments_begin(const kmg_index *ix, const char *q, int64_t qlen, int k, int rc, uint32_t max_count,
                                  uint32_t min_rows, kmg_segments **st, uint64_t *R) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (!ix) return fail(KMG_ERR_ARG, "index is NULL");
  if (rc != 0 && rc != 1) return fail(KMG_ERR_ARG, "rc must be 0 or 1");
  SegmentsPtr g(new (std::nothrow) kmg_segments());
  if (!g) return fail(KMG_ERR_NOMEM, "host allocation failed");
  g->device = ix->device;
  int rv = segments_run(ix, q, qlen, k, rc, max_count, min_rows, &g->rows, &g->R);
  if (rv == KMG_ERR_UNSTABLE) rv = segments_run(ix, q, qlen, k, rc, max_count, min_rows, &g->rows, &g->R);   // the sort now ranks by bitmap
  TRY(rv);
  if (R) *R = g->R;
  *st = g.release();
  return KMG_OK;
}

extern "C" int kmg_join_segments_begin(const kmg_index *a, const kmg_index *b, int rc, uint32_t max_count, uint32_t min_rows,
                                       kmg_segments **st, uint64_t *R) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (!a || !b) return fail(KMG_ERR_ARG, "index is NULL");
  if (rc != 0 && rc != 1) return fail(KMG_ERR_ARG, "rc must be 0 or 1");
  if (a->device != b->device) return fail(KMG_ERR_ARG, "the two indexes live on different devices (%d, %d)", a->device, b->device);
  if (rc && a->k != b->k) return fail(KMG_ERR_K, "the reverse complement needs indexes of one k (here %d and %d)", a->k, b->k);
  TRY(use_index(a));
  SegmentsPtr g(new (std::nothrow) kmg_segments());
  if (!g) return fail(KMG_ERR_NOMEM, "host allocation failed");
  g->device = a->device;
  g->anti = rc == 1;
  int rv = join_segments_run(a, b, rc, max_count, min_rows, &g->rows, &g->R);
  if (rv == KMG_ERR_UNSTABLE) rv = join_segments_run(a, b, rc, max_count, min_rows, &g->rows, &g->R);   // the sort now ranks by bitmap
  TRY(rv);
  if (R) *R = g->R;
  *st = g.release();
  return KMG_OK;
}

// Rows [first, first + n) of a finished int32 result of `width` words per row (segments: 3, chains: 6) to out.
static int emit_int32_rows(const int32_t *rows, int width, uint64_t first, uint64_t n, int32_t *out, const char *name) {
  if (n == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  const size_t row_bytes = 4 * (size_t)width;
  const int sms = g_ctx.sms;
  int rc = stream_rows(n, row_bytes, out, CHUNK_BYTES / row_bytes, [=](uint64_t f, uint64_t cnt, void *dst, uint64_t *, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(width * cnt, 256), (uint64_t)sms * 16);
    LAUNCH(name, s, segments_emit_kernel<<<grid, 256, 0, s>>>(rows + width * (first + f), width * cnt, (int32_t *)dst));
    return KMG_OK;
  });
  prof_bytes(name, 2.0 * row_bytes * n);
  return rc;
}

extern "C" int kmg_segments_emit_chunk(kmg_segments *g, uint64_t first, uint64_t n, int32_t *out) {
  if (!g) return fail(KMG_ERR_ARG, "segments handle is NULL");
  TRY(use_device(g->device, "the segments live"));
  if (first > g->R || n > g->R - first) return fail(KMG_ERR_ARG, "runs outside the result");
  return emit_int32_rows(g->rows, 3, first, n, out, "segments_emit");
}

extern "C" int kmg_segments_emit(kmg_segments *g, int32_t *out) {
  if (!g) return fail(KMG_ERR_ARG, "segments handle is NULL");
  return kmg_segments_emit_chunk(g, 0, g->R, out);
}

extern "C" int kmg_segments_free(kmg_segments *g) {
  if (!g) return KMG_OK;
  release_on_device(g->device, {g->rows});
  delete g;
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// chains: the runs of a segments handle joined across mismatches and short indels (segments.cuh)
// ------------------------------------------------------------------------------------------------
struct kmg_chains {
  int device = 0;
  uint64_t C = 0;
  int32_t *rows = nullptr;      // [6C]: (i, j, I, J, n, m) per chain
};
constexpr int CHAIN_COMPACT_ITEMS = 8, CHAIN_COMPACT_TILE = 256 * CHAIN_COMPACT_ITEMS;
constexpr int CHAIN_MAX_ROUNDS = 40;                      // pointer jumping halves every chain per round: 31 rounds reach 2^31 runs

// The chains of the R runs `runs` (12 R bytes, (i, j) order) with n >= min_rows, as (i, j, I, J, n, m) rows in the order of
// their first runs: *rows (device, 24 * *C bytes) or nullptr when *C = 0.  ANTI: antiparallel runs.
template <bool ANTI>
static int chains_of(const int32_t *runs, uint64_t R, uint32_t G, uint32_t W, uint32_t min_rows, int32_t **rows, uint64_t *C) {
  *rows = nullptr;
  *C = 0;
  if (R == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(R, 256), (uint64_t)g_ctx.sms * 16);
  DevBuf<uint64_t> key(s);
  DevBuf<uint32_t> run(s);
  TRY(key.alloc((size_t)R));
  TRY(run.alloc((size_t)R));
  LAUNCH("chains_keys", s, chains_keys_kernel<ANTI><<<grid, 256, 0, s>>>(runs, R, key, run));
  // the runs by diagonal, i ascending inside one (stable): keys below 2^32 (segment_key) are the 32 bits of a 16-mer
  kmg_index *d = nullptr;
  TRY(kmg_build_records(key, run, (int64_t)R, 16, &d));
  IndexPtr diag(d);
  key.reset(); run.reset();
  DevBuf<uint32_t> si(s), sI(s);
  TRY(si.alloc((size_t)R));
  TRY(sI.alloc((size_t)R));
  LAUNCH("chains_gather", s, chains_gather_kernel<<<grid, 256, 0, s>>>(runs, diag->pos, R, si, sI));
  DevBuf<int32_t> succ(s), pred(s);
  DevBuf<unsigned long long> nsum(s);
  TRY(succ.alloc((size_t)R));
  TRY(pred.alloc((size_t)R));
  TRY(nsum.alloc(1));
  CU(cudaMemsetAsync(nsum, 0, 8, s));
  LAUNCH("chains_link", s, chains_link_kernel<ANTI><<<(unsigned)ceil_div<uint64_t>(R, 256), 256, 0, s>>>(
                               runs, R, diag->ukeys, diag->U, diag->ustart, diag->pos, si, sI, G, W, succ, pred, nsum));
  const uint64_t U = diag->U;
  diag.reset();
  si.reset(); sI.reset();
  DevBuf<int32_t> head(s);
  TRY(head.alloc((size_t)R));
  LAUNCH("chains_heads", s, chains_heads_kernel<<<grid, 256, 0, s>>>(succ, pred, R, head));
  succ.reset(); pred.reset();
  // the first run of every chain by pointer jumping: a round that moves no pointer ends it
  DevBuf<uint32_t> flag(s);
  TRY(flag.alloc(1));
  int rounds = 0;
  for (uint32_t moved = 1; moved;) {
    if (++rounds > CHAIN_MAX_ROUNDS) return fail(KMG_ERR_CUDA, "internal error: pointer jumping did not settle in %d rounds", CHAIN_MAX_ROUNDS);
    CU(cudaMemsetAsync(flag, 0, 4, s));
    LAUNCH("chains_jump", s, chains_jump_kernel<<<grid, 256, 0, s>>>(head, R, flag));
    CU(cudaMemcpyAsync(&moved, flag, 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
  }
  DevBuf<unsigned long long> nm(s), last(s);
  TRY(nm.alloc((size_t)R));
  TRY(last.alloc((size_t)R));
  CU(cudaMemsetAsync(nm, 0, R * 8, s));
  CU(cudaMemsetAsync(last, 0, R * 8, s));
  LAUNCH("chains_aggregate", s, chains_aggregate_kernel<ANTI><<<grid, 256, 0, s>>>(runs, head, R, nm, last));
  const uint64_t tiles = ceil_div<uint64_t>(R, CHAIN_COMPACT_TILE);
  DevBuf<int32_t> tmp(s);
  DevBuf<Pair64> status(s);
  DevBuf<uint32_t> ticket(s);
  DevBuf<uint64_t> tot(s);
  TRY(tmp.alloc((size_t)(6 * R)));
  TRY(status.alloc((size_t)tiles));
  TRY(ticket.alloc(1));
  TRY(tot.alloc(3));
  CU(cudaMemsetAsync(status, 0, tiles * sizeof(Pair64), s));
  CU(cudaMemsetAsync(ticket, 0, 4, s));
  LAUNCH("chains_compact", s, chains_compact_kernel<256, CHAIN_COMPACT_ITEMS, ANTI><<<(unsigned)tiles, 256, 0, s>>>(
                                  runs, head, nm, last, R, min_rows, status, ticket, tmp, tot));
  uint64_t h[3], n_runs = 0;
  CU(cudaMemcpyAsync(h, tot, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&n_runs, nsum, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (h[1] != R || h[2] != n_runs)
    return fail(KMG_ERR_CUDA, "internal error: the chains hold %llu runs of %llu rows, the handle %llu runs of %llu rows",
                (unsigned long long)h[1], (unsigned long long)h[2], (unsigned long long)R, (unsigned long long)n_runs);
  // runs (12 B) and their keys (8 B); the gathered i and I; the link search (the runs, one lower bound over the U
  // diagonal keys and the candidates' i / I, counted as 64 B per run); head, aggregates, the rows written
  prof_bytes("chains_keys", 24.0 * R);
  prof_bytes("chains_gather", 24.0 * R);
  prof_bytes("chains_link", 12.0 * R + 8.0 * U + 64.0 * R + 8.0 * R);
  prof_bytes("chains_heads", 16.0 * R);
  prof_bytes("chains_jump", 8.0 * R * rounds);
  prof_bytes("chains_aggregate", 16.0 * R + 16.0 * (R - h[0]));
  prof_bytes("chains_compact", 16.0 * R + 24.0 * h[0]);
  DevBuf<int32_t> out(s);
  if (h[0] == R) out.reset(tmp.release());
  else if (h[0]) {                                        // keep exactly the chains that passed min_rows
    TRY(out.alloc((size_t)(6 * h[0])));
    CU(cudaMemcpyAsync(out, tmp, 24 * h[0], cudaMemcpyDeviceToDevice, s));
    CU(cudaStreamSynchronize(s));
  }
  cudaStreamSynchronize(s);
  *rows = out.release();
  *C = h[0];
  return KMG_OK;
}

extern "C" int kmg_chains_begin(const kmg_segments *seg, uint32_t max_gap, uint32_t max_shift, uint32_t min_rows,
                                kmg_chains **st, uint64_t *C) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (!seg) return fail(KMG_ERR_ARG, "segments handle is NULL");
  if (max_gap > (uint32_t)INT32_MAX) return fail(KMG_ERR_ARG, "max_gap must be below 2^31");
  if (max_shift > max_gap) return fail(KMG_ERR_ARG, "max_shift (%u) must not exceed max_gap (%u)", max_shift, max_gap);
  if (max_shift > 1024) return fail(KMG_ERR_ARG, "max_shift must be at most 1024");
  TRY(use_device(seg->device, "the segments live"));
  ChainsPtr g(new (std::nothrow) kmg_chains());
  if (!g) return fail(KMG_ERR_NOMEM, "host allocation failed");
  g->device = seg->device;
  auto run = [&]() {
    return seg->anti ? chains_of<true>(seg->rows, seg->R, max_gap, max_shift, min_rows, &g->rows, &g->C)
                     : chains_of<false>(seg->rows, seg->R, max_gap, max_shift, min_rows, &g->rows, &g->C);
  };
  int rv = run();
  if (rv == KMG_ERR_UNSTABLE) rv = run();                 // the sort now ranks by bitmap
  TRY(rv);
  if (C) *C = g->C;
  *st = g.release();
  return KMG_OK;
}

extern "C" int kmg_chains_emit_chunk(kmg_chains *g, uint64_t first, uint64_t n, int32_t *out) {
  if (!g) return fail(KMG_ERR_ARG, "chains handle is NULL");
  TRY(use_device(g->device, "the chains live"));
  if (first > g->C || n > g->C - first) return fail(KMG_ERR_ARG, "chains outside the result");
  return emit_int32_rows(g->rows, 6, first, n, out, "chains_emit");
}

extern "C" int kmg_chains_emit(kmg_chains *g, int32_t *out) {
  if (!g) return fail(KMG_ERR_ARG, "chains handle is NULL");
  return kmg_chains_emit_chunk(g, 0, g->C, out);
}

extern "C" int kmg_chains_free(kmg_chains *g) {
  if (!g) return KMG_OK;
  release_on_device(g->device, {g->rows});
  delete g;
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// sharded build
// ------------------------------------------------------------------------------------------------
// The caller's shard [g0,g1) is copied into an aligned, padded buffer whose byte 16 is window start s0.
static int shard_view(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1, int k,
                      cudaStream_t s, DevBuf<uint8_t> &buf, SeqView *sv) {
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (!(0 <= g0 && g0 <= g1 && g1 <= L && 0 <= s0 && s0 <= s1)) return fail(KMG_ERR_ARG, "inconsistent shard bounds");
  const int64_t need_lo = s0 > 0 ? s0 - 1 : 0, need_hi = std::min<int64_t>(L, s1 + k - 1);
  if (s1 > s0 && (g0 > need_lo || g1 < need_hi)) return fail(KMG_ERR_ARG, "shard bytes [%lld,%lld) do not cover [%lld,%lld)", (long long)g0, (long long)g1, (long long)need_lo, (long long)need_hi);
  const int64_t avail = std::max<int64_t>(0, need_hi - s0);
  TRY(seq_alloc(buf, avail, s));
  uint8_t *base = buf + 16;
  if (avail > 0) {
    const int64_t lead = s0 > 0 ? 1 : 0;        // one byte of left context for rule (iii)
    CU(cudaMemcpyAsync(base - lead, (const uint8_t *)d_seq + (s0 - lead - g0), (size_t)(avail + lead), cudaMemcpyDefault, s));
  }
  int64_t nstarts = std::min<int64_t>(s1, L - k + 1) - s0;
  sv->base = base; sv->nstarts = nstarts > 0 ? nstarts : 0; sv->avail = avail; sv->s0 = s0; sv->L = L; sv->k = k;
  return KMG_OK;
}

__global__ void sample_kernel(const SeqView sv, int n, uint64_t *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // evenly spaced windows; breakers are encoded like any byte (a sample only steers load balance)
  const int64_t q = sv.nstarts > 0 ? ((int64_t)i * sv.nstarts) / n : 0;
  uint64_t w = 0;
  for (int j = 0; j < sv.k; ++j) {
    const int64_t o = q + j;
    const uint8_t c = o < sv.avail ? sv.base[o] : 0;
    w = (w << 2) | ((c >> 1) & 3u);
  }
  out[i] = w & key_mask(sv.k);
}

extern "C" int kmg_shard_sample(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1, int k, int n, uint64_t *d_samples) {
  if (n <= 0 || !d_samples) return fail(KMG_ERR_ARG, "bad sample request");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint8_t> buf(s);
  SeqView sv;
  TRY(shard_view(d_seq, g0, g1, L, s0, s1, k, s, buf, &sv));
  LAUNCH("sample", s, sample_kernel<<<ceil_div(n, 256), 256, 0, s>>>(sv, n, d_samples));
  CU(cudaStreamSynchronize(s));
  return KMG_OK;
}

// The records of the shard sv, grouped by owner (nparts - 1 splitters), into (d_keys, d_pos); counts[i]: owner i's records
static int partition_records(const SeqView &sv, const uint64_t *splitters, int nparts, uint64_t *d_keys, uint32_t *d_pos, uint64_t *counts,
                             cudaStream_t s) {
  SortScratch sc(s);
  DevBuf<uint64_t> d_spl(s);
  TRY(scratch_alloc(sc, sv.nstarts, s));
  TRY(d_spl.alloc((size_t)RADIX));
  if (nparts > 1) CU(cudaMemcpyAsync(d_spl, splitters, (size_t)(nparts - 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  OwnerBin ob{d_spl, nparts};
  const int64_t tiles = ceil_div<int64_t>(sv.nstarts, HIST_TILE);
  const unsigned hgrid = (unsigned)std::min<int64_t>(tiles, (int64_t)g_ctx.sms * 2);
  LAUNCH("hist_seq_owner", s, hist_seq_kernel<HIST_THREADS, HIST_ITEMS, OwnerBin><<<hgrid, HIST_THREADS, 0, s>>>(sv, sc.hist(0), ob));
  TRY(launch_scan_hist(RADIX_BITS, s, sc.hist(0), sc.gbase(0), (uint64_t *)nullptr));
  PassParams<OwnerBin, NoBin> P{};
  P.sv = sv; P.keys_out = d_keys; P.pos_out = d_pos;
  P.gbase = sc.gbase(0); P.hist_next = nullptr;
  P.status = sc.status; P.ticket = sc.ticket(0); P.epoch = 1;
  P.bin = ob;
  TRY((launch_pass<true, OwnerBin, NoBin, false>("partition", P, sv.nstarts, s)));
  std::vector<uint32_t> h(RADIX);
  CU(cudaMemcpyAsync(h.data(), sc.hist(0), RADIX * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  double tot = 0;
  for (int i = 0; i < nparts; ++i) { counts[i] = h[i]; tot += h[i]; }
  prof_bytes("hist_seq_owner", (double)sv.avail);
  prof_bytes("partition", (double)sv.avail + 12.0 * tot);
  return KMG_OK;
}

extern "C" int kmg_shard_partition(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1, int k,
                                   const uint64_t *splitters, int nparts, uint64_t *d_keys, uint32_t *d_pos, uint64_t *counts) {
  if (nparts < 1 || nparts > RADIX || !counts) return fail(KMG_ERR_ARG, "nparts must be in [1,%d]", RADIX);
  if (nparts > 1 && !splitters) return fail(KMG_ERR_ARG, "splitters is NULL");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint8_t> buf(s);
  SeqView sv;
  TRY(shard_view(d_seq, g0, g1, L, s0, s1, k, s, buf, &sv));
  for (int i = 0; i < nparts; ++i) counts[i] = 0;
  if (sv.nstarts == 0) return KMG_OK;
  if (!d_keys || !d_pos) return fail(KMG_ERR_ARG, "record arrays are NULL");
  if (s0 + sv.nstarts > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "positions exceed int");
  const int rc = partition_records(sv, splitters, nparts, d_keys, d_pos, counts, s);
  if (rc != KMG_OK) cudaStreamSynchronize(s);             // nothing may still write the caller's arrays
  return rc;
}

extern "C" int kmg_build_records(uint64_t *d_keys, uint32_t *d_pos, int64_t n, int k, kmg_index **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (n < 0 || (n > 0 && (!d_keys || !d_pos))) return fail(KMG_ERR_ARG, "bad record arrays");
  if (n > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "too many records");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  IndexPtr ix(new (std::nothrow) kmg_index());
  if (!ix) return fail(KMG_ERR_NOMEM, "host allocation failed");
  ix->device = g_ctx.device;
  ix->k = k;
  if (n == 0) {
    TRY(dalloc(&ix->ustart, 1, s));
    cudaMemsetAsync(ix->ustart, 0, 4, s);
    cudaStreamSynchronize(s);
    *out = ix.release();
    return KMG_OK;
  }
  SortScratch sc(s);
  DevBuf<uint64_t> kbuf(s);
  DevBuf<uint32_t> pbuf(s), pfinal(s);
  TRY(scratch_alloc(sc, n, s));
  TRY(kbuf.alloc((size_t)n));
  TRY(pbuf.alloc((size_t)n));
  uint64_t *ka = d_keys, *kb = kbuf;                       // the passes ping-pong between the caller's arrays and ours
  uint32_t *pa = d_pos, *pb = pbuf;
  const unsigned hgrid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n, 256 * 16), (int64_t)g_ctx.sms * 8);
  LAUNCH("hist_rec", s, hist_rec_kernel<256, DigitBin><<<hgrid, 256, 0, s>>>(d_keys, n, nullptr, sc.hist(0), DigitBin{0}));
  TRY(launch_scan_hist(RADIX_BITS, s, sc.hist(0), sc.gbase(0), &sc.stats()->n));
  TRY(pfinal.alloc((size_t)n));                            // the index must own its positions
  TRY(sort_tail(sc, SortPlan{RADIX_BITS, num_passes(k)}, 0, true, ka, pa, kb, pb, n, s, pfinal));      // keys end in ka (may be the caller's array)
  TRY(finish_index(ix.get(), sc, ka, pfinal, n, s));
  pfinal.release();
  if (ix->unstable) { demote_rank_variant(); return fail(KMG_ERR_UNSTABLE, "position lists not ascending after the one-atomic sort pass; rebuild (the bitmap variant is now selected)"); }
  const int R = num_passes(k);
  prof_bytes("hist_rec", 8.0 * n);
  if (R > 1) prof_bytes("sort_pass_hist", 24.0 * n * (R - 1));
  prof_bytes("sort_pass", 24.0 * n);
  *out = ix.release();
  return KMG_OK;
}


// ------------------------------------------------------------------------------------------------
// sharded build over peer memory: no host synchronisation between the halo and the finished index
// ------------------------------------------------------------------------------------------------
struct kmg_shard {
  int device = 0;
  bool hashed = false;     // grouped sharded build: records and owner ranges are those of mix64(key)
  uint8_t *buf = nullptr;  // the shard's bytes (seq_alloc): sv.base = buf + 16
  SeqView sv;
};
static kmg_shard *new_shard(DevBuf<uint8_t> &buf, const SeqView &sv, bool hashed) {
  kmg_shard *sh = new (std::nothrow) kmg_shard();
  if (!sh) return nullptr;
  sh->device = g_ctx.device; sh->hashed = hashed; sh->sv = sv; sh->buf = buf.release();
  return sh;
}

extern "C" int kmg_shard_open(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1, int k, kmg_shard **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  TRY(ctx_init());
  DevBuf<uint8_t> buf(g_ctx.stream());
  SeqView sv;
  TRY(shard_view(d_seq, g0, g1, L, s0, s1, k, g_ctx.stream(), buf, &sv));
  if (s0 + sv.nstarts > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "positions exceed int");
  if (!(*out = new_shard(buf, sv, false))) return fail(KMG_ERR_NOMEM, "host allocation failed");
  return KMG_OK;
}
extern "C" int kmg_shard_close(kmg_shard *sh) {
  if (!sh) return KMG_OK;
  // no synchronisation: the sharded calls never wait for the device
  const bool mine = g_ctx.ready && g_ctx.device == sh->device;
  if (!mine) cudaSetDevice(sh->device);
  g_arena[sh->device & 63].put(sh->buf, mine ? g_ctx.stream() : nullptr, false);
  delete sh;
  return KMG_OK;
}
extern "C" int kmg_shard_set_mixed(kmg_shard *sh, int mixed) {
  if (!sh) return fail(KMG_ERR_ARG, "shard is NULL");
  sh->hashed = mixed != 0;     // count / scatter then work on mix64(key): the owner ranges of a grouped sharded index
  return KMG_OK;
}
extern "C" int kmg_shard_windows(const kmg_shard *sh, int64_t *nstarts) {
  if (!sh || !nstarts) return fail(KMG_ERR_ARG, "NULL argument");
  *nstarts = sh->sv.nstarts;
  return KMG_OK;
}

extern "C" int kmg_shard_sample_keys(const kmg_shard *sh, int n, uint64_t *d_samples) {
  if (!sh || n <= 0 || !d_samples) return fail(KMG_ERR_ARG, "bad sample request");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  LAUNCH("sample", s, sample_kernel<<<ceil_div(n, 256), 256, 0, s>>>(sh->sv, n, d_samples));
  return KMG_OK;
}

__global__ void widen_counts_kernel(const uint32_t *hist, int n, uint64_t *out) {
  if ((int)threadIdx.x < n) out[threadIdx.x] = hist[threadIdx.x];
}

extern "C" int kmg_shard_count(const kmg_shard *sh, const uint64_t *d_splitters, int nparts, uint64_t *d_counts) {
  if (!sh || !d_counts) return fail(KMG_ERR_ARG, "NULL argument");
  if (nparts < 1 || nparts > MAX_PEERS) return fail(KMG_ERR_ARG, "nparts must be in [1,%d]", MAX_PEERS);
  if (nparts > 1 && !d_splitters) return fail(KMG_ERR_ARG, "splitters is NULL");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint32_t> hist(s);
  TRY(hist.alloc((size_t)RADIX));
  CU(cudaMemsetAsync(hist, 0, RADIX * 4, s));
  if (sh->sv.nstarts > 0) {
    OwnerBin ob{d_splitters, nparts};
    const int64_t tiles = ceil_div<int64_t>(sh->sv.nstarts, HIST_TILE);
    const unsigned hgrid = (unsigned)std::min<int64_t>(tiles, (int64_t)g_ctx.sms * 2);
    if (sh->hashed)
      LAUNCH("hist_seq_owner", s, hist_seq_kernel<HIST_THREADS, HIST_ITEMS, HashOwnerBin><<<hgrid, HIST_THREADS, 0, s>>>(sh->sv, hist, HashOwnerBin{ob}));
    else
      LAUNCH("hist_seq_owner", s, hist_seq_kernel<HIST_THREADS, HIST_ITEMS, OwnerBin><<<hgrid, HIST_THREADS, 0, s>>>(sh->sv, hist, ob));
    prof_bytes("hist_seq_owner", (double)sh->sv.avail);
  }
  LAUNCH("widen_counts", s, widen_counts_kernel<<<1, MAX_PEERS, 0, s>>>(hist, nparts, d_counts));
  return KMG_OK;
}

extern "C" int kmg_shard_scatter(const kmg_shard *sh, const uint64_t *d_splitters, int nparts, int rank,
                                 void *const *peer_keys, void *const *peer_pos, uint64_t capacity,
                                 const uint64_t *d_matrix, int32_t pos_add, uint64_t *d_info) {
  if (!sh || !peer_keys || !peer_pos || !d_matrix || !d_info) return fail(KMG_ERR_ARG, "NULL argument");
  if (nparts < 1 || nparts > MAX_PEERS || rank < 0 || rank >= nparts) return fail(KMG_ERR_ARG, "bad nparts/rank");
  if (nparts > 1 && !d_splitters) return fail(KMG_ERR_ARG, "splitters is NULL");
  if (capacity > (uint64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "capacity exceeds int coordinates");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  SortScratch sc(s);
  DevBuf<PeerTable> tab(s);
  TRY(scratch_alloc(sc, sh->sv.nstarts, s));
  TRY(tab.alloc(1));
  PeerPtrs pp{};
  for (int i = 0; i < nparts; ++i) { pp.keys[i] = (uint64_t *)peer_keys[i]; pp.pos[i] = (uint32_t *)peer_pos[i]; }
  LAUNCH("owner_offsets", s, owner_offsets_kernel<<<1, RADIX, 0, s>>>(d_matrix, nparts, rank, capacity, pp, sc.gbase(0), tab, d_info));
  if (sh->sv.nstarts == 0) return KMG_OK;
  OwnerBin ob{d_splitters, nparts};
  PassParams<OwnerBin, NoBin> P{};
  P.sv = sh->sv;
  P.gbase = sc.gbase(0); P.hist_next = nullptr;
  P.status = sc.status; P.ticket = sc.ticket(0); P.epoch = 1;
  P.pos_add = (uint32_t)pos_add;
  P.hashed = sh->hashed ? 1u : 0u;                    // the owner is then looked up for mix64(key), which is what is written
  P.peer = tab;
  P.bin = ob;
  // few bins, many lanes per bin: the bitmap variant measured best here (0.51 ms at N=2; ballots 0.54 ms)
  TRY((launch_pass_cfg<PassCfg<256, 24, 2, 0, 8, 8>, true, OwnerBin, NoBin, false, true>("scatter_peer", P, sh->sv.nstarts, s)));
  prof_bytes("scatter_peer", (double)sh->sv.avail + 12.0 * (double)sh->sv.nstarts);
  return KMG_OK;
}

__global__ void set_n_kernel(const uint64_t *info, uint64_t cap, uint64_t *n) { *n = info[0] < cap ? info[0] : cap; }

// Index from the records peers scattered into (d_keys, d_pos): their number is on the device (d_info[0]).
// Everything is sized by `capacity`; the one host synchronisation is the read of the finished index's stats.
// Owner-side build from records that peers scattered into (d_keys, d_pos).  Two layouts:
//   dense   (d_counts == nullptr): records 0 .. d_info[0]-1, d_info[1] != 0 if an owner overflowed (kmg_shard_scatter);
//   regions (d_counts != nullptr): source r's records start at r * region_cap, d_counts[r] of them (kmg_shard_scatter_ranges).
// Everything is sized by `capacity`; the one host synchronisation is the read of the finished index's stats.
static int owner_build(uint64_t *d_keys, uint32_t *d_pos, uint64_t capacity, const uint64_t *d_info, int nsegs, uint64_t region_cap,
                       const uint64_t *d_counts, int k, int order, kmg_index **out) {
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  IndexPtr ix(new (std::nothrow) kmg_index());
  if (!ix) return fail(KMG_ERR_NOMEM, "host allocation failed");
  ix->device = g_ctx.device;
  ix->k = k;
  const int64_t n = (int64_t)capacity;
  SortScratch sc(s);
  DevBuf<uint64_t> kbuf(s);
  DevBuf<uint32_t> pbuf(s), pfinal(s);
  DevBuf<TileSegs> seg(s);
  uint64_t h_info[2] = {0, 0};
  uint32_t h_seg_overflow = 0;
  const bool grouped = grouped_for(k, order, n);
  // the arrays are sized with slack (1.25-1.3x what an owner expects); the digit plan follows the expected record count
  const SortPlan gp = grouped_plan(d_counts ? n * 10 / 13 : n * 4 / 5);
  TRY(scratch_alloc(sc, n, s, grouped ? gp.rb : RADIX_BITS));
  TRY(kbuf.alloc((size_t)n));
  TRY(pbuf.alloc((size_t)n));
  uint64_t *ka = d_keys, *kb = kbuf;                       // the passes ping-pong between the caller's arrays and ours
  uint32_t *pa = d_pos, *pb = pbuf;
  const unsigned hgrid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n, 256 * 16), (int64_t)g_ctx.sms * 8);
  const int rb0 = grouped ? gp.rb : RADIX_BITS;
  if (d_counts) {
    TRY(seg.alloc(1));
    LAUNCH("tile_segs", s, tile_segs_kernel<<<1, MAX_SEGS, 0, s>>>(d_counts, nsegs, region_cap, record_tile(rb0), seg, &sc.stats()->n));
    LAUNCH("hist_rec", s, hist_seg_kernel<256, DigitBin><<<hgrid, 256, 0, s>>>(d_keys, seg, sc.hist(0), DigitBin{0, (1u << rb0) - 1}));
    CU(cudaMemcpyAsync(&h_seg_overflow, &seg.get()->overflow, 4, cudaMemcpyDeviceToHost, s));
  } else {
    LAUNCH("set_n", s, set_n_kernel<<<1, 1, 0, s>>>(d_info, capacity, &sc.stats()->n));
    LAUNCH("hist_rec", s, hist_rec_kernel<256, DigitBin><<<hgrid, 256, 0, s>>>(d_keys, n, &sc.stats()->n, sc.hist(0), DigitBin{0, (1u << rb0) - 1}));
    CU(cudaMemcpyAsync(h_info, d_info, sizeof h_info, cudaMemcpyDeviceToHost, s));
  }
  TRY(launch_scan_hist(rb0, s, sc.hist(0), sc.gbase(0), (uint64_t *)nullptr));
  TRY(pfinal.alloc((size_t)n));
  if (grouped) {
    // records carry mix64(key): sort on its low bits, then partition the groups in which k-mers share them.
    // The passes ping-pong (caller's arrays <-> ours); the fix-up needs the result and a scratch pair, so the
    // last pass may not divert into pfinal: copy the positions at the end instead.
    TRY(sort_tail(sc, gp, 0, true, ka, pa, kb, pb, n, s, nullptr, seg, nsegs));
    uint32_t h_cnt[4] = {0, 0, 0, 0};
    DevBuf<uint32_t> fixmem(s);
    TRY(fix_groups(sc, gp.bits(), ka, pa, kb, pb, n, s, h_cnt, fixmem));
    if (pa != d_pos) pfinal.reset(pbuf.release());          // the sorted positions are in our array: the index keeps it
    else if (cudaMemcpyAsync(pfinal, pa, (size_t)n * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return fail(KMG_ERR_CUDA, "copy failed");
    TRY(finish_index(ix.get(), sc, ka, pfinal, n, s, true));   // synchronises
    pfinal.release();                                        // the index owns it now (it is freed with the index)
    if (h_cnt[2]) return fail(KMG_ERR_RANGE, "more colliding groups than the task lists hold");
    ix->grouped = true;
    ix->hbits = gp.bits();
  } else {
    TRY(sort_tail(sc, SortPlan{RADIX_BITS, num_passes(k)}, 0, true, ka, pa, kb, pb, n, s, pfinal, seg, nsegs));
    TRY(finish_index(ix.get(), sc, ka, pfinal, n, s));            // synchronises
    pfinal.release();
  }
  if (ix->unstable) { demote_rank_variant(); return fail(KMG_ERR_UNSTABLE, "position lists not ascending after the one-atomic sort pass; rebuild (the bitmap variant is now selected)"); }
  const int R = grouped ? gp.passes : num_passes(k);
  prof_bytes("hist_rec", 8.0 * (double)ix->N);
  if (R > 1) prof_bytes("sort_pass_hist", 24.0 * (double)ix->N * (R - 1));
  prof_bytes("sort_pass", 24.0 * (double)ix->N);
  if (grouped) prof_bytes("group_detect", 8.0 * (double)ix->N);
  if (h_info[1] || h_seg_overflow)
    return fail(KMG_ERR_RANGE, "an owner received more than the exchange capacity of %llu records", (unsigned long long)(d_counts ? region_cap : capacity));
  *out = ix.release();
  return KMG_OK;
}

// Index from the records peers scattered into (d_keys, d_pos): their number is on the device (d_info[0]).
extern "C" int kmg_build_received(uint64_t *d_keys, uint32_t *d_pos, uint64_t capacity, const uint64_t *d_info, int k, int order,
                                  kmg_index **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (capacity == 0 || capacity > (uint64_t)INT32_MAX || !d_keys || !d_pos || !d_info) return fail(KMG_ERR_ARG, "bad record arrays");
  return owner_build(d_keys, d_pos, capacity, d_info, 0, 0, nullptr, k, order, out);
}
// The same for a region-mode scatter (kmg_shard_scatter_ranges): nparts regions of region_cap slots, d_counts[r] records in region r.
extern "C" int kmg_build_regions(uint64_t *d_keys, uint32_t *d_pos, uint64_t region_cap, int nparts, const uint64_t *d_counts, int k,
                                 kmg_index **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (nparts < 1 || nparts > MAX_PEERS || region_cap == 0 || region_cap * (uint64_t)nparts > (uint64_t)INT32_MAX || !d_keys || !d_pos || !d_counts)
    return fail(KMG_ERR_ARG, "bad record arrays");
  if (!grouped_for(k, KMG_ORDER_GROUPED, (int64_t)(region_cap * nparts))) return fail(KMG_ERR_ARG, "region exchange carries mixed keys: k must be large enough for the grouped build");
  return owner_build(d_keys, d_pos, region_cap * (uint64_t)nparts, nullptr, nparts, region_cap, d_counts, k, KMG_ORDER_GROUPED, out);
}

// ---- region-mode scatter: nothing is counted or exchanged beforehand ----------------------------------------------------
__global__ void region_table_kernel(PeerPtrs pp, PeerPtrs counts /* keys[] reused as count arrays */, int nparts, int rank, uint64_t region_cap,
                                    PeerTable *tab, uint32_t *gbase, bool announce_zero) {
  const int b = threadIdx.x;
  for (int o = b; o < MAX_NB; o += blockDim.x) gbase[o] = 0;
  if (b < MAX_PEERS) {
    tab->keys[b] = b < nparts ? pp.keys[b] : nullptr;
    tab->pos[b] = b < nparts ? pp.pos[b] : nullptr;
    tab->delta[b] = (int64_t)rank * (int64_t)region_cap;
    tab->counts[b] = b < nparts ? counts.keys[b] : nullptr;
    if (announce_zero && b < nparts) counts.keys[b][rank] = 0;    // a shard without windows still tells every owner so
  }
  if (b == 0) { tab->cap = region_cap; tab->rank = (uint32_t)rank; tab->region = 1; }
}

// Encode the shard, group its records by owner = one of nparts equal ranges of the mixed key, and write each group straight
// into this rank's region of the owner's arrays (own or NVLink-mapped); the last tile stores the per-owner totals in the
// owners' count arrays.  pos_add as in kmg_shard_scatter.
extern "C" int kmg_shard_scatter_ranges(const kmg_shard *sh, int nparts, int rank, void *const *peer_keys, void *const *peer_pos,
                                        void *const *peer_counts, uint64_t region_cap, int32_t pos_add) {
  if (!sh || !peer_keys || !peer_pos || !peer_counts) return fail(KMG_ERR_ARG, "NULL argument");
  if (nparts < 1 || nparts > MAX_PEERS || rank < 0 || rank >= nparts) return fail(KMG_ERR_ARG, "bad nparts/rank");
  if (region_cap == 0 || region_cap * (uint64_t)nparts > (uint64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "capacity exceeds int coordinates");
  if (!sh->hashed) return fail(KMG_ERR_ARG, "region exchange needs a shard of mixed keys (grouped order, k large enough)");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  SortScratch sc(s);
  DevBuf<PeerTable> tab(s);
  TRY(scratch_alloc(sc, sh->sv.nstarts, s, 4));
  TRY(tab.alloc(1));
  PeerPtrs pp{}, pc{};
  for (int i = 0; i < nparts; ++i) { pp.keys[i] = (uint64_t *)peer_keys[i]; pp.pos[i] = (uint32_t *)peer_pos[i]; pc.keys[i] = (uint64_t *)peer_counts[i]; }
  LAUNCH("region_table", s, region_table_kernel<<<1, 256, 0, s>>>(pp, pc, nparts, rank, region_cap, tab, sc.gbase(0), sh->sv.nstarts == 0));
  if (sh->sv.nstarts == 0) return KMG_OK;
  PassParams<RangeBin, NoBin> P{};
  P.sv = sh->sv;
  P.gbase = sc.gbase(0); P.hist_next = nullptr;
  P.status = sc.status; P.ticket = sc.ticket(0); P.epoch = 1;
  P.pos_add = (uint32_t)pos_add;
  P.hashed = 1;
  P.peer = tab;
  P.dbg = g_sort_dbg;
  P.bin = RangeBin{(uint32_t)nparts};
  // kmg_tune "scatter_shape" (tuning runs): more resident tiles per SM = more remote stores in flight on the NVLink
  if (rank_variant() >= 3 && !g_scatter_bitmap) {
    if (g_scatter_shape == 1) TRY((launch_pass_cfg<PassCfg<256, 24, 3, 3, 4, 4>, true, RangeBin, NoBin, false, true>("scatter_peer", P, sh->sv.nstarts, s)));
    else if (g_scatter_shape == 2) TRY((launch_pass_cfg<PassCfg<256, 16, 4, 3, 4, 4>, true, RangeBin, NoBin, false, true>("scatter_peer", P, sh->sv.nstarts, s)));
    else TRY((launch_pass_cfg<PassCfg<256, 24, 2, 3, 4, 4>, true, RangeBin, NoBin, false, true>("scatter_peer", P, sh->sv.nstarts, s)));
  } else
    TRY((launch_pass_cfg<PassCfg<256, 24, 2, 0, 8, 4>, true, RangeBin, NoBin, false, true>("scatter_peer", P, sh->sv.nstarts, s)));
  prof_bytes("scatter_peer", (double)sh->sv.avail + 12.0 * (double)sh->sv.nstarts);
  return KMG_OK;
}

// match the (mixed key, i) records of a region-mode scatter: compacted into dense arrays, then as kmg_query_received
extern "C" int kmg_query_regions(const kmg_index *ix, const uint64_t *d_keys, const int32_t *d_i, uint64_t region_cap, int nparts,
                                 const uint64_t *d_counts, kmg_query **st, uint64_t *M) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (nparts < 1 || nparts > MAX_PEERS || region_cap == 0 || region_cap * (uint64_t)nparts > (uint64_t)INT32_MAX || !d_keys || !d_i || !d_counts)
    return fail(KMG_ERR_ARG, "bad record arrays");
  TRY(use_index(ix));
  cudaStream_t s = g_ctx.stream();
  const uint64_t capacity = region_cap * (uint64_t)nparts;
  DevBuf<TileSegs> seg(s);
  DevBuf<uint64_t> dn(s), dk(s);
  DevBuf<uint32_t> di(s);
  uint32_t h_seg_overflow = 0;
  TRY(seg.alloc(1));
  TRY(dn.alloc(1));
  TRY(dk.alloc((size_t)capacity));
  TRY(di.alloc((size_t)capacity));
  LAUNCH("tile_segs", s, tile_segs_kernel<<<1, MAX_SEGS, 0, s>>>(d_counts, nparts, region_cap, (uint32_t)PROBE_TILE, seg, dn));
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(region_cap, 256), (uint64_t)g_ctx.sms * 8);
  LAUNCH("seg_compact", s, seg_compact_kernel<<<grid, 256, 0, s>>>(d_keys, (const uint32_t *)d_i, seg, dk, di));
  CU(cudaMemcpyAsync(&h_seg_overflow, &seg.get()->overflow, 4, cudaMemcpyDeviceToHost, s));
  SeqView sv{};
  TRY(query_common(ix, false, sv, dk, (const int32_t *)di.get(), (int64_t)capacity, st, M, dn, true));   // synchronises
  if (h_seg_overflow) {
    kmg_query_free(*st);
    *st = nullptr;
    return fail(KMG_ERR_RANGE, "an owner received more than the exchange capacity of %llu records", (unsigned long long)region_cap);
  }
  return KMG_OK;
}

// ---- exchange buffers that other processes on the node can map (CUDA IPC over NVLink) ---------------------
extern "C" int kmg_ipc_alloc(size_t bytes, void **dptr, void *handle) {
  if (!dptr || !handle) return fail(KMG_ERR_ARG, "NULL argument");
  TRY(ctx_init());
  void *p = nullptr;
  CU(cudaMalloc(&p, bytes ? bytes : 1));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return fail(KMG_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle is 64 bytes");
  memcpy(handle, &h, 64);
  *dptr = p;
  return KMG_OK;
}
extern "C" int kmg_ipc_free(void *dptr) {
  if (dptr) { cudaDeviceSynchronize(); cudaFree(dptr); }
  return KMG_OK;
}
extern "C" int kmg_ipc_open(const void *handle, void **dptr) {
  if (!dptr || !handle) return fail(KMG_ERR_ARG, "NULL argument");
  TRY(ctx_init());
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CU(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
  return KMG_OK;
}
extern "C" int kmg_ipc_close(void *dptr) {
  if (dptr) cudaIpcCloseMemHandle(dptr);
  return KMG_OK;
}

// match the (key, i) records peers scattered into (d_keys, d_i); their number is d_info[0] on the device
extern "C" int kmg_query_received(const kmg_index *ix, const uint64_t *d_keys, const int32_t *d_i, uint64_t capacity,
                                  const uint64_t *d_info, int mixed, kmg_query **st, uint64_t *M) {
  if (!st) return fail(KMG_ERR_ARG, "st is NULL");
  *st = nullptr;
  if (capacity == 0 || capacity > (uint64_t)INT32_MAX || !d_keys || !d_i || !d_info) return fail(KMG_ERR_ARG, "bad record arrays");
  TRY(use_index(ix));
  uint64_t h_info[2] = {0, 0};
  CU(cudaMemcpyAsync(h_info, d_info, sizeof h_info, cudaMemcpyDeviceToHost, g_ctx.stream()));
  SeqView sv{};
  int rc = query_common(ix, false, sv, d_keys, d_i, (int64_t)capacity, st, M, d_info, mixed != 0);
  cudaStreamSynchronize(g_ctx.stream());
  if (rc == KMG_OK && h_info[1]) {
    kmg_query_free(*st);
    *st = nullptr;
    return fail(KMG_ERR_RANGE, "an owner received more than the exchange capacity of %llu records", (unsigned long long)capacity);
  }
  return rc;
}


// ---- halo + splitter sample in one exchange ------------------------------------------------------------
// Pack of one rank (what every other rank may need from it): bytes [0,k-1) = its first k-1 bytes,
// byte 40 = its last byte, then n ascending sample keys at byte 48.  Ranks all-gather the packs;
// kmg_shard_open_packed then assembles the shard with its halo and selects the splitters, all on the device.
constexpr int PACK_HDR = 48;

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
shard_pack_kernel(const uint8_t *__restrict__ own, int64_t n_own, int k, int n, const bool mixed, uint8_t *__restrict__ pack) {
  extern __shared__ uint64_t sk[];                       // n keys (n a power of two)
  const int tid = threadIdx.x;
  if (tid < PACK_HDR) {
    uint8_t v = 0;
    if (tid < k - 1 && tid < n_own) v = own[tid];
    if (tid == 40 && n_own > 0) v = own[n_own - 1];
    pack[tid] = v;
  }
  const int64_t nwin = n_own - k + 1 > 0 ? n_own - k + 1 : 1;
  for (int i = tid; i < n; i += THREADS) {               // evenly spaced windows of the rank's own bytes; breakers are
    const int64_t q = ((int64_t)i * nwin) / n;           // encoded like any byte (a sample only steers load balance)
    uint64_t w = 0;
    for (int j = 0; j < k; ++j) {
      const int64_t o = q + j;
      const uint8_t c = o < n_own ? own[o] : 0;
      w = (w << 2) | ((c >> 1) & 3u);
    }
    sk[i] = mixed ? mix64(w & key_mask(k)) : (w & key_mask(k));   // grouped build: owners hold ranges of the mix
  }
  __syncthreads();
  for (int size = 2; size <= n; size <<= 1)              // bitonic sort, ascending
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < n / 2; i += THREADS) {
        const int lo = 2 * i - (i & (stride - 1));       // element with bit `stride` clear
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const uint64_t a = sk[lo], b = sk[hi];
        if ((a > b) == up) { sk[lo] = b; sk[hi] = a; }
      }
      __syncthreads();
    }
  uint64_t *out = reinterpret_cast<uint64_t *>(pack + PACK_HDR);
  for (int i = tid; i < n; i += THREADS) out[i] = sk[i];
}

extern "C" int kmg_shard_pack_bytes(int n_samples) { return PACK_HDR + 8 * n_samples; }

extern "C" int kmg_shard_pack(const void *d_own, int64_t n_own, int k, int n_samples, int order, void *d_pack) {
  if (!d_pack || (n_own > 0 && !d_own) || n_own < 0) return fail(KMG_ERR_ARG, "bad arguments");
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (n_samples < 2 || n_samples > 4096 || (n_samples & (n_samples - 1))) return fail(KMG_ERR_ARG, "n_samples must be a power of two in [2,4096]");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  LAUNCH("shard_pack", s, shard_pack_kernel<1024><<<1, 1024, (size_t)n_samples * 8, s>>>((const uint8_t *)d_own, n_own, k, n_samples, grouped_for(k, order, 0), (uint8_t *)d_pack));
  return KMG_OK;
}

// left byte and right halo of the padded shard, from the gathered packs
__global__ void halo_fill_kernel(uint8_t *base, int64_t n_own, int need_right, bool left, int rank, int world, int64_t per, int64_t L,
                                 int k, const uint8_t *__restrict__ allpack, int pack_bytes) {
  const int t = threadIdx.x;
  if (t == 0 && left) base[-1] = allpack[(size_t)(rank - 1) * pack_bytes + 40];
  if (t < need_right) {                                  // byte s1 + t lives in the head of the first later rank that has it
    int64_t off = t;
    for (int r = rank + 1; r < world; ++r) {
      const int64_t rs0 = min((int64_t)r * per, L), rs1 = min((int64_t)(r + 1) * per, L);
      const int64_t have = min(rs1 - rs0, (int64_t)(k - 1));
      if (off < have) { base[n_own + t] = allpack[(size_t)r * pack_bytes + off]; break; }
      off -= have;
    }
  }
}

// splitter j = element number (j * total) / world of all samples in ascending order; every rank's list is sorted,
// so an element's global position is a sum of binary searches (ties broken by (rank, index): a total order)
__global__ void select_splitters_kernel(const uint8_t *__restrict__ allpack, int pack_bytes, int n, int world, uint64_t *__restrict__ spl) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * world) return;
  const int r = e / n, i = e - r * n;
  const uint64_t *mine = reinterpret_cast<const uint64_t *>(allpack + (size_t)r * pack_bytes + PACK_HDR);
  const uint64_t x = mine[i];
  int64_t g = i;
  for (int o = 0; o < world; ++o) {
    if (o == r) continue;
    const uint64_t *lst = reinterpret_cast<const uint64_t *>(allpack + (size_t)o * pack_bytes + PACK_HDR);
    int lo = 0, hi = n;                                  // o < r: elements <= x come first; o > r: elements < x
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const uint64_t v = lst[mid];
      if (o < r ? v <= x : v < x) lo = mid + 1; else hi = mid;
    }
    g += lo;
  }
  const int64_t total = (int64_t)n * world;
  for (int j = 1; j < world; ++j)
    if (g == (j * total) / world) spl[j - 1] = x;
}

extern "C" int kmg_shard_open_packed(const void *d_own, int64_t n_own, int64_t L, int world, int rank, int k, int n_samples,
                                     int order, const void *d_allpack, kmg_shard **out, uint64_t *d_splitters) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be in [1,32]");
  if (world < 1 || world > MAX_PEERS || rank < 0 || rank >= world || !d_allpack)      // d_splitters may be NULL: fixed owner ranges
    return fail(KMG_ERR_ARG, "bad world/rank/pack arguments");
  const int64_t per = (L + world - 1) / world;
  const int64_t s0 = std::min<int64_t>((int64_t)rank * per, L), s1 = std::min<int64_t>((int64_t)(rank + 1) * per, L);
  if (n_own != s1 - s0 || (n_own > 0 && !d_own)) return fail(KMG_ERR_ARG, "rank %d must hold bytes [%lld,%lld) of the sequence", rank, (long long)s0, (long long)s1);
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  const int pack_bytes = PACK_HDR + 8 * n_samples;
  const int64_t need_hi = std::min<int64_t>(L, s1 + k - 1);
  const int64_t avail = std::max<int64_t>(0, need_hi - s0);
  DevBuf<uint8_t> buf(s);
  TRY(seq_alloc(buf, avail, s));
  uint8_t *base = buf + 16;
  if (n_own > 0) CU(cudaMemcpyAsync(base, d_own, (size_t)n_own, cudaMemcpyDefault, s));
  const int need_right = (int)(need_hi - s1);
  if (need_right > 0 || s0 > 0)
    LAUNCH("halo_fill", s, halo_fill_kernel<<<1, 32, 0, s>>>(base, n_own, need_right, s0 > 0 && n_own > 0, rank, world, per, L, k,
                                                             (const uint8_t *)d_allpack, pack_bytes));
  int64_t nstarts = std::min<int64_t>(s1, L - k + 1) - s0;
  SeqView sv;
  sv.base = base; sv.nstarts = nstarts > 0 ? nstarts : 0; sv.avail = avail; sv.s0 = s0; sv.L = L; sv.k = k;
  if (s0 + sv.nstarts > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "positions exceed int");
  if (world > 1 && d_splitters)
    LAUNCH("select_splitters", s, select_splitters_kernel<<<ceil_div(n_samples * world, 256), 256, 0, s>>>(
                                      (const uint8_t *)d_allpack, pack_bytes, n_samples, world, d_splitters));
  if (!(*out = new_shard(buf, sv, grouped_for(k, order, 0)))) return fail(KMG_ERR_NOMEM, "host allocation failed");
  return KMG_OK;
}

// ------------------------------------------------------------------------------------------------
// count.kmers: per-source k-mer counts in one table (SURVEY.md 8f rank 3)
// ------------------------------------------------------------------------------------------------
// Replaces seq_to_counts / kmer_count_insert (src/kmer_hash.c:185-252) as called from count_kmers (:548-591): the
// reference keeps, per distinct k-mer, an array of source_n ints in the SAME khash (kmer_pos_t.v reused as counters) and
// bumps column `source` for every window of every sequence handed to count.kmers(seq, c(k, source, source_n), ptr).
// Here a sequence's counts are the list lengths of its (sorted) position index -- the same windows, the same build --
// and the table is a sorted array of distinct keys with a U x source_n count matrix; a new batch is merged in by one
// stable sort of the concatenated key lists (table entries first) and a row-wise copy/add.
struct kmg_counter {
  int device = 0, k = 0, source_n = 0;
  uint64_t U = 0, new_total = 0;     // distinct k-mers; sum over calls of the k-mers that were new (khash_ptr.kmer_count)
  uint64_t *keys = nullptr;          // [U] ascending 2-bit keys
  int32_t *counts = nullptr;         // [U][source_n]
  // made on the first depth call, dropped whenever keys / counts are replaced
  std::mutex mu;
  uint4 *hash = nullptr;             // key table (probe.cuh), slots {key, row u, count (source_n == 1) or 1}
  uint64_t hash_nb = 0;
};

__global__ void count_first_kernel(const uint32_t *__restrict__ ustart, uint64_t U, int source_n, int source, int32_t *__restrict__ counts) {
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (uint64_t)gridDim.x * blockDim.x)
    counts[u * source_n + source] = (int32_t)(ustart[u + 1] - ustart[u]);
}
__global__ void iota_kernel(uint32_t *p, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = (uint32_t)i;
}
// merged index over (table keys ++ batch keys): every distinct key has one or two payloads, the table's first
__global__ void count_merge_kernel(const uint32_t *__restrict__ mstart, const uint32_t *__restrict__ mpay, uint64_t Um, uint64_t Ut,
                                   const int32_t *__restrict__ old_counts, const uint32_t *__restrict__ bstart, int source_n, int source,
                                   int32_t *__restrict__ counts) {
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < Um; u += (uint64_t)gridDim.x * blockDim.x) {
    int32_t add = 0;
    const int32_t *row = nullptr;
    for (uint32_t j = mstart[u]; j < mstart[u + 1]; ++j) {
      const uint32_t p = mpay[j];
      if (p < Ut) row = old_counts + (uint64_t)p * source_n;
      else add += (int32_t)(bstart[p - Ut + 1] - bstart[p - Ut]);
    }
    for (int s = 0; s < source_n; ++s) counts[u * source_n + s] = (row ? row[s] : 0) + (s == source ? add : 0);
  }
}
// rows (i, count of source s) for s = 0..source_n-1: what kmer.pos(ptr, 2) returns for a count table (the reference's
// kmer_positions walks v.a[0..v.n), src/kmer_hash.c:1108-1112, and v holds the counters).  Writes cells
// [first, first + rows) to out[0, rows): a chunk starts at any cell, not only at a multiple of source_n.
__global__ void count_rows_kernel(const int32_t *__restrict__ counts, uint64_t first, uint64_t rows, int source_n, int2 *__restrict__ out) {
  for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < rows; c += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t cell = first + c;
    out[c] = make_int2((int)(cell / source_n + 1), counts[cell]);
  }
}
// spectrum[min(count, max_count)] += 1 over the k-mers (count_spectrum, src/kmer_tree.c:85-99); source < 0: summed over sources
__global__ void spectrum_counts_kernel(const int32_t *__restrict__ counts, uint64_t U, int source_n, int source, uint32_t max_count,
                                       unsigned long long *__restrict__ spec) {
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t c = 0;
    if (source >= 0) c = (uint64_t)counts[u * source_n + source];
    else for (int s = 0; s < source_n; ++s) c += (uint64_t)counts[u * source_n + s];
    atomicAdd(spec + (c >= max_count ? max_count : c), 1ull);
  }
}
__global__ void spectrum_index_kernel(const uint32_t *__restrict__ ustart, uint64_t U, uint32_t max_count, unsigned long long *__restrict__ spec) {
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = ustart[u + 1] - ustart[u];
    atomicAdd(spec + (c >= max_count ? max_count : c), 1ull);
  }
}

extern "C" int kmg_count_new(int k, int source_n, kmg_counter **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > KMG_MAX_K) return fail(KMG_ERR_K, "k must be a positive integer less than 1+MAX_K");
  if (source_n < 1) return fail(KMG_ERR_ARG, "source_n must be larger than 1 and larger than source");
  TRY(ctx_init());
  kmg_counter *c = new (std::nothrow) kmg_counter();
  if (!c) return fail(KMG_ERR_NOMEM, "host allocation failed");
  c->device = g_ctx.device; c->k = k; c->source_n = source_n;
  *out = c;
  return KMG_OK;
}
extern "C" int kmg_count_free(kmg_counter *c) {
  if (!c) return KMG_OK;
  release_on_device(c->device, {c->keys, c->counts, c->hash});
  delete c;
  return KMG_OK;
}
static int use_counter(const kmg_counter *c) { return c ? use_device(c->device, "the count table lives") : fail(KMG_ERR_ARG, "counter is NULL"); }

// seq_to_counts(seq, k, hash, source, source_n) for one sequence (src/kmer_hash.c:220-252)
extern "C" int kmg_count_add(kmg_counter *c, const char *seq, int64_t len, int source) {
  TRY(use_counter(c));
  if (source < 0 || source >= c->source_n) return fail(KMG_ERR_ARG, "source_n must be larger than 1 and larger than source");
  if (len < 0 || (len > 0 && !seq)) return fail(KMG_ERR_ARG, "bad sequence pointer/length");
  kmg_index *bi = nullptr;
  TRY(kmg_build_ordered(seq, len, c->k, KMG_ORDER_SORTED, &bi));
  const IndexPtr b(bi);
  if (b->U == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  {                                                          // the key table describes the arrays about to be replaced
    std::lock_guard<std::mutex> g(c->mu);
    DevBuf<uint4> table(s, c->hash);
    c->hash = nullptr;
    c->hash_nb = 0;
  }
  const int sn = c->source_n;
  const unsigned grid_of_b = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(b->U, 256), (uint64_t)g_ctx.sms * 16);
  if (c->U == 0) {                                           // first batch: the table is the batch
    DevBuf<int32_t> ncounts(s);
    TRY(ncounts.alloc((size_t)b->U * sn));
    CU(cudaMemsetAsync(ncounts, 0, (size_t)b->U * sn * sizeof(int32_t), s));
    LAUNCH("count_first", s, count_first_kernel<<<grid_of_b, 256, 0, s>>>(b->ustart, b->U, sn, source, ncounts));
    CU(cudaStreamSynchronize(s));
    c->keys = b->ukeys; b->ukeys = nullptr;                // the batch's key array becomes the table's
    c->counts = ncounts.release();
    c->U = b->U; c->new_total += b->U;
    return KMG_OK;
  }
  const uint64_t Ut = c->U, n = Ut + b->U;
  if (n > (uint64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "count table would exceed 2^31-1 k-mers");
  DevBuf<uint64_t> cat_keys(s);
  DevBuf<uint32_t> cat_pay(s);
  TRY(cat_keys.alloc((size_t)n));
  TRY(cat_pay.alloc((size_t)n));
  CU(cudaMemcpyAsync(cat_keys, c->keys, Ut * 8, cudaMemcpyDeviceToDevice, s));
  CU(cudaMemcpyAsync(cat_keys + Ut, b->ukeys, b->U * 8, cudaMemcpyDeviceToDevice, s));
  LAUNCH("iota", s, iota_kernel<<<(unsigned)std::min<uint64_t>(ceil_div<uint64_t>(n, 256), (uint64_t)g_ctx.sms * 16), 256, 0, s>>>(cat_pay, n));
  kmg_index *mi = nullptr;
  TRY(kmg_build_records(cat_keys, cat_pay, (int64_t)n, c->k, &mi));      // stable: a key's table entry precedes its batch entry
  const IndexPtr m(mi);
  DevBuf<int32_t> ncounts(s);
  TRY(ncounts.alloc((size_t)m->U * sn));
  LAUNCH("count_merge", s, count_merge_kernel<<<(unsigned)std::min<uint64_t>(ceil_div<uint64_t>(m->U, 256), (uint64_t)g_ctx.sms * 16), 256, 0, s>>>(
                               m->ustart, m->pos, m->U, Ut, c->counts, b->ustart, sn, source, ncounts));
  CU(cudaStreamSynchronize(s));
  DevBuf<uint64_t> old_keys(s, c->keys);                     // the table's arrays before this batch: freed on return
  DevBuf<int32_t> old_counts(s, c->counts);
  c->keys = m->ukeys; m->ukeys = nullptr;
  c->counts = ncounts.release();
  c->new_total += m->U - Ut;
  c->U = m->U;
  return KMG_OK;
}

extern "C" int kmg_count_sizes(const kmg_counter *c, uint64_t *U, int *source_n, int *k, uint64_t *new_total) {
  if (!c) return fail(KMG_ERR_ARG, "counter is NULL");
  if (U) *U = c->U;
  if (source_n) *source_n = c->source_n;
  if (k) *k = c->k;
  if (new_total) *new_total = c->new_total;
  return KMG_OK;
}
extern "C" int kmg_count_kmers_u64(const kmg_counter *c, uint64_t *keys) {
  TRY(use_counter(c));
  if (c->U == 0) return KMG_OK;
  if (!keys) return fail(KMG_ERR_ARG, "keys is NULL");
  CU(cudaMemcpyAsync(keys, c->keys, c->U * 8, cudaMemcpyDefault, g_ctx.stream()));
  CU(cudaStreamSynchronize(g_ctx.stream()));
  return KMG_OK;
}
extern "C" int kmg_count_kmers_ascii(const kmg_counter *c, char *out) {
  TRY(use_counter(c));
  if (!out && c->U) return fail(KMG_ERR_ARG, "buf is NULL");
  const size_t stride = (size_t)c->k + 1;
  const int k = c->k;
  const uint64_t *keys = c->keys;
  const int sms = g_ctx.sms;
  return stream_rows(c->U, stride, out, CHUNK_BYTES / stride, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(rows * stride, 256), (uint64_t)sms * 16);
    LAUNCH("kmers_ascii", s, kmers_ascii_kernel<<<grid, 256, 0, s>>>(keys + first, rows, k, (char *)dst));
    return KMG_OK;
  });
}
// the U x source_n matrix, one row per k-mer (ascending key)
extern "C" int kmg_count_matrix(const kmg_counter *c, int32_t *out) {
  TRY(use_counter(c));
  if (c->U == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  CU(cudaMemcpyAsync(out, c->counts, c->U * c->source_n * sizeof(int32_t), cudaMemcpyDefault, g_ctx.stream()));
  CU(cudaStreamSynchronize(g_ctx.stream()));
  return KMG_OK;
}
// kmer.pos(count.ptr, 2): 2 x (U * source_n) interleaved rows (i, count)
extern "C" int kmg_count_positions(const kmg_counter *c, int32_t *out) {
  TRY(use_counter(c));
  const uint64_t cells = c->U * (uint64_t)c->source_n;
  if (cells == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  const int32_t *counts = c->counts;
  const int sn = c->source_n, sms = g_ctx.sms;
  return stream_rows(cells, 8, out, CHUNK_BYTES / 8, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *, cudaStream_t s) -> int {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(rows, 256), (uint64_t)sms * 16);
    LAUNCH("count_rows", s, count_rows_kernel<<<grid, 256, 0, s>>>(counts, first, rows, sn, (int2 *)dst));
    return KMG_OK;
  });
}

static int spectrum_out(unsigned long long *d_spec, uint32_t max_count, double *spec, cudaStream_t s) {
  std::vector<unsigned long long> h((size_t)max_count + 1);
  CU(cudaMemcpyAsync(h.data(), d_spec, h.size() * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (size_t i = 0; i < h.size(); ++i) spec[i] = (double)h[i];
  return KMG_OK;
}
// kmer spectrum of one source column (source < 0: of the summed counts): spec[min(count, max_count)] += 1 per k-mer,
// doubles as the reference's spectra are (count_spectrum, src/kmer_tree.c:85-99; kmer_spectrum_*, src/kmer_hash.c:975-1038)
extern "C" int kmg_count_spectrum(const kmg_counter *c, int source, uint32_t max_count, double *spec) {
  TRY(use_counter(c));
  if (!spec) return fail(KMG_ERR_ARG, "spec is NULL");
  if (max_count < 1 || max_count > (1u << 30)) return fail(KMG_ERR_ARG, "Unsuitable value of max_count");
  if (source >= c->source_n) return fail(KMG_ERR_ARG, "source out of range");
  cudaStream_t s = g_ctx.stream();
  DevBuf<unsigned long long> d(s);
  TRY(d.alloc((size_t)max_count + 1));
  if (cudaMemsetAsync(d, 0, ((size_t)max_count + 1) * 8, s) != cudaSuccess) return fail(KMG_ERR_CUDA, "memset failed");
  if (c->U) {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(c->U, 256), (uint64_t)g_ctx.sms * 16);
    spectrum_counts_kernel<<<grid, 256, 0, s>>>(c->counts, c->U, c->source_n, source, max_count, d);
  }
  return spectrum_out(d, max_count, spec, s);
}
// the same for a position index: the count of a k-mer is the length of its position list
extern "C" int kmg_index_spectrum(const kmg_index *ix, uint32_t max_count, double *spec) {
  TRY(use_index(ix));
  if (!spec) return fail(KMG_ERR_ARG, "spec is NULL");
  if (max_count < 1 || max_count > (1u << 30)) return fail(KMG_ERR_ARG, "Unsuitable value of max_count");
  cudaStream_t s = g_ctx.stream();
  DevBuf<unsigned long long> d(s);
  TRY(d.alloc((size_t)max_count + 1));
  if (cudaMemsetAsync(d, 0, ((size_t)max_count + 1) * 8, s) != cudaSuccess) return fail(KMG_ERR_CUDA, "memset failed");
  if (ix->U) {
    const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(ix->U, 256), (uint64_t)g_ctx.sms * 16);
    spectrum_index_kernel<<<grid, 256, 0, s>>>(ix->ustart, ix->U, max_count, d);
  }
  return spectrum_out(d, max_count, spec, s);
}

// ------------------------------------------------------------------------------------------------
// seq.kmer.depth: for every window of a query, the count of its k-mer in a count table or a position index
// ------------------------------------------------------------------------------------------------
// Key table of a count table: the probe's CAS build (hbits = 0, power-of-two buckets, load <= 0.5).  The keys are in
// ascending raw-key order, not in an order the streamed build of a grouped index could use.
static int ensure_count_hash(kmg_counter *c) {
  std::lock_guard<std::mutex> g(c->mu);
  if (c->hash || c->U == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  uint64_t cap = 4 * BUCKET_SLOTS;
  while (cap < 2 * c->U) cap <<= 1;
  DevBuf<uint4> slots(s);
  TRY(slots.alloc(cap));
  CU(cudaMemsetAsync(slots, 0, cap * sizeof(uint4), s));
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(c->U, 256), (uint64_t)g_ctx.sms * 32);
  LAUNCH("count_hash_insert", s, hash_insert_kernel<<<grid, 256, 0, s>>>(c->keys, CountPayload{c->counts, c->source_n}, c->U,
                                                                       KeyHash{slots, cap / BUCKET_SLOTS, 0}, false));
  CU(cudaStreamSynchronize(s));
  c->hash = slots.release(); c->hash_nb = cap / BUCKET_SLOTS;
  prof_bytes("count_hash_insert", 12.0 * c->U + 16.0 * c->U);
  return KMG_OK;
}

constexpr int DEPTH_THREADS = 256, DEPTH_ITEMS = 8, DEPTH_TILE = DEPTH_THREADS * DEPTH_ITEMS;

// Argument checks shared by both entries; *nwin = max(0, qlen - k + 1)
static int depth_args(const char *q, int64_t qlen, int k, int strands, const int32_t *out, int64_t *nwin) {
  if (qlen < 0 || (qlen > 0 && !q)) return fail(KMG_ERR_ARG, "bad query pointer/length");
  if (qlen + 1 > (int64_t)INT32_MAX) return fail(KMG_ERR_RANGE, "query longer than int coordinates");
  if (strands != KMG_STRAND_FORWARD && strands != KMG_STRAND_BOTH) return fail(KMG_ERR_ARG, "strands must be KMG_STRAND_FORWARD or KMG_STRAND_BOTH");
  *nwin = qlen - k + 1 > 0 ? qlen - k + 1 : 0;
  if (*nwin > 0 && !out) return fail(KMG_ERR_ARG, "out is NULL");
  return KMG_OK;
}

// kt.nb == 0: empty table.  cols > 1: `cols` columns gathered from the count matrix, else one column from the slot.
static int depth_run(const char *qseq, int64_t qlen, int64_t nwin, int k, bool both, KeyHash kt, const int32_t *counts, int cols,
                     int32_t *out) {
  cudaStream_t s = g_ctx.stream();
  DevBuf<uint8_t> dseq(s);
  TRY(upload_seq(qseq, qlen, s, dseq));
  SeqView sv;
  sv.base = dseq + 16; sv.nstarts = nwin; sv.avail = qlen; sv.s0 = 0; sv.L = qlen; sv.k = k;
  const size_t row_bytes = 4 * (size_t)cols;
  const bool multi = cols > 1;                           // not counts != nullptr: an empty table has no matrix
  const int rc = stream_rows((uint64_t)nwin, row_bytes, out, CHUNK_BYTES / row_bytes, [=](uint64_t first, uint64_t rows, void *dst, uint64_t *, cudaStream_t st) -> int {
    const unsigned grid = (unsigned)ceil_div<uint64_t>(first % 16 + rows, DEPTH_TILE);
    const int64_t f = (int64_t)first, n = (int64_t)rows;
    int32_t *o = (int32_t *)dst;
#define KMG_DEPTH(B, M) LAUNCH("depth_lookup", st, (depth_lookup_kernel<DEPTH_THREADS, DEPTH_ITEMS, B, M><<<grid, DEPTH_THREADS, 0, st>>>(sv, f, n, kt, counts, cols, o)))
    if (both) { if (multi) KMG_DEPTH(true, true); else KMG_DEPTH(true, false); }
    else { if (multi) KMG_DEPTH(false, true); else KMG_DEPTH(false, false); }
#undef KMG_DEPTH
    return KMG_OK;
  });
  // one 128-byte line of HBM per table request (tools/micro/gups.cu); with several columns one more per request for the
  // row gather; counted for every window, so a query whose windows miss or are invalid is charged the same
  const double lines = (both ? 2.0 : 1.0) * (multi ? 2.0 : 1.0) * (double)nwin;
  prof_bytes("depth_lookup", (double)qlen + 128.0 * lines + (double)row_bytes * (double)nwin);
  return rc;
}

extern "C" int kmg_count_depth(const kmg_counter *cc, const char *q, int64_t qlen, int strands, int32_t *out) {
  TRY(use_counter(cc));
  int64_t nwin = 0;
  TRY(depth_args(q, qlen, cc->k, strands, out, &nwin));
  if (nwin == 0) return KMG_OK;
  kmg_counter *c = const_cast<kmg_counter *>(cc);
  TRY(ensure_count_hash(c));
  const KeyHash kt{c->hash, c->hash_nb, 0};
  return depth_run(q, qlen, nwin, c->k, strands == KMG_STRAND_BOTH, kt, c->counts, c->source_n, out);
}

extern "C" int kmg_index_depth(const kmg_index *cix, const char *q, int64_t qlen, int strands, int32_t *out) {
  TRY(use_index(cix));
  int64_t nwin = 0;
  TRY(depth_args(q, qlen, cix->k, strands, out, &nwin));
  if (nwin == 0) return KMG_OK;
  kmg_index *ix = const_cast<kmg_index *>(cix);
  TRY(ensure_hash(ix));
  const KeyHash kt{ix->hash, ix->hash ? ix->hash_nb : 0, ix->hash_hbits};
  return depth_run(q, qlen, nwin, ix->k, strands == KMG_STRAND_BOTH, kt, nullptr, 1, out);
}

// ------------------------------------------------------------------------------------------------
// FASTA / FASTQ ingestion (SURVEY.md 8f rank 4): inflate on the host, parse on the device (reads.cuh)
// ------------------------------------------------------------------------------------------------
#include <zlib.h>
#include "reads.cuh"

struct kmg_reads {
  int device = 0;
  uint64_t n_records = 0, total_bases = 0;
  uint8_t *seq = nullptr;            // packed sequences: record r at rec_off[r], one 'N' after each
  std::vector<uint64_t> rec_off;     // [n_records + 1] (host copy)
  uint64_t *d_rec_off = nullptr;
  std::vector<std::string> names;
};

extern "C" int kmg_reads_free(kmg_reads *r) {
  if (!r) return KMG_OK;
  release_on_device(r->device, {r->seq, r->d_rec_off});
  delete r;
  return KMG_OK;
}

// text: the (inflated) file contents, host or device memory
extern "C" int kmg_reads_from_memory(const void *text, int64_t len, kmg_reads **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (len < 0 || (len > 0 && !text)) return fail(KMG_ERR_ARG, "bad text pointer/length");
  TRY(ctx_init());
  cudaStream_t s = g_ctx.stream();
  ReadsPtr r(new (std::nothrow) kmg_reads());
  if (!r) return fail(KMG_ERR_NOMEM, "host allocation failed");
  r->device = g_ctx.device;
  r->rec_off.assign(1, 0);
  if (len == 0) { *out = r.release(); return KMG_OK; }
  const uint64_t n = (uint64_t)len, nblocks = (n + 15) / 16;
  const size_t cap = (size_t)nblocks * 16 + 64;
  DevBuf<uint8_t> d_text(s);
  TRY(d_text.alloc(cap));
  CU(cudaMemsetAsync(d_text + (cap - 80), 0, 80, s));
  if (n > (uint64_t)(8 << 20) && staged_transfers() && ptr_kind(text) == PK_HOST_PAGEABLE) TRY(staged_upload(d_text, text, n, s));
  else CU(cudaMemcpyAsync(d_text, text, n, cudaMemcpyDefault, s));
  DevBuf<ReadsInfo> info(s);
  DevBuf<uint32_t> tickets(s);
  TRY(info.alloc(1));
  TRY(tickets.alloc(4));
  CU(cudaMemsetAsync(info, 0, sizeof(ReadsInfo), s));
  CU(cudaMemsetAsync(tickets, 0, 16, s));
  // 1. newlines (a line-start byte decides FASTA / FASTQ: the first byte of the file)
  uint8_t first = 0;
  CU(cudaMemcpyAsync(&first, d_text, 1, cudaMemcpyDeviceToHost, s));
  const uint64_t tiles1 = ceil_div<uint64_t>(nblocks, 256 * 4);
  DevBuf<Pair64> status(s);
  TRY(status.alloc((size_t)std::max<uint64_t>(tiles1, 1)));
  CU(cudaMemsetAsync(status, 0, (size_t)tiles1 * sizeof(Pair64), s));
  unsigned long long *d_cnt = reinterpret_cast<unsigned long long *>(&info.get()->total_bases), h_cnt = 0;    // borrowed until line_scan sets it
  LAUNCH("nl_count", s, nl_count_kernel<<<(unsigned)std::min<uint64_t>(ceil_div<uint64_t>(nblocks, 256), (uint64_t)g_ctx.sms * 16), 256, 0, s>>>(d_text, n, d_cnt));
  CU(cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  DevBuf<uint64_t> nl(s);
  DevBuf<uint32_t> blk_nl(s);
  TRY(nl.alloc((size_t)h_cnt + 2));
  TRY(blk_nl.alloc((size_t)nblocks));
  ReadsInfo h{};
  LAUNCH("nl_scan", s, nl_scan_kernel<256><<<(unsigned)tiles1, 256, 0, s>>>(d_text, n, nl, blk_nl, status, tickets + 0, info));
  CU(cudaMemcpyAsync(&h, info, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (first != '>' && first != '@') return fail(KMG_ERR_ARG, "not a FASTA/FASTQ file: it starts with byte 0x%02x", first);
  const bool fastq = first == '@';
  const uint64_t nlines = h.n_lines;
  DevBuf<uint64_t> seq_len(s), seq_before(s), hdr_before(s);
  DevBuf<uint8_t> kind(s);
  TRY(seq_len.alloc((size_t)nlines + 1));
  TRY(kind.alloc((size_t)nlines + 1));
  TRY(seq_before.alloc((size_t)nlines + 1));
  TRY(hdr_before.alloc((size_t)nlines + 1));
  const unsigned lgrid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(std::max<uint64_t>(nlines, 1), 256), (uint64_t)g_ctx.sms * 16);
  LAUNCH("line_info", s, line_info_kernel<<<lgrid, 256, 0, s>>>(d_text, n, nl, info, fastq, seq_len, kind, info));
  const uint64_t tiles2 = ceil_div<uint64_t>(std::max<uint64_t>(nlines, 1), 256 * 8);
  TRY(status.alloc((size_t)tiles2));                        // the newline scan's status goes back first
  CU(cudaMemsetAsync(status, 0, (size_t)tiles2 * sizeof(Pair64), s));
  LAUNCH("line_scan", s, line_scan_kernel<256, 8><<<(unsigned)tiles2, 256, 0, s>>>(seq_len, kind, info, seq_before, hdr_before, status, tickets + 1));
  CU(cudaMemcpyAsync(&h, info, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (h.bad) return fail(KMG_ERR_ARG, "malformed FASTQ: only the four-line form (@name / sequence / + / qualities of the same length) is read");
  r->n_records = h.n_records; r->total_bases = h.total_bases;
  const uint64_t packed = h.total_bases + h.n_records;
  TRY(dalloc(&r->seq, (size_t)packed + 16, s));
  TRY(dalloc(&r->d_rec_off, (size_t)h.n_records + 1, s));
  DevBuf<uint64_t> name_pos(s);
  DevBuf<uint32_t> name_len(s);
  TRY(name_pos.alloc((size_t)h.n_records + 1));
  TRY(name_len.alloc((size_t)h.n_records + 1));
  LAUNCH("records", s, record_kernel<<<lgrid, 256, 0, s>>>(d_text, n, nl, info, kind, seq_before, hdr_before, r->d_rec_off, name_pos, name_len));
  const unsigned pgrid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(nblocks, 256), (uint64_t)g_ctx.sms * 16);
  LAUNCH("pack_reads", s, pack_kernel<<<pgrid, 256, 0, s>>>(d_text, n, nl, blk_nl, info, kind, seq_before, hdr_before, r->seq, info));
  if (h.n_records)
    LAUNCH("record_finish", s, record_finish_kernel<<<(unsigned)std::min<uint64_t>(ceil_div<uint64_t>(h.n_records, 256), (uint64_t)g_ctx.sms * 16), 256, 0, s>>>(info, r->d_rec_off, r->seq));
  std::unique_ptr<uint64_t[]> h_name_pos(new uint64_t[h.n_records + 1]);
  std::vector<uint32_t> h_name_len;
  r->rec_off.resize((size_t)h.n_records + 1);
  h_name_len.resize((size_t)h.n_records + 1);
  CU(cudaMemcpyAsync(r->rec_off.data(), r->d_rec_off, (h.n_records + 1) * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(h_name_pos.get(), name_pos, (h.n_records + 1) * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(h_name_len.data(), name_len, (h.n_records + 1) * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&h, info, sizeof h, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (h.bad) return fail(KMG_ERR_ARG, "sequence data before the first header line");
  // names: short strings, fetched from the text where it lives
  r->names.resize((size_t)h.n_records);
  const bool text_on_host = ptr_kind(text) != PK_DEVICE;
  std::vector<char> tmp;
  for (uint64_t i = 0; i < h.n_records; ++i) {
    if (text_on_host) r->names[i].assign((const char *)text + h_name_pos[i], h_name_len[i]);
    else {
      tmp.resize(h_name_len[i]);
      if (h_name_len[i]) CU(cudaMemcpy(tmp.data(), d_text + h_name_pos[i], h_name_len[i], cudaMemcpyDeviceToHost));
      r->names[i].assign(tmp.data(), h_name_len[i]);
    }
  }
  prof_bytes("nl_scan", (double)n); prof_bytes("pack_reads", (double)n + (double)packed);
  *out = r.release();
  return KMG_OK;
}

// gz or plain FASTA / FASTQ file (zlib reads both, as the reference's gzopen does: src/kmer_reader.c:43)
extern "C" int kmg_reads_open(const char *path, kmg_reads **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (!path) return fail(KMG_ERR_ARG, "path is NULL");
  gzFile gz = gzopen(path, "rb");
  if (!gz) return fail(KMG_ERR_ARG, "cannot open %s", path);
  gzbuffer(gz, 1 << 20);
  std::vector<char> text;
  size_t used = 0;
  for (;;) {
    if (text.size() - used < (size_t(16) << 20)) text.resize(std::max<size_t>(text.size() * 2, size_t(64) << 20));
    const int got = gzread(gz, text.data() + used, (unsigned)std::min<size_t>(text.size() - used, size_t(1) << 30));
    if (got < 0) { gzclose(gz); return fail(KMG_ERR_ARG, "read error in %s", path); }
    if (got == 0) break;
    used += (size_t)got;
  }
  gzclose(gz);
  return kmg_reads_from_memory(text.data(), (int64_t)used, out);
}

static int use_reads(const kmg_reads *r) { return r ? use_device(r->device, "the reads live") : fail(KMG_ERR_ARG, "reads is NULL"); }
extern "C" int kmg_reads_count(const kmg_reads *r, uint64_t *n_records, uint64_t *total_bases) {
  if (!r) return fail(KMG_ERR_ARG, "reads is NULL");
  if (n_records) *n_records = r->n_records;
  if (total_bases) *total_bases = r->total_bases;
  return KMG_OK;
}
extern "C" int kmg_reads_record(const kmg_reads *r, uint64_t i, int64_t *seq_len, char *name_buf, int name_cap) {
  if (!r) return fail(KMG_ERR_ARG, "reads is NULL");
  if (i >= r->n_records) return fail(KMG_ERR_ARG, "record %llu out of range (have %llu)", (unsigned long long)i, (unsigned long long)r->n_records);
  if (seq_len) *seq_len = (int64_t)(r->rec_off[i + 1] - 1 - r->rec_off[i]);
  if (name_buf && name_cap > 0) { strncpy(name_buf, r->names[i].c_str(), (size_t)name_cap - 1); name_buf[name_cap - 1] = 0; }
  return KMG_OK;
}
extern "C" int kmg_reads_sequence(const kmg_reads *r, uint64_t i, char *out) {
  TRY(use_reads(r));
  if (i >= r->n_records) return fail(KMG_ERR_ARG, "record out of range");
  const uint64_t len = r->rec_off[i + 1] - 1 - r->rec_off[i];
  if (len == 0) return KMG_OK;
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  CU(cudaMemcpyAsync(out, r->seq + r->rec_off[i], len, cudaMemcpyDefault, g_ctx.stream()));
  CU(cudaStreamSynchronize(g_ctx.stream()));
  return KMG_OK;
}
// make.kmer.hash on record i of the file: no R string, no 2^31-1 limit on the file, the sequence never leaves the device
extern "C" int kmg_build_record(const kmg_reads *r, uint64_t i, int k, int order, kmg_index **out) {
  if (!out) return fail(KMG_ERR_ARG, "out is NULL");
  *out = nullptr;
  TRY(use_reads(r));
  if (i >= r->n_records) return fail(KMG_ERR_ARG, "record out of range");
  const uint64_t len = r->rec_off[i + 1] - 1 - r->rec_off[i];
  return kmg_build_ordered((const char *)r->seq + r->rec_off[i], (int64_t)len, k, order, out);
}
// count.kmers over every record of the file (those longer than k), column `source`: ONE build of the packed buffer
extern "C" int kmg_count_add_reads(kmg_counter *c, const kmg_reads *r, int source) {
  TRY(use_counter(c));
  TRY(use_reads(r));
  if (r->n_records == 0) return KMG_OK;
  cudaStream_t s = g_ctx.stream();
  const uint64_t packed = r->total_bases + r->n_records;
  DevBuf<uint8_t> tmp(s);
  DevBuf<ReadsInfo> info(s);
  TRY(tmp.alloc((size_t)packed + 16));
  TRY(info.alloc(1));
  ReadsInfo h{};
  h.n_records = r->n_records; h.total_bases = r->total_bases;
  if (cudaMemcpyAsync(info, &h, sizeof h, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(tmp, r->seq, (size_t)packed, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return fail(KMG_ERR_CUDA, "copy failed");
  const unsigned grid = (unsigned)std::min<uint64_t>(ceil_div<uint64_t>(r->n_records, 256), (uint64_t)g_ctx.sms * 16);
  mask_for_counting_kernel<<<grid, 256, 0, s>>>(info, r->d_rec_off, c->k, tmp);
  if (cudaStreamSynchronize(s) != cudaSuccess) return fail(KMG_ERR_CUDA, "masking failed: %s", cudaGetErrorString(cudaGetLastError()));
  // the last record's separator is the final byte: drop it so that the end-of-string rule sees the record's own end... it is an 'N' either way
  return kmg_count_add(c, (const char *)tmp.get(), (int64_t)packed, source);
}
