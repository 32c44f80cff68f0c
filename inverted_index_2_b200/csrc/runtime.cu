// runtime.cu — context / streams / memory pools / scan utility for libii2.
#include <time.h>

#include <cstdarg>
#include <map>
#include <memory>
#include <mutex>

#include "runtime.cuh"

namespace ii2 {

std::atomic<uint64_t> g_kernel_launches{0};

static thread_local char t_last_error[512] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_last_error, sizeof(t_last_error), fmt, ap);
  va_end(ap);
}

// ------------------------------------------------------------------ context
// The bound device set.  Per-thread state is keyed by CUDA ordinal (so it stays right across
// ii2_shutdown + ii2_init of another set): t_sel is the device ii2_set_device chose (-1: the
// first of the set), t_dev the device of the running call (set at call entry, so finding the
// per-device state costs no CUDA runtime query).
struct Ctx {
  std::mutex m;
  bool ready = false;
  int ndev = 0;
  int devices[kMaxDevices] = {};
  bool peer[kMaxDevices][kMaxDevices] = {};  // [a][b]: kernels on devices[a] read devices[b]
};
static Ctx g_ctx;
static thread_local int t_sel = -1;
static thread_local int t_dev = 0;
constexpr int kMaxOrdinal = 64;  // CUDA ordinals the per-thread tables cover

static int slot_of(int device) {
  for (int i = 0; i < g_ctx.ndev; i++)
    if (g_ctx.devices[i] == device) return i;
  return -1;
}

bool ctx_ready() { return g_ctx.ready; }
int ctx_device_count() { return g_ctx.ready ? g_ctx.ndev : 0; }
int ctx_current_device() { return t_dev; }
bool ctx_bound(int device) { return g_ctx.ready && slot_of(device) >= 0; }
bool ctx_peer(int dev, int peer) {
  const int a = slot_of(dev), b = slot_of(peer);
  return a >= 0 && b >= 0 && (a == b || g_ctx.peer[a][b]);
}

// the device this thread selected, if it is still bound; else the first of the set
static int selected_device() {
  return (t_sel >= 0 && slot_of(t_sel) >= 0) ? t_sel : g_ctx.devices[0];
}

static int ctx_enter(int device) {
  t_dev = device;
  // Each host thread needs the device current.
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    set_last_error("cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    return II2_ERR_CUDA;
  }
  return II2_OK;
}

static int no_device() {
  set_last_error("ii2_init has not succeeded: no CUDA device bound (there is no CPU fallback)");
  return II2_ERR_NO_DEVICE;
}

int ctx_require() {
  if (!g_ctx.ready) return no_device();
  return ctx_enter(selected_device());
}

int ctx_require_device(int device) {
  if (device < 0 || !g_ctx.ready) return ctx_require();
  if (slot_of(device) < 0) {
    set_last_error("device %d is not in the set bound by ii2_init", device);
    return II2_ERR_INVALID;
  }
  return ctx_enter(device);
}

DeviceScope::DeviceScope(int device) {
  if (device < 0 || cudaGetDevice(&prev) != cudaSuccess) {
    prev = -1;
    return;
  }
  if (prev == device || cudaSetDevice(device) != cudaSuccess) prev = -1;
}
DeviceScope::~DeviceScope() {
  if (prev >= 0) cudaSetDevice(prev);
}

struct ThreadStream {
  cudaStream_t own = nullptr;
  cudaStream_t aux = nullptr;
  cudaEvent_t ev[16] = {};
  cudaEvent_t wait_ev = nullptr;  // stream_wait
  cudaStream_t user = nullptr;
  bool use_user = false;
  ~ThreadStream() {
    // Streams are intentionally not destroyed at thread exit: the CUDA context may
    // already be torn down when thread-local destructors run at process exit.
  }
};
static thread_local std::unique_ptr<ThreadStream> t_streams[kMaxOrdinal];  // by CUDA ordinal

static ThreadStream& thread_stream(int device) {
  std::unique_ptr<ThreadStream>& p = t_streams[device];
  if (!p) p.reset(new ThreadStream());
  return *p;
}

cudaStream_t cur_stream() {
  ThreadStream& t = thread_stream(t_dev);
  if (t.use_user) return t.user;
  if (!t.own) cudaStreamCreateWithFlags(&t.own, cudaStreamNonBlocking);
  return t.own;
}

cudaStream_t aux_stream() {
  ThreadStream& t = thread_stream(t_dev);
  if (!t.aux) cudaStreamCreateWithFlags(&t.aux, cudaStreamNonBlocking);
  return t.aux;
}

cudaEvent_t aux_event(int i) {
  ThreadStream& t = thread_stream(t_dev);
  if (!t.ev[i]) cudaEventCreateWithFlags(&t.ev[i], cudaEventDisableTiming);
  return t.ev[i];
}

int stream_wait(cudaStream_t waiter, cudaStream_t producer, int producer_device) {
  if (slot_of(producer_device) < 0) {
    set_last_error("device %d is not in the set bound by ii2_init", producer_device);
    return II2_ERR_INVALID;
  }
  ThreadStream& t = thread_stream(producer_device);
  const int here = t_dev;
  if (producer_device != here) II2_CUDA_TRY(cudaSetDevice(producer_device));
  cudaError_t e = cudaSuccess;
  if (!t.wait_ev) e = cudaEventCreateWithFlags(&t.wait_ev, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventRecord(t.wait_ev, producer);
  if (producer_device != here) II2_CUDA_TRY(cudaSetDevice(here));
  if (e != cudaSuccess) {
    set_last_error("event on the stream of device %d: %s", producer_device, cudaGetErrorString(e));
    return II2_ERR_CUDA;
  }
  II2_CUDA_TRY(cudaStreamWaitEvent(waiter, t.wait_ev, 0));
  return II2_OK;
}

// ------------------------------------------------------------------ pinned pool
struct PinnedPool {
  std::mutex m;
  std::map<void*, size_t> live;                    // ptr -> class bytes
  std::map<size_t, std::vector<void*>> free_list;  // class bytes -> ptrs
  size_t cached = 0;
  static constexpr size_t kMaxCached = size_t(8) << 30;
};
static PinnedPool g_pinned;

static size_t size_class(size_t bytes) {
  size_t c = 4096;
  while (c < bytes) c <<= 1;
  // above 64 MiB round to 16 MiB granularity instead of doubling
  if (c > (size_t(64) << 20)) {
    const size_t g = size_t(16) << 20;
    c = (bytes + g - 1) / g * g;
  }
  return c;
}

__global__ void __launch_bounds__(256)
k_small_copy(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, size_t bytes) {
  pdl_enter();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t nw = bytes >> 2;
  const bool aligned = ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 3) == 0;
  if (aligned) {
    if (i < nw) reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(src)[i];
    if (i < (bytes & 3)) dst[(nw << 2) + i] = src[(nw << 2) + i];
  } else {
    for (size_t j = i * 4; j < bytes && j < i * 4 + 4; j++) dst[j] = src[j];
  }
}

int small_copy(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes == 0) return II2_OK;
  II2_LAUNCH_CHAIN(k_small_copy, div_up((bytes + 3) / 4, 256), 256, 0, s, static_cast<uint8_t*>(dst),
                   static_cast<const uint8_t*>(src), bytes);
  return II2_OK;
}

uint64_t* pinned_scratch() {
  static thread_local uint64_t* p = nullptr;
  if (!p) {
    void* q = nullptr;
    if (cudaHostAlloc(&q, 512, cudaHostAllocDefault) != cudaSuccess) return nullptr;  // 64 words
    p = static_cast<uint64_t*>(q);
  }
  return p;
}

uint32_t* device_tickets() {
  static thread_local uint32_t* per_dev[64] = {};  // one block per (host thread, device)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  uint32_t*& p = per_dev[dev];
  if (!p) {
    void* q = nullptr;
    if (cudaMalloc(&q, 256) != cudaSuccess) return nullptr;
    if (cudaMemset(q, 0, 256) != cudaSuccess) {
      cudaFree(q);
      return nullptr;
    }
    p = static_cast<uint32_t*>(q);
  }
  return p;
}

void* pinned_alloc(size_t bytes) {
  size_t c = size_class(bytes ? bytes : 1);
  {
    std::lock_guard<std::mutex> lk(g_pinned.m);
    auto it = g_pinned.free_list.find(c);
    if (it != g_pinned.free_list.end() && !it->second.empty()) {
      void* p = it->second.back();
      it->second.pop_back();
      g_pinned.cached -= c;
      g_pinned.live[p] = c;
      return p;
    }
  }
  void* p = nullptr;
  if (cudaHostAlloc(&p, c, cudaHostAllocDefault) != cudaSuccess) {
    set_last_error("cudaHostAlloc(%zu) failed", c);
    return nullptr;
  }
  std::lock_guard<std::mutex> lk(g_pinned.m);
  g_pinned.live[p] = c;
  return p;
}

void pinned_free(void* p) {
  if (!p) return;
  size_t c = 0;
  bool release = false;
  {
    std::lock_guard<std::mutex> lk(g_pinned.m);
    auto it = g_pinned.live.find(p);
    if (it == g_pinned.live.end()) return;  // not ours
    c = it->second;
    g_pinned.live.erase(it);
    if (g_pinned.cached + c <= PinnedPool::kMaxCached) {
      g_pinned.free_list[c].push_back(p);
      g_pinned.cached += c;
    } else {
      release = true;
    }
  }
  if (release) cudaFreeHost(p);
}

static void pinned_drain() {
  std::lock_guard<std::mutex> lk(g_pinned.m);
  for (auto& kv : g_pinned.free_list)
    for (void* p : kv.second) cudaFreeHost(p);
  g_pinned.free_list.clear();
  g_pinned.cached = 0;
}

// ------------------------------------------------------------------ scratch arena
struct Arena {
  int device = 0;
  uint8_t* base = nullptr;
  size_t cap = 0, used = 0, want = 0;
  std::vector<void*> spill;  // stream-ordered allocations made when the block was too small
};
static std::mutex g_arena_m;
static std::vector<Arena*> g_arenas;
static thread_local Arena* t_arena[kMaxOrdinal] = {};  // by CUDA ordinal

static Arena* my_arena() {
  Arena*& a = t_arena[t_dev];
  if (!a) {
    a = new Arena();
    a->device = t_dev;
    std::lock_guard<std::mutex> lk(g_arena_m);
    g_arenas.push_back(a);
  }
  return a;
}

void* arena_alloc(size_t bytes, cudaStream_t stream) {
  Arena* a = my_arena();
  bytes = (bytes + 255) & ~size_t(255);
  a->want += bytes;
  if (a->used + bytes <= a->cap) {
    void* p = a->base + a->used;
    a->used += bytes;
    return p;
  }
  void* q = nullptr;
  cudaError_t e = cudaMallocAsync(&q, bytes, stream);
  if (e != cudaSuccess) {
    set_last_error("scratch allocation of %zu bytes: %s", bytes, cudaGetErrorString(e));
    return nullptr;
  }
  a->spill.push_back(q);
  return q;
}

void arena_reset(cudaStream_t stream) {
  Arena* a = my_arena();
  for (void* q : a->spill) cudaFreeAsync(q, stream);
  const bool grow = !a->spill.empty() || a->want > a->cap;
  a->spill.clear();
  if (grow) {  // the caller has synchronised: nothing in flight uses the old block
    cudaStreamSynchronize(stream);
    if (a->base) cudaFree(a->base);
    a->base = nullptr;
    a->cap = 0;
    const size_t cap = a->want + a->want / 8 + (size_t(1) << 20);
    void* q = nullptr;
    if (cudaMalloc(&q, cap) == cudaSuccess) {
      a->base = static_cast<uint8_t*>(q);
      a->cap = cap;
    } else {
      cudaGetLastError();  // stay on the spill path
    }
  }
  a->used = 0;
  a->want = 0;
}

void arena_release_all() {
  std::lock_guard<std::mutex> lk(g_arena_m);
  for (Arena* a : g_arenas) {
    DeviceScope on(a->device);
    if (a->base) cudaFree(a->base);
    a->base = nullptr;
    a->cap = a->used = a->want = 0;
  }
}

// ------------------------------------------------------------------ instrumentation
struct ProfRec {
  const char* name;
  int device;  // CUDA ordinal of the events
  cudaEvent_t e0, e1;
  double host_t0, host_ms;
};
static double host_now_ms() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
struct Prof {
  std::mutex m;
  std::atomic<bool> on{false};
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> spare[kMaxOrdinal];  // by CUDA ordinal (an event belongs to one device)
};
static Prof g_prof;

ProfScope::ProfScope(const char* name, cudaStream_t stream) : s(stream), slot(-1) {
  if (!g_prof.on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof.m);
  ProfRec r;
  r.name = name;
  r.device = t_dev;
  std::vector<cudaEvent_t>& spare = g_prof.spare[t_dev];
  for (cudaEvent_t* e : {&r.e0, &r.e1}) {
    if (!spare.empty()) {
      *e = spare.back();
      spare.pop_back();
    } else if (cudaEventCreate(e) != cudaSuccess) {
      return;
    }
  }
  cudaEventRecord(r.e0, s);
  r.host_t0 = host_now_ms();
  r.host_ms = 0;
  slot = (int)g_prof.recs.size();
  g_prof.recs.push_back(r);
}

void ProfScope::end() {
  if (slot < 0) return;
  std::lock_guard<std::mutex> lk(g_prof.m);
  if (slot < (int)g_prof.recs.size()) {
    cudaEventRecord(g_prof.recs[slot].e1, s);
    g_prof.recs[slot].host_ms = host_now_ms() - g_prof.recs[slot].host_t0;
  }
  slot = -1;
}

static void prof_reset_locked() {
  for (ProfRec& r : g_prof.recs) {
    g_prof.spare[r.device].push_back(r.e0);
    g_prof.spare[r.device].push_back(r.e1);
  }
  g_prof.recs.clear();
}

// ------------------------------------------------------------------ scan (3 phases)
constexpr int kScanThreads = 512;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads) k_scan_reduce(const uint64_t* __restrict__ d,
                                                              uint64_t n,
                                                              uint64_t* __restrict__ bsum) {
  pdl_enter();
  __shared__ uint64_t ws[kScanThreads / 32 + 2];
  uint64_t base = (uint64_t)blockIdx.x * kScanTile;
  uint64_t acc = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; i++) {
    uint64_t idx = base + (uint64_t)i * kScanThreads + threadIdx.x;
    if (idx < n) acc += d[idx];
  }
  uint64_t total;
  block_exclusive_scan(acc, ws, total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// single CTA: exclusive scan of bsum[0..nb) in place, total -> *d_total
__global__ void __launch_bounds__(1024) k_scan_single(uint64_t* __restrict__ a, uint64_t nb,
                                                      uint64_t* __restrict__ d_total) {
  pdl_enter();
  __shared__ uint64_t ws[1024 / 32 + 2];
  uint64_t carry = 0;
  for (uint64_t base = 0; base < nb; base += 1024) {
    uint64_t idx = base + threadIdx.x;
    uint64_t v = idx < nb ? a[idx] : 0;
    uint64_t total;
    uint64_t ex = block_exclusive_scan(v, ws, total);
    if (idx < nb) a[idx] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0 && d_total) *d_total = carry;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_apply(uint64_t* __restrict__ d, uint64_t n,
                                                             const uint64_t* __restrict__ bsum) {
  pdl_enter();
  __shared__ uint64_t ws[kScanThreads / 32 + 2];
  uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
  uint64_t v[kScanItems];
  uint64_t acc = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; i++) {
    v[i] = (base + i < n) ? d[base + i] : 0;
    acc += v[i];
  }
  uint64_t total;
  uint64_t ex = block_exclusive_scan(acc, ws, total) + bsum[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; i++) {
    if (base + i < n) d[base + i] = ex;
    ex += v[i];
  }
}

// m arrays of length n laid out back to back, each scanned independently by its own CTA.
// Every WARP owns a contiguous 1/32 of the array and walks it 32 elements at a time (coalesced
// loads, four tiles requested ahead, shuffle scan, running total in a register — no block
// barrier inside the loops); the 32 warp totals are scanned once, then each warp adds its base.
// (The first version gave every thread a contiguous chunk: 2 x 41 strided dependent loads per
// thread, 48 us per launch at n = 41 k.)
// Optional extras (ScanExtra): CTA m sums a u32 array into totals[sum_slot]; the last CTA to
// finish copies totals[0 .. n_copy) to `host_copy` (pinned) — the totals of a pipeline stage
// reach the host with this launch alone.
struct ScanExtra {
  const uint32_t* sum_in;
  uint32_t sum_n, sum_slot;
  uint64_t* host_copy;
  uint32_t n_copy;
  uint32_t* ticket;  // zero between launches (device_tickets)
};

__device__ __forceinline__ void scan_multi_finish(const ScanExtra& x, uint64_t* totals) {
  if (!x.host_copy) return;
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(x.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (threadIdx.x < x.n_copy) x.host_copy[threadIdx.x] = *(volatile uint64_t*)(totals + threadIdx.x);
  if (threadIdx.x == 0) *x.ticket = 0;
}

__global__ void __launch_bounds__(1024) k_scan_multi(const uint64_t* a, uint64_t* out, uint64_t n,
                                                     uint64_t* __restrict__ totals, int m,
                                                     const ScanExtra x) {
  pdl_enter();
  __shared__ uint64_t ws[1024 / 32 + 2];
  if ((int)blockIdx.x >= m) {  // the extra CTA: a plain sum
    uint64_t acc = 0;
    for (uint32_t i = threadIdx.x; i < x.sum_n; i += 1024) acc += x.sum_in[i];
    uint64_t tot;
    block_exclusive_scan(acc, ws, tot);
    if (threadIdx.x == 0) totals[x.sum_slot] = tot;
    scan_multi_finish(x, totals);
    return;
  }
  const uint64_t* arr = a + (uint64_t)blockIdx.x * n;
  uint64_t* dst = out + (uint64_t)blockIdx.x * n;
  const unsigned lane = lane_id(), w = warp_id();
  const uint64_t per_warp = ((n + 31) / 32 + 31) & ~31ull;  // multiple of 32: aligned tiles
  const uint64_t lo = w * per_warp, hi = lo + per_warp < n ? lo + per_warp : n;
  uint64_t run = 0;
  for (uint64_t base = lo; base < hi; base += 128) {
    uint64_t v[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const uint64_t i = base + 32 * q + lane;
      v[q] = i < hi ? arr[i] : 0ull;
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const uint64_t inc = warp_inclusive_scan(v[q]);
      const uint64_t i = base + 32 * q + lane;
      if (i < hi) dst[i] = run + inc - v[q];
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  uint64_t total;
  const uint64_t wbase = block_exclusive_scan<uint64_t>(lane == 0 ? run : (uint64_t)0, ws, total);
  const uint64_t add = __shfl_sync(0xffffffffu, wbase, 0);
  if (add)
    for (uint64_t i = lo + lane; i < hi; i += 32) dst[i] += add;
  if (threadIdx.x == 0 && totals) totals[blockIdx.x] = total;
  scan_multi_finish(x, totals);
}

int exclusive_scan_multi_u64(const uint64_t* in, uint64_t* out, uint64_t n, int m,
                             uint64_t* d_totals, cudaStream_t s) {
  const ScanExtra none = {nullptr, 0, 0, nullptr, 0, nullptr};
  II2_LAUNCH_CHAIN(k_scan_multi, m, 1024, 0, s, in, out, n, d_totals, m, none);
  return II2_OK;
}

int exclusive_scan_multi_sum_to_host(const uint64_t* in, uint64_t* out, uint64_t n, int m,
                                     uint64_t* d_totals, const uint32_t* sum_in, uint32_t sum_n,
                                     uint32_t sum_slot, uint64_t* host_copy, uint32_t n_copy,
                                     cudaStream_t s) {
  uint32_t* const tickets = device_tickets();
  if (!tickets || n_copy > 1024) return II2_ERR_NOMEM;
  const ScanExtra x = {sum_in, sum_n, sum_slot, host_copy, n_copy, tickets + 1};
  II2_LAUNCH_CHAIN(k_scan_multi, m + 1, 1024, 0, s, in, out, n, d_totals, m, x);
  return II2_OK;
}

int exclusive_scan_u64(uint64_t* d, uint64_t n, uint64_t* d_total, cudaStream_t s) {
  if (n == 0) {
    if (d_total) II2_CUDA_TRY(cudaMemsetAsync(d_total, 0, sizeof(uint64_t), s));
    return II2_OK;
  }
  if (n <= 16384) {
    II2_LAUNCH_CHAIN(k_scan_single, 1, 1024, 0, s, d, n, d_total);
    return II2_OK;
  }
  uint64_t nb = (n + kScanTile - 1) / kScanTile;
  DevBuf<uint64_t> bsum;
  II2_TRY(bsum.alloc(nb, s));
  // k_scan_reduce reads strided (coalesced), k_scan_apply reads blocked per thread
  II2_LAUNCH_CHAIN(k_scan_reduce, (unsigned)nb, kScanThreads, 0, s, d, n, bsum.p);
  II2_LAUNCH_CHAIN(k_scan_single, 1, 1024, 0, s, bsum.p, nb, d_total);
  II2_LAUNCH_CHAIN(k_scan_apply, (unsigned)nb, kScanThreads, 0, s, d, n, bsum.p);
  return II2_OK;
}

}  // namespace ii2

// ------------------------------------------------------------------ C-ABI: lifecycle
using namespace ii2;

extern "C" {

int ii2_abi_version(void) { return II2_ABI_VERSION; }

const char* ii2_strerror(int code) {
  switch (code) {
    case II2_OK: return "ok";
    case II2_ERR_INVALID: return "invalid argument";
    case II2_ERR_NOMEM: return "out of memory";
    case II2_ERR_CUDA: return "CUDA error";
    case II2_ERR_NO_DEVICE: return "no CUDA device (ii2_init missing or failed; there is no CPU fallback)";
    case II2_ERR_BITMASK_OOB: return "bitmask is out of bound";
    case II2_ERR_CORRUPT: return "corrupt encoded data";
    case II2_ERR_UNSUPPORTED: return "input exceeds an implementation limit";
    default: return "unknown error";
  }
}

const char* ii2_last_error(void) { return t_last_error; }

int ii2_init(const int* devices, int ndev) {
  std::lock_guard<std::mutex> lk(g_ctx.m);
  if (ndev < 0 || ndev > kMaxDevices || (!devices && ndev > 1)) {
    set_last_error("ii2_init: %d devices (1 .. %d, or devices == NULL for device 0)", ndev, kMaxDevices);
    return II2_ERR_INVALID;
  }
  int want[kMaxDevices];
  int n = (devices && ndev >= 1) ? ndev : 1;
  for (int i = 0; i < n; i++) want[i] = (devices && ndev >= 1) ? devices[i] : 0;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < i; j++)
      if (want[i] == want[j]) {
        set_last_error("ii2_init: device %d listed twice", want[i]);
        return II2_ERR_INVALID;
      }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_last_error("no CUDA device: %s", e != cudaSuccess ? cudaGetErrorString(e) : "count=0");
    return II2_ERR_NO_DEVICE;
  }
  for (int i = 0; i < n; i++) {
    const int dev = want[i];
    if (dev < 0 || dev >= count || dev >= kMaxOrdinal) {
      set_last_error("device %d out of range (have %d)", dev, count);
      return II2_ERR_INVALID;
    }
  }
  if (g_ctx.ready) {  // idempotent for the same set (any order); any other set is refused
    bool same = n == g_ctx.ndev;
    for (int i = 0; i < n && same; i++) same = slot_of(want[i]) >= 0;
    if (same) return II2_OK;
    set_last_error("already initialised on %d device(s), the first being %d", g_ctx.ndev, g_ctx.devices[0]);
    return II2_ERR_INVALID;
  }
  for (int i = 0; i < n; i++) {
    const int dev = want[i];
    II2_CUDA_TRY(cudaSetDevice(dev));
    cudaDeviceProp prop;
    II2_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) {
      set_last_error("device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major,
                     prop.minor);
      return II2_ERR_NO_DEVICE;
    }
    // Keep freed stream-ordered memory in the pool instead of returning it to the driver.
    cudaMemPool_t pool;
    II2_CUDA_TRY(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t thresh = UINT64_MAX;
    II2_CUDA_TRY(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
  }
  // Peer access of this process's contexts wherever the hardware allows it (the in-process
  // gathers read other devices' HBM directly).  Peer access covers cudaMalloc memory only: the
  // stream-ordered allocations (every result array) come from the device's default pool, which
  // another device may read only once the pool grants it access (cudaMemPoolSetAccess).
  bool peer[kMaxDevices][kMaxDevices] = {};
  for (int i = 0; i < n; i++) {
    for (int j = 0; j < n; j++) {
      if (i == j) continue;
      int can = 0;
      II2_CUDA_TRY(cudaDeviceCanAccessPeer(&can, want[i], want[j]));
      if (!can) continue;
      II2_CUDA_TRY(cudaSetDevice(want[i]));
      e = cudaDeviceEnablePeerAccess(want[j], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        e = cudaSuccess;
      }
      II2_CUDA_TRY(e);
      cudaMemPool_t pool;
      II2_CUDA_TRY(cudaDeviceGetDefaultMemPool(&pool, want[j]));
      cudaMemAccessDesc acc = {};
      acc.location.type = cudaMemLocationTypeDevice;
      acc.location.id = want[i];
      acc.flags = cudaMemAccessFlagsProtReadWrite;
      e = cudaMemPoolSetAccess(pool, &acc, 1);
      if (e != cudaSuccess) {  // that pair stays unreadable: the gathers refuse it
        cudaGetLastError();
        continue;
      }
      peer[i][j] = true;
    }
  }
  II2_CUDA_TRY(cudaSetDevice(want[0]));
  g_ctx.ndev = n;
  for (int i = 0; i < n; i++) {
    g_ctx.devices[i] = want[i];
    for (int j = 0; j < n; j++) g_ctx.peer[i][j] = peer[i][j];
  }
  g_ctx.ready = true;
  return II2_OK;
}

int ii2_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_ctx.m);
  if (!g_ctx.ready) return II2_OK;
  for (int i = 0; i < g_ctx.ndev; i++) {
    DeviceScope on(g_ctx.devices[i]);
    cudaDeviceSynchronize();
  }
  arena_release_all();
  pinned_drain();
  g_ctx.ready = false;
  return II2_OK;
}

int ii2_set_device(int device) {
  if (!g_ctx.ready) return no_device();
  if (slot_of(device) < 0) {
    set_last_error("device %d is not in the set bound by ii2_init", device);
    return II2_ERR_INVALID;
  }
  t_sel = device;
  return II2_OK;
}

int ii2_set_stream(void* cuda_stream) {
  ThreadStream& t = thread_stream(g_ctx.ready ? selected_device() : 0);
  t.user = static_cast<cudaStream_t>(cuda_stream);
  t.use_user = cuda_stream != nullptr;
  return II2_OK;
}

uint64_t ii2_kernel_launches(void) { return g_kernel_launches.load(); }

int ii2_prof_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof.m);
  prof_reset_locked();
  g_prof.on.store(on != 0);
  return II2_OK;
}

int ii2_prof_read(ii2_prof_entry* out, int cap) {
  if (cap < 0 || (cap && !out)) return II2_ERR_INVALID;
  std::lock_guard<std::mutex> lk(g_prof.m);
  int n = 0;
  for (ProfRec& r : g_prof.recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.e1) != cudaSuccess || cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    int j = 0;
    while (j < n && strcmp(out[j].name, r.name) != 0) j++;
    if (j == n) {
      if (n == cap) continue;
      out[n].name = r.name;
      out[n].ms = 0;
      out[n].host_ms = 0;
      out[n].count = 0;
      n++;
    }
    out[j].ms += ms;
    out[j].host_ms += r.host_ms;
    out[j].count += 1;
  }
  return n;
}

void ii2_free(void* p) { pinned_free(p); }

int ii2_sync(void) {
  II2_TRY(ctx_require());
  II2_CUDA_TRY(cudaStreamSynchronize(cur_stream()));
  for (int i = 0; i < g_ctx.ndev; i++) {  // this thread's streams on the other bound devices
    const int d = g_ctx.devices[i];
    if (d == t_dev || !t_streams[d]) continue;
    const ThreadStream& t = *t_streams[d];
    if (t.use_user) II2_CUDA_TRY(cudaStreamSynchronize(t.user));
    if (t.own) II2_CUDA_TRY(cudaStreamSynchronize(t.own));
  }
  return II2_OK;
}

uint32_t ii2_shard_key(const uint8_t* term, size_t len) {
  // shardKey, shard.go:362-378
  uint16_t key = 0;
  if (len >= 2) key = (uint16_t)(((uint16_t)term[0] << 8) + term[1]);
  return (uint32_t)(key >> 6);
}

}  // extern "C"
