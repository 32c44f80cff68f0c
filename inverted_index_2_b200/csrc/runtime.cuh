// runtime.cuh — process context, per-(thread, device) streams and scratch, stream-ordered
// device buffers, pinned host pool.  One process drives one GPU or a bound set of up to
// kMaxDevices GPUs (ii2_init); every call runs on one device of the set.
#pragma once
#include <vector>

#include "common.cuh"

namespace ii2 {

constexpr int kMaxDevices = 16;  // GPUs one process can bind (ii2_init)

bool ctx_ready();
// Enter a call on the device the calling thread selected (ii2_set_device; devices[0] by
// default) and make it current: II2_OK or II2_ERR_NO_DEVICE (sets last error).
int ctx_require();
// Enter a call on CUDA device `device` (the device of the call's handles); device < 0 means the
// selected one.  II2_ERR_INVALID if the device is not in the bound set.
int ctx_require_device(int device);
int ctx_current_device();      // CUDA ordinal of the running call (devices[0] outside calls)
int ctx_device_count();        // devices bound by ii2_init (0 before)
bool ctx_bound(int device);    // device is in the bound set
// kernels on `dev` can read all of `peer`'s memory: peer access is on and `peer`'s default
// memory pool (every stream-ordered allocation) grants `dev` access
bool ctx_peer(int dev, int peer);
// Make `waiter` (a stream of the running call's device) wait for the work queued so far on
// `producer`, a stream of bound device `producer_device` (one reusable event per host thread
// and device; the wait is taken at once, so the event can be recorded again).
int stream_wait(cudaStream_t waiter, cudaStream_t producer, int producer_device);
// Makes `device` current for a scope and restores the previous device (handle releases from
// any thread).
struct DeviceScope {
  int prev = -1;
  explicit DeviceScope(int device);
  ~DeviceScope();
};
// The streams and events below belong to the calling thread AND the running call's device.
cudaStream_t cur_stream();    // this thread's stream (caller-provided or library-owned)
cudaStream_t aux_stream();    // a second library-owned stream of this thread (kernel overlap)
cudaEvent_t aux_event(int i);  // this thread's reusable timing-free events, i < 16

// Per-(thread, device) scratch arena: one grow-only device block, bump-allocated during a pipeline call
// and reset when the call is over.  GB-sized cudaMallocAsync requests were measured at tens of
// milliseconds per call on B200 (the pool re-maps physical memory); the arena makes every
// intermediate buffer free of charge after the first call.
void* arena_alloc(size_t bytes, cudaStream_t stream);  // nullptr + last error on failure
// Call once per pipeline, after the stream has been synchronised: frees spill-over
// allocations and grows the block to the high-water mark of the call.
void arena_reset(cudaStream_t stream);
void arena_release_all();  // ii2_shutdown

// Device buffer: stream-ordered allocation (cudaMallocAsync) for data that outlives the call,
// or arena scratch for intermediates.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaStream_t s = nullptr;
  bool scratch = false;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n), s(o.s), scratch(o.scratch) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      release();
      p = o.p; n = o.n; s = o.s; scratch = o.scratch;
      o.p = nullptr; o.n = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  // `pad_bytes` extra readable bytes past the end (over-reading vector loads).  Every buffer
  // carries 16 bytes more than asked: the fused merge kernel stages the 16-byte aligned
  // ENVELOPE of a run, which may end up to 15 bytes past the array.
  int alloc(size_t count, cudaStream_t stream, size_t pad_bytes = 0) {
    release();
    s = stream;
    n = count;
    scratch = false;
    size_t bytes = count * sizeof(T) + pad_bytes + 16;
    void* q = nullptr;
    II2_CUDA_TRY(cudaMallocAsync(&q, bytes, stream));
    p = static_cast<T*>(q);
    return II2_OK;
  }
  // intermediate of the current pipeline call: lives until arena_reset
  int alloc_scratch(size_t count, cudaStream_t stream, size_t pad_bytes = 0) {
    release();
    s = stream;
    n = count;
    scratch = true;
    size_t bytes = count * sizeof(T) + pad_bytes + 16;
    p = static_cast<T*>(arena_alloc(bytes, stream));
    return p ? II2_OK : II2_ERR_NOMEM;
  }
  void release() {
    if (p && !scratch) cudaFreeAsync(p, s);
    p = nullptr;
    n = 0;
  }
  T* take() { T* q = p; p = nullptr; n = 0; return q; }
};

// Instrumentation (ii2_prof_enable / ii2_prof_read): CUDA events around a kernel phase on the
// launching stream.  No-ops unless enabled.
struct ProfScope {
  cudaStream_t s;
  int slot;
  ProfScope(const char* name, cudaStream_t stream);
  void end();
  ~ProfScope() { end(); }
};

// Pinned host memory with a size-class cache (cudaHostAlloc is far too slow per call).
void* pinned_alloc(size_t bytes);
void pinned_free(void* p);  // also accepts nullptr
// A pinned block that is freed when it goes out of scope; p == nullptr if the allocation failed.
struct PinnedBlock {
  void* p;
  explicit PinnedBlock(size_t bytes) : p(pinned_alloc(bytes)) {}
  PinnedBlock(const PinnedBlock&) = delete;
  PinnedBlock& operator=(const PinnedBlock&) = delete;
  ~PinnedBlock() { pinned_free(p); }
};
// 256 bytes of pinned memory owned by the calling thread: the landing place of the small
// device->host readbacks (totals, flags).  A pageable destination would make the copy wait for
// every other transfer in flight, including the next range's staging on the second stream.
uint64_t* pinned_scratch();
// 64 device words that are zero between kernels (per host thread): "last CTA" tickets; a kernel
// that takes one puts the zero back before it ends, so no launch needs a memset in front of it.
uint32_t* device_tickets();

// Copy a few bytes between PINNED host memory and device memory (either direction) with a
// kernel instead of a copy engine.  The copy engines serve requests in order: a 64-byte
// readback queued behind the next range's hundreds of MB of staging would wait for all of it.
// A kernel reads / writes the pinned page directly over the bus and only obeys stream order.
int small_copy(void* dst, const void* src, size_t bytes, cudaStream_t s);

// In-place exclusive scan of d[0..n) (u64); total written to *d_total (device) if non-null.
int exclusive_scan_u64(uint64_t* d, uint64_t n, uint64_t* d_total, cudaStream_t s);
// m short arrays (each n <= a few thousand) laid out back to back, scanned independently by
// one CTA in one launch; totals[j] (device) receives each array's sum.
// (in == out is allowed.)
int exclusive_scan_multi_u64(const uint64_t* in, uint64_t* out, uint64_t n, int m,
                             uint64_t* d_totals, cudaStream_t s);
// The same with one more CTA that sums `sum_in[0 .. sum_n)` into d_totals[sum_slot]; the last CTA
// copies d_totals[0 .. n_copy) into `host_copy` (pinned memory): scan + sum + the copy of the
// totals to the host as ONE launch.  The caller synchronises the stream before reading.
int exclusive_scan_multi_sum_to_host(const uint64_t* in, uint64_t* out, uint64_t n, int m,
                                     uint64_t* d_totals, const uint32_t* sum_in, uint32_t sum_n,
                                     uint32_t sum_slot, uint64_t* host_copy, uint32_t n_copy,
                                     cudaStream_t s);

}  // namespace ii2
