// common.cuh — shared host/device helpers for the ii2 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/ii2.h"

namespace ii2 {

// ---------------------------------------------------------------- host side
extern std::atomic<uint64_t> g_kernel_launches;
void set_last_error(const char* fmt, ...);

#define II2_CUDA_TRY(expr)                                                                 \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::ii2::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                  \
                            cudaGetErrorString(_e));                                       \
      return _e == cudaErrorMemoryAllocation ? II2_ERR_NOMEM : II2_ERR_CUDA;               \
    }                                                                                      \
  } while (0)

#define II2_TRY(expr)          \
  do {                         \
    int _rc = (expr);          \
    if (_rc != II2_OK) return _rc; \
  } while (0)

// Count the launch and catch launch-configuration errors right away.
#define II2_LAUNCHED()                                   \
  do {                                                   \
    ::ii2::g_kernel_launches.fetch_add(1, std::memory_order_relaxed); \
    II2_CUDA_TRY(cudaGetLastError());                    \
  } while (0)

// ---- chained launches (programmatic dependent launch) -------------------------------------
// A range read of a thousand terms is ~20 dependent kernels of a few microseconds each: the
// launch gaps, not the kernels, are most of its latency.  Kernels of the merge / read chain
// start with pdl_enter() and are launched with II2_LAUNCH_CHAIN: the grid is set up and its
// CTAs become resident while the previous kernel still runs, `griddepcontrol.wait` holds them
// until that kernel has completed and its writes are visible, so only the gap disappears —
// ordering and visibility are those of a plain stream.  A kernel WITHOUT pdl_enter() must never
// be launched this way (it would run next to its producer).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#define II2_LAUNCH_CHAIN(kern, grid, block, smem, s, ...)                                  \
  do {                                                                                     \
    const cudaError_t _le = ::ii2::launch_chain(kern, grid, block, smem, s, __VA_ARGS__);  \
    ::ii2::g_kernel_launches.fetch_add(1, std::memory_order_relaxed);                      \
    II2_CUDA_TRY(_le);                                                                     \
  } while (0)

constexpr int kNumSMs = 148;  // B200

static inline unsigned div_up(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

// Device-resident segment as the merge kernels see it (always decoded form).
struct SegDesc {
  const uint8_t* tb;     // term bytes, allocation readable 32 B past the end
  const uint32_t* toff;  // [n+1]
  const uint32_t* post;  // decoded postings
  const uint64_t* poff;  // [n+1]
  uint32_t n;            // terms in the segment
  uint32_t lo, hi;       // active window of this call: terms [lo,hi)
  uint32_t base;         // global instance id of term `lo` (exclusive prefix of hi-lo)
};

// Removed list on the device: sorted values + optional membership bitmap.
struct RemovedSet {
  const uint32_t* sorted;
  uint64_t n;
  const uint32_t* bitmap;  // bit v set <=> v removed, for v < bitmap_bits
  uint64_t bitmap_bits;
};

constexpr int kMaxSegs = 1024;     // segments per merge pass (smem rows, u16 group sizes)
constexpr int kMaxSamples = 8192;  // splitter samples (one CTA sorts them in smem)

#ifdef __CUDACC__
// ---------------------------------------------------------------- device side
// First statement of every kernel launched with II2_LAUNCH_CHAIN: wait for the producer grid,
// then let the consumer grid be set up behind this one.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned warp_id() { return threadIdx.x >> 5; }

template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane_id() >= (unsigned)d) v += o;
  }
  return v;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// Block-wide exclusive scan.  `ws` = shared scratch of (blockDim.x/32 + 1) elements.
// Every thread of the block must call it.  Returns the exclusive prefix of `v`;
// `total` receives the block total.  Safe to call repeatedly with the same scratch.
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* ws, T& total) {
  const unsigned lane = lane_id(), w = warp_id(), nw = (blockDim.x + 31) >> 5;
  T inc = warp_inclusive_scan(v);
  __syncthreads();  // protect ws from the previous use
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    T x = lane < nw ? ws[lane] : T(0);
    T xi = warp_inclusive_scan(x);
    if (lane < nw) ws[lane] = xi - x;
    if (lane == 31) ws[nw] = xi;  // nw <= 32
  }
  __syncthreads();
  total = ws[nw];
  return ws[w] + inc - v;
}

// (segment, index) of global instance id g: the last s with base[s] <= g (empty windows share
// their base with the next segment, so the last one is the non-empty owner).
__device__ __forceinline__ void locate_instance(const SegDesc* __restrict__ segs, int k, uint32_t g,
                                                int& s_out, uint32_t& idx_out) {
  int lo = 0, hi = k;  // first s with base > g
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (segs[mid].base <= g)
      lo = mid + 1;
    else
      hi = mid;
  }
  int s = lo - 1;
  s_out = s;
  idx_out = segs[s].lo + (g - segs[s].base);
}

// bytes.Compare(a, b) on device memory.  Returns <0, 0, >0.
__device__ __forceinline__ int term_compare(const uint8_t* a, uint32_t na, const uint8_t* b,
                                            uint32_t nb) {
  uint32_t m = na < nb ? na : nb;
  for (uint32_t i = 0; i < m; i++) {
    int d = (int)a[i] - (int)b[i];
    if (d) return d;
  }
  return na < nb ? -1 : (na > nb ? 1 : 0);
}

// First index in [lo,hi) of segment `s` whose term is >= (t,nt)  (vellum Iterator(min) seek,
// file/reader.go:147).
__device__ __forceinline__ uint32_t seg_lower_bound(const SegDesc& s, uint32_t lo, uint32_t hi,
                                                    const uint8_t* t, uint32_t nt) {
  while (lo < hi) {
    uint32_t mid = lo + ((hi - lo) >> 1);
    uint32_t o = s.toff[mid], n = s.toff[mid + 1] - o;
    if (term_compare(s.tb + o, n, t, nt) < 0)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// First index in [lo,hi) whose term is > (t,nt)  (inclusive max bound, file/reader.go:54-58).
__device__ __forceinline__ uint32_t seg_upper_bound(const SegDesc& s, uint32_t lo, uint32_t hi,
                                                    const uint8_t* t, uint32_t nt) {
  while (lo < hi) {
    uint32_t mid = lo + ((hi - lo) >> 1);
    uint32_t o = s.toff[mid], n = s.toff[mid + 1] - o;
    if (term_compare(s.tb + o, n, t, nt) <= 0)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// First index in [lo,hi) for which pred is false, pred being true on a prefix of the range
// (a partition point), found by a whole warp: the lanes probe 32 evenly spaced indexes, a
// ballot narrows the interval 33-fold — 4 rounds of dependent loads for 500 k terms instead of
// the 19 of a binary search.  Every lane must call with the same lo / hi; returns the same value
// in every lane.
template <class Pred>
__device__ __forceinline__ uint32_t warp_partition_point(uint32_t lo, uint32_t hi, Pred pred) {
  const unsigned lane = lane_id();
  while (lo < hi) {  // uniform inside the warp
    const uint32_t width = hi - lo;
    const bool narrow = width <= 32;
    const uint32_t probe = narrow ? lo + lane : lo + (uint32_t)(((uint64_t)(lane + 1) * width) / 33);
    const bool t = (!narrow || lane < width) ? pred(probe) : false;
    const uint32_t c = __popc(__ballot_sync(0xffffffffu, t));  // monotone: lanes 0 .. c-1
    if (narrow) return lo + c;
    const uint32_t first_false = lo + (uint32_t)(((uint64_t)(c + 1) * width) / 33);  // lane c's probe
    const uint32_t last_true = lo + (uint32_t)(((uint64_t)c * width) / 33);          // lane c-1's
    if (c < 32) hi = first_false;
    if (c > 0) lo = last_true + 1;
  }
  return lo;
}

// slices.BinarySearch(removedValues, v) membership (shard.go:183), answered from the bitmap
// when one covers v.
__device__ __forceinline__ bool is_removed(const RemovedSet& r, uint32_t v) {
  if (r.n == 0) return false;
  if (r.bitmap) {
    if ((uint64_t)v >= r.bitmap_bits) return false;
    return (__ldg(r.bitmap + (v >> 5)) >> (v & 31u)) & 1u;
  }
  uint64_t lo = 0, hi = r.n;
  while (lo < hi) {
    uint64_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(r.sorted + mid) < v)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo < r.n && __ldg(r.sorted + lo) == v;
}

// The same test kept out of line, for kernels that apply it to dozens of register-resident
// values per lane (32 inlined search loops were a quarter of k2_mwarp_kernel's SASS; the loop
// only runs for removed lists whose largest id is >= 2^29).
static __device__ __noinline__ bool is_removed_call(const uint32_t* __restrict__ sorted, uint64_t n,
                                                    uint32_t v) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    uint64_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(sorted + mid) < v)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo < n && __ldg(sorted + lo) == v;
}

// Bitonic sorting network without direction flags, valid for ANY n (indices >= n behave as
// +inf and never move): for each block size k, a mirrored "flip" step then half-cleaners.
// `nthreads` cooperating threads with ids tid in [0,nthreads); `sync` separates stages.
template <typename T, typename Less, typename Sync>
__device__ __forceinline__ void bitonic_sort_any(T* a, uint32_t n, uint32_t tid, uint32_t nthreads,
                                                 Less less, Sync sync) {
  if (n < 2) return;
  for (uint32_t k = 2; (k >> 1) < n; k <<= 1) {
    // flip: i pairs with i ^ (k-1)
    for (uint32_t t = tid; t < (n + 1) / 2 + (k >> 1); t += nthreads) {
      // enumerate lower elements: t -> i with bit (k/2) clear
      uint32_t i = ((t / (k >> 1)) * k) + (t % (k >> 1));
      uint32_t l = i ^ (k - 1);
      if (l < n && i < n) {
        T x = a[i], y = a[l];
        if (less(y, x)) {
          a[i] = y;
          a[l] = x;
        }
      }
    }
    sync();
    for (uint32_t j = k >> 2; j >= 1; j >>= 1) {
      for (uint32_t t = tid; t < (n + 1) / 2 + j; t += nthreads) {
        uint32_t i = ((t / j) * (j << 1)) + (t % j);
        uint32_t l = i + j;
        if (l < n) {
          T x = a[i], y = a[l];
          if (less(y, x)) {
            a[i] = y;
            a[l] = x;
          }
        }
      }
      sync();
    }
  }
}
#endif  // __CUDACC__

}  // namespace ii2
