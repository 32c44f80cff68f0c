// handles.cuh — the opaque handle types of include/ii2.h (resident segment, removed set, result),
// shared by the translation units that implement the C-ABI (api.cu, comm.cu).  Every handle
// records the CUDA device its memory lives on: calls that take handles run there.
#pragma once
#include <string>
#include <vector>

#include "prefix.cuh"
#include "union.cuh"

using namespace ii2;

struct ii2_seg {
  int device = ctx_current_device();
  uint32_t n_terms = 0;
  uint64_t n_post = 0;
  uint64_t term_bytes_len = 0;
  DevBuf<uint8_t> tb;
  DevBuf<uint32_t> toff;
  DevBuf<uint32_t> post;
  DevBuf<uint64_t> poff;
};

struct ii2_removed {
  int device = ctx_current_device();
  uint64_t n = 0;
  DevBuf<uint32_t> sorted;
  DevBuf<uint32_t> bitmap;
  uint64_t bitmap_bits = 0;
  RemovedSet set() const {
    RemovedSet r;
    r.sorted = sorted.p;
    r.n = n;
    r.bitmap = bitmap_bits ? bitmap.p : nullptr;
    r.bitmap_bits = bitmap_bits;
    return r;
  }
};

struct ii2_result {
  int device = ctx_current_device();
  cudaStream_t stream = nullptr;  // the stream that produced it (in-process gathers wait for it)
  EmitOut out;
  uint64_t T = 0, TB = 0, P = 0, E = 0;
  uint64_t postings_in = 0, terms_merged = 0;
  bool has_dec = false, has_enc = false;
  bool has_minmax = false;
  bool rebased = false;  // offsets already carry the base of a pipelined download
  std::string min_term, max_term;
};

// The device of one call's handles (segments and removed set; NULL entries are left to the
// call's own checks): -1 when there is none (the call runs on the selected device),
// II2_ERR_INVALID when they live on different devices.
inline int handles_device(ii2_seg* const* segs, int nseg, const ii2_removed* rem, int* device) {
  int d = rem ? rem->device : -1;
  for (int i = 0; segs && i < nseg; i++) {
    if (!segs[i]) continue;
    if (d >= 0 && segs[i]->device != d) {
      set_last_error("handles of one call live on different devices (%d and %d)", d, segs[i]->device);
      return II2_ERR_INVALID;
    }
    d = segs[i]->device;
  }
  *device = d;
  return II2_OK;
}

// Host-side outputs of the C-ABI (ii2_merge_out, ii2_read_out, ii2_prefix_out ...): pinned
// buffers owned by one object behind the struct's `_owner` field.
struct HostOwner {
  std::vector<void*> ptrs;
  ~HostOwner() {
    for (void* p : ptrs) pinned_free(p);
  }
  template <typename T>
  T* alloc(size_t n) {
    void* p = pinned_alloc(n * sizeof(T) + 8);
    if (p) ptrs.push_back(p);
    return static_cast<T*>(p);
  }
};
