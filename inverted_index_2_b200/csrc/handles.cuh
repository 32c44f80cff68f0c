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
};

// The removed set of a call that takes an optional ii2_removed (empty for NULL).
inline RemovedSet removed_set(const ii2_removed* rem) {
  if (!rem) return RemovedSet{};
  return RemovedSet{rem->sorted.p, rem->n, rem->bitmap_bits ? rem->bitmap.p : nullptr, rem->bitmap_bits};
}

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

// The segment table of a call: row i is segs[i] with its whole dictionary as the window, and its
// instances are numbered after those of the rows before it (.base, which only the merge and
// range-read pipeline reads).  II2_ERR_INVALID for a NULL segment; *n_inst = all instances.
inline int seg_table(SegDesc* h, ii2_seg* const* segs, int nseg, uint64_t* n_inst = nullptr) {
  uint64_t n = 0;
  for (int i = 0; i < nseg; i++) {
    const ii2_seg* g = segs[i];
    if (!g) return II2_ERR_INVALID;
    h[i] = SegDesc{g->tb.p, g->toff.p, g->post.p, g->poff.p, g->n_terms, 0, g->n_terms, (uint32_t)n};
    n += g->n_terms;
  }
  if (n_inst) *n_inst = n;
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
