// lookup.cuh — K8: batched exact-term reads over resident segments (Read(t, t) for many t at
// once, ii2_lookup_dev).
#pragma once
#include "union.cuh"

namespace ii2 {

struct LookupOut {
  DevBuf<uint8_t> found;      // [nkeys] != 0 <=> Read(key, key) yields the term
  DevBuf<uint64_t> post_off;  // [nkeys + 1]
  DevBuf<uint32_t> post;      // [total] the keys' lists back to back
  uint64_t total = 0;
  uint64_t postings_in = 0;   // Σ lengths of the source lists that were unioned
};

// d_segs: [k] resident segments (tb/toff/post/poff/n), 1 <= k <= kMaxSegs; key i =
// d_kb[d_koff[i] .. d_koff[i+1]), nkeys >= 1.  n_post: Σ postings of the segments (bounds the
// output pool of the one-CTA unions).  keep_empty: a key held only with empty lists is found
// (plain reads); otherwise a key whose list ends empty is not.  Synchronises the stream;
// intermediates come from the calling thread's scratch arena.
int k8_lookup(const SegDesc* d_segs, int k, uint64_t n_post, const uint8_t* d_kb,
              const uint32_t* d_koff, uint32_t nkeys, const RemovedSet& rem, bool keep_empty,
              LookupOut& out, cudaStream_t s);

}  // namespace ii2
