// prefix.cuh — K5: per-prefix posting unions over resident segments (PrefixSearch,
// inverted_index.go:192-295).
#pragma once
#include "union.cuh"

namespace ii2 {

struct PrefixOut {
  DevBuf<uint32_t> values;     // unions of all prefixes back to back, each sorted-unique
  DevBuf<uint64_t> value_off;  // [np + 1]
  DevBuf<uint32_t> matched;    // [np] != 0 <=> some term starts with the prefix
  uint64_t total = 0;
};

// d_segs: [k] resident segments (tb/toff/post/poff/n); prefixes = d_pbytes[d_poff[i]..d_poff[i+1]).
// d_kind: null (every item is a prefix) or [np] II2_ATOM_*: a TERM item takes only the term equal
// to it, so its list is the sorted-unique union of that term's values (boolean queries).
// h_value_off: null or [np + 1] pinned words that receive out.value_off in the round trip that
// learns the total (no extra synchronisation).
// Synchronises the stream; intermediates come from the calling thread's scratch arena.
int k5_prefix_search(const SegDesc* d_segs, int k, const uint8_t* d_pbytes, const uint32_t* d_poff,
                     uint32_t np, PrefixOut& out, cudaStream_t s, const uint8_t* d_kind = nullptr,
                     uint64_t* h_value_off = nullptr);

}  // namespace ii2
