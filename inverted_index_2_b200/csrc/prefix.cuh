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

// K5's tail, shared with K10: recs[i].cnt values of union i (records of k2_large_run) are copied
// back to back into out.values, out.value_off = their scanned offsets.  d_flag: null or a device
// word that is nonzero when the call must fail with `flag_msg` (II2_ERR_UNSUPPORTED); it is read
// in the same round trip as the total.  `place_name` names the ProfScope of the copy.
// out.value_off must hold np + 1 words.  Synchronises the stream.
int place_unions(const GroupRec* recs, uint32_t np, PrefixOut& out, const uint32_t* d_flag,
                 const char* flag_msg, const char* place_name, uint64_t* h_value_off,
                 cudaStream_t s);

#ifdef __CUDACC__
// bytes.HasPrefix(t, p)
__device__ __forceinline__ bool has_prefix(const uint8_t* t, uint32_t nt, const uint8_t* p,
                                           uint32_t np) {
  if (nt < np) return false;
  for (uint32_t i = 0; i < np; i++)
    if (t[i] != p[i]) return false;
  return true;
}

// The window of the terms of segment sd that start with p, found by a whole warp: lo = first
// term >= p (every term with prefix p is >= p), then prefix_window_hi = first term at or after lo
// that does not start with p (terms with a common prefix are contiguous in bytes.Compare order);
// both are 32-way searches (warp_partition_point).  Every lane must call; every lane gets the
// result.
__device__ __forceinline__ uint32_t prefix_window_lo(const SegDesc& sd, const uint8_t* pb,
                                                     uint32_t pn) {
  return warp_partition_point(0u, sd.n, [&](uint32_t i) {
    const uint32_t o = __ldg(sd.toff + i), n = __ldg(sd.toff + i + 1) - o;
    return term_compare(sd.tb + o, n, pb, pn) < 0;
  });
}
__device__ __forceinline__ uint32_t prefix_window_hi(const SegDesc& sd, uint32_t lo,
                                                     const uint8_t* pb, uint32_t pn) {
  return warp_partition_point(lo, sd.n, [&](uint32_t i) {
    const uint32_t o = __ldg(sd.toff + i), n = __ldg(sd.toff + i + 1) - o;
    return has_prefix(sd.tb + o, n, pb, pn);
  });
}
#endif  // __CUDACC__

}  // namespace ii2
