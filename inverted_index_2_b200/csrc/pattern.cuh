// pattern.cuh — K10: wildcard (glob) and fuzzy term patterns over resident segments
// (ii2_pattern_search_dev).  The host compiles every pattern into a PatTab; k10_pattern.cu scans
// the candidate terms with it and unions the lists of the matching ones.
#pragma once
#include "prefix.cuh"

namespace ii2 {

constexpr uint32_t kPatGroup = 16;      // unanchored patterns one CTA runs over a staged tile
constexpr uint32_t kPatMaxGlob = 63;    // glob elements: NFA states 1..63 of one u64, 0 = start
constexpr uint32_t kPatMaxFuzzy = 64;   // fuzzy bytes after the exact prefix: one u64 column
constexpr uint32_t kPatMaxEdits = 2;
constexpr uint32_t kPatMaxBytes = 65535;

// One compiled pattern.
//   GLOB: a bit-parallel NFA.  State j (bit j) = the first j elements (non-`*` items) matched;
//         mask[c] bit j+1 = element j accepts byte c; loop bit j = a `*` follows element j-1
//         (bit 0: the pattern starts with `*`); accept = bit `elements`.  A byte steps
//         D = ((D << 1) & mask[c]) | (D & loop) from D = 1.
//   FUZZY: Myers / Hyyrö bit vectors of q[P..] (m bytes): mask[c] bit i = (q[P + i] == c).
// skip: leading bytes every term of the pattern's window already matched (the glob's literal
// prefix, whose elements are single literal bytes, or the fuzzy exact prefix): the scan starts
// there, a glob in state `skip`.
struct __align__(16) PatTab {
  uint64_t mask[256];
  uint64_t loop;
  uint64_t accept;
  uint32_t kind;  // II2_PATTERN_*
  uint32_t m;     // FUZZY: len(q) - P
  uint32_t k;     // FUZZY: max edits
  uint32_t skip;
};
static_assert(sizeof(PatTab) % 16 == 0, "PatTab is staged with 16-byte copies");

// Internal patterns [p0, p0 + n) scan the same windows: the terms that start with the pre_len
// bytes at pre_off of the prefix blob (pre_len == 0: whole segments).
struct PatGroup {
  uint32_t p0, n, pre_off, pre_len;
};

struct PatternDev {
  const SegDesc* segs;
  int k;
  const PatTab* tabs;    // [nu] distinct patterns, group after group
  uint32_t nu;
  const PatGroup* groups;
  uint32_t ng;
  const uint8_t* pre;    // prefix blob
  const uint32_t* uid;   // [npat] output pattern -> internal pattern
  uint32_t npat;
};

// out: value_off [npat + 1], matched [npat], values; Synchronises the stream; intermediates come
// from the calling thread's scratch arena.
int k10_pattern_search(const PatternDev& d, PrefixOut& out, cudaStream_t s);

// Device outputs of k10_pattern_terms: output pattern i's terms are [pattern_term_off[i],
// pattern_term_off[i + 1]), ascending by bytes.Compare; term j = tb[toff[j] .. toff[j + 1]).
struct TermsOut {
  DevBuf<uint64_t> pattern_term_off;  // [npat + 1]
  DevBuf<uint8_t> tb;
  DevBuf<uint64_t> toff;              // [n_terms + 1]
  DevBuf<uint32_t> segments;          // [n_terms] term instances over the call's segments
  DevBuf<uint64_t> postings;          // [n_terms] sum of their stored list lengths
  DevBuf<uint8_t> distance;           // [n_terms] FUZZY: edit distance, GLOB: 0
  uint64_t n_terms = 0, n_bytes = 0;
};

// The distinct matching terms of every pattern over all segments, with their instance and
// posting counts.  II2_ERR_UNSUPPORTED when the matched term instances or their bytes reach 2^32.
// Synchronises the stream; every buffer (outputs too) comes from the calling thread's scratch
// arena.
int k10_pattern_terms(const PatternDev& d, TermsOut& out, cudaStream_t s);

// One byte of a glob, and of a fuzzy pattern (hb = bit m - 1; global distance, Hyyrö: row 0
// grows by one per byte, hence the 1 shifted into ph).  Host-callable so the compiler's tables
// can be checked on the CPU.
__host__ __device__ __forceinline__ uint64_t glob_step(uint64_t d, uint64_t mask_c, uint64_t loop) {
  return ((d << 1) & mask_c) | (d & loop);
}
__host__ __device__ __forceinline__ void fuzzy_step(uint64_t eq, uint64_t hb, uint64_t& pv,
                                                    uint64_t& mv, int& score) {
  const uint64_t xv = eq | mv;
  const uint64_t xh = (((eq & pv) + pv) ^ pv) | eq;
  uint64_t ph = mv | ~(xh | pv);
  const uint64_t mh = pv & xh;
  if (ph & hb)
    score++;
  else if (mh & hb)
    score--;
  ph = (ph << 1) | 1u;
  pv = (mh << 1) | ~(xv | ph);
  mv = ph & xv;
}

}  // namespace ii2
