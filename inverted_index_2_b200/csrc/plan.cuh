// plan.cuh — the bucket plan handed from K1 (splitter selection + partition of every segment's
// term dictionary) to K12 (fused term merge + posting union) and the emit kernel.
//
// Vocabulary
//   instance  one (segment, term) pair inside the call's windows; global instance id
//             g = segs[s].base + (idx - segs[s].lo); N_T instances in total.
//   sample    an evenly spaced term of one segment; all samples, ordered by (term, segment),
//             are the splitters.
//   bucket    all instances whose term lies in [splitter_{b-1}, splitter_b): a contiguous index
//             range in EVERY segment (rows of `part`), so no term straddles two buckets and
//             buckets are in ascending term order.  One K12 CTA owns one bucket.
#pragma once
#include "runtime.cuh"

namespace ii2 {

struct MergePlan {
  int k = 0;                      // segments
  uint32_t n_total = 0;           // N_T
  uint32_t n_samples = 0;         // S
  uint32_t n_buckets = 0;         // B = S + 1
  const SegDesc* segs = nullptr;  // [k] device, windows filled in
  // rows of k lower bounds: row 0 = window starts, row r+1 = lower_bound of splitter r (sorted)
  // in every segment, row S+1 = window ends; bucket b spans rows b .. b+1
  DevBuf<uint32_t> part;          // [(S+2) * k]
  // the same boundaries in the other arrays of the segments: toff[part[..]] and poff[part[..]]
  // (first term byte / first posting of the run that starts there)
  DevBuf<uint32_t> btb;           // [(S+2) * k]
  DevBuf<uint64_t> bpo;           // [(S+2) * k]
  DevBuf<uint32_t> bk_cpl;        // [B]   common prefix length of all terms in the bucket
  // [4][B+1] exclusive prefixes: instances / input postings / `_val` staging words (upper
  // bound) / term bytes of all instances (upper bound of the merged term bytes)
  DevBuf<uint64_t> bk_WP;
  const uint64_t* bk_pos() const { return bk_WP.p; }
  const uint64_t* bk_P() const { return bk_WP.p + (n_buckets + 1); }
  const uint64_t* bk_E() const { return bk_WP.p + 2 * (size_t)(n_buckets + 1); }
  const uint64_t* bk_TB() const { return bk_WP.p + 3 * (size_t)(n_buckets + 1); }
  DevBuf<uint64_t> totals;        // [4] {Σ instances, Σ postings in, Σ staging words, Σ term bytes}
};

// K1: choose splitters and partition every segment (the k-way merge of the term dictionaries,
// go-iterators MergingIterator built at shard.go:267 with file.CompareTermValues, is finished
// per bucket inside K12).  plan.k / n_total / segs must be set; h_segs = host copy of segs
// (windows), used to spread the samples; sbase = 2(k+1) words of PINNED host scratch that stay
// valid until the stream has drained (the call does not synchronise).
int k1_build_plan(MergePlan& plan, const SegDesc* h_segs, uint32_t* sbase, cudaStream_t s);

}  // namespace ii2
