// ingest.cuh — K7: documents of a batch -> sorted, de-duplicated direct-mode segments in HBM.
#pragma once
#include <vector>

#include "runtime.cuh"

namespace ii2 {

struct IngestOut {
  // every document's sorted distinct terms back to back; document d = terms [first[d], first[d+1])
  DevBuf<uint8_t> tb;     // term bytes (+ 32 readable pad bytes)
  DevBuf<uint32_t> toff;  // [n_terms + 1] byte offsets into tb
  DevBuf<uint32_t> post;  // [n_terms] the value of the term's document
  DevBuf<uint64_t> poff;  // [n_terms + 1] = 0, 1, 2, ...
  std::vector<uint64_t> first;  // [D + 1], host
  uint64_t n_terms = 0, n_bytes = 0;
};

// d_tb / d_toff[N+1]: all documents' terms as given (any order inside a document), d_doff[D+1] =
// first term of every document (device), h_doff = the same on the host, d_vals[D] = document
// values.  Synchronises the stream; temporaries come from the calling thread's scratch arena.
int k7_ingest_sort(const uint8_t* d_tb, const uint32_t* d_toff, const uint64_t* d_doff,
                   const uint64_t* h_doff, const uint32_t* d_vals, int D, uint64_t N, uint64_t TB,
                   IngestOut& out, cudaStream_t s);

// K7's segmented sort on its own: the N terms d_tb / d_toff[N+1] of D documents (d_doff[D+1] on
// the device, maxL = the longest document) ordered by bytes.Compare inside every document.
// idx[N] receives the term indices in sorted order; keep[N+1] / klen[N+1] = 1 / the term's byte
// length for the first record of every distinct term of a document, 0 elsewhere (unscanned).
// Queues the work on s; temporaries come from the calling thread's scratch arena.
int k7_sort_distinct(const uint8_t* d_tb, const uint32_t* d_toff, const uint64_t* d_doff, int D,
                     uint64_t N, uint64_t maxL, uint32_t* idx, uint64_t* keep, uint64_t* klen,
                     cudaStream_t s);

}  // namespace ii2
