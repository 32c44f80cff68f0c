// query.cuh — K9: boolean term queries over resident segments (ii2_query_dev): per query the
// intersection of its required clauses minus its excluded ones, a clause being the union of
// exact terms and prefixes.
#pragma once
#include "union.cuh"

namespace ii2 {

// Where clause c's values come from: a distinct atom's list (K5), a clause union (k2_large_run
// group g: kClauseGroup | g), or nothing (a clause without atoms).
constexpr uint32_t kClauseGroup = 0x80000000u;
constexpr uint32_t kClauseEmpty = 0xFFFFFFFFu;
struct QueryClause {
  uint32_t src;
  uint32_t excluded;  // 0 = required, 1 = excluded
};

// A validated batch whose atoms are deduplicated, staged on the device by the caller.
struct QueryDev {
  const SegDesc* segs;
  int k;                          // 1 <= k <= kMaxSegs
  const uint8_t* abytes;          // distinct atom u = abytes[aoff[u] .. aoff[u+1])
  const uint32_t* aoff;           // [nu + 1]
  const uint8_t* akind;           // [nu] II2_ATOM_*
  uint32_t nu;                    // >= 1
  const QueryClause* clauses;     // [nclauses]
  uint32_t nclauses;
  const uint32_t* qoff;           // [nq + 1] clauses of query q = [qoff[q], qoff[q+1])
  uint32_t nq;                    // >= 1
  // clause unions (clauses of two or more atoms): group g unions the distinct atoms
  // gatom[gin[g].src .. gin[g].src + gin[g].c), c <= kMaxSegs
  const GroupIn* gin;             // [ngroups]
  const uint32_t* grec;           // [ngroups] identity
  const uint32_t* gatom;          // [nsrc]
  uint32_t ngroups, nsrc;
};

// Host copies of the same arrays (the output bound is computed from them).
struct QueryHost {
  const QueryClause* clauses;
  const uint32_t* qoff;
  const GroupIn* gin;
  const uint32_t* gatom;
  uint64_t* value_off;  // pinned [nu + 1]: receives the atoms' list offsets
};

struct QueryOut {
  DevBuf<uint32_t> values;     // the results back to back, each ascending and unique
  DevBuf<uint64_t> value_off;  // [nq + 1]
  uint64_t total = 0;
  uint64_t clause_values = 0;  // Σ sizes of the clause unions
};

// Atom lists (K5), clause unions (k2_large_run), then K9 plan / intersect / place.  rem: values
// to drop from every result (rem.n == 0: none).  Synchronises the stream; the results are
// complete when it returns with the stream's work done (the caller downloads them).
int k9_query(const QueryDev& d, const QueryHost& h, const RemovedSet& rem, QueryOut& out,
             cudaStream_t s);

}  // namespace ii2
