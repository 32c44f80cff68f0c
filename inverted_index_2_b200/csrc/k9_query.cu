// k9_query.cu — K9: boolean term queries (ii2_query_dev) over resident segments.
//
// A query is the intersection of its required clauses minus the union of its excluded ones; a
// clause is the union of exact terms and prefixes (atoms).  The pipeline:
//   atoms          every distinct atom of the batch in ONE k5_prefix_search call: a prefix's list
//                  is PrefixSearch's found[p], a term's the sorted-unique union of its values.
//   clause unions  clauses of two or more atoms only, as one more k2_large_run whose sources are
//                  the atoms' lists (a group has at most 1024 sources, the size of the gather's
//                  offset table).  A one-atom clause uses its atom's list as it is.
//   k9_plan        one thread per query: the smallest required clause is the DRIVER, the other
//                  clauses are ordered required by ascending size, then excluded; the driver is
//                  cut into tiles of kTile values.
//   k9_intersect   a grid of a fixed number of CTAs per SM strides over the tiles.  A CTA holds a
//                  tile's 2048 driver values (8 consecutive per thread) with an alive mask, and
//                  for every other clause finds the window of its values inside [first, last] of
//                  the tile.  A window of at most kStage values is staged in shared memory with
//                  16-byte copies, a larger one is searched in global memory; each thread finds
//                  its first candidate by binary search and gallops to the next ones (they are
//                  ascending).  The tile stops as soon as no candidate is alive.  Survivors leave
//                  the removed set and are compacted into the tile's slot.
//   k9_place       tile counts are scanned, a query's offset is the scan at its first tile, and
//                  the tiles are copied back to back.
// Host synchronisations per call: K5's, k2_large_run's when a clause has two or more atoms, and
// one for the output size — none of them depends on the number of queries.
#include <algorithm>
#include <vector>

#include "prefix.cuh"
#include "query.cuh"
#include "runtime.cuh"

namespace ii2 {

namespace {

constexpr uint32_t kTile = 2048;              // driver values per tile
constexpr uint32_t kPer = 8;                  // consecutive candidates per thread
constexpr uint32_t kThreads = kTile / kPer;   // 256
constexpr uint32_t kStage = 8192;             // clause values a CTA stages in shared memory
constexpr unsigned kCtasPerSM = 4;
static_assert(kThreads == 256, "k9_intersect is written for 256 threads");

struct ClauseDesc {
  const uint32_t* v;  // ascending, unique
  uint32_t n;
  uint32_t excluded;
};

struct PlanArgs {
  const uint32_t* qoff;
  const QueryClause* clauses;
  uint32_t nq;
  const uint32_t* avals;     // K5: distinct atom u's list = avals[aoff[u] .. aoff[u+1])
  const uint64_t* aoff;
  const GroupRec* groups;    // clause unions
  ClauseDesc* cl;            // [nclauses]
  uint32_t* order;           // [nclauses] per query: driver first, then the probe order
  uint64_t* tiles;           // [nq + 1] driver tiles (scanned into tile bases afterwards)
  unsigned long long* clause_values;
};

// one thread per query
__global__ void __launch_bounds__(256) k9_plan(const PlanArgs a) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q > a.nq) return;
  if (q == a.nq) {
    a.tiles[q] = 0;
    return;
  }
  const uint32_t c0 = a.qoff[q], c1 = a.qoff[q + 1];
  uint64_t sum = 0;
  for (uint32_t c = c0; c < c1; c++) {
    const QueryClause qc = a.clauses[c];
    ClauseDesc d;
    d.excluded = qc.excluded;
    if (qc.src == kClauseEmpty) {
      d.v = a.avals;
      d.n = 0;
    } else if (qc.src & kClauseGroup) {
      const GroupRec r = a.groups[qc.src & ~kClauseGroup];
      d.v = reinterpret_cast<const uint32_t*>(r.dec);
      d.n = r.cnt;
    } else {
      d.v = a.avals + a.aoff[qc.src];
      d.n = (uint32_t)(a.aoff[qc.src + 1] - a.aoff[qc.src]);
    }
    a.cl[c] = d;
    sum += d.n;
  }
  // rank by (excluded, size, index): the smallest required clause comes first (every query has
  // one), excluded clauses last.  Quadratic in the clauses of ONE query, which are few.
  for (uint32_t c = c0; c < c1; c++) {
    const ClauseDesc d = a.cl[c];
    const uint64_t key = ((uint64_t)d.excluded << 32) | d.n;
    uint32_t rank = 0;
    for (uint32_t o = c0; o < c1; o++) {
      const ClauseDesc e = a.cl[o];
      const uint64_t ko = ((uint64_t)e.excluded << 32) | e.n;
      rank += (ko < key || (ko == key && o < c)) ? 1u : 0u;
    }
    a.order[c0 + rank] = c;
  }
  a.tiles[q] = (a.cl[a.order[c0]].n + (uint64_t)kTile - 1) / kTile;
  if (sum) atomicAdd(a.clause_values, (unsigned long long)sum);
}

// first index in [lo, hi) with v[i] >= x (v ascending)
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* v, uint32_t lo, uint32_t hi,
                                                    uint32_t x) {
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (v[mid] < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// The same from a position known to be at or before the answer: steps of 1, 2, 4, ... then a
// binary search inside the last step.
__device__ __forceinline__ uint32_t gallop_u32(const uint32_t* v, uint32_t pos, uint32_t end,
                                               uint32_t x) {
  if (pos >= end || v[pos] >= x) return pos;
  uint32_t lo = pos, step = 1, hi;  // v[lo] < x
  while (true) {
    const uint32_t nxt = end - lo > step ? lo + step : end;
    if (nxt == end || v[nxt] >= x) {
      hi = nxt;
      break;
    }
    lo = nxt;
    step <<= 1;
  }
  return lower_bound_u32(v, lo + 1, hi, x);
}

// The thread's alive candidates (ascending) against the clause values v[lo, hi): a candidate
// stays alive iff it is found in a required clause / not found in an excluded one.
__device__ __forceinline__ uint32_t probe(const uint32_t* v, uint32_t lo, uint32_t hi,
                                          const uint32_t (&x)[kPer], uint32_t alive,
                                          bool excluded) {
  uint32_t pos = lo, out = alive;
  bool first = true;
#pragma unroll
  for (uint32_t j = 0; j < kPer; j++) {
    if (!((alive >> j) & 1u)) continue;
    pos = first ? lower_bound_u32(v, pos, hi, x[j]) : gallop_u32(v, pos, hi, x[j]);
    first = false;
    const bool hit = pos < hi && v[pos] == x[j];
    if (hit == excluded) out &= ~(1u << j);
  }
  return out;
}

struct K9Args {
  const uint64_t* tile_base;  // [nq + 1]; [nq] = number of tiles
  uint32_t nq;
  const uint32_t* qoff;
  const uint32_t* order;
  const ClauseDesc* cl;
  RemovedSet rem;
  uint32_t* slots;  // tile t's survivors at slots + t * kTile
  uint64_t* tcnt;   // survivors of tile t (zeroed beyond the last tile)
};

__global__ void __launch_bounds__(kThreads) k9_intersect(const K9Args a) {
  __shared__ __align__(16) uint32_t s_win[kStage + 8];
  __shared__ uint32_t s_lohi[2];
  __shared__ uint32_t s_ws[kThreads / 32 + 1];
  const uint64_t ntiles = a.tile_base[a.nq];
  for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    // the query of tile t: the last q with tile_base[q] <= t (a query without tiles shares its
    // base with the next one)
    uint32_t l = 1, h = a.nq;
    while (l < h) {
      const uint32_t m = (l + h) >> 1;
      if (a.tile_base[m] <= t)
        l = m + 1;
      else
        h = m;
    }
    const uint32_t q = l - 1;
    const uint32_t c0 = a.qoff[q], c1 = a.qoff[q + 1];
    const ClauseDesc dr = a.cl[a.order[c0]];
    const uint64_t i0 = (t - a.tile_base[q]) * kTile;
    const uint32_t m = (uint32_t)min((uint64_t)kTile, (uint64_t)dr.n - i0);
    for (uint32_t i = threadIdx.x; i < m; i += kThreads) s_win[i] = dr.v[i0 + i];
    __syncthreads();
    uint32_t x[kPer], alive = 0;
#pragma unroll
    for (uint32_t j = 0; j < kPer; j++) {
      const uint32_t idx = threadIdx.x * kPer + j;
      x[j] = idx < m ? s_win[idx] : 0u;
      alive |= (idx < m ? 1u : 0u) << j;
    }
    const uint32_t first = s_win[0], last = s_win[m - 1];
    for (uint32_t c = c0 + 1; c < c1; c++) {
      const ClauseDesc e = a.cl[a.order[c]];
      if (warp_id() == 0) {
        const uint32_t wlo = warp_partition_point(0u, e.n, [&](uint32_t i) { return e.v[i] < first; });
        const uint32_t whi = warp_partition_point(wlo, e.n, [&](uint32_t i) { return e.v[i] <= last; });
        if (lane_id() == 0) {
          s_lohi[0] = wlo;
          s_lohi[1] = whi;
        }
      }
      __syncthreads();  // (also: every thread has read its candidates out of s_win)
      const uint32_t wlo = s_lohi[0], whi = s_lohi[1];
      if (wlo == whi) {
        if (!e.excluded) alive = 0;  // no value of a required clause lies in the tile's range
      } else if (whi - wlo <= kStage) {
        // aligned 16-byte copies: the allocations are 16-byte aligned and padded by 16 bytes,
        // so the envelope of the window stays inside the clause's buffer
        const uintptr_t p0 = reinterpret_cast<uintptr_t>(e.v + wlo);
        const uint4* src = reinterpret_cast<const uint4*>(p0 & ~(uintptr_t)15);
        const uint32_t shift = (uint32_t)((p0 & 15) >> 2);
        const uint32_t nvec = (shift + (whi - wlo) + 3) >> 2;
        uint4* dst = reinterpret_cast<uint4*>(s_win);
        for (uint32_t i = threadIdx.x; i < nvec; i += kThreads) dst[i] = __ldg(src + i);
        __syncthreads();
        if (alive) alive = probe(s_win, shift, shift + (whi - wlo), x, alive, e.excluded != 0);
      } else if (alive) {
        alive = probe(e.v, wlo, whi, x, alive, e.excluded != 0);
      }
      if (!__syncthreads_or(alive != 0)) break;  // (also: s_win and s_lohi are free again)
    }
    if (alive && a.rem.n) {
#pragma unroll
      for (uint32_t j = 0; j < kPer; j++)
        if (((alive >> j) & 1u) && is_removed(a.rem, x[j])) alive &= ~(1u << j);
    }
    uint32_t tot;
    const uint32_t ex = block_exclusive_scan((uint32_t)__popc(alive), s_ws, tot);
    uint32_t* dst = a.slots + t * kTile + ex;
#pragma unroll
    for (uint32_t j = 0; j < kPer; j++)
      if ((alive >> j) & 1u) *dst++ = x[j];
    if (threadIdx.x == 0) a.tcnt[t] = tot;
  }
}

// the list of distinct atom gatom[j] as source j of the clause unions
__global__ void __launch_bounds__(256)
k9_sources(const uint32_t* __restrict__ gatom, uint32_t nsrc, const uint32_t* avals,
           const uint64_t* __restrict__ aoff, uint64_t* __restrict__ src_ptr,
           uint32_t* __restrict__ src_len) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nsrc) return;
  const uint32_t u = gatom[j];
  src_ptr[j] = reinterpret_cast<uint64_t>(avals + aoff[u]);
  src_len[j] = (uint32_t)(aoff[u + 1] - aoff[u]);
}

// value_off[q] = position of query q's first tile in the scanned tile counts
__global__ void __launch_bounds__(256)
k9_offsets(const uint64_t* __restrict__ tile_base, uint32_t nq, const uint64_t* __restrict__ tpos,
           uint64_t* __restrict__ value_off) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q <= nq) value_off[q] = tpos[tile_base[q]];
}

__global__ void __launch_bounds__(256)
k9_place(const uint64_t* __restrict__ tile_base, uint32_t nq, const uint32_t* __restrict__ slots,
         const uint64_t* __restrict__ tpos, uint32_t* __restrict__ out) {
  const uint64_t ntiles = tile_base[nq];
  for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const uint64_t p = tpos[t], n = tpos[t + 1] - p;
    for (uint32_t i = threadIdx.x; i < n; i += 256) out[p + i] = slots[t * kTile + i];
  }
}

}  // namespace

int k9_query(const QueryDev& d, const QueryHost& h, const RemovedSet& rem, QueryOut& out,
             cudaStream_t s) {
  PrefixOut po;
  II2_TRY(k5_prefix_search(d.segs, d.k, d.abytes, d.aoff, d.nu, po, s, d.akind, h.value_off));
  // clause unions (the sort space stays in the arena until the call ends)
  DevBuf<GroupRec> recs;
  DevBuf<uint32_t> large_tmp, large_enc;
  if (d.ngroups) {
    ProfScope scope("k9_clauses", s);
    DevBuf<uint64_t> src_ptr;
    DevBuf<uint32_t> src_len;
    II2_TRY(src_ptr.alloc_scratch(d.nsrc, s));
    II2_TRY(src_len.alloc_scratch(d.nsrc, s));
    II2_TRY(recs.alloc_scratch(d.ngroups, s));
    k9_sources<<<div_up(d.nsrc, 256), 256, 0, s>>>(d.gatom, d.nsrc, po.values.p, po.value_off.p,
                                                   src_ptr.p, src_len.p);
    II2_LAUNCHED();
    LargeArgs la;
    la.rec = d.grec;
    la.bucket = nullptr;
    la.gin = d.gin;
    la.src_ptr = src_ptr.p;
    la.src_len = src_len.p;
    la.recs = recs.p;
    la.rem = RemovedSet{};
    la.want_enc = 0;
    la.keep_empty = 1;
    la.always_sort = 1;
    la.presorted = nullptr;
    la.bk_raw = nullptr;
    la.nb1 = 0;
    II2_TRY(k2_large_run(la, d.ngroups, large_tmp, large_enc, s));
  }
  // Upper bound of the driver tiles, from the atoms' sizes: a one-atom clause's size is exact, a
  // union's is at most the sum of its atoms'.  Slot t of the output holds tile t's survivors.
  const uint64_t* vo = h.value_off;
  uint64_t tile_bound = 0;
  for (uint32_t q = 0; q < d.nq; q++) {
    uint64_t best = ~0ull;
    for (uint32_t c = h.qoff[q]; c < h.qoff[q + 1]; c++) {
      const QueryClause qc = h.clauses[c];
      if (qc.excluded) continue;
      uint64_t b = 0;
      if (qc.src == kClauseEmpty) {
        b = 0;
      } else if (qc.src & kClauseGroup) {
        const GroupIn& g = h.gin[qc.src & ~kClauseGroup];
        for (uint32_t j = g.src; j < g.src + g.c; j++) b += vo[h.gatom[j] + 1] - vo[h.gatom[j]];
      } else {
        b = vo[qc.src + 1] - vo[qc.src];
      }
      best = std::min(best, b);
    }
    tile_bound += (best + kTile - 1) / kTile;
  }
  DevBuf<ClauseDesc> cl;
  DevBuf<uint32_t> order, slots;
  DevBuf<uint64_t> tiles, tcnt, ctr;
  II2_TRY(cl.alloc_scratch(d.nclauses, s));
  II2_TRY(order.alloc_scratch(d.nclauses, s));
  II2_TRY(tiles.alloc_scratch((size_t)d.nq + 1, s));
  II2_TRY(ctr.alloc_scratch(2, s));  // [0] clause values, [1] output values
  II2_TRY(slots.alloc_scratch(tile_bound * kTile, s));
  II2_TRY(tcnt.alloc_scratch(tile_bound + 1, s));
  II2_CUDA_TRY(cudaMemsetAsync(ctr.p, 0, 16, s));
  II2_CUDA_TRY(cudaMemsetAsync(tcnt.p, 0, (tile_bound + 1) * 8, s));
  {
    ProfScope scope("k9_plan", s);
    PlanArgs pa;
    pa.qoff = d.qoff;
    pa.clauses = d.clauses;
    pa.nq = d.nq;
    pa.avals = po.values.p;
    pa.aoff = po.value_off.p;
    pa.groups = recs.p;
    pa.cl = cl.p;
    pa.order = order.p;
    pa.tiles = tiles.p;
    pa.clause_values = reinterpret_cast<unsigned long long*>(ctr.p);
    k9_plan<<<div_up((uint64_t)d.nq + 1, 256), 256, 0, s>>>(pa);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(tiles.p, (uint64_t)d.nq + 1, nullptr, s));
  }
  if (tile_bound) {
    ProfScope scope("k9_intersect", s);
    K9Args ka;
    ka.tile_base = tiles.p;
    ka.nq = d.nq;
    ka.qoff = d.qoff;
    ka.order = order.p;
    ka.cl = cl.p;
    ka.rem = rem;
    ka.slots = slots.p;
    ka.tcnt = tcnt.p;
    const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kCtasPerSM, tile_bound);
    k9_intersect<<<grid, kThreads, 0, s>>>(ka);
    II2_LAUNCHED();
  }
  ProfScope scope("k9_place", s);
  II2_TRY(out.value_off.alloc_scratch((size_t)d.nq + 1, s));
  II2_TRY(exclusive_scan_u64(tcnt.p, tile_bound + 1, ctr.p + 1, s));
  k9_offsets<<<div_up((uint64_t)d.nq + 1, 256), 256, 0, s>>>(tiles.p, d.nq, tcnt.p, out.value_off.p);
  II2_LAUNCHED();
  uint64_t* hc = pinned_scratch();
  if (!hc) return II2_ERR_NOMEM;
  II2_TRY(small_copy(hc, ctr.p, 16, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  out.clause_values = hc[0];
  out.total = hc[1];
  II2_TRY(out.values.alloc_scratch(out.total, s));
  if (out.total) {
    k9_place<<<(unsigned)std::min<uint64_t>((uint64_t)kNumSMs * 8, tile_bound), 256, 0, s>>>(
        tiles.p, d.nq, slots.p, tcnt.p, out.values.p);
    II2_LAUNCHED();
  }
  return II2_OK;
}

}  // namespace ii2
