// k10_pattern.cu — K10: wildcard and fuzzy term patterns (ii2_pattern_search_dev) over resident
// segments, the counterpart of vellum's fst.Search(automaton, ...).
//
// For every pattern, the result is the sorted-unique union of the values of every term that
// matches it, over all segments, and matched[i] says whether any term instance matched (as
// PrefixSearch, even one with an empty list).  No removed filter (reads never filter, Q2).
//
// A pattern's candidates are the terms that start with its literal prefix (glob) or exact prefix
// (fuzzy): one window of every sorted segment, found like K5's.  A pattern without such a prefix
// must test every term instance: a scan of the term dictionary, byte-parallel and HBM-bound.
// So the host puts the unanchored patterns in groups of kPatGroup that share their windows (whole
// segments) and a CTA runs a staged tile of terms against the whole group: the dictionary is read
// once per group, not once per pattern.  An anchored pattern is a group of its own.
//   k10_windows  one warp per (group, segment): the window and its tiles of <= kTile instances.
//   (scan)       tile bases; k10_groups: per group its tiles and (tile, pattern) entries, scanned.
//   k10_match    a persistent grid over the tiles: stage the group's tables, the tile's term
//                offsets and bytes in shared memory, one thread per term and pattern; a ballot
//                per warp writes the entry's match bitmap, the postings of the matches are summed.
//   (scan)       entries' postings -> every entry's place in one buffer, patterns back to back.
//   k10_gather   one CTA per entry copies the lists of its matching terms to their places.
//   union        k2_large_run, one single-source group per pattern, sorted (always_sort): the
//                bitmap path takes dense wide unions such as `*` by itself.
//   place        K5's tail (place_unions) on the records in output order.
// k10_pattern_terms (ii2_pattern_terms_dev) shares the front half (k10_windows .. k10_match) and
// returns the matching terms instead: entries counted and scanned, every match a record (term
// bytes, list length, distance), each pattern's records sorted by K7's segmented sort, runs of one
// term reduced to (term, instances, postings), placed in output order.
#include <algorithm>
#include <vector>

#include "ingest.cuh"
#include "pattern.cuh"
#include "runtime.cuh"

namespace ii2 {

namespace {

constexpr uint32_t kTile = 2048;             // term instances per tile
constexpr uint32_t kThreads = 256;
constexpr uint32_t kPer = kTile / kThreads;  // terms per thread
constexpr uint32_t kWords = kTile / 32;      // match bitmap words of one (tile, pattern)
constexpr uint32_t kStageBytes = 40960;      // term bytes of a tile staged in shared memory
constexpr unsigned kMatchCtasPerSM = 2;
constexpr unsigned kGatherCtasPerSM = 8;
constexpr size_t kMatchSmem = kPatGroup * sizeof(PatTab) + (kTile + 4) * 4 + kStageBytes + 16;
static_assert(kPer == 8 && kWords == 64, "k10_match / k10_gather index bits by kPer x 8 warps");

struct WinArgs {
  const SegDesc* segs;
  int k;
  const PatGroup* groups;
  uint32_t ng;
  const uint8_t* pre;
  uint32_t* ulo;    // [units] first term of the window of unit (group, segment)
  uint32_t* ucnt;   // [units] its terms
  uint64_t* tiles;  // [units + 1] its tiles, scanned into tile bases afterwards
};

__global__ void __launch_bounds__(256) k10_windows(const WinArgs a) {
  const uint64_t id = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint64_t units = (uint64_t)a.ng * a.k;
  if (id > units) return;  // whole warps leave together
  if (id == units) {
    if (lane_id() == 0) a.tiles[units] = 0;
    return;
  }
  const uint32_t g = (uint32_t)(id / a.k);
  const SegDesc sd = a.segs[id % a.k];
  const PatGroup gr = a.groups[g];
  uint32_t lo = 0, hi = sd.n;
  if (gr.pre_len) {  // uniform inside the warp
    const uint8_t* pb = a.pre + gr.pre_off;
    lo = prefix_window_lo(sd, pb, gr.pre_len);
    hi = prefix_window_hi(sd, lo, pb, gr.pre_len);
  }
  if (lane_id() != 0) return;
  a.ulo[id] = lo;
  a.ucnt[id] = hi - lo;
  a.tiles[id] = ((uint64_t)(hi - lo) + kTile - 1) / kTile;
}

// per group: its tiles gt[g] and entries (tiles x patterns), scanned into entry bases afterwards.
// Entry of tile t (of group g) and the group's pattern j: ebase[g] + j * gt[g] + (t - first tile).
__global__ void __launch_bounds__(256)
k10_groups(const uint64_t* __restrict__ tile_base, int k, const PatGroup* __restrict__ groups,
           uint32_t ng, uint64_t* __restrict__ gt, uint64_t* __restrict__ ebase) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g > ng) return;
  if (g == ng) {
    ebase[ng] = 0;
    return;
  }
  const uint64_t n = tile_base[(uint64_t)(g + 1) * k] - tile_base[(uint64_t)g * k];
  gt[g] = n;
  ebase[g] = n * groups[g].n;
}

// the last i in [lo, hi) with base[i] <= x (base ascending, base[lo] <= x): empty ranges share
// their base with the next one, so this is the non-empty owner
__device__ __forceinline__ uint64_t owner_of(const uint64_t* base, uint64_t lo, uint64_t hi,
                                             uint64_t x) {
  lo++;
  while (lo < hi) {
    const uint64_t m = (lo + hi) >> 1;
    if (base[m] <= x)
      lo = m + 1;
    else
      hi = m;
  }
  return lo - 1;
}

// Bytes [t.skip, n) of the term at byte o of `words` (4-byte words, readable one word past the
// term) against one pattern.  Four bytes per load pair, funnel-shifted to the term's phase.
__device__ __forceinline__ bool match_term(const PatTab& t, const uint32_t* words, uint32_t o,
                                           uint32_t n) {
  if (t.kind == II2_PATTERN_GLOB) {
    uint64_t d = 1ull << t.skip;
    for (uint32_t p = t.skip; p < n && d; p += 4) {
      const uint32_t at = o + p;
      uint32_t w = __funnelshift_r(words[at >> 2], words[(at >> 2) + 1], (at & 3u) * 8u);
      const uint32_t e = min(4u, n - p);
      for (uint32_t b = 0; b < e; b++, w >>= 8) d = glob_step(d, t.mask[w & 0xFFu], t.loop);
    }
    return (d & t.accept) != 0;
  }
  const uint32_t tl = n - t.skip;
  if (tl > t.m + t.k || t.m > tl + t.k) return false;  // the lengths alone differ by more than k
  if (t.m == 0) return true;
  uint64_t pv = ~0ull, mv = 0;
  int score = (int)t.m;
  const uint64_t hb = 1ull << (t.m - 1);
  for (uint32_t p = t.skip; p < n; p += 4) {
    const uint32_t at = o + p;
    uint32_t w = __funnelshift_r(words[at >> 2], words[(at >> 2) + 1], (at & 3u) * 8u);
    const uint32_t e = min(4u, n - p);
    for (uint32_t b = 0; b < e; b++, w >>= 8) fuzzy_step(t.mask[w & 0xFFu], hb, pv, mv, score);
    // the distance falls by at most one per byte left
    if (score - (int)(n - p - e) > (int)t.k) return false;
  }
  return score <= (int)t.k;
}

struct MatchArgs {
  const SegDesc* segs;
  int k;
  const PatTab* tabs;
  const PatGroup* groups;
  const uint64_t* tile_base;  // [units + 1]
  uint64_t units;
  const uint32_t* ulo;
  const uint32_t* ucnt;
  const uint64_t* gt;
  const uint64_t* ebase;
  uint32_t* bits;     // [entries][kWords]: bit i = term lo + i of the tile matches
  uint64_t* epost;    // [entries + 1]: postings of the entry's matches
  uint32_t* matched;  // [nu]
};

__global__ void __launch_bounds__(kThreads) k10_match(const MatchArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  PatTab* s_tab = reinterpret_cast<PatTab*>(smem);
  uint32_t* s_off = reinterpret_cast<uint32_t*>(smem + kPatGroup * sizeof(PatTab));
  uint32_t* s_tb = s_off + kTile + 4;  // 16-byte aligned
  __shared__ unsigned long long s_post[kPatGroup];
  __shared__ uint32_t s_any[kPatGroup];
  const unsigned tid = threadIdx.x, lane = lane_id(), warp = warp_id();
  uint32_t cur = ~0u;  // group whose tables are staged
  const uint64_t ntiles = a.tile_base[a.units];
  for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const uint64_t u = owner_of(a.tile_base, 0, a.units, t);
    const uint32_t g = (uint32_t)(u / a.k);
    const SegDesc sd = a.segs[u % a.k];
    const PatGroup gr = a.groups[g];
    const uint32_t lo = a.ulo[u] + (uint32_t)(t - a.tile_base[u]) * kTile;
    const uint32_t cnt = min(kTile, a.ulo[u] + a.ucnt[u] - lo);
    const uint64_t stride = a.gt[g];
    const uint64_t e0 = a.ebase[g] + (t - a.tile_base[(uint64_t)g * a.k]);
    __syncthreads();  // the previous tile is done with the shared arrays
    if (g != cur) {
      const uint4* src = reinterpret_cast<const uint4*>(a.tabs + gr.p0);
      uint4* dst = reinterpret_cast<uint4*>(s_tab);
      const uint32_t nv = gr.n * (uint32_t)(sizeof(PatTab) / 16);
      for (uint32_t i = tid; i < nv; i += kThreads) dst[i] = __ldg(src + i);
      cur = g;
    }
    // the tile's offsets and, when they fit, its term bytes (16-byte copies of the envelope, one
    // spare word for the funnel shift past the last term; segment buffers are padded by 32 bytes)
    const uint32_t b0 = __ldg(sd.toff + lo), b1 = __ldg(sd.toff + lo + cnt);
    const bool staged =
        (reinterpret_cast<uintptr_t>(sd.tb) & 15u) == 0 && b1 - (b0 & ~15u) + 8 <= kStageBytes;
    const uint32_t base = staged ? (b0 & ~15u) : (b0 & ~3u);
    for (uint32_t i = tid; i <= cnt; i += kThreads) s_off[i] = __ldg(sd.toff + lo + i) - base;
    if (staged) {
      const uint4* src = reinterpret_cast<const uint4*>(sd.tb + base);
      uint4* dst = reinterpret_cast<uint4*>(s_tb);
      const uint32_t nv = (b1 - base + 8 + 15) / 16;
      for (uint32_t i = tid; i < nv; i += kThreads) dst[i] = __ldg(src + i);
    }
    if (tid < kPatGroup) {
      s_post[tid] = 0;
      s_any[tid] = 0;
    }
    __syncthreads();
    const uint32_t* words = staged ? s_tb : reinterpret_cast<const uint32_t*>(sd.tb + base);
#pragma unroll 1
    for (uint32_t j = 0; j < kPer; j++) {
      const uint32_t i = j * kThreads + tid;  // a warp takes 32 consecutive terms
      const bool valid = i < cnt;
      uint32_t o = 0, n = 0;
      if (valid) {
        o = s_off[i];
        n = s_off[i + 1] - o;
      }
      uint64_t len = ~0ull;  // list length, read on the first match
#pragma unroll 1
      for (uint32_t q = 0; q < gr.n; q++) {
        const bool hit = valid && match_term(s_tab[q], words, o, n);
        const uint32_t ball = __ballot_sync(0xffffffffu, hit);
        if (hit && len == ~0ull) len = __ldg(sd.poff + lo + i + 1) - __ldg(sd.poff + lo + i);
        if (lane == 0) a.bits[(e0 + q * stride) * kWords + j * (kThreads / 32) + warp] = ball;
        if (ball) {  // uniform inside the warp
          const uint64_t sum = warp_sum<uint64_t>(hit ? len : 0ull);
          if (lane == 0) {
            atomicAdd(&s_post[q], (unsigned long long)sum);
            s_any[q] = 1;
          }
        }
      }
    }
    __syncthreads();
    if (tid < gr.n) {
      a.epost[e0 + tid * stride] = s_post[tid];
      if (s_any[tid]) atomicOr(&a.matched[gr.p0 + tid], 1u);
    }
  }
}

// internal pattern u: its postings are [pstart[u], pstart[u] + plen[u]) of the scanned entries
__global__ void __launch_bounds__(256)
k10_lengths(const PatGroup* __restrict__ groups, uint32_t ng, const uint64_t* __restrict__ gt,
            const uint64_t* __restrict__ ebase, const uint64_t* __restrict__ epos,
            uint64_t* __restrict__ pstart, uint64_t* __restrict__ plen) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  const PatGroup gr = groups[g];
  for (uint32_t j = 0; j < gr.n; j++) {
    const uint64_t e = ebase[g] + j * gt[g];
    pstart[gr.p0 + j] = epos[e];
    plen[gr.p0 + j] = epos[e + gt[g]] - epos[e];
  }
}

// one single-source union group per internal pattern
__global__ void __launch_bounds__(256)
k10_sources(const uint64_t* __restrict__ pstart, const uint64_t* __restrict__ plen, uint32_t nu,
            const uint32_t* buf, uint64_t* __restrict__ src_ptr, uint32_t* __restrict__ src_len,
            GroupIn* __restrict__ gin, uint32_t* __restrict__ rec) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= nu) return;
  src_ptr[u] = reinterpret_cast<uint64_t>(buf + pstart[u]);
  src_len[u] = (uint32_t)plen[u];  // < 2^32: checked on the host
  GroupIn g;
  g.inst = 0;
  g.tlen = 0;
  g.src = u;
  g.c = 1;
  g.L = 0xFFFFFFFFu;
  g.pst = 0;
  g.eslot = 0;
  g.pad = 0;
  gin[u] = g;
  rec[u] = u;
}

struct GatherArgs {
  const SegDesc* segs;
  int k;
  uint32_t ng;
  const uint64_t* tile_base;
  uint64_t units;
  const uint32_t* ulo;
  const uint64_t* gt;
  const uint64_t* ebase;  // [ng + 1]
  const uint32_t* bits;
  const uint64_t* epos;   // [entries + 1] scanned: first slot of every entry in buf
  uint32_t* buf;
};

// one CTA per entry: the lists of the matching terms, back to back in term order, copied flat
// (every thread finds the term of its slot in the staged prefix of the list lengths)
__global__ void __launch_bounds__(kThreads) k10_gather(const GatherArgs a) {
  __shared__ uint64_t s_src[kTile];  // first posting of the m-th match in the segment
  __shared__ uint64_t s_dst[kTile];  // its first slot relative to the entry
  __shared__ uint32_t s_ws32[kThreads / 32 + 1];
  __shared__ uint64_t s_ws64[kThreads / 32 + 1];
  const unsigned tid = threadIdx.x;
  const uint64_t nent = a.ebase[a.ng];
  for (uint64_t e = blockIdx.x; e < nent; e += gridDim.x) {
    const uint64_t p0 = a.epos[e], total = a.epos[e + 1] - p0;
    if (total == 0) continue;  // uniform inside the CTA
    const uint64_t g = owner_of(a.ebase, 0, a.ng, e);
    const uint64_t t = a.tile_base[g * a.k] + (e - a.ebase[g]) % a.gt[g];
    const uint64_t u = owner_of(a.tile_base, g * a.k, (g + 1) * a.k, t);
    const SegDesc sd = a.segs[u % a.k];
    const uint32_t lo = a.ulo[u] + (uint32_t)(t - a.tile_base[u]) * kTile + tid * kPer;
    const uint32_t m8 = (a.bits[e * kWords + (tid >> 2)] >> ((tid & 3u) * 8u)) & 0xFFu;
    uint64_t start[kPer], len[kPer], sum = 0;
#pragma unroll
    for (uint32_t b = 0; b < kPer; b++) {
      start[b] = len[b] = 0;
      if ((m8 >> b) & 1u) {
        start[b] = __ldg(sd.poff + lo + b);
        len[b] = __ldg(sd.poff + lo + b + 1) - start[b];
        sum += len[b];
      }
    }
    uint32_t nm_tot;
    uint64_t sum_tot;
    uint32_t mi = block_exclusive_scan((uint32_t)__popc(m8), s_ws32, nm_tot);
    uint64_t di = block_exclusive_scan(sum, s_ws64, sum_tot);
#pragma unroll
    for (uint32_t b = 0; b < kPer; b++)
      if ((m8 >> b) & 1u) {
        s_src[mi] = start[b];
        s_dst[mi++] = di;
        di += len[b];
      }
    __syncthreads();
    uint32_t* dst = a.buf + p0;
    for (uint64_t j = tid; j < total; j += kThreads) {
      uint32_t l = 1, h = nm_tot;  // the last match with s_dst <= j
      while (l < h) {
        const uint32_t m = (l + h) >> 1;
        if (s_dst[m] <= j)
          l = m + 1;
        else
          h = m;
      }
      dst[j] = __ldg(sd.post + s_src[l - 1] + (j - s_dst[l - 1]));
    }
    __syncthreads();  // s_src / s_dst are free again
  }
}

// the union records and matched flags in output order (patterns may repeat)
__global__ void __launch_bounds__(256)
k10_output(const uint32_t* __restrict__ uid, uint32_t npat, const GroupRec* __restrict__ recs,
           const uint32_t* __restrict__ matched_u, GroupRec* __restrict__ recs_out,
           uint32_t* __restrict__ matched) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npat) return;
  recs_out[i] = recs[uid[i]];
  matched[i] = matched_u[uid[i]];
}

// The front half of both calls: the windows of every (group, segment) unit, their tiles, the
// (tile, pattern) entries and k10_match's bitmaps.  Synchronises the stream once (the tile and
// entry totals).
struct Front {
  uint64_t units = 0, ntiles = 0, nent = 0;
  DevBuf<uint32_t> ulo, ucnt, matched_u, bits;
  DevBuf<uint64_t> tiles, gt, ebase, epos;
};

int k10_front(const PatternDev& d, Front& f, cudaStream_t s) {
  const uint32_t nu = d.nu, ng = d.ng;
  const int k = d.k;
  const uint64_t units = (uint64_t)ng * k;
  f.units = units;
  II2_TRY(f.ulo.alloc_scratch(units, s));
  II2_TRY(f.ucnt.alloc_scratch(units, s));
  II2_TRY(f.tiles.alloc_scratch(units + 1, s));
  II2_TRY(f.gt.alloc_scratch(ng, s));
  II2_TRY(f.ebase.alloc_scratch((size_t)ng + 1, s));
  II2_TRY(f.matched_u.alloc_scratch(nu, s));
  II2_CUDA_TRY(cudaMemsetAsync(f.matched_u.p, 0, (size_t)nu * 4, s));
  uint64_t* h = pinned_scratch();
  if (!h) return II2_ERR_NOMEM;
  {
    ProfScope scope("k10_windows", s);
    WinArgs wa;
    wa.segs = d.segs;
    wa.k = k;
    wa.groups = d.groups;
    wa.ng = ng;
    wa.pre = d.pre;
    wa.ulo = f.ulo.p;
    wa.ucnt = f.ucnt.p;
    wa.tiles = f.tiles.p;
    k10_windows<<<div_up((units + 1) * 32, 256), 256, 0, s>>>(wa);  // a warp per unit
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(f.tiles.p, units + 1, nullptr, s));
    k10_groups<<<div_up((uint64_t)ng + 1, 256), 256, 0, s>>>(f.tiles.p, k, d.groups, ng, f.gt.p,
                                                             f.ebase.p);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(f.ebase.p, (uint64_t)ng + 1, nullptr, s));
    II2_TRY(small_copy(h, f.tiles.p + units, 8, s));
    II2_TRY(small_copy(h + 1, f.ebase.p + ng, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
  }
  const uint64_t ntiles = h[0], nent = h[1];
  f.ntiles = ntiles;
  f.nent = nent;
  II2_TRY(f.bits.alloc_scratch(nent * kWords, s));
  II2_TRY(f.epos.alloc_scratch(nent + 1, s));
  II2_CUDA_TRY(cudaMemsetAsync(f.epos.p + nent, 0, 8, s));
  if (ntiles) {
    ProfScope scope("k10_match", s);
    // (a per-device attribute: set on every call, the call's device may change)
    II2_CUDA_TRY(cudaFuncSetAttribute(k10_match, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)kMatchSmem));
    MatchArgs ma;
    ma.segs = d.segs;
    ma.k = k;
    ma.tabs = d.tabs;
    ma.groups = d.groups;
    ma.tile_base = f.tiles.p;
    ma.units = units;
    ma.ulo = f.ulo.p;
    ma.ucnt = f.ucnt.p;
    ma.gt = f.gt.p;
    ma.ebase = f.ebase.p;
    ma.bits = f.bits.p;
    ma.epost = f.epos.p;
    ma.matched = f.matched_u.p;
    const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kMatchCtasPerSM, ntiles);
    k10_match<<<grid, kThreads, kMatchSmem, s>>>(ma);
    II2_LAUNCHED();
  }
  return II2_OK;
}


// -------------------------------------------------------- matched terms (k10_pattern_terms)
// entry e -> its group g, tile t (numbered over all units) and unit u, as k10_gather finds them
__device__ __forceinline__ void entry_tile(const uint64_t* ebase, uint32_t ng, const uint64_t* gt,
                                           const uint64_t* tile_base, int k, uint64_t e,
                                           uint64_t& g, uint64_t& t, uint64_t& u) {
  g = owner_of(ebase, 0, ng, e);
  t = tile_base[g * k] + (e - ebase[g]) % gt[g];
  u = owner_of(tile_base, g * k, (g + 1) * k, t);
}

struct TermArgs {
  const SegDesc* segs;
  int k;
  uint32_t ng;
  const PatTab* tabs;
  const PatGroup* groups;
  const uint64_t* tile_base;
  const uint32_t* ulo;
  const uint64_t* gt;
  const uint64_t* ebase;  // [ng + 1]
  const uint32_t* bits;
  uint64_t* ecnt;         // [entries + 1] matches of every entry; scanned: its first record
  uint64_t* ebyt;         // [entries + 1] their term bytes; scanned: the first byte of its records
  // records: one per matching term instance, the entries' matches back to back in term order
  uint8_t* tb;            // term bytes
  uint32_t* toff;         // [n + 1]
  uint64_t* len;          // [n] stored list length
  uint8_t* dist;          // [n] FUZZY: the edit distance, GLOB: 0
  uint64_t n, nbytes;
};

// a warp per entry: the matches of the entry and their term bytes
__global__ void __launch_bounds__(256) k10_term_count(const TermArgs a) {
  const unsigned lane = lane_id();
  const uint64_t nent = a.ebase[a.ng];
  const uint64_t nw = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < nent; e += nw) {
    // word w holds terms 32w .. 32w + 31 of the tile; a lane takes words lane and lane + 32
    const uint32_t m0 = a.bits[e * kWords + lane], m1 = a.bits[e * kWords + 32 + lane];
    uint32_t cnt = 0, bytes = 0;
    if (__any_sync(0xffffffffu, (m0 | m1) != 0)) {
      uint64_t g, t, u;
      entry_tile(a.ebase, a.ng, a.gt, a.tile_base, a.k, e, g, t, u);
      const SegDesc sd = a.segs[u % a.k];
      const uint32_t lo = a.ulo[u] + (uint32_t)(t - a.tile_base[u]) * kTile;
#pragma unroll
      for (uint32_t h = 0; h < 2; h++) {
        uint32_t m = h ? m1 : m0;
        cnt += __popc(m);
        while (m) {
          const uint32_t i = lo + (lane + 32 * h) * 32 + (__ffs(m) - 1);
          m &= m - 1;
          bytes += __ldg(sd.toff + i + 1) - __ldg(sd.toff + i);
        }
      }
    }
    cnt = warp_sum(cnt);
    const uint64_t b = warp_sum<uint64_t>(bytes);
    if (lane == 0) {
      a.ecnt[e] = cnt;
      a.ebyt[e] = b;
    }
  }
}

// byte Levenshtein distance between t[skip..n) and the pattern's q[P..]: the Myers / Hyyrö
// column of match_term run to the end of the term
__device__ __forceinline__ uint32_t fuzzy_distance(const PatTab* t, const uint8_t* term,
                                                   uint32_t n) {
  const uint32_t skip = __ldg(&t->skip), m = __ldg(&t->m);
  if (m == 0) return n - skip;
  uint64_t pv = ~0ull, mv = 0;
  int score = (int)m;
  const uint64_t hb = 1ull << (m - 1);
  for (uint32_t p = skip; p < n; p++)
    fuzzy_step(__ldg(&t->mask[__ldg(term + p)]), hb, pv, mv, score);
  return (uint32_t)score;
}

// one CTA per entry: its matches become records (term bytes, list length, distance), the term
// bytes copied flat (every thread finds the term of its byte in the staged byte offsets)
__global__ void __launch_bounds__(kThreads) k10_term_records(const TermArgs a) {
  __shared__ uint32_t s_src[kTile];  // first byte of the m-th match in the segment
  __shared__ uint32_t s_dst[kTile];  // its first byte relative to the entry's first
  __shared__ uint32_t s_ws[kThreads / 32 + 1];
  __shared__ uint32_t s_wb[kThreads / 32 + 1];
  const unsigned tid = threadIdx.x;
  if (blockIdx.x == 0 && tid == 0) a.toff[a.n] = (uint32_t)a.nbytes;
  const uint64_t nent = a.ebase[a.ng];
  for (uint64_t e = blockIdx.x; e < nent; e += gridDim.x) {
    const uint64_t r0 = a.ecnt[e];
    if (a.ecnt[e + 1] == r0) continue;  // uniform inside the CTA
    uint64_t g, t, u;
    entry_tile(a.ebase, a.ng, a.gt, a.tile_base, a.k, e, g, t, u);
    const SegDesc sd = a.segs[u % a.k];
    const PatTab* tab = a.tabs + a.groups[g].p0 + (e - a.ebase[g]) / a.gt[g];
    const bool fuzzy = __ldg(&tab->kind) == II2_PATTERN_FUZZY;
    const uint32_t lo = a.ulo[u] + (uint32_t)(t - a.tile_base[u]) * kTile + tid * kPer;
    const uint32_t m8 = (a.bits[e * kWords + (tid >> 2)] >> ((tid & 3u) * 8u)) & 0xFFu;
    uint32_t o[kPer], n[kPer], sum = 0;
#pragma unroll
    for (uint32_t b = 0; b < kPer; b++) {
      o[b] = n[b] = 0;
      if ((m8 >> b) & 1u) {
        o[b] = __ldg(sd.toff + lo + b);
        n[b] = __ldg(sd.toff + lo + b + 1) - o[b];
        sum += n[b];
      }
    }
    uint32_t nm_tot, b_tot;
    uint32_t mi = block_exclusive_scan((uint32_t)__popc(m8), s_ws, nm_tot);
    uint32_t di = block_exclusive_scan(sum, s_wb, b_tot);
    const uint32_t b0 = (uint32_t)a.ebyt[e];
#pragma unroll
    for (uint32_t b = 0; b < kPer; b++)
      if ((m8 >> b) & 1u) {
        const uint64_t r = r0 + mi;
        a.toff[r] = b0 + di;
        a.len[r] = __ldg(sd.poff + lo + b + 1) - __ldg(sd.poff + lo + b);
        a.dist[r] = fuzzy ? (uint8_t)fuzzy_distance(tab, sd.tb + o[b], n[b]) : 0;
        s_src[mi] = o[b];
        s_dst[mi++] = di;
        di += n[b];
      }
    __syncthreads();
    uint8_t* dst = a.tb + b0;
    for (uint32_t j = tid; j < b_tot; j += kThreads) {
      uint32_t l = 1, h = nm_tot;  // the last match with s_dst <= j
      while (l < h) {
        const uint32_t m = (l + h) >> 1;
        if (s_dst[m] <= j)
          l = m + 1;
        else
          h = m;
      }
      dst[j] = __ldg(sd.tb + s_src[l - 1] + (j - s_dst[l - 1]));
    }
    __syncthreads();  // s_src / s_dst are free again
  }
}

// internal pattern u: its records are [pdoff[u], pdoff[u + 1]) (the entries of a pattern are
// consecutive, the patterns back to back)
__global__ void __launch_bounds__(256)
k10_term_docs(const PatGroup* __restrict__ groups, uint32_t ng, uint32_t nu,
              const uint64_t* __restrict__ gt, const uint64_t* __restrict__ ebase,
              const uint64_t* __restrict__ ecnt, uint64_t* __restrict__ pdoff) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g > ng) return;
  if (g == ng) {
    pdoff[nu] = ecnt[ebase[ng]];
    return;
  }
  const PatGroup gr = groups[g];
  for (uint32_t j = 0; j < gr.n; j++) pdoff[gr.p0 + j] = ecnt[ebase[g] + j * gt[g]];
}

// slen[p] = list length of the p-th sorted record (slen[n] = 0, scanned afterwards); the first
// sorted record of kept term r: first[r] (first[kept] = n)
__global__ void __launch_bounds__(256)
k10_term_runs(const uint32_t* __restrict__ idx, const uint64_t* __restrict__ len, uint64_t n,
              const uint64_t* __restrict__ pos, uint64_t* __restrict__ slen,
              uint32_t* __restrict__ first) {
  const uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (p > n) return;
  if (p == n) {
    slen[n] = 0;
    first[pos[n]] = (uint32_t)n;
    return;
  }
  slen[p] = len[idx[p]];
  if (pos[p + 1] != pos[p]) first[pos[p]] = (uint32_t)p;
}

// output pattern i (internal uid[i]): its terms and their bytes
__global__ void __launch_bounds__(256)
k10_term_sizes(const uint32_t* __restrict__ uid, uint32_t npat, const uint64_t* __restrict__ pdoff,
               const uint64_t* __restrict__ pos, const uint64_t* __restrict__ boff,
               uint64_t* __restrict__ ocnt, uint64_t* __restrict__ obyt) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > npat) return;
  if (i == npat) {
    ocnt[npat] = obyt[npat] = 0;
    return;
  }
  const uint64_t a = pdoff[uid[i]], b = pdoff[uid[i] + 1];
  ocnt[i] = pos[b] - pos[a];
  obyt[i] = boff[b] - boff[a];
}

struct TermEmit {
  const uint32_t* uid;
  uint32_t npat;
  const uint64_t* pdoff;  // [nu + 1] first record of every internal pattern
  const uint32_t* idx;    // [n] sorted records
  const uint64_t* pos;    // [n + 1] scanned kept flags
  const uint64_t* boff;   // [n + 1] scanned bytes of the kept records
  const uint64_t* slen;   // [n + 1] scanned list lengths in sorted order
  const uint32_t* first;  // [kept + 1]
  const uint8_t* tb;      // records
  const uint32_t* toff;
  const uint8_t* dist;
  const uint64_t* ooff;   // [npat + 1] first output term of every output pattern
  const uint64_t* obyt;   // [npat + 1] its first output byte
  uint64_t nout, nbytes;
  uint8_t* o_tb;
  uint64_t* o_toff;
  uint32_t* o_seg;
  uint64_t* o_post;
  uint8_t* o_dist;
};

// one warp per output term: the kept record of its run, copied into its output pattern's place
__global__ void __launch_bounds__(256) k10_term_emit(const TermEmit e) {
  const uint64_t r = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const unsigned lane = lane_id();
  if (r > e.nout) return;
  if (r == e.nout) {
    if (lane == 0) e.o_toff[r] = e.nbytes;
    return;
  }
  const uint64_t i = owner_of(e.ooff, 0, e.npat, r);
  const uint64_t d0 = e.pdoff[e.uid[i]];
  const uint64_t kr = e.pos[d0] + (r - e.ooff[i]);
  const uint32_t p = e.first[kr], pn = e.first[kr + 1];
  const uint32_t j = e.idx[p];
  const uint32_t o = e.toff[j], n = e.toff[j + 1] - o;
  const uint64_t dst = e.obyt[i] + (e.boff[p] - e.boff[d0]);
  for (uint32_t q = lane; q < n; q += 32) e.o_tb[dst + q] = e.tb[o + q];
  if (lane == 0) {
    e.o_toff[r] = dst;
    e.o_seg[r] = pn - p;
    e.o_post[r] = e.slen[pn] - e.slen[p];
    e.o_dist[r] = e.dist[j];
  }
}

}  // namespace

int k10_pattern_search(const PatternDev& d, PrefixOut& out, cudaStream_t s) {
  const uint32_t npat = d.npat, nu = d.nu, ng = d.ng;
  const int k = d.k;
  out.total = 0;
  II2_TRY(out.value_off.alloc((size_t)npat + 1, s));
  II2_TRY(out.matched.alloc(npat ? npat : 1, s));
  if (npat == 0 || k == 0) {
    II2_CUDA_TRY(cudaMemsetAsync(out.value_off.p, 0, ((size_t)npat + 1) * 8, s));
    II2_CUDA_TRY(cudaMemsetAsync(out.matched.p, 0, (npat ? npat : 1) * 4, s));
    II2_TRY(out.values.alloc(0, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    return II2_OK;
  }
  Front f;
  II2_TRY(k10_front(d, f, s));
  const uint64_t units = f.units, nent = f.nent;
  // every entry's first slot; every pattern's postings (the entries of a pattern are consecutive,
  // the patterns back to back)
  DevBuf<uint64_t> pstart, plen;
  DevBuf<uint32_t> buf;
  PinnedBlock h_len((size_t)nu * 8);
  if (!h_len.p) return II2_ERR_NOMEM;
  uint64_t* hl = static_cast<uint64_t*>(h_len.p);
  {
    ProfScope scope("k10_gather", s);
    II2_TRY(pstart.alloc_scratch(nu, s));
    II2_TRY(plen.alloc_scratch(nu, s));
    II2_TRY(exclusive_scan_u64(f.epos.p, nent + 1, nullptr, s));
    k10_lengths<<<div_up(ng, 256), 256, 0, s>>>(d.groups, ng, f.gt.p, f.ebase.p, f.epos.p, pstart.p,
                                                 plen.p);
    II2_LAUNCHED();
    II2_CUDA_TRY(cudaMemcpyAsync(hl, plen.p, (size_t)nu * 8, cudaMemcpyDeviceToHost, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    uint64_t total = 0;
    for (uint32_t u = 0; u < nu; u++) {
      if (hl[u] >= (1ull << 32)) {
        set_last_error("pattern search: a pattern matches %llu postings (max 2^32-1)",
                       (unsigned long long)hl[u]);
        return II2_ERR_UNSUPPORTED;
      }
      total += hl[u];
    }
    II2_TRY(buf.alloc_scratch(total, s));
    if (total) {
      GatherArgs ga;
      ga.segs = d.segs;
      ga.k = k;
      ga.ng = ng;
      ga.tile_base = f.tiles.p;
      ga.units = units;
      ga.ulo = f.ulo.p;
      ga.gt = f.gt.p;
      ga.ebase = f.ebase.p;
      ga.bits = f.bits.p;
      ga.epos = f.epos.p;
      ga.buf = buf.p;
      const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kGatherCtasPerSM, nent);
      k10_gather<<<grid, kThreads, 0, s>>>(ga);
      II2_LAUNCHED();
    }
  }
  DevBuf<uint64_t> src_ptr;
  DevBuf<uint32_t> src_len, rec;
  DevBuf<GroupIn> gin;
  DevBuf<GroupRec> recs, recs_out;
  II2_TRY(src_ptr.alloc_scratch(nu, s));
  II2_TRY(src_len.alloc_scratch(nu, s));
  II2_TRY(rec.alloc_scratch(nu, s));
  II2_TRY(gin.alloc_scratch(nu, s));
  II2_TRY(recs.alloc_scratch(nu, s));
  II2_TRY(recs_out.alloc_scratch(npat, s));
  k10_sources<<<div_up(nu, 256), 256, 0, s>>>(pstart.p, plen.p, nu, buf.p, src_ptr.p, src_len.p,
                                              gin.p, rec.p);
  II2_LAUNCHED();
  LargeArgs la;
  la.rec = rec.p;
  la.bucket = nullptr;
  la.gin = gin.p;
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
  DevBuf<uint32_t> tmp, enc;
  {
    ProfScope scope("k10_union", s);
    II2_TRY(k2_large_run(la, nu, tmp, enc, s));
  }
  k10_output<<<div_up(npat, 256), 256, 0, s>>>(d.uid, npat, recs.p, f.matched_u.p, recs_out.p,
                                               out.matched.p);
  II2_LAUNCHED();
  return place_unions(recs_out.p, npat, out, nullptr, "", "k10_place", nullptr, s);
}

int k10_pattern_terms(const PatternDev& d, TermsOut& out, cudaStream_t s) {
  const uint32_t npat = d.npat, nu = d.nu, ng = d.ng;
  const int k = d.k;
  out.n_terms = out.n_bytes = 0;
  II2_TRY(out.pattern_term_off.alloc_scratch((size_t)npat + 1, s));
  if (npat == 0 || k == 0) {
    II2_CUDA_TRY(cudaMemsetAsync(out.pattern_term_off.p, 0, ((size_t)npat + 1) * 8, s));
    II2_TRY(out.toff.alloc_scratch(1, s));
    II2_CUDA_TRY(cudaMemsetAsync(out.toff.p, 0, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    return II2_OK;
  }
  Front f;
  II2_TRY(k10_front(d, f, s));
  const uint64_t nent = f.nent;
  // every entry's matches and bytes, scanned: every internal pattern's records are contiguous
  DevBuf<uint64_t> ecnt, ebyt, pdoff;
  II2_TRY(ecnt.alloc_scratch(nent + 1, s));
  II2_TRY(ebyt.alloc_scratch(nent + 1, s));
  II2_TRY(pdoff.alloc_scratch((size_t)nu + 1, s));
  PinnedBlock h_blk(((size_t)nu + 2) * 8);
  if (!h_blk.p) return II2_ERR_NOMEM;
  uint64_t* h_doff = static_cast<uint64_t*>(h_blk.p);  // [nu + 1], then the byte total
  TermArgs ta;
  ta.segs = d.segs;
  ta.k = k;
  ta.ng = ng;
  ta.tabs = d.tabs;
  ta.groups = d.groups;
  ta.tile_base = f.tiles.p;
  ta.ulo = f.ulo.p;
  ta.gt = f.gt.p;
  ta.ebase = f.ebase.p;
  ta.bits = f.bits.p;
  ta.ecnt = ecnt.p;
  ta.ebyt = ebyt.p;
  {
    ProfScope scope("k10_term_count", s);
    II2_CUDA_TRY(cudaMemsetAsync(ecnt.p + nent, 0, 8, s));
    II2_CUDA_TRY(cudaMemsetAsync(ebyt.p + nent, 0, 8, s));
    if (nent) {
      const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kGatherCtasPerSM,
                                                         div_up(nent, 8));
      k10_term_count<<<grid, 256, 0, s>>>(ta);  // a warp per entry
      II2_LAUNCHED();
    }
    II2_TRY(exclusive_scan_u64(ecnt.p, nent + 1, nullptr, s));
    II2_TRY(exclusive_scan_u64(ebyt.p, nent + 1, nullptr, s));
    k10_term_docs<<<div_up((uint64_t)ng + 1, 256), 256, 0, s>>>(d.groups, ng, nu, f.gt.p, f.ebase.p,
                                                                ecnt.p, pdoff.p);
    II2_LAUNCHED();
    II2_CUDA_TRY(cudaMemcpyAsync(h_doff, pdoff.p, ((size_t)nu + 1) * 8, cudaMemcpyDeviceToHost, s));
    II2_CUDA_TRY(cudaMemcpyAsync(h_doff + nu + 1, ebyt.p + nent, 8, cudaMemcpyDeviceToHost, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
  }
  const uint64_t n = h_doff[nu], nbytes = h_doff[nu + 1];
  if (n >= (1ull << 32) || nbytes >= (1ull << 32)) {
    set_last_error("pattern terms: %llu matched term instances of %llu bytes (max 2^32-1 each)",
                   (unsigned long long)n, (unsigned long long)nbytes);
    return II2_ERR_UNSUPPORTED;
  }
  uint64_t maxL = 0;
  for (uint32_t u = 0; u < nu; u++) maxL = std::max(maxL, h_doff[u + 1] - h_doff[u]);
  DevBuf<uint8_t> rtb, rdist;
  DevBuf<uint32_t> rtoff, idx, first;
  DevBuf<uint64_t> rlen, pos, boff, slen;
  II2_TRY(rtb.alloc_scratch(nbytes, s, 32));
  II2_TRY(rtoff.alloc_scratch(n + 1, s));
  II2_TRY(rlen.alloc_scratch(n, s));
  II2_TRY(rdist.alloc_scratch(n, s));
  if (n) {
    ProfScope scope("k10_term_records", s);
    ta.tb = rtb.p;
    ta.toff = rtoff.p;
    ta.len = rlen.p;
    ta.dist = rdist.p;
    ta.n = n;
    ta.nbytes = nbytes;
    const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kGatherCtasPerSM, nent);
    k10_term_records<<<grid, kThreads, 0, s>>>(ta);
    II2_LAUNCHED();
  }
  // each internal pattern's records by bytes.Compare (K7's sort, a pattern per document); the
  // first record of every distinct term is kept
  II2_TRY(idx.alloc_scratch(n, s));
  II2_TRY(pos.alloc_scratch(n + 1, s));
  II2_TRY(boff.alloc_scratch(n + 1, s));
  II2_TRY(slen.alloc_scratch(n + 1, s));
  II2_TRY(first.alloc_scratch(n + 1, s));
  II2_TRY(k7_sort_distinct(rtb.p, rtoff.p, pdoff.p, (int)nu, n, maxL, idx.p, pos.p, boff.p, s));
  // output pattern i: terms [ooff[i], ooff[i + 1]), their bytes from obase[i]
  DevBuf<uint64_t>& ooff = out.pattern_term_off;
  DevBuf<uint64_t> obase;
  II2_TRY(obase.alloc_scratch((size_t)npat + 1, s));
  uint64_t* h = pinned_scratch();
  if (!h) return II2_ERR_NOMEM;
  {
    ProfScope scope("k10_term_reduce", s);
    II2_TRY(exclusive_scan_u64(pos.p, n + 1, nullptr, s));
    II2_TRY(exclusive_scan_u64(boff.p, n + 1, nullptr, s));
    k10_term_runs<<<div_up(n + 1, 256), 256, 0, s>>>(idx.p, rlen.p, n, pos.p, slen.p, first.p);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(slen.p, n + 1, nullptr, s));
    k10_term_sizes<<<div_up((uint64_t)npat + 1, 256), 256, 0, s>>>(d.uid, npat, pdoff.p, pos.p,
                                                                   boff.p, ooff.p, obase.p);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(ooff.p, (uint64_t)npat + 1, nullptr, s));
    II2_TRY(exclusive_scan_u64(obase.p, (uint64_t)npat + 1, nullptr, s));
    II2_TRY(small_copy(h, ooff.p + npat, 8, s));
    II2_TRY(small_copy(h + 1, obase.p + npat, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
  }
  const uint64_t nout = h[0], obytes = h[1];
  out.n_terms = nout;
  out.n_bytes = obytes;
  II2_TRY(out.tb.alloc_scratch(obytes, s));
  II2_TRY(out.toff.alloc_scratch(nout + 1, s));
  II2_TRY(out.segments.alloc_scratch(nout, s));
  II2_TRY(out.postings.alloc_scratch(nout, s));
  II2_TRY(out.distance.alloc_scratch(nout, s));
  ProfScope scope("k10_term_emit", s);
  TermEmit te;
  te.uid = d.uid;
  te.npat = npat;
  te.pdoff = pdoff.p;
  te.idx = idx.p;
  te.pos = pos.p;
  te.boff = boff.p;
  te.slen = slen.p;
  te.first = first.p;
  te.tb = rtb.p;
  te.toff = rtoff.p;
  te.dist = rdist.p;
  te.ooff = ooff.p;
  te.obyt = obase.p;
  te.nout = nout;
  te.nbytes = obytes;
  te.o_tb = out.tb.p;
  te.o_toff = out.toff.p;
  te.o_seg = out.segments.p;
  te.o_post = out.postings.p;
  te.o_dist = out.distance.p;
  k10_term_emit<<<div_up((nout + 1) * 32, 256), 256, 0, s>>>(te);  // a warp per output term
  II2_LAUNCHED();
  return II2_OK;
}

}  // namespace ii2
