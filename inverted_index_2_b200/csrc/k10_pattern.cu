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
#include <algorithm>
#include <vector>

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
  const uint64_t units = (uint64_t)ng * k;
  DevBuf<uint32_t> ulo, ucnt, matched_u;
  DevBuf<uint64_t> tiles, gt, ebase;
  II2_TRY(ulo.alloc_scratch(units, s));
  II2_TRY(ucnt.alloc_scratch(units, s));
  II2_TRY(tiles.alloc_scratch(units + 1, s));
  II2_TRY(gt.alloc_scratch(ng, s));
  II2_TRY(ebase.alloc_scratch((size_t)ng + 1, s));
  II2_TRY(matched_u.alloc_scratch(nu, s));
  II2_CUDA_TRY(cudaMemsetAsync(matched_u.p, 0, (size_t)nu * 4, s));
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
    wa.ulo = ulo.p;
    wa.ucnt = ucnt.p;
    wa.tiles = tiles.p;
    k10_windows<<<div_up((units + 1) * 32, 256), 256, 0, s>>>(wa);  // a warp per unit
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(tiles.p, units + 1, nullptr, s));
    k10_groups<<<div_up((uint64_t)ng + 1, 256), 256, 0, s>>>(tiles.p, k, d.groups, ng, gt.p, ebase.p);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(ebase.p, (uint64_t)ng + 1, nullptr, s));
    II2_TRY(small_copy(h, tiles.p + units, 8, s));
    II2_TRY(small_copy(h + 1, ebase.p + ng, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
  }
  const uint64_t ntiles = h[0], nent = h[1];
  DevBuf<uint32_t> bits;
  DevBuf<uint64_t> epos;
  II2_TRY(bits.alloc_scratch(nent * kWords, s));
  II2_TRY(epos.alloc_scratch(nent + 1, s));
  II2_CUDA_TRY(cudaMemsetAsync(epos.p + nent, 0, 8, s));
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
    ma.tile_base = tiles.p;
    ma.units = units;
    ma.ulo = ulo.p;
    ma.ucnt = ucnt.p;
    ma.gt = gt.p;
    ma.ebase = ebase.p;
    ma.bits = bits.p;
    ma.epost = epos.p;
    ma.matched = matched_u.p;
    const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)kNumSMs * kMatchCtasPerSM, ntiles);
    k10_match<<<grid, kThreads, kMatchSmem, s>>>(ma);
    II2_LAUNCHED();
  }
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
    II2_TRY(exclusive_scan_u64(epos.p, nent + 1, nullptr, s));
    k10_lengths<<<div_up(ng, 256), 256, 0, s>>>(d.groups, ng, gt.p, ebase.p, epos.p, pstart.p, plen.p);
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
      ga.tile_base = tiles.p;
      ga.units = units;
      ga.ulo = ulo.p;
      ga.gt = gt.p;
      ga.ebase = ebase.p;
      ga.bits = bits.p;
      ga.epos = epos.p;
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
  k10_output<<<div_up(npat, 256), 256, 0, s>>>(d.uid, npat, recs.p, matched_u.p, recs_out.p,
                                               out.matched.p);
  II2_LAUNCHED();
  return place_unions(recs_out.p, npat, out, nullptr, "", "k10_place", nullptr, s);
}

}  // namespace ii2
