// k5_prefix.cu — K5: InvertedIndex.PrefixSearch (inverted_index.go:192-295) on resident segments.
//
// The reference walks every candidate shard from the smallest prefix to the end of the greatest
// one, tests every term against every prefix (bytes.HasPrefix, :274-279), appends the term's
// values to found[prefix] and finally sorts + compacts every list (:289-292).  The shard
// selection by min/max (:211-236) and the early stop (:266-271) only skip terms that cannot
// match, so the result is, for every prefix p:
//     found[p] = sorted-unique union of the values of ALL terms t with HasPrefix(t, p),
// and p is a key of the map iff at least one term matched (even one with an empty list).
// No removed filter on this path (reads never filter, shard.go:72-75, survey Q2).
//
// B200 shape: terms with prefix p are one contiguous window of every sorted segment, so their
// postings are one contiguous slice of the segment's posting array.  k5_windows finds the
// window of every (prefix, segment) pair with two binary searches; the union of a prefix is
// then exactly the "heavy term" union of k12_union.cu (multi-CTA gather, tile sort, global
// bitonic stages, dedup) over those slices, with sorting forced for single-source groups;
// k5_place copies the unions back to back.  Integer/byte work, HBM-bound.
#include <algorithm>

#include "keys.cuh"
#include "prefix.cuh"

namespace ii2 {

namespace {

struct K5Args {
  const SegDesc* segs;
  int k;
  const uint8_t* pbytes;
  const uint32_t* poff;  // [np + 1]
  const uint8_t* kind;   // [np] II2_ATOM_*, or null: every item is a prefix
  uint32_t np;
  uint64_t* src_ptr;   // [np * k]
  uint32_t* src_len;   // [np * k]
  GroupIn* gin;        // [np]
  uint32_t* rec;       // [np] identity
  uint32_t* matched;   // [np] zeroed
  uint32_t* flags;     // [0] = a slice longer than 2^32-1 postings
};

// One WARP per (prefix, segment): the window of the prefix (prefix_window_lo / _hi).  An exact
// TERM item's window is [lo, lo + (term lo == p)).
__global__ void __launch_bounds__(256) k5_windows(const K5Args a) {
  const uint64_t id = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (id >= (uint64_t)a.np * a.k) return;  // whole warps leave together
  const uint32_t p = (uint32_t)(id / a.k);
  const int s = (int)(id % a.k);
  const SegDesc sd = a.segs[s];
  const uint8_t* pb = a.pbytes + a.poff[p];
  const uint32_t pn = a.poff[p + 1] - a.poff[p];
  const uint32_t lo = prefix_window_lo(sd, pb, pn);
  uint32_t hi;
  if (a.kind && a.kind[p] == II2_ATOM_TERM) {  // uniform inside the warp
    uint32_t eq = 0;
    if (lo < sd.n) {
      const uint32_t o = __ldg(sd.toff + lo), n = __ldg(sd.toff + lo + 1) - o;
      eq = term_compare(sd.tb + o, n, pb, pn) == 0;
    }
    hi = lo + eq;
  } else {
    hi = prefix_window_hi(sd, lo, pb, pn);
  }
  if (lane_id() != 0) return;
  const uint64_t p0 = sd.poff[lo], p1 = sd.poff[hi];
  uint64_t len = p1 - p0;
  if (len > 0xFFFFFFFFull) {
    atomicExch(&a.flags[0], 1u);
    len = 0;
  }
  a.src_ptr[id] = reinterpret_cast<uint64_t>(sd.post + p0);
  a.src_len[id] = (uint32_t)len;
  if (hi > lo) atomicOr(&a.matched[p], 1u);
  if (s == 0) {
    GroupIn g;
    g.inst = 0;
    g.tlen = 0;
    g.src = (uint32_t)(id);
    g.c = (uint32_t)a.k;
    g.L = 0xFFFFFFFFu;
    g.pst = 0;
    g.eslot = 0;
    g.pad = 0;
    a.gin[p] = g;
    a.rec[p] = p;
  }
}

__global__ void __launch_bounds__(256)
k5_counts(const GroupRec* __restrict__ recs, uint32_t np, uint64_t* __restrict__ cnt) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < np) cnt[p] = recs[p].cnt;
  if (p == np) cnt[np] = 0;
}

// grid (x = CTAs per prefix, y = prefix): copy the union of prefix y to its place
__global__ void __launch_bounds__(256)
k5_place(const GroupRec* __restrict__ recs, const uint64_t* __restrict__ off,
         uint32_t* __restrict__ out) {
  const GroupRec r = recs[blockIdx.y];
  const uint32_t* src = reinterpret_cast<const uint32_t*>(r.dec);
  uint32_t* dst = out + off[blockIdx.y];
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < r.cnt; i += (uint64_t)gridDim.x * 256)
    dst[i] = src[i];
}

}  // namespace

int k5_prefix_search(const SegDesc* d_segs, int k, const uint8_t* d_pbytes, const uint32_t* d_poff,
                     uint32_t np, PrefixOut& out, cudaStream_t s, const uint8_t* d_kind,
                     uint64_t* h_value_off) {
  out.total = 0;
  II2_TRY(out.value_off.alloc((size_t)np + 1, s));
  II2_TRY(out.matched.alloc(np ? np : 1, s));
  if (np == 0 || k == 0) {
    II2_CUDA_TRY(cudaMemsetAsync(out.value_off.p, 0, ((size_t)np + 1) * 8, s));
    II2_CUDA_TRY(cudaMemsetAsync(out.matched.p, 0, (np ? np : 1) * 4, s));
    II2_TRY(out.values.alloc(0, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    if (h_value_off) memset(h_value_off, 0, ((size_t)np + 1) * 8);
    return II2_OK;
  }
  const uint64_t pairs = (uint64_t)np * k;
  if (pairs >= (1ull << 32)) {
    set_last_error("prefix search: %u prefixes x %d segments exceed 2^32 pairs", np, k);
    return II2_ERR_UNSUPPORTED;
  }
  DevBuf<uint64_t> src_ptr;
  DevBuf<uint32_t> src_len, rec, flags;
  DevBuf<GroupIn> gin;
  DevBuf<GroupRec> recs;
  II2_TRY(src_ptr.alloc_scratch(pairs, s));
  II2_TRY(src_len.alloc_scratch(pairs, s));
  II2_TRY(rec.alloc_scratch(np, s));
  II2_TRY(flags.alloc_scratch(2, s));
  II2_TRY(gin.alloc_scratch(np, s));
  II2_TRY(recs.alloc_scratch(np, s));
  II2_CUDA_TRY(cudaMemsetAsync(out.matched.p, 0, (size_t)np * 4, s));
  II2_CUDA_TRY(cudaMemsetAsync(flags.p, 0, 8, s));
  K5Args a;
  a.segs = d_segs;
  a.k = k;
  a.pbytes = d_pbytes;
  a.poff = d_poff;
  a.kind = d_kind;
  a.np = np;
  a.src_ptr = src_ptr.p;
  a.src_len = src_len.p;
  a.gin = gin.p;
  a.rec = rec.p;
  a.matched = out.matched.p;
  a.flags = flags.p;
  {
    ProfScope scope("k5_windows", s);
    k5_windows<<<div_up(pairs, 8), 256, 0, s>>>(a);  // a warp per pair
    II2_LAUNCHED();
  }
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
    ProfScope scope("k5_union", s);
    II2_TRY(k2_large_run(la, np, tmp, enc, s));
  }
  return place_unions(recs.p, np, out, flags.p,
                      "prefix search: one segment holds more than 2^32-1 postings under a prefix",
                      "k5_place", h_value_off, s);
}

int place_unions(const GroupRec* recs, uint32_t np, PrefixOut& out, const uint32_t* d_flag,
                 const char* flag_msg, const char* place_name, uint64_t* h_value_off,
                 cudaStream_t s) {
  uint64_t* h = pinned_scratch();
  if (!h) return II2_ERR_NOMEM;
  DevBuf<uint64_t> d_tot;
  II2_TRY(d_tot.alloc_scratch(1, s));
  k5_counts<<<div_up((uint64_t)np + 1, 256), 256, 0, s>>>(recs, np, out.value_off.p);
  II2_LAUNCHED();
  II2_TRY(exclusive_scan_u64(out.value_off.p, (uint64_t)np + 1, d_tot.p, s));
  II2_TRY(small_copy(h, d_tot.p, 8, s));
  h[1] = 0;
  if (d_flag) II2_TRY(small_copy(h + 1, d_flag, 8, s));
  if (h_value_off)
    II2_CUDA_TRY(cudaMemcpyAsync(h_value_off, out.value_off.p, ((size_t)np + 1) * 8,
                                 cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  if ((uint32_t)h[1]) {
    set_last_error("%s", flag_msg);
    return II2_ERR_UNSUPPORTED;
  }
  out.total = h[0];
  II2_TRY(out.values.alloc((size_t)out.total, s));
  if (out.total) {
    ProfScope scope(place_name, s);
    const unsigned gx = (unsigned)std::max<uint64_t>(
        1, std::min<uint64_t>(1024, (out.total / np + 2047) / 2048));
    for (uint32_t y0 = 0; y0 < np; y0 += 32768) {
      const uint32_t ny = std::min<uint32_t>(32768, np - y0);
      k5_place<<<dim3(gx, ny), 256, 0, s>>>(recs + y0, out.value_off.p + y0, out.values.p);
      II2_LAUNCHED();
    }
  }
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  return II2_OK;
}

}  // namespace ii2
