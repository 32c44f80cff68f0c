// k1_plan.cu — K1: splitters for the k-way merge of the sorted term dictionaries.
//
// Replaces the head selection of go-iterators' MergingIterator over per-segment readers
// (shard.go:253-278, ordering = file.CompareTermValues = bytes.Compare, file/types.go:24-26)
// by a merge-path style partition of the OUTPUT term space:
//
//   k1_sample_keys     every segment contributes evenly spaced sample terms in proportion to
//                      its size (about one per 640 instances overall); 16-byte key windows.
//   k1_rank_samples    one warp per sample x, lanes over segments: binary search among every
//                      segment's samples -> how many are smaller -> the rank of x in the merged
//                      sample order is the sum over segments (a k-way merge by ranking, no
//                      sort).  Sorted splitter arrays by scatter.
//   k1_partition_chunks_raw  merge-path partition: one CTA per 1024-term chunk of one segment
//                      stages the chunk's offsets and term bytes in shared memory (coalesced,
//                      every term byte read once) and locates the splitters that fall inside
//                      it.  Row r+1 of `part` = lower_bound of splitter r in every segment;
//                      `btb` / `bpo` = the term-byte and posting offsets at that boundary, so
//                      that a bucket's four runs per segment (term offsets, posting offsets,
//                      term bytes, postings) are known without touching the offset arrays.
//   k1_bucket_stats    per bucket: instances, input postings, term bytes (all from the
//                      boundary tables), common prefix length; then one scan -> bucket bases.
//
// Integer/byte work; every probe is an L2 hit after the first touch (samples and offsets of
// 64 segments are a few MB).
#include <algorithm>
#include <cstdlib>

#include "keys.cuh"
#include "plan.cuh"

namespace ii2 {

constexpr uint32_t kInstancesPerBucket = 768;  // target; K1b tiles hold 1024
constexpr uint32_t kMaxBuckets = 1u << 20;

struct SampleArrays {
  uint64_t* hi;
  uint64_t* lo;
  uint64_t* ptr;   // first byte of the sample term
  uint32_t* len;
  uint32_t* idx;   // term index inside its segment
  uint32_t* seg;
};

__global__ void __launch_bounds__(256)
k1_sample_keys(const SegDesc* __restrict__ segs, int k, const uint32_t* __restrict__ sbase,
               uint32_t S, SampleArrays sa) {
  pdl_enter();
  const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= S) return;
  int lo = 0, hi = k;  // segment of sample x: last s with sbase[s] <= x
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sbase[mid + 1] <= x)
      lo = mid + 1;
    else
      hi = mid;
  }
  const int s = lo;
  const SegDesc sd = segs[s];
  const uint32_t m = sbase[s + 1] - sbase[s], j = x - sbase[s], n = sd.hi - sd.lo;
  // Segments of one shard are samples of the same term distribution: equal relative positions
  // would pile all k samples of a quantile onto the same few terms and leave k-times oversized
  // buckets between the piles.  Every segment gets its own phase (golden-ratio sequence), so
  // the merged samples interleave evenly.
  const double phase = (double)s * 0.6180339887498949;
  const double phi = phase - floor(phase);
  uint32_t off = (uint32_t)(((double)j + phi) * (double)n / (double)m);
  if (off >= n) off = n - 1;
  const uint32_t idx = sd.lo + off;
  const KeyedTerm t = keyed_term(sd, idx);
  sa.hi[x] = t.hi;
  sa.lo[x] = t.lo;
  sa.ptr[x] = reinterpret_cast<uint64_t>(t.p);
  sa.len[x] = t.len;
  sa.idx[x] = idx;
  sa.seg[x] = (uint32_t)s;
}

__device__ __forceinline__ KeyedTerm sample_term(const SampleArrays& sa, uint32_t x) {
  KeyedTerm t;
  t.hi = sa.hi[x];
  t.lo = sa.lo[x];
  t.p = reinterpret_cast<const uint8_t*>(sa.ptr[x]);
  t.len = sa.len[x];
  return t;
}

// One warp per sample x, lanes over segments: how many samples of every segment sort before x
// (ties between equal terms broken by segment) = the rank of x among all samples.  The sorted
// splitter arrays are filled by scattering x to its rank.
__global__ void __launch_bounds__(256)
k1_rank_samples(int k, const uint32_t* __restrict__ sbase, uint32_t S, SampleArrays sa,
                SampleArrays sorted) {
  pdl_enter();
  const uint32_t x = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = lane_id();
  if (x >= S) return;
  const KeyedTerm tx = sample_term(sa, x);
  const uint32_t sx = sa.seg[x];
  uint32_t racc = 0;
  for (int s = lane; s < k; s += 32) {
    const uint32_t b0 = sbase[s], m = sbase[s + 1] - b0;
    if ((uint32_t)s == sx) {
      racc += x - b0;
    } else {
      uint32_t lo = 0, hi = m;  // samples of s strictly below x
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (keyed_compare(sample_term(sa, b0 + mid), tx) < 0)
          lo = mid + 1;
        else
          hi = mid;
      }
      // ties between equal sample terms are ordered by segment
      const bool equal = lo < m && (uint32_t)s < sx && keyed_compare(sample_term(sa, b0 + lo), tx) == 0;
      racc += lo + (equal ? 1u : 0u);
    }
  }
  racc = warp_sum(racc);
  if (lane == 0) {
    sorted.hi[racc] = tx.hi;
    sorted.lo[racc] = tx.lo;
    sorted.ptr[racc] = reinterpret_cast<uint64_t>(tx.p);
    sorted.len[racc] = tx.len;
  }
}

constexpr uint32_t K1_CHUNK = 1024;

// crank[c] = splitters <= the term just before chunk c (0 for the first chunk of a segment):
// chunk c then owns the splitters [crank[c], crank[c+1]) (all the rest for a segment's last
// chunk).  One thread per chunk: 16 dependent probes each, all chunks in parallel — inside the
// partition kernel the same two searches kept a whole CTA waiting at its barrier.
__global__ void __launch_bounds__(256)
k1_chunk_ranks(const SegDesc* __restrict__ segs, int k, const uint32_t* __restrict__ cbase,
               uint32_t n_chunks, uint32_t S, SampleArrays sp, uint32_t* __restrict__ crank) {
  pdl_enter();
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chunks) return;
  int lo = 0, hi = k;  // segment of chunk c: last s with cbase[s] <= c
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cbase[mid + 1] <= c)
      lo = mid + 1;
    else
      hi = mid;
  }
  const SegDesc sd = segs[lo];
  const uint32_t ci = c - cbase[lo];
  uint32_t r = 0;
  if (ci != 0 && sd.hi > sd.lo) {
    const KeyedTerm t = keyed_term(sd, sd.lo + ci * K1_CHUNK - 1);
    uint32_t a = 0, b = S;  // first splitter > t
    while (a < b) {
      const uint32_t mid = (a + b) >> 1;
      if (keyed_compare(sample_term(sp, mid), t) <= 0)
        a = mid + 1;
      else
        b = mid;
    }
    r = a;
  }
  crank[c] = r;
}

// The same partition with the chunk staged RAW: the chunk's offsets and term bytes are two
// contiguous pieces of the segment, copied into shared memory with coalesced word loads (every
// byte of the dictionary still read exactly once, but by ~38 independent coalesced loads per
// thread instead of 16 offset loads + 40 scattered key-window loads), and only the few splitters
// that fall inside the chunk build key windows — from shared memory, during their search.
constexpr uint32_t K1_RAW_BYTES = K1_CHUNK * 19;  // term bytes of a chunk (14.5 B per term on average in C2)

__device__ __forceinline__ void smem_key16(const uint32_t* __restrict__ raw, uint32_t a, uint32_t len,
                                           uint64_t& hi, uint64_t& lo) {
  // raw = words of the staged bytes, a = byte offset of the term inside them (window at byte 0)
  if (len == 0) {
    hi = lo = 0;
    return;
  }
  const uint32_t* wp = raw + (a >> 2);
  const uint32_t sh = (a & 3u) * 8u;
  const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4];
  const uint32_t x0 = __byte_perm(__funnelshift_r(w0, w1, sh), 0, 0x0123);
  const uint32_t x1 = __byte_perm(__funnelshift_r(w1, w2, sh), 0, 0x0123);
  const uint32_t x2 = __byte_perm(__funnelshift_r(w2, w3, sh), 0, 0x0123);
  const uint32_t x3 = __byte_perm(__funnelshift_r(w3, w4, sh), 0, 0x0123);
  hi = ((uint64_t)x0 << 32) | x1;
  lo = ((uint64_t)x2 << 32) | x3;
  if (len < 16) {
    if (len <= 8) {
      lo = 0;
      if (len < 8) hi &= ~0ull << (8 * (8 - len));
    } else {
      lo &= ~0ull << (8 * (16 - len));
    }
  }
}

__global__ void __launch_bounds__(256)
k1_partition_chunks_raw(const SegDesc* __restrict__ segs, int k, const uint32_t* __restrict__ cbase,
                        uint32_t S, SampleArrays sp, const uint32_t* __restrict__ crank,
                        uint32_t* __restrict__ part, uint32_t* __restrict__ btb,
                        uint64_t* __restrict__ bpo) {
  pdl_enter();
  extern __shared__ __align__(16) uint32_t k1_smem[];
  uint32_t* s_off = k1_smem;                  // [K1_CHUNK + 1] term offsets of the chunk
  uint32_t* s_raw = k1_smem + K1_CHUNK + 4;   // staged term bytes (+ 8 words of slack)
  __shared__ uint32_t s_range[2];
  const uint32_t c = blockIdx.x;
  int lo = 0, hi = k;  // segment of chunk c: last s with cbase[s] <= c
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cbase[mid + 1] <= c)
      lo = mid + 1;
    else
      hi = mid;
  }
  const int s = lo;
  const SegDesc sd = segs[s];
  const uint32_t nchunks = cbase[s + 1] - cbase[s], ci = c - cbase[s];
  const uint32_t i0 = sd.lo + ci * K1_CHUNK;
  const uint32_t i1 = (ci + 1 == nchunks) ? sd.hi : i0 + K1_CHUNK;
  const uint32_t n = i1 - i0;
  // start of the staged bytes: 16-byte aligned ADDRESS when the buffer allows it (128-bit loads)
  const uint32_t t0 = __ldg(sd.toff + i0), b1 = __ldg(sd.toff + i1);
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(sd.tb + t0) & 15u);
  const bool wide = mis <= t0;
  const uint32_t b0 = wide ? t0 - mis : (t0 & ~3u);
  const uint32_t words = (b1 - b0 + 3u) >> 2;
  const bool staged = words * 4u + 16u <= K1_RAW_BYTES;
  // offsets and term bytes go straight from global to shared memory (cp.async / LDGSTS: no
  // register round trip — the LSU data pipe was this kernel's busiest unit, 71 % of its peak
  // with LDG + STS, profiles/r02_ncu_full_metrics.csv)
  {
    constexpr int PER = K1_CHUNK / 256;
    const uint32_t s_off_a = (uint32_t)__cvta_generic_to_shared(s_off);
#pragma unroll
    for (int j = 0; j < PER; j++) {
      const uint32_t t = threadIdx.x + j * 256;
      if (t < n)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_off_a + 4 * t), "l"(sd.toff + i0 + t)
                     : "memory");
    }
    if (threadIdx.x == 0) s_off[n] = b1;
  }
  if (staged) {
    if (wide) {
      const uint4* src = reinterpret_cast<const uint4*>(sd.tb + b0);
      const uint32_t dst_a = (uint32_t)__cvta_generic_to_shared(s_raw);
      const uint32_t quads = (words + 3u) >> 2;
#pragma unroll 4
      for (uint32_t q = threadIdx.x; q < quads; q += 256)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_a + 16 * q), "l"(src + q) : "memory");
    } else {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(sd.tb + b0);
#pragma unroll 8
      for (uint32_t q = threadIdx.x; q < words; q += 256) s_raw[q] = __ldg(src + q);
    }
  }
  if (threadIdx.x < 2 && ci == 0) {  // window start / end rows
    const bool first = threadIdx.x == 0;
    const uint64_t at = (uint64_t)(first ? 0 : S + 1) * k + s;
    const uint32_t idx = first ? sd.lo : sd.hi;
    part[at] = idx;
    btb[at] = __ldg(sd.toff + idx);
    bpo[at] = __ldg(sd.poff + idx);
  }
  if (threadIdx.x == 0) {
    s_range[0] = crank[c];
    s_range[1] = ci + 1 == nchunks ? S : crank[c + 1];
  }
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const uint32_t ra = s_range[0], rb = s_range[1];
  for (uint32_t r = ra + threadIdx.x; r < rb; r += 256) {
    const KeyedTerm x = sample_term(sp, r);
    uint32_t a = 0, b = n;  // first term of the chunk >= x
    while (a < b) {
      const uint32_t mid = (a + b) >> 1;
      KeyedTerm t;
      const uint32_t o = s_off[mid];
      t.len = s_off[mid + 1] - o;
      if (staged)
        smem_key16(s_raw, o - b0, t.len, t.hi, t.lo);
      else
        load_key16(sd.tb, o, t.len, 0, t.hi, t.lo);
      int cmp;
      if (t.hi != x.hi) {
        cmp = t.hi < x.hi ? -1 : 1;
      } else if (t.lo != x.lo) {
        cmp = t.lo < x.lo ? -1 : 1;
      } else if (t.len > 16 && x.len > 16) {
        t.p = sd.tb + o;
        cmp = term_compare(t.p + 16, t.len - 16, x.p + 16, x.len - 16);
      } else {
        cmp = t.len < x.len ? -1 : (t.len > x.len ? 1 : 0);
      }
      if (cmp < 0)
        a = mid + 1;
      else
        b = mid;
    }
    // the boundary in every array of the segment: term index, first term byte, first posting
    const uint64_t at = (uint64_t)(r + 1) * k + s;
    part[at] = i0 + a;
    btb[at] = s_off[a];
    bpo[at] = __ldg(sd.poff + i0 + a);
  }
}

// One warp per bucket.  raw[0][b] = instances, raw[1][b] = input postings, raw[2][b] = staging
// words (upper bound), raw[3][b] = term bytes of all instances (upper bound of the bucket's
// merged term bytes).  Everything comes from the boundary tables the partition wrote.
__global__ void __launch_bounds__(256)
k1_bucket_stats(int k, uint32_t S, SampleArrays sp, const uint32_t* __restrict__ part,
                const uint32_t* __restrict__ btb, const uint64_t* __restrict__ bpo,
                uint64_t* __restrict__ raw, uint32_t* __restrict__ bk_cpl) {
  pdl_enter();
  const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t B = S + 1;
  if (b > B) return;
  const unsigned lane = lane_id();
  if (b == B) {
    if (lane < 4) raw[(uint64_t)lane * (B + 1) + B] = 0;
    return;
  }
  uint64_t w = 0, p = 0, t = 0;
  for (int s = lane; s < k; s += 32) {
    const uint64_t r0 = (uint64_t)b * k + s, r1 = r0 + k;
    w += part[r1] - part[r0];
    p += bpo[r1] - bpo[r0];
    t += btb[r1] - btb[r0];
  }
  w = warp_sum(w);
  p = warp_sum(p);
  t = warp_sum(t);
  if (lane == 0) {
    raw[b] = w;
    raw[(uint64_t)(B + 1) + b] = p;
    // `_val` staging words the bucket can need: every term of L values reserves
    // L + L/4 + 6 words (union_dev.cuh enc_slot_words) and there are at most w terms
    raw[2ull * (B + 1) + b] = p + (p >> 2) + 6 * w;
    raw[3ull * (B + 1) + b] = t;
    uint32_t c = 0;
    // the delimiting splitters of bucket b (samples b - 1 and b), if both exist
    if (b >= 1 && b < S && w) {
      const uint8_t* x = reinterpret_cast<const uint8_t*>(sp.ptr[b - 1]);
      const uint8_t* y = reinterpret_cast<const uint8_t*>(sp.ptr[b]);
      const uint32_t m = sp.len[b - 1] < sp.len[b] ? sp.len[b - 1] : sp.len[b];
      while (c < m && x[c] == y[c]) c++;
    }
    bk_cpl[b] = c;
  }
}

// ---- a window small enough for ONE bucket ------------------------------------------------------
// (a point read, a handful of terms): no splitter exists, so the plan is the two boundary rows,
// the bucket's sizes and their trivial prefixes — one CTA instead of the five launches of the
// general path (copy of the bases, chunk ranks, partition, stats, scan); a read of this size is
// bound by the number of launches.
__global__ void __launch_bounds__(256)
k1_plan_single(const SegDesc* __restrict__ segs, int k, uint32_t* __restrict__ part,
               uint32_t* __restrict__ btb, uint64_t* __restrict__ bpo, uint64_t* __restrict__ bk_WP,
               uint32_t* __restrict__ bk_cpl, uint64_t* __restrict__ totals) {
  pdl_enter();
  __shared__ uint64_t ws[256 / 32 + 2];
  uint64_t w = 0, p = 0, t = 0;
  for (int s = threadIdx.x; s < k; s += 256) {
    const SegDesc sd = segs[s];
    const uint32_t t0 = __ldg(sd.toff + sd.lo), t1 = __ldg(sd.toff + sd.hi);
    const uint64_t p0 = __ldg(sd.poff + sd.lo), p1 = __ldg(sd.poff + sd.hi);
    part[s] = sd.lo;
    part[k + s] = sd.hi;
    btb[s] = t0;
    btb[k + s] = t1;
    bpo[s] = p0;
    bpo[k + s] = p1;
    w += sd.hi - sd.lo;
    p += p1 - p0;
    t += t1 - t0;
  }
  uint64_t tw, tp, tt;
  block_exclusive_scan(w, ws, tw);
  block_exclusive_scan(p, ws, tp);
  block_exclusive_scan(t, ws, tt);
  if (threadIdx.x == 0) {
    const uint64_t v[4] = {tw, tp, tp + (tp >> 2) + 6 * tw, tt};  // as k1_bucket_stats
#pragma unroll
    for (int j = 0; j < 4; j++) {
      bk_WP[2 * j] = 0;
      bk_WP[2 * j + 1] = v[j];
      totals[j] = v[j];
    }
    bk_cpl[0] = 0;
  }
}

int k1_build_plan(MergePlan& plan, const SegDesc* h_segs, uint32_t* sbase, cudaStream_t s) {
  const int k = plan.k;
  const uint32_t N = plan.n_total;
  if (k > kMaxSegs) {
    set_last_error("k1: %d segments in one pass (max %d)", k, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  // samples per segment, proportional to its window; chunks of the merge-path partition
  const uint32_t per_bucket = [] {  // tuning knob: II2_BUCKET=<instances per bucket>
    const char* e = getenv("II2_BUCKET");
    const long v = e ? atol(e) : 0;
    return (v >= 32 && v <= 1024) ? (uint32_t)v : kInstancesPerBucket;
  }();
  uint64_t want = N / per_bucket;
  // a small call (a narrow range read) is latency-bound: smaller buckets spread it over the SMs,
  // up to 592 buckets of at least 128 instances
  constexpr uint32_t small_bucket = 128, small_want = 592;
  if (want < small_want && N / small_bucket > want)
    want = std::min<uint64_t>(small_want, N / small_bucket);
  // ... and a window of a few hundred instances (a point read) is ONE bucket: planning it costs
  // more launches than the bucket takes (k1_plan_single)
  constexpr uint32_t single_max = 768;
  if (N <= single_max) want = 0;
  if (want > kMaxBuckets - 1) want = kMaxBuckets - 1;
  uint32_t* cbase = sbase + (k + 1);
  sbase[0] = 0;
  cbase[0] = 0;
  // Where the samples come from.  Evenly spaced samples of MANY segments interleave like a
  // Poisson process (a segment's j-th sample drifts by ~sqrt(j) terms against the others), so
  // bucket sizes would be exponentially distributed: a quarter of the buckets above 4/3 of the
  // mean, most instances inside them.  Evenly spaced samples of ONE segment cut the merged
  // order into nearly equal pieces whenever the segments resemble each other (measured CV 0.2),
  // so the largest segment supplies 15/16 of the splitters and every segment still gets its
  // proportional share of the remaining 1/16, which bounds the buckets when they do not.
  int big = 0;
  for (int i = 1; i < k; i++)
    if (h_segs[i].hi - h_segs[i].lo > h_segs[big].hi - h_segs[big].lo) big = i;
  const uint64_t n_big = k ? h_segs[big].hi - h_segs[big].lo : 0;
  uint64_t want_big = want - want / 16;
  if (want_big + 1 > n_big) want_big = n_big ? n_big - 1 : 0;
  const uint64_t want_rest = want - want_big;
  uint64_t cum = 0, given = 0;
  for (int i = 0; i < k; i++) {
    const uint64_t n = h_segs[i].hi - h_segs[i].lo;
    cum += n;
    // cumulative rounding: the samples add up to `want_rest` even when every segment's share is < 1
    uint64_t m = N ? want_rest * cum / N - given : 0;
    given += m;
    if (i == big) m += want_big;
    if (m + 1 > n) m = n ? n - 1 : 0;
    sbase[i + 1] = sbase[i] + (uint32_t)m;
    cbase[i + 1] = cbase[i] + (uint32_t)std::max<uint64_t>(1, (n + K1_CHUNK - 1) / K1_CHUNK);
  }
  const uint32_t S = sbase[k], n_chunks = cbase[k];  // S samples = S + 1 buckets of the partition
  const uint32_t B = S + 1;
  plan.n_samples = S;
  plan.n_buckets = B;
  ProfScope scope("k1_plan", s);
  II2_TRY(plan.part.alloc_scratch((size_t)(B + 1) * k, s));
  II2_TRY(plan.bk_cpl.alloc_scratch(B, s));
  II2_TRY(plan.btb.alloc_scratch((size_t)(B + 1) * k, s));
  II2_TRY(plan.bpo.alloc_scratch((size_t)(B + 1) * k, s));
  II2_TRY(plan.bk_WP.alloc_scratch(4 * (size_t)(B + 1), s));
  II2_TRY(plan.totals.alloc_scratch(4, s));
  if (S == 0) {
    II2_LAUNCH_CHAIN(k1_plan_single, 1, 256, 0, s, plan.segs, k, plan.part.p, plan.btb.p, plan.bpo.p,
                     plan.bk_WP.p, plan.bk_cpl.p, plan.totals.p);
    return II2_OK;
  }
  DevBuf<uint32_t> d_base, d_u32;
  DevBuf<uint64_t> d_u64;
  II2_TRY(d_base.alloc_scratch(2 * (size_t)(k + 1), s));
  II2_TRY(d_u64.alloc_scratch(6 * (size_t)S, s));
  II2_TRY(d_u32.alloc_scratch(4 * (size_t)S, s));
  II2_TRY(small_copy(d_base.p, sbase, 2 * (size_t)(k + 1) * 4, s));  // sbase is pinned
  const uint32_t* d_sbase = d_base.p;
  const uint32_t* d_cbase = d_base.p + (k + 1);
  SampleArrays sa{d_u64.p, d_u64.p + S, d_u64.p + 2 * S, d_u32.p, d_u32.p + S, d_u32.p + 2 * S};
  SampleArrays sp{d_u64.p + 3 * S, d_u64.p + 4 * S, d_u64.p + 5 * S, d_u32.p + 3 * S, nullptr, nullptr};
  II2_LAUNCH_CHAIN(k1_sample_keys, div_up(S, 256), 256, 0, s, plan.segs, k, d_sbase, S, sa);
  II2_LAUNCH_CHAIN(k1_rank_samples, div_up((uint64_t)S * 32, 256), 256, 0, s, k, d_sbase, S, sa, sp);
  {
    constexpr size_t smem = (K1_CHUNK + 4 + 8) * 4 + K1_RAW_BYTES;
    static bool attr_set = false;
    if (!attr_set) {
      II2_CUDA_TRY(cudaFuncSetAttribute(k1_partition_chunks_raw,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_set = true;
    }
    DevBuf<uint32_t> crank;
    II2_TRY(crank.alloc_scratch((size_t)n_chunks + 1, s));
    II2_LAUNCH_CHAIN(k1_chunk_ranks, div_up(n_chunks, 256), 256, 0, s, plan.segs, k, d_cbase, n_chunks, S, sp, crank.p);
    II2_LAUNCH_CHAIN(k1_partition_chunks_raw, n_chunks, 256, smem, s, plan.segs, k, d_cbase, S, sp, crank.p,
                     plan.part.p, plan.btb.p, plan.bpo.p);
  }
  II2_LAUNCH_CHAIN(k1_bucket_stats, div_up((uint64_t)(B + 1) * 32, 256), 256, 0, s, k, S, sp, plan.part.p,
                   plan.btb.p, plan.bpo.p, plan.bk_WP.p, plan.bk_cpl.p);
  II2_TRY(exclusive_scan_multi_u64(plan.bk_WP.p, plan.bk_WP.p, B + 1, 4, plan.totals.p, s));
  return II2_OK;
}

}  // namespace ii2
